"""The geometry of a group job on inputs of 2^32 bytes or more (kc_group_plan, host only, no GPU).

From KC_POS32_BYTES = 2^32 - 16 on, a group builds the k-mer set by the signature construction alone (64-bit window positions):
no fixed slots, and a heap that holds that construction's receive regions instead of the fixed-slot / exact items.  Where the
group's 32-bit bounds (kc_grp_large_bound, the same check the compute path makes before a job) do not hold, the plan is refused.
Below KC_POS32_BYTES the plan is that of the parent layout, pinned here at the last 32-bit size."""
import pytest

import kmercamel_b200 as kb
from kmercamel_b200 import sharded

POS32 = 2**32 - 16
SIZES = [2**32 - 16, 2**32, 4_500_000_000, 6_400_000_000, 20_000_000_000]
WORLDS = [1, 2, 3, 8]
KS = [31, 63, 127]

# (fixed_slots, n_digits, cap_sub, heap_bytes) at n_bytes = 2^32 - 17, as the layout below KC_POS32_BYTES gives them
LAST32 = {(1, 31): (1, 256, 17145600, 66585384704), (1, 63): (1, 256, 17145600, 109543970304), (1, 127): (1, 256, 17145600, 195461141760),
          (2, 31): (1, 256, 8579616, 34373129984), (2, 63): (1, 256, 8579616, 55856879360), (2, 127): (1, 256, 8579616, 98824377856),
          (3, 31): (1, 256, 5723264, 23635712000), (3, 63): (1, 256, 5723264, 37961182464), (3, 127): (1, 256, 5723264, 66612123392),
          (8, 31): (1, 256, 2150752, 10213938944), (8, 63): (1, 256, 2150752, 15591560960), (8, 127): (1, 256, 2150752, 26346804992)}


def _refused(world, k, n_bytes):
    with pytest.raises(kb.KcError) as e:
        sharded.group_plan(world, 0, k, n_bytes)
    return e.value.code == -6


def _expected_refusal(world, n_bytes):
    """kc_grp_large_bound in Python: one (sender, owner) stream or one rank's dense stream would reach 2^32 records."""
    tile = 256 * 32
    tiles = -(-n_bytes // tile)
    region = (int(n_bytes / world / 5.16 / world * 1.15) + 8192 + 31) // 32 * 32
    slice_max = min(n_bytes, -(-tiles // world) * tile)
    dense = int(slice_max / 5.16 * 1.3) + world * 8192 + 65536
    return region >= 2**32 or dense >= 2**32


@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("k", KS)
def test_last_32_bit_size_keeps_its_plan(world, k):
    n = POS32 - 1
    plans = sharded.check_plans(world, k, n)
    g = int(kb.load_library().kc_shard_granule(k))
    for r, p in enumerate(plans):
        tiles = -(-n // g)
        assert p["pos_begin"] == min(n, tiles * r // world * g) and p["pos_end"] == min(n, tiles * (r + 1) // world * g)
        assert (int(p["fixed_slots"]), p["n_digits"], p["cap_sub"], p["heap_bytes"]) == LAST32[(world, k)]


@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("k", KS)
def test_plan_from_2_32(world, k):
    g = int(kb.load_library().kc_shard_granule(k))
    heaps = []
    for n in SIZES:
        if _expected_refusal(world, n):
            assert _refused(world, k, n), (world, k, n)
            continue
        plans = sharded.check_plans(world, k, n)
        for p in plans:
            assert not p["fixed_slots"] and p["cap_sub"] == 0
            assert p["pos_begin"] % g == 0 and (p["pos_end"] % g == 0 or p["pos_end"] == n)
        # code words, two flag arrays and one record stream per sender: no room for fixed-slot receive arrays
        heap = plans[0]["heap_bytes"]
        assert heap <= n * (0.5 + 2 / world) + 2**30, (world, k, n, heap)
        heaps.append((n, heap))
    for (n0, h0), (n1, h1) in zip(heaps, heaps[1:]):  # at most linear growth
        assert h1 <= h0 * n1 / n0 + 2**20, (world, k, n0, n1, h0, h1)


def test_refusals_follow_the_bound():
    assert _refused(1, 31, 20_000_000_000)                  # one rank on 20 GB: its dense stream passes 2^32 records
    assert not _expected_refusal(2, 20_000_000_000)
    sharded.check_plans(2, 31, 20_000_000_000)
    assert _refused(2, 21, 5_000_000_000)                   # k < 26: no signature construction
    sharded.check_plans(2, 21, POS32 - 1)                   # ... which the 32-bit sizes do not need
