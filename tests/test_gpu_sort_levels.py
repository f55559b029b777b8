"""The radix sort of sort.cuh word for word against np.lexsort, and the overlap stage past the single-CTA engine at wide k byte for
byte against the oracle.

kc_sort is the tuple sort of every overlap level (engine.cuh, 64 + 2d key bits over 2, 3 or 5 limbs) and the sparse switch's presort
(runs.cuh, 40 bits of one limb).  Its radix levels, skipped buckets, limb-straddling digits, uniform buckets and the local kernel's
insertion and bitonic sorts only run on buckets of more than SortCfg<L>::CAP items, which engine inputs reach only at some widths;
the test hook kc_debug_sort runs it on chosen words, and its statistics are held to a counts-only model of the bucket bookkeeping
(_model), so that each case also shows it took the path it targets.  The second half runs the multi-kernel level loop (more than
1024 virtual nodes) at k = 32..127, where the level loop sorts 3- and 5-limb tuples through those radix levels."""
import numpy as np
import pytest

from kmercamel_b200 import synth
from oracle import orc
from test_gpu_fasta_exact import SMALL_NS, _cached, _exact, _set, fctx, reads, tie_heavy_simplitigs, xctx  # noqa: F401 (fixtures)

pytestmark = pytest.mark.gpu

LIMBS = (1, 2, 3, 5)
CAP = {1: 8192, 2: 4096, 3: 2048, 5: 1024}     # SortCfg<L>::CAP
TILE = {1: 4096, 2: 2048, 3: 1024, 5: 1024}    # SortCfg<L>::TILE
SUB_SMALL = 24                                  # KC_SUB_SMALL: larger sub-buckets of the local kernel take the bitonic network
SUB_BITS_MAX = 11                               # KC_SUB_BITS_MAX
M64 = (1 << 64) - 1


# ---- reference and model ---------------------------------------------------------------------------------------------------
def _digits(w, pos, nbits):
    """Bits [pos, pos + nbits) of every word of w [n, L] (nbits <= 32), as int64."""
    limb, off = pos >> 6, pos & 63
    v = w[:, limb] >> np.uint64(off)
    if off + nbits > 64 and limb + 1 < w.shape[1]:
        v = v | (w[:, limb + 1] << np.uint64(64 - off))
    return (v & np.uint64((1 << nbits) - 1)).astype(np.int64)


def _model(ref, key_bits):
    """Counts-only model of kc_sort's bucket bookkeeping on the sorted words `ref`: every bucket is a contiguous range of them
    (its items share the key bits already partitioned).  -> the statistics kc_debug_sort reports."""
    L = ref.shape[1]
    cap = CAP[L]
    n = ref.shape[0]
    st = dict(levels=0, max_big=0, small=0, uniform=0, whole_bitonic=0)
    small = []
    big = []
    if n == 0:
        return st
    if n <= cap:
        small.append((0, n, key_bits))
    elif key_bits == 0:
        st["uniform"] += 1
    else:
        big.append((0, n, key_bits))
    while big:
        st["levels"] += 1
        st["max_big"] = max(st["max_big"], len(big))
        nxt = []
        for off, size, rem in big:
            want = -(-size // (cap // 4))
            bits = 1
            while (1 << bits) < want and bits < 8:
                bits += 1
            bits = min(bits, rem)
            d = _digits(ref[off:off + size], rem - bits, bits)
            cuts = np.flatnonzero(np.diff(d)) + 1
            for a, b in zip(np.r_[0, cuts], np.r_[cuts, size]):
                child = (off + int(a), int(b - a), rem - bits)
                if child[1] <= cap:
                    small.append(child)
                elif child[2] == 0:
                    st["uniform"] += 1
                else:
                    nxt.append(child)
        big = nxt
    st["small"] = len(small)
    for off, size, rem in small:
        if size < 2:
            continue
        bits = 1
        while (1 << bits) < 2 * size and bits < SUB_BITS_MAX:
            bits += 1
        bits = min(bits, rem)
        cnt = np.bincount(_digits(ref[off:off + size], rem - bits, bits), minlength=1 << bits)
        st["whole_bitonic"] += int(np.count_nonzero(cnt > SUB_SMALL) > 64)
    return st


def _check(ctx, words, key_bits):
    """kc_debug_sort must give np.lexsort's order word for word and the model's statistics; -> the statistics."""
    words = np.ascontiguousarray(words, dtype=np.uint64)
    ref = words[np.lexsort(words.T)] if len(words) else words
    got, st = ctx.debug_sort(words, key_bits)
    assert np.array_equal(got, ref)
    assert st == _model(ref, key_bits)
    return st


def _random(rng, n, L, key_bits):
    w = rng.integers(0, 1 << 63, size=(n, L), dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, size=(n, L), dtype=np.uint64)
    return w & _mask(L, key_bits)


def _mask(L, key_bits):
    return np.array([(((1 << key_bits) - 1) >> (64 * i)) & M64 for i in range(L)], dtype=np.uint64)


def _from_ints(vals, L):
    return np.array([[(v >> (64 * i)) & M64 for i in range(L)] for v in vals], dtype=np.uint64).reshape(-1, L)


def _widths(L):
    """40 (the sparse switch's presort) and the tuple widths 64 + 2d of the overlap levels that fit L limbs."""
    return [40] + [64 + 2 * d for d in (0, 1, 31, 32, 63, 64, 126) if 64 + 2 * d <= 64 * L]


@pytest.fixture(scope="module")
def sctx():
    import kmercamel_b200 as kb
    c = kb.Context(0)
    yield c
    c.close()


# ---- sizes and key widths ------------------------------------------------------------------------------------------------
def _sizes(L):
    cap, tile = CAP[L], TILE[L]
    s = {1, 2, 24, 25, cap - 1, cap, cap + 1, 32 * cap, 32 * cap + 1}
    for j in (1, 2, 3, 7):
        s |= {tile * j - 1, tile * j + 1}
    return sorted(s)


@pytest.mark.parametrize("L", LIMBS)
def test_sizes_and_widths(sctx, L):
    rng = np.random.default_rng(L)
    cap = CAP[L]
    for key_bits in _widths(L):
        for n in _sizes(L):
            st = _check(sctx, _random(rng, n, L, key_bits), key_bits)
            assert (st["levels"] > 0) == (n > cap), (key_bits, n)
            if n in (32 * cap, 32 * cap + 1):
                # 32 CAP items take 7-bit digits at the first level, one more item 8-bit digits: that many buckets of about CAP / 8
                assert st["small"] == (128 if n == 32 * cap else 256) and st["levels"] == 1, (key_bits, n)


@pytest.mark.parametrize("L", LIMBS)
def test_millions_of_random_words(sctx, L):
    rng = np.random.default_rng(100 + L)
    key_bits = 64 * L if L > 1 else 40
    st = _check(sctx, _random(rng, 3_000_001, L, key_bits), key_bits)
    assert st["levels"] >= 2 and st["max_big"] > 1


def test_bad_arguments(sctx):
    import kmercamel_b200 as kb
    w = np.zeros((4, 4), dtype=np.uint64)
    with pytest.raises(kb.KcError) as e:
        sctx.debug_sort(w, 64)          # 4 limbs: not a width the library sorts
    assert e.value.code == -2
    w = np.zeros((4, 2), dtype=np.uint64)
    with pytest.raises(kb.KcError) as e:
        sctx.debug_sort(w, 129)         # more key bits than the words hold
    assert e.value.code == -2
    w[2, 1] = 1 << 20
    with pytest.raises(kb.KcError) as e:
        sctx.debug_sort(w, 84)          # a bit set above key_bits
    assert e.value.code == -2
    got, st = sctx.debug_sort(w, 85)
    assert np.array_equal(got[-1], w[2]) and st["small"] == 1


# ---- shared prefixes: skipped levels with the parity kept, digits across limb boundaries ----------------------------------------
@pytest.mark.parametrize("L", LIMBS)
def test_shared_prefixes(sctx, L):
    rng = np.random.default_rng(200 + L)
    cap = CAP[L]
    for key_bits in _widths(L):
        for b in (3, 8, 13, 63, 64, 65, 129):
            if b >= key_bits:
                continue
            for n in (cap + 1, 5 * cap + 3, 40 * cap + 7):
                prefix = _random(rng, 1, L, key_bits) & ~_mask(L, b)
                w = _random(rng, n, L, b) | prefix
                st = _check(sctx, w, key_bits)
                assert st["levels"] >= -(-(key_bits - b) // 8), (key_bits, b, n)  # a digit has at most 8 bits
                if b <= 8:  # at most 256 distinct words: the larger runs end as uniform buckets
                    assert st["uniform"] > 0 or n < 256 * cap


# ---- uniform buckets -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("L", LIMBS)
def test_uniform_buckets(sctx, L):
    rng = np.random.default_rng(300 + L)
    cap = CAP[L]
    for key_bits in (_widths(L)[0], _widths(L)[-1]):
        runs = [cap + 1, cap + 7, 2 * cap, 5 * cap + 3]
        heads = _random(rng, len(runs), L, key_bits)
        heads[1] = heads[0]
        heads[1, 0] ^= np.uint64(1)                        # two runs that differ in the lowest key bit only
        w = np.concatenate([np.repeat(heads[i:i + 1], r, axis=0) for i, r in enumerate(runs)] + [_random(rng, 300, L, key_bits)])
        w = w[rng.permutation(len(w))]
        st = _check(sctx, w, key_bits)
        assert st["uniform"] == len(runs)
    # every word equal: one uniform bucket after all key bits, and with no key bits at all the root is uniform
    for key_bits in (0, 64 * L):
        w = np.repeat(_random(rng, 1, L, key_bits), 3 * cap + 1, axis=0)
        st = _check(sctx, w, key_bits)
        assert st["uniform"] == 1 and st["small"] == 0


# ---- the local kernel: insertion sort up to 24 items, bitonic networks above -----------------------------------------------
def _local_bucket(rng, L, key_bits, groups):
    """One bucket of at most CAP words whose local-kernel sub-buckets (the top digit the kernel picks) hold `groups` items each."""
    n = sum(groups)
    bits = 1
    while (1 << bits) < 2 * n and bits < SUB_BITS_MAX:
        bits += 1
    bits = min(bits, key_bits)
    assert len(groups) <= 1 << bits
    digits = rng.choice(1 << bits, size=len(groups), replace=False)
    parts = []
    for dg, g in zip(digits, groups):
        hi = _from_ints([int(dg) << (key_bits - bits)], L)
        parts.append(_random(rng, g, L, key_bits - bits) | hi)
    w = np.concatenate(parts)
    return w[rng.permutation(n)]


@pytest.mark.parametrize("L", LIMBS)
def test_local_kernel_paths(sctx, L):
    rng = np.random.default_rng(400 + L)
    cap = CAP[L]
    key_bits = _widths(L)[-1]
    cases = [([24] * 5, 0), ([25] * 5, 0), ([24, 25, 1, 2, 23, 26], 0), ([37, 100, 333], 0), ([cap - 3], 0),
             ([25] * 30 + [3] * 10, 0)]
    if 65 * 25 <= cap:  # 65 oversized sub-buckets need more than CAP = 1024 items at 5 limbs
        cases += [([25] * 64, 0), ([25] * 65, 1), ([25] * 64 + [24] * 4, 0), ([25] * 64 + [26, 7], 1), ([27] * 70 + [5] * 9, 1)]
    for groups, whole in cases:
        w = _local_bucket(rng, L, key_bits, groups)
        st = _check(sctx, w, key_bits)
        assert st["levels"] == 0 and st["small"] == 1 and st["whole_bitonic"] == whole, groups
    # the same sub-buckets inside buckets that radix levels produce (several local buckets per launch)
    groups = [25] * 65 if 65 * 25 <= cap else [25] * 40
    want = -(-8 * sum(groups) // (cap // 4))
    bits = max(b for b in range(1, 9) if b == 1 or (1 << (b - 1)) < want)  # kc_sort_prep_kernel's digit width for the root
    step = (1 << bits) // 8
    w = np.concatenate([_local_bucket(rng, L, key_bits - bits, groups) | _from_ints([(i * step) << (key_bits - bits)], L)
                        for i in range(8)])
    st = _check(sctx, w, key_bits)
    assert st["levels"] == 1 and st["small"] == 8 and st["whole_bitonic"] == (8 if 65 * 25 <= cap else 0)


# ---- engine-shaped tuples ------------------------------------------------------------------------------------------------
META_SHIFT = 27            # KC_META_SHIFT (engine.cuh)
ROLE_P = 1 << 36           # KC_ROLE_P


def _tuples(first, last, k, d, strict):
    """The tuples of one overlap level d (engine.cuh): (d-suffix of the last k-mer, node) and (d-prefix of the first k-mer,
    KC_ROLE_P | batch | ~node) for every node; limb 0 = meta << KC_META_SHIFT, the key above it."""
    n = first.shape[0]
    L = first.shape[1] + 1
    batch = n // 16 + 1 if strict else n + 1
    x = np.arange(n, dtype=np.uint64)
    suf = last & _mask(L - 1, 2 * d)
    pre = np.zeros_like(first)
    sh = 2 * (k - d)
    for i in range(L - 1):  # first >> 2 (k - d), limb by limb
        src, off = i + sh // 64, sh % 64
        if src < L - 1:
            pre[:, i] = first[:, src] >> np.uint64(off)
            if off and src + 1 < L - 1:
                pre[:, i] |= first[:, src + 1] << np.uint64(64 - off)
    t_s = np.concatenate([(x << np.uint64(META_SHIFT))[:, None], suf], axis=1)
    meta_p = np.uint64(ROLE_P) | ((x // np.uint64(batch)) << np.uint64(32)) | (~x & np.uint64(0xFFFFFFFF))
    t_p = np.concatenate([(meta_p << np.uint64(META_SHIFT))[:, None], pre], axis=1)
    return np.concatenate([t_s, t_p])


@pytest.mark.parametrize("k", [31, 63, 95, 127])
def test_engine_shaped_tuples(sctx, k):
    seq, off, ln = reads()
    noff, nln, _, _ = _cached(("nodes", k), lambda: orc.fasta_nodes(seq, off, ln, k, True))
    first = orc.window_words(seq, noff, k)
    last = orc.window_words(seq, noff + nln - np.uint64(k), k)
    for d in sorted({0, 1, 31, 32, 63, 64, 126, k - 1} & set(range(k))):
        for strict in (True, False):
            t = _tuples(first, last, k, d, strict)
            st = _check(sctx, t, 64 + 2 * d)
            assert st["levels"] > 0, (k, d)


# ---- the comb: 255 singletons leave one big bucket at every 8-bit level -------------------------------------------------------
def _comb(rng, L, n_equal):
    """n_equal copies of one word plus, for every 8-bit level but the last, the 255 words that agree with it above that level's digit
    and differ in it: each level moves 255 small buckets into the list."""
    key_bits = 64 * L
    main = int.from_bytes(rng.bytes(8 * L), "little")
    teeth = []
    for j in range(key_bits // 8 - 1):
        pos = key_bits - 8 * (j + 1)
        dg = (main >> pos) & 255
        low = int.from_bytes(rng.bytes(8 * L), "little") & ((1 << pos) - 1)
        for v in range(256):
            if v != dg:
                teeth.append(((main >> (pos + 8)) << (pos + 8)) | (v << pos) | low)
    w = np.concatenate([_from_ints([main], L).repeat(n_equal, axis=0), _from_ints(teeth, L)])
    return w[rng.permutation(len(w))], key_bits


@pytest.mark.parametrize("L,n_equal", [(5, 40_000), (3, 70_000), (2, 140_000), (5, 33_000), (5, 200_000), (3, 66_000)])
def test_comb(sctx, L, n_equal):
    """More small buckets than the list holds (16 n / CAP + 4096) at 5 and 3 limbs: the local kernel empties the list between
    levels.  The counts are exact: every tooth is a small bucket of one item and the equal words one uniform bucket."""
    rng = np.random.default_rng(500 + L + n_equal)
    w, key_bits = _comb(rng, L, n_equal)
    st = _check(sctx, w, key_bits)
    assert st["levels"] == key_bits // 8 and st["max_big"] == 1
    assert st["small"] == 255 * (key_bits // 8 - 1) and st["uniform"] == 1


def test_small_list_bound_worst_case(sctx):
    """Levels that add as many small buckets as they can while the list is nearly full: the list bound holds with the local kernel
    run between levels.  Many big buckets of just over 32 CAP items each take 8-bit digits, and every digit is a singleton or a big
    bucket again."""
    rng = np.random.default_rng(600)
    L, cap = 5, CAP[5]
    key_bits = 64 * L
    parts = []
    for top in range(6):  # six interleaved combs under different top bytes: 6 big buckets per level, 6 * 255 small ones
        w, _ = _comb(rng, L, 33_000)
        hi = _from_ints([top << (key_bits - 8)], L)
        parts.append((w & _mask(L, key_bits - 8)) | hi)
    st = _check(sctx, np.concatenate(parts), key_bits)
    assert st["max_big"] == 6 and st["small"] > 16 * (len(np.concatenate(parts)) // cap) + 4096


# ---- the overlap stage past the single-CTA engine at wide k, byte for byte against the oracle ---------------------------------
def _level_loop_ran(ctx, n_nodes):
    assert n_nodes > SMALL_NS and ctx.stat("path_levels") > 0


@pytest.mark.parametrize("k", [64, 95, 127])
@pytest.mark.parametrize("compl", [True, False])
@pytest.mark.parametrize("small_engine", [1, 0])
def test_reads_wide_k(xctx, k, compl, small_engine):
    _set(xctx, small_engine=small_engine)
    got = _exact(xctx, reads(), k, compl)
    _level_loop_ran(xctx, got.n_nodes)


@pytest.mark.parametrize("small_engine", [1, 0])
def test_reads_maxone_k127(xctx, small_engine):
    _set(xctx, small_engine=small_engine)
    got = _exact(xctx, reads(), 127, maxone=True)
    _level_loop_ran(xctx, got.n_nodes)


@pytest.mark.parametrize("k", [95, 127])
@pytest.mark.parametrize("small_engine", [1, 0])
def test_lower_bound_wide_k(xctx, k, small_engine):
    _set(xctx, small_engine=small_engine)
    seq, off, ln = reads()
    want = _cached(("lb", k), lambda: orc.lower_bound_from_fasta(seq, off, ln, k, True))
    lb, st = xctx.lower_bound(seq, k=k)
    assert lb == want
    _level_loop_ran(xctx, st.n_nodes)


def short_reads(k):
    """Reads of k + 4 bases (five k-mers each) from a 150 kbp genome at 6x: past the sparse switch, the k-mers are the nodes."""
    return _cached(("short_reads", k), lambda: synth.frame_records(list(synth.reads_from_genome(150_000, 6.0, k + 4, 0.01, seed=k))))


@pytest.mark.parametrize("k", [64, 96, 127])
@pytest.mark.parametrize("sparse", [1, 0])
@pytest.mark.parametrize("small_engine", [1, 0])
def test_sparse_switch_wide_k(xctx, k, sparse, small_engine):
    _set(xctx, sparse_switch=sparse, small_engine=small_engine)
    got = _exact(xctx, short_reads(k), k, sparse=bool(sparse))
    assert got.n_simplitigs * 5 >= got.n_kmers
    assert got.n_nodes == (got.n_kmers if sparse else got.n_simplitigs)
    _level_loop_ran(xctx, got.n_nodes)


@pytest.mark.parametrize("k,compl", [(33, True), (64, False), (100, True), (127, True)])
@pytest.mark.parametrize("small_engine", [1, 0])
def test_simplitigs_wide_k(xctx, k, compl, small_engine):
    recs = _cached(("S", 20_000, k), lambda: tie_heavy_simplitigs(20_000, k, 20_000 + k))
    want_ms, want_mo = _cached(("S_orc", 20_000, k, compl), lambda: orc.compute_from_simplitigs(recs, k, compl, True))
    seq, off, ln = orc.records_to_arrays(recs)
    _set(xctx, small_engine=small_engine)
    got = xctx.compute(seq, off, ln, k=k, complements=compl, assume_simplitigs=True, want_maxone=True)
    assert got.ms == want_ms and got.maxone == want_mo
    _level_loop_ran(xctx, got.n_nodes)


def tie_heavy_nodes(n, k, seed):
    """n node ends cut from records of k to 2k + 2 bases over a two- or three-letter alphabet, half of them periodic with a few
    substitutions: many equal overlaps at every level.  -> (first, last) [n, limbs] u64"""
    def make():
        rng = np.random.default_rng(seed)
        letters = np.frombuffer([b"AC", b"ACG", b"AT"][seed % 3], dtype=np.uint8)
        motifs = [rng.choice(letters, size=int(rng.integers(1, 7))).tobytes() for _ in range(6)]
        recs = []
        for _ in range(n):
            m = k + int(rng.integers(0, k + 3))
            if rng.random() < 0.5:
                mo = motifs[int(rng.integers(0, len(motifs)))]
                ph = int(rng.integers(0, len(mo)))
                r = bytearray((mo * (m // len(mo) + 2))[ph:ph + m])
                for _ in range(int(rng.integers(0, 3))):
                    r[int(rng.integers(0, m))] = int(rng.choice(letters))
                recs.append(bytes(r))
            else:
                recs.append(rng.choice(letters, size=m).tobytes())
        seq, off, ln = orc.records_to_arrays(recs)
        return orc.window_words(seq, off, k), orc.window_words(seq, off + ln - np.uint64(k), k)
    return _cached(("tie_nodes", n, k, seed), make)


@pytest.mark.parametrize("k,n", [(32, 50_000), (33, 20_000), (63, 5_000), (64, 30_000), (65, 8_000), (96, 12_000), (127, 20_000)])
@pytest.mark.parametrize("small_engine", [1, 0])
def test_overlap_path_wide_k(xctx, k, n, small_engine):
    first, last = tie_heavy_nodes(n, k, k + n)
    compl = k % 2 == 1
    _set(xctx, small_engine=small_engine)
    for strict, lb in ((True, False), (False, False), (True, True), (False, True)):
        ef, ov = xctx.overlap_path(first, last, k=k, complements=compl, lower_bound=lb, strict=strict)
        _level_loop_ran(xctx, n)
        want_ef, want_ov = _cached(("tie_orc", n, k, strict, lb),
                                   lambda: orc.overlap_path(first, last, k, compl, lower_bound=lb, parts=16 if strict else 1))
        assert np.array_equal(ef, want_ef) and np.array_equal(ov, want_ov), (strict, lb)


def low_complexity_wide(k, seed, n_records=8000):
    """Records of k to k + 50 bases of homopolymers, (AT)^n, (ACG)^n and mutated short tandem repeats: equal overlaps everywhere, and
    the greedy closes cycles at wide k."""
    def make():
        rng = np.random.default_rng(seed)
        recs = []
        for i in range(n_records):
            n = k + int(rng.integers(0, 51))
            kind = i % 4
            if kind == 0:
                r = bytes([b"ACGT"[int(rng.integers(0, 4))]]) * n
            elif kind == 1:
                r = (b"AT" * n)[int(rng.integers(0, 2)):][:n]
            else:
                m = rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), size=int(rng.integers(2, 6))).tobytes()
                r = bytearray((m * (n // len(m) + 1))[:n])
                for _ in range(int(rng.integers(0, 3))):
                    r[int(rng.integers(0, n))] = b"ACGT"[int(rng.integers(0, 4))]
                r = bytes(r)
            recs.append(np.frombuffer(r, dtype=np.uint8).copy())
        return synth.frame_records(recs)
    return _cached(("low_wide", k, seed, n_records), make)


@pytest.mark.parametrize("k", [40, 64, 100])
@pytest.mark.parametrize("compl", [True, False])
@pytest.mark.parametrize("small_engine", [1, 0])
def test_cycles_wide_k(xctx, k, compl, small_engine):
    _set(xctx, small_engine=small_engine)
    got = _exact(xctx, low_complexity_wide(k, k), k, compl)
    _level_loop_ran(xctx, got.n_nodes)
    assert xctx.stat("path_bans") > 0
