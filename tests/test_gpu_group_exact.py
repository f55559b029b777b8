"""The multi-GPU construction byte for byte against the one-batch greedy oracle (orc.compute_from_fasta).

A group (kc_init_multi, group.cuh) cuts the input into slices of window END positions, one per rank, ships every k-mer to the
owner of its hash range, resolves it there, clears the losers' bits in every rank's flags and prints its own slice of the
superstring.  Whatever the slicing, the bytes must be those of the oracle.  The slices are cut over tiles of 8192, 4096 or 2048
window ends (fixed slots and exact route at k < 32, < 64, <= 127) and of 8192 (signature scan), so the inputs here plant their
features at every multiple of 2048 positions: every slice edge of every rank count, in every geometry, lands on one.

Every case checks through the ranks' statistics that the rung it is meant to cover ran, the same on every rank:
  signature buckets  sig_runs + 1                           (k >= 26, no -z)
  fixed slots        fast_runs + 1                          (fast_heuristics off, so -z takes them too)
  exact route        neither, and no fallback of either.
The ranks share one device (a device ordinal may repeat); in-process ranks wait on host barriers and events, never on a
spinning kernel, so they cannot starve each other."""
import numpy as np
import pytest
import torch

import kmercamel_b200 as kb
from kmercamel_b200 import synth
from oracle import orc
from test_gpu_fasta_exact import DEFAULTS, _set, genome_with_reads, low_complexity

SITE = 2048              # KsCfg<4>::EX_TILE; the other tiles (4096, 8192, the signature scan's 8192) are multiples of it
EMIT_CHUNK = 16384       # KC_EMIT_CHUNK: a node is printed in chunks of this many bytes, slices are cut at 16-byte multiples
STATS = ("sig_runs", "sig_fallbacks", "fast_runs", "fast_fallbacks")
RUNG_STATS = {"sig": {"sig_runs": 1}, "fast": {"fast_runs": 1}, "exact": {}}
LEAF = 64                # fast_leaf_target: a plan of two levels on every input below that has more than a few kB
RUNG_OPTIONS = {"sig": dict(sig_min_items=0),
                "fast": dict(sig_set=0, fast_min_items=0, fast_leaf_target=LEAF),
                "exact": dict(sig_set=0, fast_set=0)}
_ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
_COMP = np.zeros(256, dtype=np.uint8)
for _a, _b in zip(b"ACGTacgt", b"TGCAtgca"):
    _COMP[_a] = _b


def revcomp(a):
    return _COMP[np.asarray(a, dtype=np.uint8)][::-1].copy()


def records_of(seq):
    """A framed sequence (records separated and ended by '\\n') -> (seq, rec_off, rec_len)."""
    nl = np.flatnonzero(seq == 10)
    starts = np.concatenate([[0], nl[:-1] + 1])
    assert len(nl) and nl[-1] == len(seq) - 1 and np.all(nl >= starts)
    return seq, starts.astype(np.uint64), (nl - starts).astype(np.uint64)


# ---- inputs (seeded, each under 1 MB) ---------------------------------------------------------------------------------------
_CACHE = {}


def _cached(key, make):
    if key not in _CACHE:
        _CACHE[key] = make()
    return _CACHE[key]


SHORT_LENGTHS = (4, 10, 20, 25, 26, 30, 31, 47, 60, 64, 100, 126)  # records across a site: shorter than some k, longer than others
N_KINDS = 5
N_BLOCKS = 296


def site_kind(i):
    """The feature planted at site i.  With 296 blocks this puts five different kinds on the five slice edges 3 ranks have over
    the three tile sizes, and over 2, 3, 5, 8 and 16 ranks every kind on an edge of every tile size (test_sites_on_slice_edges)."""
    return (i + i // 3) % N_KINDS


def boundary_genome(n_blocks=N_BLOCKS, units=12, seed=2048):
    """One record of random bases cut by a feature at every site B = i * SITE (i >= 1), of kind site_kind(i):
      0  a forward copy of a stretch from much earlier, over [B - 150, B + 150): the windows ending at B - 1 and at B repeat it
      1  the same, reverse-complemented
      2  an N run starting at B (valid windows end at B - 1, none at B)
      3  a record break at B
      4  a record shorter than some k across B
    Cross-slice counts: for c = 1..4, `units` random 160-mers occur c times each, spread over the input in c equal parts (so each
    occurrence lies in another slice once there are c ranks or more), one occurrence of every other unit reverse-complemented.  A
    unit's k-mers reach -z c only when the owner adds up what the senders shipped, and vanish at -z c + 1."""
    def make():
        rng = np.random.default_rng(seed)
        n = n_blocks * SITE
        s = _ACGT[rng.integers(0, 4, size=n, dtype=np.uint8)]
        slots = [b * SITE + o for b in range(n_blocks) for o in (400, 1000)]   # unit slots, clear of the sites' +-150
        used = np.zeros(len(slots), dtype=bool)
        for c in range(1, 5):
            for u in range(units):
                unit = _ACGT[rng.integers(0, 4, size=160, dtype=np.uint8)]
                for j in range(c):
                    want = int((j + 0.5) * len(slots) / c) + 3 * (u - units // 2) + c
                    at = min((x for x in range(len(slots)) if not used[x]), key=lambda x: abs(x - want))
                    used[at] = True
                    p = slots[at]
                    s[p:p + 160] = revcomp(unit) if (j == 1 and u % 2) else unit
        for i in range(1, n_blocks):
            b = i * SITE
            kind = site_kind(i)
            if i % 7 == 0:
                s[b + 200:b + 350] += 32                                         # a lower-case stretch
            if kind in (0, 1):
                j = int(rng.integers(0, max(1, i - 8)))
                src = s[j * SITE + 1250:j * SITE + 1550].copy()                  # block interiors that nothing is planted on
                s[b - 150:b + 150] = src if kind == 0 else revcomp(src)
            elif kind == 2:
                s[b:b + 1 + (i * 7) % 40] = ord("N")
            elif kind == 3:
                s[b] = 10
            else:
                ln = SHORT_LENGTHS[i % len(SHORT_LENGTHS)]
                a = ln // 2 + 1
                s[b - a] = 10
                s[b - a + ln + 1] = 10
        s = np.concatenate([s, np.frombuffer(b"\n", dtype=np.uint8)])
        return records_of(s)
    return _cached(("boundary", n_blocks, units, seed), make)


def count_255(seed=255):
    """A 31-mer that occurs 255 times (half of them reverse-complemented) and one that occurs 254 times, each occurrence a record
    of its own between random 560-base records, so that the occurrences spread over every slice."""
    def make():
        rng = np.random.default_rng(seed)
        a, b = (_ACGT[rng.integers(0, 4, size=31, dtype=np.uint8)] for _ in range(2))
        specials = [a if i % 2 else revcomp(a) for i in range(255)] + [b] * 254
        order = rng.permutation(len(specials))
        recs = []
        for i in order:
            recs.append(_ACGT[rng.integers(0, 4, size=560, dtype=np.uint8)])
            recs.append(specials[i])
        return synth.frame_records(recs)
    return _cached("count_255", make)


def tiny():
    """Less than one tile of the smallest geometry: every rank but the last has an empty slice."""
    def make():
        r = synth.random_genome_records(3, 600, 1601)
        return synth.frame_records([r[0], r[1], np.concatenate([r[2][:200], r[0][100:300], r[2][200:400]]), r[0][50:70]])
    return _cached("tiny", make)


def short_superstring(length):
    """One random record: a superstring shorter than 16 bytes a rank, so some ranks' emission slices are empty."""
    return _cached(("short_ms", length), lambda: synth.frame_records(synth.random_genome_records(1, length, 1700 + length)))


def long_reverse_pair(k, n_ranks=16):
    """Two records of more than EMIT_CHUNK * n_ranks bases; the second ends with the reverse complement of the first one's last
    k - 1 bases, so the greedy joins the first with the second's reverse strand and prints one long node backwards."""
    def make():
        ln = EMIT_CHUNK * n_ranks + 1000
        r0, r1 = synth.random_genome_records(2, ln, 1800 + k)
        r1 = r1.copy()
        r1[ln - (k - 1):] = revcomp(r0[ln - (k - 1):])
        return synth.frame_records([r0, r1])
    return _cached(("long_pair", k, n_ranks), make)


def short_sparse():
    """Records of 31 to 34 bases: at k = 31 one run for every 2.5 k-mers."""
    return _cached("short_sparse", lambda: synth.frame_records(synth.short_records(3000, 31, 34, 1900)))


def concatenated(*names):
    """Framed inputs back to back (more than 1 MB for the heap to outgrow its first size)."""
    def make():
        parts = [_input(n) for n in names]
        shift = np.cumsum([0] + [len(p[0]) for p in parts[:-1]]).astype(np.uint64)
        return (np.concatenate([p[0] for p in parts]), np.concatenate([p[1] + d for p, d in zip(parts, shift)]),
                np.concatenate([p[2] for p in parts]))
    return _cached(("cat",) + names, make)


INPUTS = {"boundary": boundary_genome, "count_255": count_255, "tiny": tiny, "gr": genome_with_reads,
          "low": lambda: low_complexity(3, 8000),       # one run for every 3 to 4.3 k-mers at k = 8 and k = 9 -u
          "short_sparse": short_sparse,
          "ms24": lambda: short_superstring(24), "ms30": lambda: short_superstring(30), "ms100": lambda: short_superstring(100),
          "long31": lambda: long_reverse_pair(31), "long63": lambda: long_reverse_pair(63), "long127": lambda: long_reverse_pair(127),
          "boundary+long31": lambda: concatenated("boundary", "long31")}


def _input(name):
    return INPUTS[name]()


def test_sites_on_slice_edges():
    """The rank counts below put every kind of site on a slice edge of every tile size (the plan of kc_group_plan; the signature
    scan cuts like k < 32), and the five edges of 3 ranks on five kinds."""
    n_bytes = len(boundary_genome()[0])
    kinds_3 = {}
    for k in (31, 63, 127):
        kinds = set()
        for n in (2, 3, 5, 8, 16):
            for r in range(1, n):
                e = kb.group_plan(n, r, k, n_bytes)["pos_begin"]
                assert e % SITE == 0
                kinds.add(site_kind(e // SITE))
                if n == 3:
                    kinds_3[e] = site_kind(e // SITE)
        assert kinds == set(range(N_KINDS)), k
    assert sorted(kinds_3.values()) == list(range(N_KINDS))


# ---- fixtures -----------------------------------------------------------------------------------------------------------
def _devices(n_ranks):
    return [r % torch.cuda.device_count() for r in range(n_ranks)]


@pytest.fixture(scope="module")
def groups():
    """One group per rank count for the whole module, created on first use; the ranks share the visible devices round robin."""
    made = {}

    def get(n_ranks):
        if n_ranks not in made:
            made[n_ranks] = kb.Group(_devices(n_ranks))
        return made[n_ranks]
    yield get
    for g in made.values():
        g.close()


def _reset(grp, **options):
    """Every option at its default, fast_heuristics off (no rung skipped on account of -z or of an earlier overflow), then options."""
    _set(grp, **DEFAULTS)
    grp.set_option("fast_heuristics", 0)
    _set(grp, **options)


@pytest.fixture
def group(groups):
    """-> get(n_ranks, **options): the module's group of that size, set up by _reset; the defaults are restored afterwards."""
    used = []

    def get(n_ranks, **options):
        g = groups(n_ranks)
        used.append(g)
        _reset(g, **options)
        return g
    yield get
    for g in used:
        _set(g, **DEFAULTS)


# ---- the check ----------------------------------------------------------------------------------------------------------
def _stats(grp):
    return {n: grp.stat(n) for n in STATS}


def _single(ctx, name, k, compl, z, sparse):
    """(n_occurrences, length) of the same job on one GPU, computed once."""
    def make():
        ctx.set_option("sparse_switch", int(sparse))
        try:
            r = ctx.compute(_input(name)[0], k=k, complements=compl, min_frequency=z)
        finally:
            ctx.set_option("sparse_switch", 1)
        return r.n_occurrences, r.length
    return _cached(("single", name, k, compl, z, sparse), make)


def check(grp, ctx, name, k, compl, z, rung, sparse=True):
    """grp.compute must give orc.compute_from_fasta's bytes, k-mer, node and run counts, the single GPU's n_occurrences and length,
    and advance the statistics of `rung` by one on every rank and nothing else; -> the group's result.  The oracle's answer depends
    on neither the rung nor the rank count: it is computed once per job."""
    seq, off, ln = _input(name)
    want = _cached(("orc", name, k, compl, z, sparse), lambda: orc.compute_from_fasta(seq, off, ln, k, compl, z, sparse_switch=sparse))
    s0 = _stats(grp)
    got = grp.compute(seq, k=k, complements=compl, min_frequency=z)
    s1 = _stats(grp)
    deltas = [{n: s1[n][r] - s0[n][r] for n in STATS if s1[n][r] != s0[n][r]} for r in range(grp.n)]
    assert deltas == [RUNG_STATS[rung]] * grp.n, (name, k, compl, z, rung, deltas)
    assert got.n_kmers == want["n_kmers"]
    assert (got.n_nodes, got.n_simplitigs) == (want["n_nodes"], want["n_simplitigs"])
    assert got.length == len(want["ms"])
    assert got.ms == want["ms"]
    assert (got.n_occurrences, got.length) == _single(ctx, name, k, compl, z, sparse)
    return got


def _id(rung, k, compl, z):
    return f"{rung}-k{k}{'' if compl else 'u'}-z{z}"


# ---- the rung matrix at 3 ranks -------------------------------------------------------------------------------------------
SIG_KS = (26, 27, 31, 32, 47, 63, 64, 95, 127)
FAST_KS = (11, 21, 31, 32, 63, 64, 127)
EXACT_KS = (5, 11, 21, 31, 32, 63, 64, 127)
MATRIX = ([("sig", k, c, 1) for k in SIG_KS for c in (True, False)]
          + [("fast", k, c, z) for k in FAST_KS for c in (True, False) for z in (1, 2, 3)]
          + [("exact", k, c, z) for k in EXACT_KS for c in (True, False) for z in (1, 2, 3)])


@pytest.mark.gpu
@pytest.mark.parametrize("rung,k,compl,z", MATRIX, ids=[_id(*c) for c in MATRIX])
def test_rungs_three_ranks(group, ctx, rung, k, compl, z):
    check(group(3, **RUNG_OPTIONS[rung]), ctx, "boundary", k, compl, z, rung)


# every rung, every word width and -z 1 / 3 at the other rank counts: 2, 5 (uneven digit ownership), 8 and 16 (KC_MAX_PEERS)
SUBSET = ([("sig", k, c, 1) for k, c in ((31, True), (63, False), (127, True))]
          + [(r, k, c, z) for r in ("fast", "exact") for k, c in ((21, True), (63, True), (127, False)) for z in (1, 3)])


@pytest.mark.gpu
@pytest.mark.parametrize("n_ranks", [2, 5, 8, 16])
@pytest.mark.parametrize("rung,k,compl,z", SUBSET, ids=[_id(*c) for c in SUBSET])
def test_rungs_other_rank_counts(group, ctx, n_ranks, rung, k, compl, z):
    check(group(n_ranks, **RUNG_OPTIONS[rung]), ctx, "boundary", k, compl, z, rung)


# ---- reads with coverage: realistic -z ------------------------------------------------------------------------------------------
GR_CASES = [("sig", 31, True, 1), ("fast", 21, True, 2), ("fast", 31, True, 3), ("fast", 63, False, 2), ("exact", 21, True, 2),
            ("exact", 31, True, 3), ("exact", 63, False, 2)]


@pytest.mark.gpu
@pytest.mark.parametrize("n_ranks", [3, 8])
@pytest.mark.parametrize("rung,k,compl,z", GR_CASES, ids=[_id(*c) for c in GR_CASES])
def test_genome_with_reads(group, ctx, n_ranks, rung, k, compl, z):
    check(group(n_ranks, **RUNG_OPTIONS[rung]), ctx, "gr", k, compl, z, rung)


# ---- -z 255 ----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("rung", ["exact", "fast"])
def test_count_255(group, ctx, rung):
    got = check(group(3, **RUNG_OPTIONS[rung]), ctx, "count_255", 31, True, 255, rung)
    assert got.n_kmers == 1 and got.length == 31            # the 255-fold k-mer alone: the 254-fold one is gone


# ---- less than one tile: most slices empty ----------------------------------------------------------------------------------
TINY_CASES = [("sig", 31, True, 1), ("sig", 64, False, 1), ("fast", 21, True, 2), ("fast", 31, False, 1), ("exact", 11, True, 1),
              ("exact", 21, True, 2), ("exact", 127, True, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("n_ranks", [8, 16])
@pytest.mark.parametrize("rung,k,compl,z", TINY_CASES, ids=[_id(*c) for c in TINY_CASES])
def test_tiny_input(group, ctx, n_ranks, rung, k, compl, z):
    assert len(tiny()[0]) < SITE
    options = dict(RUNG_OPTIONS[rung], fast_leaf_target=4) if rung == "fast" else RUNG_OPTIONS[rung]  # two levels on 2 kB
    check(group(n_ranks, **options), ctx, "tiny", k, compl, z, rung)


# ---- emission slices ------------------------------------------------------------------------------------------------------
SHORT_MS = ([(n, "ms24", "exact", 11) for n in (2, 3, 5, 8, 16)] + [(n, "ms30", "sig", 27) for n in (2, 3, 5, 8, 16)]
            + [(n, "ms100", r, k) for n in (8, 16) for r, k in (("sig", 31), ("exact", 63))])


@pytest.mark.gpu
@pytest.mark.parametrize("n_ranks,name,rung,k", SHORT_MS)
def test_superstring_shorter_than_the_slices(group, ctx, n_ranks, name, rung, k):
    got = check(group(n_ranks, **RUNG_OPTIONS[rung]), ctx, name, k, True, 1, rung)
    assert got.length < 16 * n_ranks


@pytest.mark.gpu
@pytest.mark.parametrize("n_ranks", [2, 3, 5, 8, 16])
@pytest.mark.parametrize("rung,k", [("sig", 31), ("fast", 31), ("sig", 127), ("exact", 63)])
def test_long_node_on_the_reverse_strand(group, ctx, n_ranks, rung, k):
    name = f"long{k}"
    seq, off, ln = _input(name)
    assert all(int(x) > EMIT_CHUNK * n_ranks for x in ln)
    got = check(group(n_ranks, **RUNG_OPTIONS[rung]), ctx, name, k, True, 1, rung)
    ms = got.ms.upper()
    assert any(bytes(revcomp(seq[int(o):int(o) + int(n)])) in ms for o, n in zip(off, ln))


# ---- the sparse switch (the k-mers are the nodes) --------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n_ranks", [3, 8])
@pytest.mark.parametrize("name,rung,k,compl", [("low", "exact", 8, True), ("low", "exact", 9, False), ("short_sparse", "sig", 31, True),
                                               ("short_sparse", "fast", 31, False)])
@pytest.mark.parametrize("sparse", [1, 0])
def test_sparse_switch(group, ctx, n_ranks, name, rung, k, compl, sparse):
    got = check(group(n_ranks, **RUNG_OPTIONS[rung], sparse_switch=sparse), ctx, name, k, compl, 1, rung, sparse=bool(sparse))
    assert got.n_simplitigs * 5 >= got.n_kmers
    assert got.n_nodes == (got.n_kmers if sparse else got.n_simplitigs)


# ---- one group through a fixed sequence of jobs ----------------------------------------------------------------------------------
# (input, k, complements, -z, rung, options).  The heap is rebuilt when a job outgrows it (n_bytes, then the word width), the rungs
# alternate, and the fixed slots run twice on one input with another plan each time and no exact job in between (the exact route
# rebuilds the level-0 destination tables of every rank): fast_sigmas 8 -> 16 changes the sub-slot stride, fast_leaf_target
# 64 -> 16 the number of digits as well.  Tables kept from the first job of such a pair would scatter the second one's items at
# the first one's stride, or to digits that had no owner.
REUSE_JOBS = [
    ("tiny", 21, True, 1, "exact", {}),
    ("gr", 21, True, 2, "fast", {}),
    ("gr", 31, True, 1, "sig", {}),
    ("boundary+long31", 31, True, 1, "sig", {}),           # more bytes than the heap was sized for
    ("boundary+long31", 31, True, 2, "fast", {}),
    ("boundary", 63, False, 1, "sig", {}),                 # a wider word
    ("gr", 31, True, 3, "exact", {}),
    ("boundary", 31, True, 1, "fast", dict(fast_sigmas=8)),
    ("boundary", 31, True, 1, "fast", dict(fast_sigmas=16)),
    ("boundary", 31, True, 2, "fast", dict(fast_sigmas=16)),
    ("boundary", 27, True, 1, "sig", {}),
    ("boundary", 21, False, 2, "fast", dict(fast_leaf_target=64)),
    ("boundary", 21, False, 2, "fast", dict(fast_leaf_target=16)),
    ("boundary", 21, True, 3, "fast", dict(fast_leaf_target=16, fast_sigmas=16)),
    ("long127", 127, True, 1, "fast", {}),                 # the widest word
    ("long127", 127, True, 1, "exact", {}),
    ("long127", 127, True, 1, "fast", dict(fast_leaf_target=16)),
    ("gr", 11, True, 1, "exact", {}),
    ("gr", 11, True, 1, "fast", {}),
    ("gr", 11, True, 1, "fast", dict(fast_sigmas=16)),
]


@pytest.mark.gpu
def test_one_group_through_a_sequence_of_jobs(ctx):
    grp = kb.Group(_devices(3))
    try:
        for name, k, compl, z, rung, options in REUSE_JOBS:
            _reset(grp, **{**RUNG_OPTIONS[rung], **options})
            check(grp, ctx, name, k, compl, z, rung)
    finally:
        grp.close()
