"""The from-FASTA superstring byte for byte against a restatement of the whole pipeline (orc.compute_from_fasta).

From FASTA the nodes of the greedy are the first-occurrence runs of the input (runs.cuh), or its k-mers past the sparse switch, and
the engine runs non-strict: every prefix in one batch, all cycle closers of a round banned at once.  That output is a pure function of
the input, and the reference's greedy with one prefix batch (orc.overlap_path parts = 1) is its exact specification.  Every path the
device can take from FASTA must therefore give the oracle's bytes: the speculative tail, the single-CTA engine, the multi-kernel level
loop with its fused levels and cycle fallback, each k-mer set construction, the sparse switch, -M, the lower bound.  Each case checks
through the context's statistics that it reached the path it is meant to cover."""
import numpy as np
import pytest

from kmercamel_b200 import synth
import kmercamel_b200 as kb
from oracle import orc

pytestmark = pytest.mark.gpu

SPEC_RUNS = 512       # KC_SPEC_RUNS (tail_spec.cuh)
SMALL_NS = 1024       # more nodes than this: the first levels run in the multi-kernel level loop (small_engine.cuh)
DEFAULTS = dict(tail_spec=1, small_engine=1, small_threads=0, sparse_switch=1, sig_set=1, sig_load_pct=0, sig_min_items=1 << 16,
                fast_set=1, fast_min_items=1 << 16, fast_leaf_target=768, fast_sigmas=8, fast_heuristics=1)
STATS = ("tail_spec_runs", "tail_spec_fallbacks", "sig_runs", "sig_fallbacks", "fast_runs", "fast_fallbacks")


@pytest.fixture(scope="module")
def fctx():
    c = kb.Context(0)
    yield c
    c.close()


@pytest.fixture
def xctx(fctx):
    """The module's context with every option at its default and no memory of earlier overflows; restored afterwards."""
    _set(fctx, **DEFAULTS)
    fctx.set_option("fast_heuristics", 0)
    try:
        yield fctx
    finally:
        _set(fctx, **DEFAULTS)


def _set(ctx, **kw):
    for name, value in kw.items():
        ctx.set_option(name, value)


def _stats(ctx):
    return {n: ctx.stat(n) for n in STATS}


def _advanced(s0, s1):
    return {n for n in STATS if s1[n] != s0[n]}


# ---- inputs ------------------------------------------------------------------------------------------------------------
_CACHE = {}


def _cached(name, make):
    if name not in _CACHE:
        _CACHE[name] = make()
    return _CACHE[name]


def spneumoniae():
    import gzip
    import os
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "spneumoniae.fa.gz")
    return _cached("spn", lambda: kb.frame_fasta(gzip.open(path).read()))


def messy_genome(seed, n_records=12, max_len=30_000):
    """Ragged records with lower-case stretches and N runs, plus records shorter than k."""
    def make():
        rng = np.random.default_rng(seed)
        recs = []
        for i in range(n_records):
            r = synth.random_genome_records(1, int(rng.integers(max_len // 3, max_len)), seed * 100 + i)[0].copy()
            a = int(rng.integers(0, len(r) - 2000))
            r[a:a + 1500] += 32
            if i % 3 == 0:
                b = int(rng.integers(0, len(r) - 20))
                r[b:b + int(rng.integers(1, 20))] = ord("N")
            recs.append(r)
        recs.append(np.frombuffer(b"ACGTACGTAC", dtype=np.uint8).copy())
        recs.append(recs[0][:20].copy())
        return synth.frame_records(recs)
    return _cached(("messy", seed), make)


def short_records(n, length, seed):
    """n random records of `length` bases: one first-occurrence run each."""
    return _cached(("short", n, length, seed), lambda: synth.frame_records(synth.random_genome_records(n, length, seed)))


def human_like():
    return _cached("human", lambda: synth.frame_records(synth.human_like_genome(3_000_000, seed=3100)))


def reads():
    return _cached("reads", lambda: synth.frame_records(list(synth.reads_from_genome(150_000, 8.0, 150, 0.01, seed=47))))


def genome_with_reads():
    """Random records, a duplicated piece, an N / low-complexity record and reads with coverage: k-mers that occur 2 and 3 times."""
    def make():
        recs = synth.random_genome_records(4, 20_000, 77)
        recs.append(recs[0][1000:6000].copy())
        recs.append(np.frombuffer(b"ACGTNNNNNACGT" * 40, dtype=np.uint8).copy())
        recs += list(synth.reads_from_genome(20_000, 4.0, 150, 0.01, seed=78))
        return synth.frame_records(recs)
    return _cached("gr", make)


def sparse_input(name):
    return _cached(name, lambda: synth.big_config_input(name))


def low_complexity(seed, n_records=600):
    """Many short records of homopolymers, (AT)^n, (ACG)^n and mutated short tandem repeats: equal overlaps everywhere, and the
    greedy closes cycles at most levels."""
    def make():
        rng = np.random.default_rng(seed)
        recs = []
        for i in range(n_records):
            n = int(rng.integers(8, 60))
            kind = i % 5
            if kind == 0:
                r = bytes([b"ACGT"[int(rng.integers(0, 4))]]) * n
            elif kind == 1:
                r = (b"AT" * n)[int(rng.integers(0, 2)):][:n]
            elif kind == 2:
                r = (b"ACG" * n)[int(rng.integers(0, 3)):][:n]
            else:
                m = rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), size=int(rng.integers(2, 6))).tobytes()
                r = bytearray((m * (n // len(m) + 1))[:n])
                for _ in range(int(rng.integers(0, 3))):
                    r[int(rng.integers(0, n))] = b"ACGT"[int(rng.integers(0, 4))]
                r = bytes(r)
            recs.append(np.frombuffer(r, dtype=np.uint8).copy())
        return synth.frame_records(recs)
    return _cached(("low", seed, n_records), make)


# ---- the check ---------------------------------------------------------------------------------------------------------
def _exact(ctx, inp, k, compl=True, z=1, maxone=False, sparse=True):
    """ctx.compute on the framed input must be orc.compute_from_fasta byte for byte; -> the device result."""
    seq, off, ln = inp
    key = ("orc", id(seq), k, compl, z, maxone, sparse)
    want = _cached(key, lambda: orc.compute_from_fasta(seq, off, ln, k, compl, z, want_maxone=maxone, sparse_switch=sparse))
    got = ctx.compute(seq, k=k, complements=compl, min_frequency=z, want_maxone=maxone)
    assert got.n_kmers == want["n_kmers"]
    assert (got.n_nodes, got.n_simplitigs) == (want["n_nodes"], want["n_simplitigs"])
    assert got.length == len(want["ms"])
    assert got.ms == want["ms"]
    if maxone:
        assert got.maxone == want["maxone"]
    return got


# ---- speculative tail (<= 512 runs) after the signature construction ------------------------------------------------------
# spneumoniae has more than 512 runs at k = 31 (1127, and 967 with -u): the speculation is tried there and falls back
SPEC_CASES = [("spn", 31, True), ("spn", 31, False), ("spn", 63, True), ("spn", 63, False), ("spn", 127, True), ("spn", 127, False),
              ("messy", 26, True), ("messy", 31, True), ("messy", 32, False), ("messy", 63, False), ("messy", 64, True),
              ("messy", 127, True)]


def _spec_input(ctx, name):
    if name == "spn":
        # its repeats overflow the signature buckets at the planned load: plan them a fifth full
        ctx.set_option("sig_load_pct", 20)
        return spneumoniae()
    return messy_genome(5)


@pytest.mark.parametrize("name,k,compl", SPEC_CASES)
def test_speculative_tail(xctx, name, k, compl):
    _set(xctx, sig_min_items=0)
    inp = _spec_input(xctx, name)
    s0 = _stats(xctx)
    got = _exact(xctx, inp, k, compl)
    spec = got.n_simplitigs <= SPEC_RUNS
    assert _advanced(s0, _stats(xctx)) == {"tail_spec_runs" if spec else "tail_spec_fallbacks", "sig_runs"}
    assert spec or (name, k) == ("spn", 31)


# ---- single-CTA engine without the speculation ------------------------------------------------------------------------------
@pytest.mark.parametrize("name,k,compl", SPEC_CASES)
def test_small_engine_without_spec(xctx, name, k, compl):
    _set(xctx, sig_min_items=0, tail_spec=0)
    inp = _spec_input(xctx, name)
    s0 = _stats(xctx)
    _exact(xctx, inp, k, compl)
    assert _advanced(s0, _stats(xctx)) == {"sig_runs"}
    assert xctx.stat("path_levels") > 0


@pytest.mark.parametrize("n_runs", [SPEC_RUNS + 1, 1000])
def test_small_engine_past_the_spec_cap(xctx, n_runs):
    _set(xctx, sig_min_items=0)
    s0 = _stats(xctx)
    got = _exact(xctx, short_records(n_runs, 60, 5), 31)
    assert _advanced(s0, _stats(xctx)) == {"tail_spec_fallbacks", "sig_runs"}
    assert got.n_simplitigs == n_runs and 2 * got.n_nodes <= 2 * SMALL_NS


# ---- multi-kernel level loop ---------------------------------------------------------------------------------------------
# more than SMALL_NS nodes with complements: the free ends do not fit the single-CTA engine at the first levels.  (The human-like
# genome has only 348 runs at k = 63; the reads take that width.)
@pytest.mark.parametrize("name,k", [("human", 31), ("spn", 31), ("reads", 31), ("reads", 47), ("reads", 63)])
@pytest.mark.parametrize("small_engine", [1, 0])
def test_level_loop(xctx, name, k, small_engine):
    _set(xctx, small_engine=small_engine)
    got = _exact(xctx, {"human": human_like, "spn": spneumoniae, "reads": reads}[name](), k)
    assert got.n_nodes > SMALL_NS and xctx.stat("path_levels") > 0


# ---- fixed-slot and exact k-mer set constructions ----------------------------------------------------------------------------
@pytest.mark.parametrize("k,z", [(5, 1), (9, 1), (15, 1), (21, 1), (31, 1), (21, 2), (31, 2), (31, 3)])
@pytest.mark.parametrize("construction", ["fast", "exact"])
def test_set_constructions(xctx, k, z, construction):
    _set(xctx, sig_set=0, fast_min_items=0) if construction == "fast" else _set(xctx, sig_set=0, fast_set=0)
    s0 = _stats(xctx)
    _exact(xctx, genome_with_reads(), k, k % 2 == 1, z)
    # at k = 5 the 512 distinct k-mers repeat far beyond a fixed slot: the attempt overflows and the exact construction takes over
    fast = {"fast_fallbacks"} if k == 5 else {"fast_runs"}
    assert _advanced(s0, _stats(xctx)) == (fast if construction == "fast" else set())


# ---- sparse switch ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,k,compl", [("tiny_sparse_k31", 31, True), ("tiny_sparse_k9u", 9, False)])
@pytest.mark.parametrize("sparse", [1, 0])
def test_sparse_switch(xctx, name, k, compl, sparse):
    _set(xctx, sparse_switch=sparse)
    got = _exact(xctx, sparse_input(name), k, compl, sparse=bool(sparse))
    assert got.n_simplitigs * 5 >= got.n_kmers
    assert got.n_nodes == (got.n_kmers if sparse else got.n_simplitigs)


# ---- cycles and bans ------------------------------------------------------------------------------------------------------
# the last two have more than SMALL_NS nodes: their first levels run in the level loop even with the single-CTA engine on
BAN_CASES = [(4, True, 2, 600), (4, False, 9, 600), (5, False, 2, 600), (6, True, 3, 600), (7, True, 4, 600), (8, False, 5, 600),
             (10, True, 6, 600), (12, True, 7, 600), (12, False, 8, 600), (9, True, 22, 8000), (11, True, 23, 8000)]


@pytest.mark.parametrize("k,compl,seed,n_records", BAN_CASES)
@pytest.mark.parametrize("small_engine", [1, 0])
def test_cycles_and_bans(xctx, k, compl, seed, n_records, small_engine):
    _set(xctx, small_engine=small_engine)
    _exact(xctx, low_complexity(seed, n_records), k, compl)
    bans = xctx.stat("path_bans")
    print(f"k={k} complements={compl} seed={seed} small_engine={small_engine}: path_bans={bans} "
          f"path_ban_rounds={xctx.stat('path_ban_rounds')} path_levels={xctx.stat('path_levels')}")
    assert bans > 0 and xctx.stat("path_ban_rounds") > 0


# ---- -M -----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["spn31", "spn63u", "reads31", "gr21z2", "sparse9u", "low6", "low12u"])
def test_maxone(xctx, case):
    inp, k, compl, z = {"spn31": (spneumoniae, 31, True, 1), "spn63u": (spneumoniae, 63, False, 1), "reads31": (reads, 31, True, 1),
                        "gr21z2": (genome_with_reads, 21, True, 2), "sparse9u": (lambda: sparse_input("tiny_sparse_k9u"), 9, False, 1),
                        "low6": (lambda: low_complexity(3), 6, True, 1), "low12u": (lambda: low_complexity(8), 12, False, 1)}[case]
    _exact(xctx, inp(), k, compl, z, maxone=True)


# ---- the overlap stage alone, non-strict and strict ----------------------------------------------------------------------
@pytest.mark.parametrize("small_engine", [1, 0])
def test_overlap_path_non_strict_and_strict(xctx, small_engine):
    from test_host import tie_heavy_node_set
    from test_oracle import node_ends
    _set(xctx, small_engine=small_engine)
    banned = 0
    for seed in range(40):
        k, compl, recs = tie_heavy_node_set(seed)
        first, last = node_ends([r.decode() for r in recs], k)
        for strict, parts in ((False, 1), (True, 16)):
            ef, ov = xctx.overlap_path(first, last, k=k, complements=compl, strict=strict)
            want_ef, want_ov = orc.overlap_path(first, last, k, compl, parts=parts)
            assert np.array_equal(ef, want_ef) and np.array_equal(ov, want_ov), (seed, k, compl, strict)
            banned += not strict and xctx.stat("path_bans") > 0
    assert 3 * banned >= 40


# ---- lower bound ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,k,z", [("spn", 13, 1), ("spn", 31, 1), ("spn", 31, 2), ("reads", 31, 1), ("low", 8, 1)])
def test_lower_bound(xctx, name, k, z):
    seq, off, ln = {"spn": spneumoniae, "reads": reads, "low": lambda: low_complexity(4)}[name]()
    want = orc.lower_bound_from_fasta(seq, off, ln, k, True, z)
    lb, st = xctx.lower_bound(seq, k=k, min_frequency=z)
    assert lb == want and st.n_nodes == len(orc.fasta_nodes(seq, off, ln, k, True, z)[0])


# ---- device-resident input ------------------------------------------------------------------------------------------------
def test_compute_device(xctx):
    import torch
    seq, off, ln = messy_genome(5)
    want = orc.compute_from_fasta(seq, off, ln, 31, True)
    d = torch.from_numpy(seq).cuda()
    torch.cuda.synchronize()
    for tail_spec in (1, 0):
        _set(xctx, sig_min_items=0, tail_spec=tail_spec)
        res = xctx.compute_device(d.data_ptr(), d.numel(), k=31)
        assert (res.n_kmers, res.n_nodes) == (want["n_kmers"], want["n_nodes"])
        assert xctx.copy_to_host(res.ms_ptr, res.length) == want["ms"]


# ---- -S at scale: the strict engine on the fused level path ------------------------------------------------------------------
def tie_heavy_simplitigs(n, k, seed):
    """n records of k to k + 20 bases cut from a 2 kbp genome over {A, C}: the ends share (k-1)-overlaps with many others."""
    rng = np.random.default_rng(seed)
    genome = rng.choice(np.frombuffer(b"AC", dtype=np.uint8), size=2000).tobytes()
    starts = rng.integers(0, 2000 - k - 20, size=n)
    lens = rng.integers(k, k + 21, size=n)
    return [genome[s:s + l] for s, l in zip(starts, lens)]


@pytest.mark.parametrize("n,k,compl", [(10_000, 21, True), (30_000, 15, False), (100_000, 11, True)])
@pytest.mark.parametrize("small_engine", [1, 0])
def test_simplitigs_at_scale(xctx, n, k, compl, small_engine):
    recs = _cached(("S", n, k), lambda: tie_heavy_simplitigs(n, k, n + k))
    want_ms, want_mo = _cached(("S_orc", n, k, compl), lambda: orc.compute_from_simplitigs(recs, k, compl, True))
    seq, off, ln = orc.records_to_arrays(recs)
    _set(xctx, small_engine=small_engine)
    got = xctx.compute(seq, off, ln, k=k, complements=compl, assume_simplitigs=True, want_maxone=True)
    assert got.ms == want_ms and got.maxone == want_mo
    assert xctx.stat("path_levels") > 0
