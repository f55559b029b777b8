"""No result may depend on what the device arena held before a block was handed out.

One arena (kc_common.cuh Arena) serves every call of a context and is never cleared, and within a call its stack discipline hands the
same bytes out again (the speculative tail's region, a discarded set construction, scan and compaction scratch).  A kernel that reads
a word nobody wrote in this call sees an earlier call's bits, which on a fresh slab or on a repeated input are often exactly the right
ones.  The option "arena_poison" fills every block with a byte before it is handed out: 0x00 looks like a finished zero-fill, 0xFF
like KC_NONE, 0xA5 like neither, and 'A' like a base, so a loader that reads past the input sees extra k-mers instead of a record
break.  Every entry point, on every path it can take, must still give the oracle's bytes; so must a context after a long mixed call
history, and a call repeated with the worst-case estimate after it ran out of arena (run_with_arena).  Each case checks through the
context's statistics that it reached the path it is meant to cover."""
import numpy as np
import pytest

import kmercamel_b200 as kb
from kmercamel_b200 import synth
from oracle import orc
from test_gpu_fasta_exact import (DEFAULTS, SPEC_RUNS, SMALL_NS, _advanced, _cached, _exact, _set, _stats, genome_with_reads,
                                  low_complexity, messy_genome, reads, short_records, sparse_input, spneumoniae, tie_heavy_simplitigs)

pytestmark = pytest.mark.gpu

POISONS = [0x00, 0xFF, 0xA5, 0x41]
POISON_IDS = ["00", "ff", "a5", "A"]
OFF = dict(arena_poison=-1, arena_estimate_ppm=1_000_000)


@pytest.fixture(scope="module")
def actx():
    c = kb.Context(0)
    yield c
    c.close()


@pytest.fixture(params=POISONS, ids=POISON_IDS)
def pctx(actx, request):
    """The module's context at its defaults, no memory of earlier overflows, its arena poisoned with the parameter; restored afterwards."""
    _set(actx, **DEFAULTS, **OFF)
    actx.set_option("fast_heuristics", 0)
    actx.set_option("arena_poison", request.param)
    try:
        yield actx
    finally:
        _set(actx, **DEFAULTS, **OFF)


# ---- 1. every from-FASTA path, byte for byte against orc.compute_from_fasta ------------------------------------------------------
# (id, input, k, complements, -z, -M, sparse switch, options, statistics that must advance (None: not checked), extra check)
FASTA_CASES = [
    ("spec_k31", lambda: messy_genome(5), 31, True, 1, False, True, dict(sig_min_items=0), {"sig_runs", "tail_spec_runs"}, None),
    ("spec_k32u", lambda: messy_genome(5), 32, False, 1, False, True, dict(sig_min_items=0), {"sig_runs", "tail_spec_runs"}, None),
    ("spec_k63u", lambda: messy_genome(5), 63, False, 1, False, True, dict(sig_min_items=0), {"sig_runs", "tail_spec_runs"}, None),
    ("spec_k64", lambda: messy_genome(5), 64, True, 1, False, True, dict(sig_min_items=0), {"sig_runs", "tail_spec_runs"}, None),
    ("spec_k95", lambda: messy_genome(5), 95, True, 1, False, True, dict(sig_min_items=0), {"sig_runs", "tail_spec_runs"}, None),
    ("spec_k127", lambda: messy_genome(5), 127, True, 1, False, True, dict(sig_min_items=0), {"sig_runs", "tail_spec_runs"}, None),
    ("spec_fallback", lambda: short_records(SPEC_RUNS + 1, 60, 5), 31, True, 1, False, True, dict(sig_min_items=0),
     {"sig_runs", "tail_spec_fallbacks"}, None),
    ("small_engine", lambda: messy_genome(5), 31, True, 1, False, True, dict(sig_min_items=0, tail_spec=0), {"sig_runs"}, "levels"),
    ("level_loop", reads, 31, True, 1, False, True, dict(), None, "many_nodes"),
    ("level_loop_k47_no_small", reads, 47, True, 1, False, True, dict(small_engine=0), None, "many_nodes"),
    ("sig_overflow", lambda: messy_genome(5), 31, True, 1, False, True, dict(sig_min_items=0, sig_load_pct=400, fast_min_items=0),
     {"sig_fallbacks", "tail_spec_fallbacks", "fast_runs"}, None),
    ("fast", genome_with_reads, 21, True, 1, False, True, dict(sig_set=0, fast_min_items=0), {"fast_runs"}, None),
    ("fast_overflow", genome_with_reads, 5, True, 1, False, True, dict(sig_set=0, fast_min_items=0), {"fast_fallbacks"}, None),
    ("exact_k32", genome_with_reads, 32, True, 1, False, True, dict(sig_set=0, fast_set=0), set(), None),
    ("exact_k63u", genome_with_reads, 63, False, 1, False, True, dict(sig_set=0, fast_set=0), set(), None),
    ("z2", genome_with_reads, 31, True, 2, False, True, dict(fast_min_items=0), {"fast_runs"}, None),
    ("z3_exact", genome_with_reads, 31, True, 3, False, True, dict(fast_set=0), set(), None),
    ("sparse", lambda: sparse_input("tiny_sparse_k31"), 31, True, 1, False, True, dict(), None, "sparse"),
    ("sparse_k9u", lambda: sparse_input("tiny_sparse_k9u"), 9, False, 1, False, True, dict(), None, "sparse"),
    ("maxone_spn31", spneumoniae, 31, True, 1, True, True, dict(), None, None),
    ("maxone_z2", genome_with_reads, 21, True, 2, True, True, dict(), None, None),
    ("maxone_k127u", lambda: messy_genome(5), 127, False, 1, True, True, dict(), None, None),
    ("bans", lambda: low_complexity(6), 6, True, 1, False, True, dict(), None, "bans"),
]


@pytest.mark.parametrize("case", FASTA_CASES, ids=[c[0] for c in FASTA_CASES])
def test_poisoned_fasta_paths(pctx, case):
    _, inp, k, compl, z, maxone, sparse, opts, advance, extra = case
    _set(pctx, **opts)
    s0 = _stats(pctx)
    got = _exact(pctx, inp(), k, compl, z, maxone=maxone, sparse=sparse)
    if advance is not None:
        assert _advanced(s0, _stats(pctx)) == advance
    if extra == "levels":
        assert pctx.stat("path_levels") > 0
    elif extra == "many_nodes":
        assert got.n_nodes > SMALL_NS and pctx.stat("path_levels") > 0
    elif extra == "sparse":
        assert got.n_nodes == got.n_kmers
    elif extra == "bans":
        assert pctx.stat("path_bans") > 0


# ---- 2. the neighbours of the compute path --------------------------------------------------------------------------------------
def _records(inp):
    seq, off, ln = inp
    return [bytes(seq[int(o):int(o) + int(n)]) for o, n in zip(off, ln)]


def test_poisoned_simplitigs_maxone(pctx):
    recs = _cached(("S", 3000, 21), lambda: tie_heavy_simplitigs(3000, 21, 3021))
    want_ms, want_mo = _cached(("S_orc", 3000, 21, True), lambda: orc.compute_from_simplitigs(recs, 21, True, True))
    seq, off, ln = orc.records_to_arrays(recs)
    for small_engine in (1, 0):
        _set(pctx, small_engine=small_engine)
        got = pctx.compute(seq, off, ln, k=21, assume_simplitigs=True, want_maxone=True)
        assert got.ms == want_ms and got.maxone == want_mo
        assert pctx.stat("path_levels") > 0


def test_poisoned_lower_bound(pctx):
    seq, off, ln = genome_with_reads()
    for k, z in ((31, 1), (31, 2), (63, 1)):
        want = _cached(("lb", k, z), lambda: orc.lower_bound_from_fasta(seq, off, ln, k, True, z))
        lb, st = pctx.lower_bound(seq, k=k, min_frequency=z)
        assert lb == want
    recs = _cached(("S", 3000, 21), lambda: tie_heavy_simplitigs(3000, 21, 3021))
    s2, o2, l2 = orc.records_to_arrays(recs)
    want = _cached(("lbS", 21), lambda: orc.lower_bound_from_simplitigs(recs, 21, True))
    lb, _ = pctx.lower_bound(s2, o2, l2, k=21, assume_simplitigs=True)
    assert lb == want


@pytest.mark.parametrize("route", ["sig", "exact"])
def test_poisoned_streaming(pctx, route):
    seq, off, ln = genome_with_reads()
    if route == "sig":
        _set(pctx, sig_min_items=0)
    else:
        _set(pctx, sig_set=0, fast_set=0)
    for k, z in ((31, 1), (31, 2), (31, 3), (64, 2)):
        want = _cached(("stream", k, z), lambda: orc.streaming(seq, off, ln, k, True, z))
        s0 = _stats(pctx)
        got = pctx.streaming(seq, k=k, min_frequency=z)
        assert got.ms == want, (k, z)
        assert _advanced(s0, _stats(pctx)) == ({"sig_runs"} if route == "sig" else set())


def _masked_superstring():
    seq, off, ln = messy_genome(5)
    return _cached(("ms", 31), lambda: orc.compute_from_fasta(seq, off, ln, 31, True)["ms"])


def test_poisoned_maskopt(pctx):
    ms = _masked_superstring()
    assert ms[-1:] != b"\n"                    # the last byte is a letter: a loader that runs past n meets the poison
    for minimize in (False, True):
        want = _cached(("maskopt", minimize), lambda: orc.maskopt(ms, 31, True, minimize))
        assert pctx.maskopt(ms, k=31, minimize=minimize).ms == want


@pytest.mark.parametrize("k", [21, 31, 63])
def test_poisoned_count_kmers(pctx, k):
    seq, off, ln = genome_with_reads()
    keys, vals = _cached(("count", k), lambda: orc.count_kmers(seq, off, ln, k, True))
    for z in (1, 2):
        got_k, got_v = pctx.count_kmers(seq, k=k, min_frequency=z)
        keep = vals.astype(np.int64) + 1 >= z
        assert np.array_equal(got_k, keys[keep]) and np.array_equal(got_v, vals[keep])


@pytest.mark.parametrize("sig_set", [1, 0])
def test_poisoned_kmer_digest(pctx, sig_set):
    _set(pctx, sig_set=sig_set, sig_min_items=0)
    seq, off, ln = messy_genome(5)
    for k in (31, 63):
        keys, vals = _cached(("count_messy", k), lambda: orc.count_kmers(seq, off, ln, k, True))
        want = orc.kmer_digest(keys, vals)
        s0 = _stats(pctx)
        assert pctx.kmer_digest(seq, k=k) == want
        assert _advanced(s0, _stats(pctx)) == ({"sig_runs"} if sig_set else set())
        # the same set without the final '\n': the last byte is a base
        assert pctx.kmer_digest(seq[:-1], k=k) == want
    keys, vals = _cached(("count_messy", 31), lambda: orc.count_kmers(seq, off, ln, 31, True))
    ms = _masked_superstring()
    assert pctx.kmer_digest(np.frombuffer(ms, dtype=np.uint8), k=31, masked=True) == orc.kmer_digest(keys, vals)
    gseq, goff, gln = genome_with_reads()
    gk, gv = _cached(("count", 21), lambda: orc.count_kmers(gseq, goff, gln, 21, True))
    assert pctx.kmer_digest(gseq, k=21, min_frequency=2) == orc.kmer_digest(gk, gv, 2)


def test_poisoned_overlap_path(pctx):
    from test_host import tie_heavy_node_set
    from test_oracle import node_ends
    for seed in range(6):
        k, compl, recs = tie_heavy_node_set(seed)
        first, last = node_ends([r.decode() for r in recs], k)
        for strict, parts in ((False, 1), (True, 16)):
            ef, ov = pctx.overlap_path(first, last, k=k, complements=compl, strict=strict)
            want_ef, want_ov = _cached(("ovl", seed, parts), lambda: orc.overlap_path(first, last, k, compl, parts=parts))
            assert np.array_equal(ef, want_ef) and np.array_equal(ov, want_ov), (seed, strict)


def test_poisoned_partial_presort(pctx):
    rng = np.random.default_rng(7)
    for k in (3, 31, 63, 127):
        kmers = rng.integers(0, 1 << 62, size=(5000, orc.limbs_for_k(k)), dtype=np.uint64)
        assert np.array_equal(pctx.partial_presort(kmers, k=k), orc.partial_presort(kmers, k))


def test_poisoned_compute_device(pctx):
    import torch
    seq, off, ln = messy_genome(5)
    want = _cached(("orc_dev",), lambda: orc.compute_from_fasta(seq, off, ln, 31, True))
    d = torch.from_numpy(seq).cuda()
    torch.cuda.synchronize()
    for tail_spec in (1, 0):
        _set(pctx, sig_min_items=0, tail_spec=tail_spec)
        res = pctx.compute_device(d.data_ptr(), d.numel(), k=31)
        assert (res.n_kmers, res.n_nodes) == (want["n_kmers"], want["n_nodes"])
        assert pctx.copy_to_host(res.ms_ptr, res.length) == want["ms"]


# ---- 3. a chunked host-to-device copy (8 MB and more) into a poisoned arena -------------------------------------------------------
def _chunked_input():
    return _cached("chunked", lambda: synth.frame_records(synth.random_genome_records(4, 2_200_000, 808)))


@pytest.mark.parametrize("poison", [0xFF, 0x41], ids=["ff", "A"])
def test_poisoned_chunked_copy(poison):
    seq, off, ln = _chunked_input()
    assert seq.size >= 8 << 20
    clean = kb.Context(0)
    try:
        want = clean.compute(seq, k=31)
    finally:
        clean.close()
    keys = _cached("chunked_keys", lambda: orc.count_kmers(seq, off, ln, 31, True)[0])
    c = kb.Context(0)
    try:
        c.set_option("arena_poison", poison)
        for tail_spec in (1, 0):
            c.set_option("tail_spec", tail_spec)
            got = c.compute(seq, k=31)
            assert got.ms == want.ms and got.n_kmers == want.n_kmers == len(keys)
        assert orc.verify_ms(got.ms, 31, True, keys)
    finally:
        c.close()


# ---- 4. groups of in-process ranks, every rank's arena poisoned -----------------------------------------------------------------
@pytest.mark.parametrize("n_ranks", [2, 3])
def test_poisoned_group(n_ranks):
    import torch
    n_dev = torch.cuda.device_count()
    seq, off, ln = _cached("group_in", lambda: synth.frame_records(synth.random_genome_records(3, 200_000, 909)))
    grp = kb.Group([r % n_dev for r in range(n_ranks)])
    try:
        grp.set_option("fast_heuristics", 0)
        grp.set_option("sig_min_items", 0)
        grp.set_option("fast_min_items", 0)
        for poison in (0x00, 0xFF, 0x41):
            grp.set_option("arena_poison", poison)
            for construction, k in (("sig", 31), ("fast", 31), ("fast", 21)):
                grp.set_option("sig_set", int(construction == "sig"))
                want = _cached(("group_orc", k), lambda: orc.compute_from_fasta(seq, off, ln, k, True))
                stat = f"{construction}_runs"
                r0 = grp.stat(stat)
                got = grp.compute(seq, k=k)
                assert got.ms == want["ms"] and got.n_kmers == want["n_kmers"], (poison, construction, k)
                assert [b - a for a, b in zip(r0, grp.stat(stat))] == [1] * n_ranks, (poison, construction, k)
    finally:
        grp.close()


# ---- 5. a long mixed call history on one context -------------------------------------------------------------------------------
ERR_ARG, ERR_EMPTY, ERR_BAD_SEQ = -2, -4, -5


def _schedule_inputs():
    def make():
        rng = np.random.default_rng(2024)
        pieces = []
        for i in range(6):
            n_rec = int(rng.integers(1, 6))
            recs = synth.random_genome_records(n_rec, int(rng.integers(2_000, 60_000)), 500 + i)
            if i % 2:
                recs.append(recs[0][: len(recs[0]) // 2].copy())       # repeated k-mers
            pieces.append(synth.frame_records(recs))
        return pieces
    return _cached("sched_inputs", make)


def _schedule(seed, n_calls=150):
    rng = np.random.default_rng(seed)
    kinds = ["compute", "compute", "compute", "compute_S", "lower_bound", "streaming", "maskopt", "count", "digest", "digest_masked",
             "overlap", "presort", "fail_empty", "fail_bad_seq", "fail_k0", "fail_z300", "overflow_sig", "overflow_fast"]
    calls = []
    for i in range(n_calls):
        kind = kinds[int(rng.integers(0, len(kinds)))]
        c = dict(kind=kind, piece=int(rng.integers(0, 6)), k=int(rng.choice([15, 21, 27, 31, 32, 45, 63, 64, 96, 127])),
                 compl=bool(rng.integers(0, 2)), z=int(rng.choice([1, 1, 2, 3])), maxone=bool(rng.integers(0, 2)),
                 poison=int(rng.choice(POISONS)) if i % 2 else -1)
        if kind.startswith("overflow_"):   # where the construction is tried: no -z, no -M (and k >= 26 for the signature buckets)
            c.update(z=1, maxone=False, k=int(rng.choice([31, 63, 127])) if kind == "overflow_sig" else c["k"])
        calls.append(c)
    return calls


_EXPECT = {}


def _expected(c, inp):
    seq, off, ln = inp
    kind, k, compl, z, maxone = c["kind"], c["k"], c["compl"], c["z"], c["maxone"]
    if kind in ("compute", "overflow_sig", "overflow_fast"):
        key = ("fasta", c["piece"], k, compl, z, maxone)
        make = lambda: orc.compute_from_fasta(seq, off, ln, k, compl, z, want_maxone=maxone)
    elif kind == "compute_S":
        key = ("S", c["piece"], k, compl, maxone)
        make = lambda: orc.compute_from_simplitigs(_records(inp), k, compl, maxone)
    elif kind == "lower_bound":
        key = ("lb", c["piece"], k, compl, z)
        make = lambda: orc.lower_bound_from_fasta(seq, off, ln, k, compl, z)
    elif kind == "streaming":
        key = ("stream", c["piece"], k, compl, z)
        make = lambda: orc.streaming(seq, off, ln, k, compl, z)
    elif kind in ("count", "digest", "digest_masked", "overlap", "presort"):
        key = ("count", c["piece"], k, compl)
        make = lambda: orc.count_kmers(seq, off, ln, k, compl)
    elif kind == "maskopt":
        key = ("maskopt", c["piece"], k, compl, maxone)
        make = lambda: orc.maskopt(_expected(dict(c, kind="compute", z=1, maxone=False), inp)["ms"], k, compl, maxone)
    else:
        return None
    if key not in _EXPECT:
        try:
            _EXPECT[key] = make()
        except ValueError:          # no k-mer is left after -z: the call must fail with KC_ERR_EMPTY
            _EXPECT[key] = ERR_EMPTY
    return _EXPECT[key]


def _run_call(ctx, c, inp):
    """One call of the schedule; asserts its result (or error code) against the oracle."""
    seq, off, ln = inp
    kind, k, compl, z, maxone = c["kind"], c["k"], c["compl"], c["z"], c["maxone"]
    want = _expected(c, inp)
    if isinstance(want, int) and want == ERR_EMPTY:
        with pytest.raises(kb.KcError) as e:
            if kind == "lower_bound":
                ctx.lower_bound(seq, k=k, complements=compl, min_frequency=z)
            else:
                ctx.compute(seq, k=k, complements=compl, min_frequency=z, want_maxone=maxone)
        assert e.value.code == ERR_EMPTY
    elif kind.startswith("fail_"):
        code = {"fail_empty": ERR_EMPTY, "fail_bad_seq": ERR_BAD_SEQ, "fail_k0": ERR_ARG, "fail_z300": ERR_ARG}[kind]
        with pytest.raises(kb.KcError) as e:
            if kind == "fail_empty":
                ctx.compute(np.frombuffer(b"ACGT\nNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNN\nAC\n", dtype=np.uint8), k=min(k, 31))
            elif kind == "fail_bad_seq":
                ctx.maskopt(b"ACGTacgt" * 20 + b"X" + b"ACGT" * 20, k=min(k, 31), complements=compl)
            elif kind == "fail_k0":
                ctx.compute(seq, k=0)
            else:
                ctx.compute(seq, k=k, min_frequency=300)
        assert e.value.code == code
    elif kind in ("compute", "overflow_sig", "overflow_fast"):
        if kind == "overflow_sig":
            _set(ctx, sig_min_items=0, sig_load_pct=400, fast_min_items=0)
        elif kind == "overflow_fast":
            _set(ctx, sig_set=0, fast_min_items=0, fast_sigmas=0)
        try:
            got = ctx.compute(seq, k=k, complements=compl, min_frequency=z, want_maxone=maxone)
        finally:
            _set(ctx, sig_set=1, sig_min_items=DEFAULTS["sig_min_items"], sig_load_pct=0, fast_min_items=DEFAULTS["fast_min_items"],
                 fast_sigmas=DEFAULTS["fast_sigmas"])
        assert got.ms == want["ms"] and got.n_kmers == want["n_kmers"]
        if maxone:
            assert got.maxone == want["maxone"]
    elif kind == "compute_S":
        s2, o2, l2 = orc.records_to_arrays(_records(inp))
        got = ctx.compute(s2, o2, l2, k=k, complements=compl, assume_simplitigs=True, want_maxone=maxone)
        assert got.ms == want[0] and got.maxone == want[1]
    elif kind == "lower_bound":
        assert ctx.lower_bound(seq, k=k, complements=compl, min_frequency=z)[0] == want
    elif kind == "streaming":
        assert ctx.streaming(seq, k=k, complements=compl, min_frequency=z).ms == want
    elif kind == "maskopt":
        ms = _expected(dict(c, kind="compute", z=1, maxone=False), inp)["ms"]
        assert ctx.maskopt(ms, k=k, complements=compl, minimize=maxone).ms == want
    elif kind == "count":
        keys, vals = want
        got_k, got_v = ctx.count_kmers(seq, k=k, complements=compl, min_frequency=z)
        keep = vals.astype(np.int64) + 1 >= z
        assert np.array_equal(got_k, keys[keep]) and np.array_equal(got_v, vals[keep])
    elif kind == "digest":
        assert ctx.kmer_digest(seq, k=k, complements=compl, min_frequency=z) == orc.kmer_digest(*want, z)
    elif kind == "digest_masked":
        ms = _expected(dict(c, kind="compute", z=1, maxone=False), inp)["ms"]
        assert ctx.kmer_digest(np.frombuffer(ms, dtype=np.uint8), k=k, complements=compl, masked=True) == orc.kmer_digest(*want)
    elif kind == "overlap":
        keys = want[0][:400]
        ef, ov = ctx.overlap_path(keys, keys, k=k, complements=compl, strict=maxone)
        want_ef, want_ov = orc.overlap_path(keys, keys, k, compl, parts=16 if maxone else 1)
        assert np.array_equal(ef, want_ef) and np.array_equal(ov, want_ov)
    elif kind == "presort":
        assert np.array_equal(ctx.partial_presort(want[0], k=k), orc.partial_presort(want[0], k))


@pytest.mark.parametrize("seed", [11, 12])
def test_mixed_call_history(seed):
    """About 150 calls over every entry point on one context: k across the three word widths, -u, -z, -S, -M, input sizes that move
    the arena offsets, the poison on for every other call, failing calls and forced overflows in between."""
    pieces = _schedule_inputs()
    c = kb.Context(0)
    try:
        c.set_option("fast_heuristics", 1)
        for i, call in enumerate(_schedule(seed)):
            c.set_option("arena_poison", call["poison"])
            try:
                _run_call(c, call, pieces[call["piece"]])
            except AssertionError as e:
                raise AssertionError(f"schedule seed {seed}, call {i}: {call}") from e
        assert c.stat("sig_fallbacks") > 0 and c.stat("fast_fallbacks") > 0
    finally:
        c.close()


# ---- 6. the retry after running out of arena ------------------------------------------------------------------------------------
# Stage a kernel class belongs to, in call order; a failed first attempt is found by the launches it added to the call's profile.
_STAGE_OF = {"extract": "set", "sort_hist": "set", "sort_scatter": "set", "sort_local": "set", "sort_misc": "set", "ks_hist0": "set",
             "ks_scatter0": "set", "ks_resolve": "set", "runs": "runs", "tuples": "engine", "simulate": "engine", "doubling": "engine",
             "commit": "engine", "small_engine": "engine", "rank": "emission", "emit": "emission", "maxone": "emission"}
_ORDER = ["set", "runs", "engine", "emission"]


def _profiled(c, call):
    c.profile_reset()
    c.profile_enable(True)
    try:
        r = call(c)
        prof = c.profile()
    finally:
        c.profile_enable(False)
    return r, {name: v["launches"] for name, v in prof.items()}


def _reached(base, prof):
    """The last stage that the failed first attempt launched kernels in (launches beyond those of an unfailed call)."""
    stages = [_STAGE_OF[n] for n in prof if n in _STAGE_OF and prof[n] > base[n]]
    return max(stages, key=_ORDER.index) if stages else "set"


# (id, input, k, -M, options, stages the first attempts must have run out of arena in)
RETRY_CASES = [
    ("spec", lambda: messy_genome(5), 31, False, dict(sig_min_items=0), {"set", "tail_spec"}),
    ("sig", lambda: messy_genome(5), 31, False, dict(sig_min_items=0, tail_spec=0), {"set", "runs", "engine"}),
    ("fast", reads, 31, False, dict(sig_set=0, fast_min_items=0), {"set"}),
    ("sparse_exact", lambda: sparse_input("tiny_sparse_k31"), 31, False, dict(sig_set=0, fast_set=0), {"set", "runs", "engine"}),
    ("maxone", spneumoniae, 31, True, dict(), {"set"}),
    ("maxone_sparse", lambda: sparse_input("tiny_sparse_k31"), 31, True, dict(), {"set"}),
    ("chunked", _chunked_input, 31, False, dict(tail_spec=0), {"set"}),
]
FRACTIONS = [0.05, 0.2, 0.4, 0.6, 0.8, 0.9, 0.97, 0.99, 0.999]


@pytest.mark.parametrize("case", RETRY_CASES, ids=[c[0] for c in RETRY_CASES])
def test_retry_after_arena_exhausted(case):
    """A fresh context whose first arena estimate is scaled below what the call needs: the call runs out of arena part way, is repeated
    once with the worst-case estimate, and gives the oracle's bytes; so does the next, ordinary call on that context."""
    name, inp, k, maxone, opts, stages = case
    seq, off, ln = inp()
    want = _cached(("orc", id(seq), k, True, 1, maxone, True), lambda: orc.compute_from_fasta(seq, off, ln, k, True, want_maxone=maxone))

    def compute(x):
        r = x.compute(seq, k=k, want_maxone=maxone)
        assert r.ms == want["ms"] and r.maxone == want["maxone"] and r.n_kmers == want["n_kmers"]
        return r

    def fresh():
        c = kb.Context(0)
        _set(c, **opts)
        c.set_option("arena_poison", 0xA5)
        return c

    c = fresh()
    try:
        _, base = _profiled(c, compute)
        assert c.stat("arena_retries") == 0
        cap, high = c.stat("arena_bytes"), c.stat("arena_high")
        spec = c.stat("tail_spec_runs") == 1
    finally:
        c.close()
    assert high < cap
    reached = set()
    # arena sizes below the call's high-water mark, down to one 4 KB page short of it (sizes are rounded up to pages)
    for target in [f * high for f in FRACTIONS] + [high - 8192]:
        ppm = max(1, int(target / cap * 1_000_000))
        c = fresh()
        try:
            c.set_option("arena_estimate_ppm", ppm)
            _, prof = _profiled(c, compute)
            assert c.stat("arena_retries") == 1, target
            stage = _reached(base, prof)
            reached.add("tail_spec" if spec and stage != "set" else stage)
            compute(c)                                                       # the next, ordinary call on the context
            assert c.stat("arena_retries") == 1
        finally:
            c.close()
    print(f"{name}: first attempts ran out of arena in {sorted(reached)}")
    assert stages <= reached
