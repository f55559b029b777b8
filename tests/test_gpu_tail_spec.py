"""The speculative tail of the from-FASTA path (kcgpu.cu run_tail_spec, option "tail_spec") against the ordinary tail.

With few first-occurrence runs the whole call after the signature construction is queued for a cap of runs and read back once; every
other input falls back to the ordinary tail on the same flags.  Either way the superstring must be byte-identical to the one of
tail_spec = 0 on the same context."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from kmercamel_b200 import synth  # noqa: E402

pytestmark = pytest.mark.gpu

SPEC_RUNS = 512  # KC_SPEC_RUNS (tail_spec.cuh)
DEFAULTS = dict(tail_spec=1, sig_set=1, sig_load_pct=0, sig_min_items=1 << 16, fast_set=1, fast_heuristics=1, sparse_switch=1)


@pytest.fixture(scope="module")
def sctx():
    import kmercamel_b200 as kb
    c = kb.Context(0)
    yield c
    c.close()


def _set(ctx, **kw):
    for name, value in kw.items():
        ctx.set_option(name, value)


@pytest.fixture
def tctx(sctx):
    _set(sctx, **DEFAULTS)
    sctx.set_option("fast_heuristics", 0)  # every call tries the speculation (no memory of an earlier failure)
    yield sctx
    _set(sctx, **DEFAULTS)


def _stats(ctx):
    return {n: ctx.stat(n) for n in ("tail_spec_runs", "tail_spec_fallbacks", "sig_runs", "sig_fallbacks")}


def _both(ctx, seq, expect, **kw):
    """compute with tail_spec = 1 (checking which path it took: "spec" or "fallback") and tail_spec = 0; returns both results."""
    ctx.set_option("tail_spec", 1)
    s0 = _stats(ctx)
    got = ctx.compute(seq, **kw)
    s1 = _stats(ctx)
    if expect == "spec":
        assert (s1["tail_spec_runs"], s1["tail_spec_fallbacks"]) == (s0["tail_spec_runs"] + 1, s0["tail_spec_fallbacks"])
    else:
        assert (s1["tail_spec_runs"], s1["tail_spec_fallbacks"]) == (s0["tail_spec_runs"], s0["tail_spec_fallbacks"] + 1)
    ctx.set_option("tail_spec", 0)
    want = ctx.compute(seq, **kw)
    assert _stats(ctx)["tail_spec_runs"] == s1["tail_spec_runs"]
    assert got.ms == want.ms
    for f in ("n_kmers", "n_nodes", "n_simplitigs", "length"):
        assert getattr(got, f) == getattr(want, f), f
    return got, want


def _messy_genome(seed, n_records=20, max_len=60_000):
    """Ragged records with lowercase stretches and N bytes (each N stretch ends a run)."""
    rng = np.random.default_rng(seed)
    recs = []
    for i in range(n_records):
        r = synth.random_genome_records(1, int(rng.integers(max_len // 3, max_len)), seed * 100 + i)[0].copy()
        a = int(rng.integers(0, len(r) - 2000))
        r[a:a + 1500] += 32  # lowercase
        if i % 3 == 0:
            b = int(rng.integers(0, len(r) - 20))
            r[b:b + int(rng.integers(1, 20))] = ord("N")
        recs.append(r)
    return synth.frame_records(recs)[0]


def _short_records(n, length, seed):
    """n random records of `length` bases: one first-occurrence run each."""
    return synth.frame_records(synth.random_genome_records(n, length, seed))[0]


@pytest.mark.parametrize("k", [26, 31, 32, 63, 127])
@pytest.mark.parametrize("compl", [True, False])
def test_spec_matches_ordinary_tail(tctx, k, compl):
    _set(tctx, sig_min_items=0)
    seq = _messy_genome(7 + k)
    _both(tctx, seq, "spec", k=k, complements=compl)


def test_spec_config1_200kbp(tctx):
    seq = synth.frame_records(synth.random_genome_records(50, 200_000, 12345))[0]
    got, _ = _both(tctx, seq, "spec", k=31)
    assert got.n_simplitigs == 50


def test_spec_run_cap(tctx):
    _set(tctx, sig_min_items=0)
    got, _ = _both(tctx, _short_records(SPEC_RUNS, 60, 5), "spec", k=31)
    assert got.n_simplitigs == SPEC_RUNS
    got, _ = _both(tctx, _short_records(SPEC_RUNS + 1, 60, 5), "fallback", k=31)
    assert got.n_simplitigs == SPEC_RUNS + 1


def test_spec_signature_overflow(tctx):
    _set(tctx, sig_min_items=0, sig_load_pct=400)  # every bucket overflows: fixed slots build the flags
    fb0 = tctx.stat("sig_fallbacks")
    _both(tctx, _messy_genome(3, 4), "fallback", k=31)
    assert tctx.stat("sig_fallbacks") == fb0 + 2  # once per arm


def test_spec_sparse_switch(tctx):
    _set(tctx, sig_min_items=0)
    seq = synth.frame_records(synth.short_records(200, 31, 34, 11))[0]
    got, _ = _both(tctx, seq, "fallback", k=31)
    assert got.n_nodes == got.n_kmers  # the k-mers themselves went to the greedy


def test_spec_empty_input(tctx):
    import kmercamel_b200 as kb
    _set(tctx, sig_min_items=0)
    seq = np.frombuffer(b"ACGTNACGTNACGTN" * 100 + b"\n", dtype=np.uint8).copy()
    with pytest.raises(kb.KcError) as e:
        tctx.compute(seq, k=31)
    assert "no k-mers" in str(e.value)


def test_spec_alternating(tctx):
    _set(tctx, sig_min_items=0)
    few, many = _messy_genome(21, 6), _short_records(3 * SPEC_RUNS, 60, 6)
    r1, _ = _both(tctx, few, "spec", k=31)
    _both(tctx, many, "fallback", k=31)
    r3, _ = _both(tctx, few, "spec", k=31)
    assert r1.ms == r3.ms
    # with the heuristics on, a failure is remembered for inputs of similar size, and a different size tries again
    tctx.set_option("fast_heuristics", 1)
    tctx.set_option("tail_spec", 1)
    tctx.compute(many, k=31)
    s0 = _stats(tctx)
    tctx.compute(many, k=31)
    s1 = _stats(tctx)
    assert (s1["tail_spec_runs"], s1["tail_spec_fallbacks"]) == (s0["tail_spec_runs"], s0["tail_spec_fallbacks"])
    tctx.compute(_messy_genome(22, 2, 20_000), k=31)
    assert tctx.stat("tail_spec_runs") == s1["tail_spec_runs"] + 1


def test_spec_one_read_back_config1(tctx):
    import torch
    seq = synth.frame_records(synth.random_genome_records(50, 1_000_000, 12345))[0]
    d = torch.from_numpy(seq).cuda()
    torch.cuda.synchronize()
    tctx.set_option("tail_spec", 1)
    tctx.compute_device(d.data_ptr(), d.numel(), k=31)
    r0, s0 = tctx.stat("read_backs"), tctx.stat("tail_spec_runs")
    res = tctx.compute_device(d.data_ptr(), d.numel(), k=31)
    assert tctx.stat("read_backs") == r0 + 1
    assert tctx.stat("tail_spec_runs") == s0 + 1
    assert res.n_launches <= 9, res.n_launches
    tctx.set_option("tail_spec", 0)
    want = tctx.compute_device(d.data_ptr(), d.numel(), k=31)
    assert tctx.stat("read_backs") > r0 + 2
    assert res.n_launches < want.n_launches
    assert (res.length, res.n_kmers, res.n_nodes) == (want.length, want.n_kmers, want.n_nodes)
