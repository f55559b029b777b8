"""Signature-bucket k-mer set construction (kmercamel_b200/csrc/kmerset_sig.cuh) against the exact construction and the oracle.

The first-occurrence flags are a pure function of the input (reference src/parser.h:22-141: which k-mers exist, and where each occurs
first), so every construction must yield byte-identical superstrings; the exact construction itself is pinned on the reference in
test_gpu.py / test_gpu_big.py."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from kmercamel_b200 import synth  # noqa: E402
from oracle import orc  # noqa: E402

pytestmark = pytest.mark.gpu


def _options(ctx, **kw):
    defaults = dict(sig_set=1, sig_load_pct=0, sig_min_items=1 << 16, fast_set=1, fast_heuristics=0)
    defaults.update(kw)
    for name, value in defaults.items():
        ctx.set_option(name, value)


def _restore(ctx):
    _options(ctx)
    ctx.set_option("fast_heuristics", 1)


def _mixed_input(seed):
    recs = synth.random_genome_records(6, 50_000, seed)
    recs.append(recs[0][1000:9000].copy())                                            # duplicates
    recs.append(np.frombuffer(b"ACGTNNNNNACGT" * 50, dtype=np.uint8).copy())          # N breaks
    recs.append(np.frombuffer(b"ACGTTGCATGCAGTCGATCGATTTGAC" * 40, dtype=np.uint8).copy())  # a short period: few k-mers, many times
    rc = recs[1][2000:30_000][::-1].copy()                                            # reverse complement of a stretch
    comp = np.zeros(256, dtype=np.uint8)
    for a, b in zip(b"ACGT", b"TGCA"):
        comp[a] = b
    recs.append(comp[rc])
    recs += list(synth.reads_from_genome(20000, 3.0, 150, 0.01, seed=seed + 1))
    return synth.frame_records(recs)


@pytest.mark.parametrize("k,compl", [(31, True), (31, False), (26, True), (27, False), (28, True), (29, True), (30, False), (32, True),
                                     (47, True), (63, False), (64, True), (95, False), (127, True)])
def test_sig_matches_exact(ctx, k, compl):
    seq, off, ln = _mixed_input(100 + k)
    try:
        _options(ctx, sig_set=0, fast_set=0)
        want = ctx.compute(seq, k=k, complements=compl)
        for load_pct in (0, 20):
            _options(ctx, sig_min_items=0, sig_load_pct=load_pct)
            runs0, fb0 = ctx.stat("sig_runs"), ctx.stat("sig_fallbacks")
            got = ctx.compute(seq, k=k, complements=compl)
            assert (ctx.stat("sig_runs"), ctx.stat("sig_fallbacks")) == (runs0 + 1, fb0), load_pct
            assert got.n_kmers == want.n_kmers and got.ms == want.ms, load_pct
    finally:
        _restore(ctx)
    want_k, _ = orc.count_kmers(seq, off, ln, k, compl)
    assert got.n_kmers == len(want_k) and orc.verify_ms(got.ms, k, compl, want_k)


def test_sig_small_k_takes_the_other_constructions(ctx):
    seq, off, ln = _mixed_input(7)
    try:
        _options(ctx, sig_min_items=0)
        for k in (11, 21, 25):
            runs0, fb0 = ctx.stat("sig_runs"), ctx.stat("sig_fallbacks")
            got = ctx.compute(seq, k=k)
            assert (ctx.stat("sig_runs"), ctx.stat("sig_fallbacks")) == (runs0, fb0)
            want_k, _ = orc.count_kmers(seq, off, ln, k, True)
            assert got.n_kmers == len(want_k)
    finally:
        _restore(ctx)


def test_sig_edge_inputs(ctx):
    """Ragged ends: inputs that stop inside a 32-base strip, records shorter than k, one k-mer, windows at the very start."""
    rng = np.random.default_rng(5)
    base = rng.integers(0, 4, 3000)
    text = np.frombuffer(b"ACGT", dtype=np.uint8)[base]
    try:
        for n in (31, 32, 33, 63, 64, 65, 95, 1000, 1023, 1025, 2999):
            for k in (31, 63, 127):
                if n < k:
                    continue
                s = np.concatenate([text[:n], np.frombuffer(b"\n", dtype=np.uint8)])
                _options(ctx, sig_set=0, fast_set=0)
                want = ctx.compute(s, k=k)
                _options(ctx, sig_min_items=0)
                runs0 = ctx.stat("sig_runs")
                got = ctx.compute(s, k=k)
                assert ctx.stat("sig_runs") == runs0 + 1
                assert got.ms == want.ms and got.n_kmers == want.n_kmers, (n, k)
        # many short records, some shorter than k
        recs = [text[i * 40:i * 40 + 20 + (i * 7) % 45] for i in range(60)]
        seq, off, ln = synth.frame_records(recs)
        _options(ctx, sig_set=0, fast_set=0)
        want = ctx.compute(seq, k=31)
        _options(ctx, sig_min_items=0)
        got = ctx.compute(seq, k=31)
        assert got.ms == want.ms and got.n_kmers == want.n_kmers
    finally:
        _restore(ctx)


def test_sig_overflow_falls_back(ctx):
    recs = synth.random_genome_records(4, 60_000, 99)
    seq, off, ln = synth.frame_records(recs)
    try:
        _options(ctx, sig_set=0, fast_set=0)
        want = ctx.compute(seq, k=31)
        _options(ctx, sig_min_items=0, sig_load_pct=400)        # four times the capacity on average: every bucket overflows
        fb0 = ctx.stat("sig_fallbacks")
        got = ctx.compute(seq, k=31)
        assert ctx.stat("sig_fallbacks") == fb0 + 1
        assert got.ms == want.ms and got.n_kmers == want.n_kmers
        # one k-mer repeated far beyond any bucket
        s2 = np.frombuffer(b"A" * 300_000 + b"\n" + bytes(recs[0]) + b"\n", dtype=np.uint8)
        _options(ctx, sig_set=0, fast_set=0)
        want = ctx.compute(s2, k=31)
        _options(ctx)
        fb0 = ctx.stat("sig_fallbacks")
        got = ctx.compute(s2, k=31)
        assert ctx.stat("sig_fallbacks") == fb0 + 1
        assert got.ms == want.ms and got.n_kmers == want.n_kmers
        # remembered (fast_heuristics): the next call on a similar input does not try again
        ctx.set_option("fast_heuristics", 1)
        got = ctx.compute(s2, k=31)
        fb1 = ctx.stat("sig_fallbacks")
        got2 = ctx.compute(s2, k=31)
        assert ctx.stat("sig_fallbacks") == fb1 and got2.ms == got.ms == want.ms
    finally:
        _restore(ctx)


@pytest.mark.parametrize("call", ["digest", "streaming"])
def test_sig_overflow_memory_is_compute_only(ctx, call):
    """Only compute remembers a signature overflow: a digest or streaming call that overflows leaves the next compute on the same
    input trying the buckets, and a remembered compute overflow does not stop the next digest or streaming call from trying them."""
    recs = synth.random_genome_records(4, 60_000, 99)
    seq, off, ln = synth.frame_records(recs)
    other = {"digest": lambda: ctx.kmer_digest(seq, k=31), "streaming": lambda: ctx.streaming(seq, k=31)}[call]
    try:
        _options(ctx, sig_min_items=0, sig_load_pct=400, fast_heuristics=1)  # every bucket overflows; the memories start clear
        want = ctx.compute(seq, k=31)
        ctx.set_option("fast_heuristics", 1)
        fb0 = ctx.stat("sig_fallbacks")
        other()
        assert ctx.stat("sig_fallbacks") == fb0 + 1
        got = ctx.compute(seq, k=31)                 # tries the buckets: the overflow above was not remembered
        assert ctx.stat("sig_fallbacks") == fb0 + 2 and got.ms == want.ms
        got = ctx.compute(seq, k=31)                 # this overflow was: the buckets are skipped
        assert ctx.stat("sig_fallbacks") == fb0 + 2 and got.ms == want.ms
        other()                                      # ... but not by a digest or streaming call
        assert ctx.stat("sig_fallbacks") == fb0 + 3
        got = ctx.compute(seq, k=31)                 # which leaves the memory of compute as it was
        assert ctx.stat("sig_fallbacks") == fb0 + 3 and got.ms == want.ms
    finally:
        _restore(ctx)


@pytest.mark.parametrize("coverage", [2.0, 30.0])
def test_sig_reads_with_coverage(ctx, coverage):
    """Reads: every run of windows comes `coverage` times, so the bucket sizes spread by sqrt(coverage): 2x still fits, 30x overflows
    and falls back.  Either way the result is the exact one."""
    reads = synth.reads_from_genome(200_000, coverage, 150, 0.01, seed=11)
    seq, off, ln = synth.frame_records(list(reads))
    try:
        _options(ctx, sig_set=0, fast_set=0)
        want = ctx.compute(seq, k=31)
        _options(ctx)
        runs0, fb0 = ctx.stat("sig_runs"), ctx.stat("sig_fallbacks")
        got = ctx.compute(seq, k=31)
        assert (ctx.stat("sig_runs") - runs0, ctx.stat("sig_fallbacks") - fb0) == ((1, 0) if coverage < 3 else (0, 1))
        assert got.ms == want.ms and got.n_kmers == want.n_kmers
    finally:
        _restore(ctx)


def test_sig_config2_full_size(ctx):
    """configs[1] at full size through the path bench.py times: signature buckets, exact set."""
    recs = synth.random_genome_records(50, 1_000_000, 12345)
    seq, off, ln = synth.frame_records(recs)
    runs0, fb0 = ctx.stat("sig_runs"), ctx.stat("sig_fallbacks")
    r = ctx.compute(seq, k=31)
    assert (ctx.stat("sig_runs"), ctx.stat("sig_fallbacks")) == (runs0 + 1, fb0)
    assert r.n_kmers == 49_998_500 and abs(r.length - 49_999_860) <= 0.001 * 49_999_860
    got, n_on = orc.ms_kmers(r.ms, 31, True)
    keys, _ = ctx.count_kmers(seq, k=31)
    assert n_on == r.n_kmers and np.array_equal(got, keys)


@pytest.mark.parametrize("k", [63, 127])
def test_sig_wide_words_5mbp(ctx, k):
    recs = synth.random_genome_records(5, 1_000_000, 31337 + k)
    seq, off, ln = synth.frame_records(recs)
    try:
        _options(ctx, sig_set=0)
        want = ctx.compute(seq, k=k, complements=False)
        _options(ctx)
        runs0, fb0 = ctx.stat("sig_runs"), ctx.stat("sig_fallbacks")
        got = ctx.compute(seq, k=k, complements=False)
        assert (ctx.stat("sig_runs"), ctx.stat("sig_fallbacks")) == (runs0 + 1, fb0)
        assert got.ms == want.ms and got.n_kmers == want.n_kmers == 5 * (1_000_000 - k + 1)
    finally:
        _restore(ctx)
