"""The one-GPU from-FASTA call of a genome replayed as a cached CUDA graph (kcgpu.cu run_sig_spec).

The first call of a shape captures the signature construction and the speculative tail; later calls of the same shape replay the graph
with their own input pointer.  Every result must be byte-identical to the direct launches of a fresh context (kernel-class timers on:
no graph), whatever buffer the input sits in, whatever the arena held before, and whichever tail the status block chooses."""
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from kmercamel_b200 import synth  # noqa: E402

pytestmark = pytest.mark.gpu


def _genome(n, length, seed):
    return synth.frame_records(synth.random_genome_records(n, length, seed))[0]


def _with_runs(seq, every):
    """The same bytes with an N every `every` bases: one first-occurrence run per stretch, far more than the speculative tail's cap."""
    s = seq.copy()
    s[every::every] = ord("N")
    return s


def _direct(seq, k, **options):
    """kc_compute_device of a fresh context with the kernel-class timers on, which launch directly."""
    import torch
    import kmercamel_b200 as kb
    c = kb.Context(0)
    try:
        for name, value in options.items():
            c.set_option(name, value)
        c.profile_enable(True)
        d = torch.from_numpy(seq).cuda()
        r = c.compute_device(d.data_ptr(), d.numel(), k=k)
        assert c.stat("spec_graph_captures") == 0
        return c.copy_to_host(r.ms_ptr, r.length), r.n_kmers, r.n_nodes
    finally:
        c.close()


def _run(ctx, d, k):
    r = ctx.compute_device(d.data_ptr(), d.numel(), k=k)
    return ctx.copy_to_host(r.ms_ptr, r.length), r.n_kmers, r.n_nodes


@pytest.fixture(params=["private", "legacy"])
def gctx(request):
    """A context on its own stream, and one on the legacy default stream (torch's, as bench.py passes it), which cannot be captured."""
    import kmercamel_b200 as kb
    c = kb.Context(0) if request.param == "private" else kb.Context(0, 0)
    yield c
    c.close()


def _graph_counts(ctx):
    return ctx.stat("spec_graph_captures"), ctx.stat("spec_graph_replays")


def test_replay_rotating_inputs_then_other_shapes(gctx):
    import torch
    seqs = [_genome(4, 120_000, 500 + i) for i in range(4)]
    assert len({s.size for s in seqs}) == 1
    want = [_direct(s, 31) for s in seqs]
    bufs = [torch.from_numpy(s).cuda() for s in seqs]
    for step in range(10):  # capture once, then replay with every buffer in turn
        i = step % 4
        assert _run(gctx, bufs[i], 31) == want[i], step
    assert _graph_counts(gctx) == (1, 9)
    assert gctx.stat("tail_spec_runs") == 10
    # a different size and a different k: new shapes, each captured (a larger arena for k = 47 also drops the cached graphs)
    other = _genome(3, 90_000, 77)
    d_other = torch.from_numpy(other).cuda()
    assert _run(gctx, d_other, 31) == _direct(other, 31)
    assert _run(gctx, bufs[1], 47) == _direct(seqs[1], 47)
    assert _graph_counts(gctx)[0] == 3
    assert _run(gctx, bufs[2], 31) == want[2]
    assert _run(gctx, bufs[3], 31) == want[3]
    assert sum(_graph_counts(gctx)) == 14


def test_timers_launch_directly(gctx):
    import torch
    seqs = [_genome(4, 100_000, 600 + i) for i in range(2)]
    bufs = [torch.from_numpy(s).cuda() for s in seqs]
    want = [_direct(s, 31) for s in seqs]
    assert _run(gctx, bufs[0], 31) == want[0]
    gctx.profile_enable(True)
    gctx.profile_reset()
    for step in range(4):
        assert _run(gctx, bufs[step % 2], 31) == want[step % 2]
    assert _graph_counts(gctx) == (1, 0)
    assert gctx.profile()["ks_resolve"]["launches"] == 4
    gctx.profile_enable(False)
    assert _run(gctx, bufs[1], 31) == want[1]
    assert _graph_counts(gctx) == (1, 1)


def test_too_many_runs_after_a_cached_call(gctx):
    import torch
    seq = _genome(4, 100_000, 700)
    many = _with_runs(_genome(4, 100_000, 701), 200)
    assert many.size == seq.size
    d, dm = torch.from_numpy(seq).cuda(), torch.from_numpy(many).cuda()
    want, want_many = _direct(seq, 31), _direct(many, 31)
    assert _run(gctx, d, 31) == want
    fb = gctx.stat("tail_spec_fallbacks")
    assert _run(gctx, dm, 31) == want_many  # the replayed graph says "too many runs": the ordinary tail runs on its flags
    assert gctx.stat("tail_spec_fallbacks") == fb + 1
    assert _graph_counts(gctx) == (1, 1)
    gctx.set_option("fast_heuristics", 0)  # no memory of the failure: the next call of the size speculates again
    assert _run(gctx, d, 31) == want
    assert _run(gctx, dm, 31) == want_many
    assert _run(gctx, d, 31) == want


def test_signature_overflow_from_a_replayed_graph(gctx):
    import torch
    opts = dict(fast_heuristics=0, sig_load_pct=400)  # every bucket overflows: the fixed slots build the flags
    for name, value in opts.items():
        gctx.set_option(name, value)
    seqs = [_genome(3, 80_000, 800 + i) for i in range(2)]
    bufs = [torch.from_numpy(s).cuda() for s in seqs]
    want = [_direct(s, 31, **opts) for s in seqs]
    fb = gctx.stat("sig_fallbacks")
    for step in range(4):
        assert _run(gctx, bufs[step % 2], 31) == want[step % 2]
    assert gctx.stat("sig_fallbacks") == fb + 4
    assert _graph_counts(gctx) == (1, 3)


@pytest.mark.parametrize("poison", [0x00, 0xFF, 0x41], ids=["00", "ff", "A"])
def test_poisoned_arena_between_replays(gctx, poison):
    import torch
    seqs = [_genome(4, 100_000, 900 + i) for i in range(3)]
    bufs = [torch.from_numpy(s).cuda() for s in seqs]
    want = [_direct(s, 31) for s in seqs]
    gctx.set_option("arena_poison", poison)  # every block the captured calls allocate is filled again on every replay
    for step in range(6):
        assert _run(gctx, bufs[step % 3], 31) == want[step % 3], step
    assert _graph_counts(gctx) == (1, 5)
