"""Inputs of 2^32 bytes or more on a multi-GPU group: the signature construction across the ranks with 64-bit window positions.

The big / small inputs are those of test_gpu_positions64.py: windows straddle byte 2^32, and the copies past it fold into the
first occurrences, so the group's superstring of the big input must be byte-identical to one GPU's superstring of the small one.
The ranks share the visible devices (rank r on device r % count); ranks that share a device need their arenas once each, so every
test states the device memory it needs and skips below it."""
import json
import os
import shutil
import socket
import subprocess
import sys

import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

import kmercamel_b200 as kb  # noqa: E402
from test_gpu_positions64 import EXE, _byte, _compute, _need_gpu_gb, inputs, lctx, PART  # noqa: E402,F401

KC_ERR_TOO_LARGE = -6


def _devices(n_ranks):
    n = torch.cuda.device_count()
    return [r % n for r in range(n_ranks)]


def _need_for_ranks(n_ranks, k, extra_gb=5):
    """Device memory the fullest device needs: per rank a heap of ~2.2-2.6 x the input (sequence, code words, flags, record
    streams) and an arena of the overlap stage and emission of one GPU (group_arena_need), ~45 / 52 / 60 GB at k = 31 / 63 / 127."""
    per_rank = 11 + {31: 45, 63: 52, 127: 60}[k]
    ranks_on_one = -(-n_ranks // torch.cuda.device_count())
    _need_gpu_gb(ranks_on_one * per_rank + extra_gb)


def _group_compute(grp, seq, **kw):
    """Group.compute, with the library's own refusal of arenas the devices cannot hold together turned into a skip."""
    try:
        return grp.compute(seq, **kw)
    except kb.KcError as e:
        if "cannot hold every rank's arena" in str(e):
            pytest.skip(f"the ranks' arenas do not fit their devices together: {e}")
        raise


@pytest.fixture(scope="module")
def host_inputs(inputs):
    big, small = inputs
    return big.cpu().numpy(), small


@pytest.fixture(scope="module")
def group2():
    _need_for_ranks(2, 127)  # before the group holds any of it: the widest word the tests below ask for
    g = kb.Group(_devices(2))
    yield g
    g.close()


def _poison(grp, value):
    grp.set_option("arena_poison", value)


def _check_group(grp, lctx, big_host, small, k, compl):
    want, want_ms = _compute(lctx, small, k=k, complements=compl)
    runs0, fb0 = grp.stat("sig_runs"), grp.stat("sig_fallbacks")
    got = _group_compute(grp, big_host, k=k, complements=compl)
    assert got.n_kmers == want.n_kmers and got.length == want.length
    assert got.ms == want_ms
    assert grp.stat("sig_runs") == [r + 1 for r in runs0]
    assert grp.stat("sig_fallbacks") == fb0


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


@pytest.mark.parametrize("poison", [-1, 0xA5], ids=["plain", "poisoned"])
def test_torchrun_processes_past_2_32(tmp_path, poison):
    """Two processes, IPC heaps allocated for a cap above 2^32, each with its own copy of the big input: the concatenated slices
    equal one GPU's superstring of the small input."""
    _need_for_ranks(2, 31, extra_gb=20)
    out = tmp_path / "verdict.json"
    env = dict(os.environ, PYTHONPATH=ROOT, KC_TEST_POISON=str(poison))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nproc_per_node=2", "--nnodes=1", f"--master_port={_free_port()}",
           os.path.join(ROOT, "tests", "sharded_worker64.py"), str(out)]
    p = subprocess.run(cmd, env=env, capture_output=True, timeout=1800)
    assert p.returncode == 0, p.stderr.decode()[-4000:]
    v = json.load(open(out))
    assert v["identical"], v


@pytest.mark.parametrize("poison", [-1, 0xA5], ids=["plain", "poisoned"])
def test_three_ranks_past_2_32(lctx, host_inputs, poison):
    _need_for_ranks(3, 31)
    big_host, small = host_inputs
    g = kb.Group(_devices(3))
    try:
        _poison(g, poison)
        _check_group(g, lctx, big_host, small, 31, True)
    finally:
        g.close()


@pytest.mark.parametrize("poison", [-1, 0xA5], ids=["plain", "poisoned"])
@pytest.mark.parametrize("compl", [True, False])
@pytest.mark.parametrize("k", [127, 63, 31])
def test_group_past_2_32_matches_one_gpu(lctx, host_inputs, group2, k, compl, poison):
    """Two ranks; with arena_poison every arena allocation is filled with a byte pattern first: the result must not change."""
    big_host, small = host_inputs
    try:
        _poison(group2, poison)
        _check_group(group2, lctx, big_host, small, k, compl)
    finally:
        _poison(group2, -1)


@pytest.mark.parametrize("what", ["min_frequency", "k21", "sig_set", "overflow"])
def test_group_refusals_past_2_32(lctx, inputs, group2, what):
    """The refusals of one GPU, on the group: KC_ERR_TOO_LARGE with the reason, and the same group then computes the small input."""
    big, small = inputs
    kw = dict(k=31)
    reason = {"min_frequency": "-z", "k21": "k is below 26", "sig_set": "sig_set = 0", "overflow": "overflowed"}[what]
    if what == "min_frequency":
        kw["min_frequency"] = 2
    elif what == "k21":
        kw["k"] = 21
    elif what == "overflow":  # repeat-rich: ~300 records in each bucket of a 2 kbp stretch (test_refusals_above_2_32)
        n = _byte("N")
        rep = torch.cat([small[:2000], n]).repeat(300)
        big = big.clone()
        big[PART + 16:PART + 16 + rep.numel()] = rep
        small = torch.cat([small[:-1], n, rep, small[-1:]])
    big_host = big.cpu().numpy()
    small_host = small.cpu().numpy()
    fb0 = group2.stat("sig_fallbacks")
    try:
        if what == "sig_set":
            group2.set_option("sig_set", 0)
        with pytest.raises(kb.KcError) as e:
            group2.compute(big_host, **kw)
        assert e.value.code == KC_ERR_TOO_LARGE
        msg = str(e.value)
        assert "2^32 bytes or more" in msg and reason in msg, msg
        if what == "overflow":
            assert group2.stat("sig_fallbacks") == [f + 1 for f in fb0]
    finally:
        group2.set_option("sig_set", 1)
    want = lctx.compute(small_host, **kw)
    got = group2.compute(small_host, **kw)
    assert got.ms == want.ms and got.n_kmers == want.n_kmers


def test_cli_group_past_2_32(lctx, inputs, group2, tmp_path):
    """`compute -g 0,1` with two distinct GPUs runs such an input on the group (no one-GPU note) and writes the one-GPU superstring."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two visible devices for -g 0,1 (with one device the CLI runs such an input on one GPU)")
    if shutil.disk_usage(tmp_path).free < 10e9:
        pytest.skip("needs 10 GB of free disk for a 4.3 GB FASTA")
    group2.close()  # its arenas: the CLI builds a group of its own
    _need_gpu_gb(80)
    big, small = inputs
    if not os.path.exists(EXE):
        subprocess.check_call(["make", "-C", ROOT, "host/kmercamel"], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    _, want_ms = _compute(lctx, small, k=31)
    fa = tmp_path / "big.fa"
    with open(fa, "wb") as f:
        f.write(b">big\n")
        f.write(memoryview(big.cpu().numpy()))
    p = subprocess.run([EXE, "compute", "-k", "31", "-g", "0,1", str(fa)], capture_output=True)
    err = p.stderr.decode()
    assert p.returncode == 0, err
    assert "run on one GPU" not in err
    assert p.stdout.split(b"\n")[1] == want_ms
    fa.unlink()
