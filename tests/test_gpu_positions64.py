"""Inputs of 2^32 bytes and more on one GPU (64-bit window positions in the signature construction, kmerset_sig.cuh).

The inputs are generated on the device with torch (seeded), so that nothing of 4 GB goes through numpy on the way in.  Every
test has a context of its own, closed when it ends, so that an arena of these sizes is not kept by the session context or by the
next test.  Every test skips, with the reason, when the GPU (shared) or the disk has too little free space."""
import os
import shutil
import subprocess

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

import kmercamel_b200 as kb  # noqa: E402

MBP = 1_000_000
PART = 8 * MBP               # A and B of the positions test
EXE = os.path.join(ROOT, "host", "kmercamel")


def _need_gpu_gb(gb):
    free, _ = torch.cuda.mem_get_info()
    if free < gb * 1e9:
        pytest.skip(f"needs {gb} GB of free device memory, {free / 1e9:.1f} GB free")


def _acgt(n, gen):
    lut = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device="cuda")
    return lut[torch.randint(0, 4, (n,), dtype=torch.uint8, device="cuda", generator=gen).long()]


def _revcomp(x):
    comp = torch.zeros(256, dtype=torch.uint8, device="cuda")
    for a, b in zip(b"ACGT", b"TGCA"):
        comp[a] = b
    return comp[x.flip(0).long()]


def _byte(c):
    return torch.tensor([ord(c)], dtype=torch.uint8, device="cuda")


@pytest.fixture
def lctx():
    c = kb.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def inputs():
    """big   = A + N-run + B + N + A + N + rc(B[:half]) + newline, B starting 4 Mbp before byte 2^32 (windows of B straddle it);
    small = A + NNNN + B + N + rc(B[:half]) + newline.
    The copy of A adds no k-mer, and the N separators keep windows from spanning the junctions, so the first occurrences of the
    big input are those of the small one, in the same order: the superstrings must be byte-identical (with -u too, where the
    reverse complement adds k-mers to both)."""
    _need_gpu_gb(50)
    g = torch.Generator(device="cuda")
    g.manual_seed(20261020)
    a, b = _acgt(PART, g), _acgt(PART, g)
    rcb = _revcomp(b[: PART // 2])
    gap = 2**32 - 4 * MBP - PART
    n, nl = _byte("N"), _byte("\n")
    small = torch.cat([a, n.repeat(4), b, n, rcb, nl])
    big = torch.empty(PART + gap + PART + 1 + PART + 1 + PART // 2 + 1, dtype=torch.uint8, device="cuda")
    o = 0
    for part in (a, None, b, n, a, n, rcb, nl):
        if part is None:
            big[o:o + gap].fill_(ord("N"))
            o += gap
        else:
            big[o:o + part.numel()] = part
            o += part.numel()
    assert o == big.numel() and big.numel() >= 2**32 and PART + gap == 2**32 - 4 * MBP
    torch.cuda.synchronize()
    yield big, small
    del big, small
    torch.cuda.empty_cache()


def _compute(ctx, seq, **kw):
    r = ctx.compute_device(seq.data_ptr(), seq.numel(), **kw)
    return r, ctx.copy_to_host(r.ms_ptr, r.length)


@pytest.mark.parametrize("k", [31, 63, 127])
@pytest.mark.parametrize("compl", [True, False])
def test_positions_past_2_32_match_the_small_input(lctx, inputs, k, compl):
    big, small = inputs
    want, want_ms = _compute(lctx, small, k=k, complements=compl)
    runs0 = lctx.stat("sig_runs")
    got, got_ms = _compute(lctx, big, k=k, complements=compl)
    assert lctx.stat("sig_runs") == runs0 + 1
    assert got.n_kmers == want.n_kmers and got.length == want.length
    assert got_ms == want_ms
    assert got.n_occurrences > want.n_occurrences  # the copies were seen
    if k == 63 and not compl:  # host buffers: kc_compute copies the input in chunks
        r = lctx.compute(big.cpu().numpy(), k=k, complements=compl, want_maxone=False)
        assert r.ms == want_ms and r.n_kmers == want.n_kmers


@pytest.mark.parametrize("what", ["min_frequency", "want_maxone", "k21", "sig_set", "overflow"])
def test_refusals_above_2_32(lctx, inputs, what):
    """Inputs of 2^32 bytes or more have the signature construction alone: without it, or when a bucket overflows, the call fails
    with KC_ERR_TOO_LARGE and says why; the small input still takes the other constructions."""
    big, small = inputs
    kw = dict(k=31)
    opts = {}
    reason = {"min_frequency": "-z", "want_maxone": "-M", "k21": "k is below 26", "sig_set": "sig_set = 0", "overflow": "overflowed"}[what]
    if what == "min_frequency":
        kw["min_frequency"] = 2
    elif what == "want_maxone":
        kw["want_maxone"] = True
    elif what == "k21":
        kw["k"] = 21
    elif what == "sig_set":
        opts["sig_set"] = 0
    else:
        # Repeat-rich: a 2 kbp stretch 300 times (inside the N run of the big input) puts ~300 records into each of its buckets.
        # (Forcing the option sig_load_pct does not do it here: the buckets are planned from the input size, which is mostly N.)
        n = _byte("N")
        rep = torch.cat([small[:2000], n]).repeat(300)
        big = big.clone()
        big[PART + 16:PART + 16 + rep.numel()] = rep
        small = torch.cat([small[:-1], n, rep, small[-1:]])
    try:
        for name, v in opts.items():
            lctx.set_option(name, v)
        with pytest.raises(kb.KcError) as e:
            lctx.compute_device(big.data_ptr(), big.numel(), **kw)
        assert e.value.code == -6
        msg = str(e.value)
        assert "2^32 bytes or more" in msg and reason in msg, msg
        r = lctx.compute_device(small.data_ptr(), small.numel(), **kw)  # the 32-bit constructions still take the small input
        assert r.n_kmers > 0
    finally:
        lctx.set_option("sig_set", 1)
        lctx.set_option("sig_load_pct", 0)


def test_cli_above_2_32(lctx, inputs, tmp_path):
    """`compute -g 0,0` runs such an input on one GPU (with the note) and writes the library's superstring; -V refuses it."""
    big, small = inputs
    if shutil.disk_usage(tmp_path).free < 10e9:
        pytest.skip("needs 10 GB of free disk for a 4.3 GB FASTA")
    _need_gpu_gb(45)
    if not os.path.exists(EXE):
        subprocess.check_call(["make", "-C", ROOT, "host/kmercamel"], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    _, want_ms = _compute(lctx, small, k=31)
    fa = tmp_path / "big.fa"
    with open(fa, "wb") as f:
        f.write(b">big\n")
        f.write(memoryview(big.cpu().numpy()))
    p = subprocess.run([EXE, "compute", "-k", "31", "-g", "0,0", str(fa)], capture_output=True)
    err = p.stderr.decode()
    assert p.returncode == 0, err
    assert "run on one GPU" in err
    assert p.stdout.split(b"\n")[1] == want_ms
    p = subprocess.run([EXE, "compute", "-k", "31", "-V", str(fa)], capture_output=True)
    err = p.stderr.decode()
    assert p.returncode != 0
    assert "verification not available for inputs of 2^32 bytes or more" in err and "Verification FAILED" not in err
    fa.unlink()


def _add(d, e):
    m = (1 << 64) - 1
    return [(d[0] + e[0]) & m, (d[1] + e[1]) & m, d[2] ^ e[2], (d[3] + e[3]) & m]


def test_4_4_gbases_genome_by_additive_digests(lctx):
    """k = 63, 44 x 100 Mbp uniform random records: no duplicate k-mer (with overwhelming probability).  kc_kmer_digest adds over
    disjoint k-mer sets (n, sum, sum * c mod 2^64; xor), so the input digested record by record must equal the superstring
    digested in pieces [iP, (i + 1) P + k - 1) with masked = 1: in a min-one superstring every k-mer is ON exactly once."""
    _need_gpu_gb(60)
    k, n_rec, rec_len = 63, 44, 100 * MBP
    g = torch.Generator(device="cuda")
    g.manual_seed(44)
    seq = torch.empty(n_rec * (rec_len + 1), dtype=torch.uint8, device="cuda")
    for i in range(n_rec):
        o = i * (rec_len + 1)
        seq[o:o + rec_len] = _acgt(rec_len, g)
        seq[o + rec_len] = ord("\n")
    assert seq.numel() >= 2**32
    r, ms = _compute(lctx, seq, k=k)
    host = seq.cpu().numpy()
    del seq
    torch.cuda.empty_cache()
    n_kmers = n_rec * (rec_len - k + 1)
    assert r.n_kmers == n_kmers
    a = np.frombuffer(ms, dtype=np.uint8)
    assert r.length == len(ms) and int(np.count_nonzero(a < ord("a"))) == n_kmers
    assert all(c >= ord("a") for c in ms[-(k - 1):])
    d_in = [0, 0, 0, 0]
    for i in range(n_rec):
        o = i * (rec_len + 1)
        d_in = _add(d_in, lctx.kmer_digest(host[o:o + rec_len + 1], k=k))
    d_out = [0, 0, 0, 0]
    piece = 1 << 28
    for s in range(0, len(ms), piece):
        d_out = _add(d_out, lctx.kmer_digest(a[s:min(len(ms), s + piece + k - 1)], k=k, masked=True))
    assert d_in[0] == n_kmers
    assert d_out == d_in
