"""The neighbours of `compute` through the signature construction: kc_kmer_digest, kc_lower_bound and kc_streaming (and the CLI's
`lowerbound`, `compute -a streaming` and `verify`), below 2^32 bytes against the sorted-keys / fixed-slot / exact constructions
(option sig_set = 0), and on inputs of 2^32 bytes and more against small equivalents.

The large inputs are generated on the device with torch (seeded).  Every large test has a context of its own, closed when it ends, and
skips, with the reason, when the GPU (shared) or the disk has too little free space."""
import gzip
import os
import shutil
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN_DIR, ROOT

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

import kmercamel_b200 as kb  # noqa: E402
from kmercamel_b200 import synth  # noqa: E402

MBP = 1_000_000
PART = 8 * MBP
EXE = os.path.join(ROOT, "host", "kmercamel")
DEFAULTS = dict(sig_set=1, sig_load_pct=0, sig_min_items=1 << 16, fast_set=1, fast_heuristics=1)
_COMP = bytes.maketrans(b"ACGTacgt", b"TGCAtgca")


# ---- small inputs: the signature route against the others -------------------------------------------------------------------

@pytest.fixture(scope="module")
def sctx():
    c = kb.Context(0)
    yield c
    c.close()


@pytest.fixture
def nctx(sctx):
    """The module context with the defaults, sig_min_items = 0 (small inputs take the signature construction)."""
    for name, v in DEFAULTS.items():
        sctx.set_option(name, v)
    sctx.set_option("sig_min_items", 0)
    yield sctx
    for name, v in DEFAULTS.items():
        sctx.set_option(name, v)


@pytest.fixture(scope="module")
def genome():
    """Seeded human-like records (repeats, N runs) with lower-case stretches and ragged lengths, framed."""
    recs = synth.human_like_genome(600_000, seed=77, n_runs=6)
    rng = np.random.default_rng(77)
    out = []
    for i, r in enumerate(recs):
        r = r.copy()
        if i % 3 == 0 and len(r) > 2000:  # soft-masked stretch
            a = int(rng.integers(0, len(r) - 1000))
            r[a:a + int(rng.integers(100, 1000))] |= 0x20
        out.append(r[: len(r) - int(rng.integers(0, 97))])
    out.append(np.frombuffer(b"ACGTNacgt", dtype=np.uint8).copy())  # shorter than every k
    seq, _, _ = synth.frame_records(out)
    return seq


def _digest(ctx, seq, sig, **kw):
    ctx.set_option("sig_set", sig)
    runs, fb = ctx.stat("sig_runs"), ctx.stat("sig_fallbacks")
    d = ctx.kmer_digest(seq, **kw)
    return d, ctx.stat("sig_runs") - runs, ctx.stat("sig_fallbacks") - fb


@pytest.mark.parametrize("k", [26, 29, 31, 32, 47, 63, 64, 100, 127])
@pytest.mark.parametrize("compl", [True, False])
def test_digest_routes_agree(nctx, genome, k, compl):
    d1, runs, _ = _digest(nctx, genome, 1, k=k, complements=compl)
    assert runs == 1
    d0, runs, _ = _digest(nctx, genome, 0, k=k, complements=compl)
    assert runs == 0
    assert d1 == d0 and d1[0] > 0 and d1[3] == d1[1]
    nctx.set_option("sig_set", 1)
    r = nctx.compute(genome, k=k, complements=compl)
    assert r.n_kmers == d1[0]
    ms = np.frombuffer(r.ms, dtype=np.uint8)
    m1, runs, _ = _digest(nctx, ms, 1, k=k, complements=compl, masked=True)
    assert runs == 1
    m0, _, _ = _digest(nctx, ms, 0, k=k, complements=compl, masked=True)
    assert m1 == m0
    assert m1[:3] == d1[:3]


@pytest.mark.parametrize("j", [1, 3])
@pytest.mark.parametrize("d", [-64, -31, -1, 0, 1, 31, 64])
def test_digest_at_tile_edges(nctx, j, d):
    """One record of 8192 j + d bases (windows at strip and tile edges of the scan), as input and as a masked superstring."""
    rng = np.random.default_rng(1000 * j + d)
    rec = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=8192 * j + d)]
    cased = rec | (rng.integers(0, 2, size=rec.size).astype(np.uint8) << 5)
    seq, _, _ = synth.frame_records([rec])
    for k in (31, 64):
        for s, masked in ((seq, False), (cased, True)):
            d1, runs, _ = _digest(nctx, s, 1, k=k, masked=masked)
            d0, _, _ = _digest(nctx, s, 0, k=k, masked=masked)
            assert runs == 1 and d1 == d0


def test_digest_overflow_falls_back(nctx, genome):
    want, _, _ = _digest(nctx, genome, 0, k=31)
    nctx.set_option("sig_load_pct", 400)  # 4 x the records a bucket holds: every bucket overflows
    got, runs, fb = _digest(nctx, genome, 1, k=31)
    assert (runs, fb) == (0, 1) and got == want


def test_digest_empty_sets(nctx):
    ns = np.frombuffer(b"N" * 100_000 + b"\n", dtype=np.uint8)
    for sig in (1, 0):
        assert _digest(nctx, ns, sig, k=31)[0] == [0, 0, 0, 0]
    rng = np.random.default_rng(5)
    low = np.frombuffer(b"acgt", dtype=np.uint8)[rng.integers(0, 4, size=100_000)]
    for sig in (1, 0):
        d, runs, _ = _digest(nctx, low, sig, k=31, masked=True)
        assert d == [0, 0, 0, 0] and runs == sig


@pytest.fixture(scope="module")
def repeated():
    """The genome with copies (some k-mers twice, some three times) for -z 2 and 3, and a seeded 150x read set.  Its reads are long
    and have few errors, so that every k up to 127 sees each k-mer in ~70 windows or more: the signature buckets overflow."""
    recs = synth.human_like_genome(300_000, seed=78, n_runs=3)
    extra = [recs[0].copy(), recs[0][5000:].copy(), np.frombuffer(bytes(recs[1]).translate(_COMP)[::-1], dtype=np.uint8).copy()]
    seq, _, _ = synth.frame_records(recs + extra)
    reads = synth.frame_reads(synth.reads_chunks(100_000, 150.0, 300, 0.001, 79), 300)
    return seq, reads


@pytest.mark.parametrize("k", [26, 31, 63, 127])
@pytest.mark.parametrize("z", [1, 2, 3])
def test_streaming_routes_agree(nctx, repeated, k, z):
    seq, reads = repeated
    for s, what in ((seq, "genome"), (reads, "reads")):
        nctx.set_option("sig_set", 1)
        runs, fb = nctx.stat("sig_runs"), nctx.stat("sig_fallbacks")
        got = nctx.streaming(s, k=k, min_frequency=z)
        if what == "genome":
            assert nctx.stat("sig_runs") - runs == z and nctx.stat("sig_fallbacks") == fb
        else:  # coverage overflows the buckets: the first pass falls back, the later ones do not try again
            assert nctx.stat("sig_fallbacks") - fb == 1 and nctx.stat("sig_runs") == runs
        nctx.set_option("sig_set", 0)
        want = nctx.streaming(s, k=k, min_frequency=z)
        assert got.ms == want.ms and got.n_kmers == want.n_kmers and got.n_occurrences == want.n_occurrences
        if what == "genome":
            assert got.n_kmers > 0


# ---- inputs of 2^32 bytes and more -------------------------------------------------------------------------------------------

def _need_gpu_gb(gb):
    free, _ = torch.cuda.mem_get_info()
    if free < gb * 1e9:
        pytest.skip(f"needs {gb} GB of free device memory, {free / 1e9:.1f} GB free")


def _acgt(n, gen, alphabet=b"ACGT"):
    lut = torch.tensor(list(alphabet), dtype=torch.uint8, device="cuda")
    return lut[torch.randint(0, 4, (n,), dtype=torch.uint8, device="cuda", generator=gen).long()]


def _revcomp(x):
    comp = torch.zeros(256, dtype=torch.uint8, device="cuda")
    for a, b in zip(b"ACGT", b"TGCA"):
        comp[a] = b
    return comp[x.flip(0).long()]


def _fill(parts, n):
    out = torch.empty(n, dtype=torch.uint8, device="cuda")
    o = 0
    for p in parts:
        out[o:o + p.numel()] = p
        o += p.numel()
    assert o == n
    return out


@pytest.fixture
def lctx():
    c = kb.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def inputs():
    """big   = A + N gap + B + N * 128 + A + N * 128 + rc(B[:half]) + newline, B starting 4 Mbp before byte 2^32;
    small = the same with an N * 128 gap.  The copy of A adds no k-mer and every separator is at least k long, so the two have
    the same k-mer set, the same first-occurrence runs and the same streaming output.  -> host arrays (big, small)."""
    _need_gpu_gb(40)
    g = torch.Generator(device="cuda")
    g.manual_seed(20261021)
    a, b = _acgt(PART, g), _acgt(PART, g)
    rcb = _revcomp(b[: PART // 2])
    n128 = torch.full((128,), ord("N"), dtype=torch.uint8, device="cuda")
    nl = torch.tensor([ord("\n")], dtype=torch.uint8, device="cuda")
    gap = torch.full((2**32 - 4 * MBP - PART,), ord("N"), dtype=torch.uint8, device="cuda")
    tail = [b, n128, a, n128, rcb, nl]
    small = torch.cat([a, n128] + tail)
    big = _fill([a, gap] + tail, PART + gap.numel() + small.numel() - PART - 128)
    assert big.numel() >= 2**32
    big_h, small_h = big.cpu().numpy(), small.cpu().numpy()
    del a, b, rcb, gap, big, small
    torch.cuda.empty_cache()
    return big_h, small_h


@pytest.mark.parametrize("k", [31, 63, 127])
@pytest.mark.parametrize("compl", [True, False])
def test_large_digest_matches_small(lctx, inputs, k, compl):
    big, small = inputs
    _need_gpu_gb(30)
    want = lctx.kmer_digest(small, k=k, complements=compl)
    runs = lctx.stat("sig_runs")
    assert lctx.kmer_digest(big, k=k, complements=compl) == want
    assert lctx.stat("sig_runs") == runs + 1 and want[0] > 0


@pytest.mark.parametrize("k", [31, 63])
def test_large_lowerbound_and_streaming_match_small(lctx, inputs, k):
    big, small = inputs
    _need_gpu_gb(40)
    lb_small, st_small = lctx.lower_bound(small, k=k)
    lb_big, st_big = lctx.lower_bound(big, k=k)
    assert lb_big == lb_small and st_big.n_kmers == st_small.n_kmers
    for z in (1, 2):
        want = lctx.streaming(small, k=k, min_frequency=z)
        got = lctx.streaming(big, k=k, min_frequency=z)
        assert got.ms == want.ms and got.n_kmers == want.n_kmers
        assert got.n_occurrences == want.n_occurrences  # the N gap holds no window: both see the same windows


def test_large_masked_superstring(lctx, inputs):
    """ms(small) + lower-case filler past 2^32 + ms(small): the second copy's k-mers lie beyond 2^32 and fold into the first."""
    big, small = inputs
    _need_gpu_gb(40)
    k = 31
    r = lctx.compute(small, k=k)
    ms = torch.from_numpy(np.frombuffer(r.ms, dtype=np.uint8).copy()).cuda()
    g = torch.Generator(device="cuda")
    g.manual_seed(5)
    filler = _acgt(2**32 - ms.numel() + MBP, g, b"acgt")
    sup = _fill([ms, filler, ms], 2 * ms.numel() + filler.numel()).cpu().numpy()
    del filler, ms
    torch.cuda.empty_cache()
    want = lctx.kmer_digest(small, k=k)
    assert want[0] == r.n_kmers
    assert lctx.kmer_digest(sup, k=k, masked=True) == want


def test_4_4_gbases_genome_with_repeats(lctx):
    """k = 63: 43 random records of 100 Mbp plus a copy, a reverse complement and a partial copy of earlier ones; the input and the
    superstring are digested in one call each."""
    _need_gpu_gb(70)
    k, n_rec, rec_len = 63, 43, 100 * MBP
    g = torch.Generator(device="cuda")
    g.manual_seed(4400)
    recs = [_acgt(rec_len, g) for _ in range(n_rec)]
    recs += [recs[3], _revcomp(recs[10]), recs[20][rec_len // 3:]]
    nl = torch.tensor([ord("\n")], dtype=torch.uint8, device="cuda")
    parts = []
    for r in recs:
        parts += [r, nl]
    seq = _fill(parts, sum(p.numel() for p in parts))
    del recs, parts
    assert seq.numel() >= 2**32
    r = lctx.compute_device(seq.data_ptr(), seq.numel(), k=k)
    ms_bytes = lctx.copy_to_host(r.ms_ptr, r.length)
    ms = np.frombuffer(ms_bytes, dtype=np.uint8)
    host = seq.cpu().numpy()
    del seq
    torch.cuda.empty_cache()
    assert r.n_kmers == n_rec * (rec_len - k + 1) and r.length >= 2**32
    rh = lctx.compute(host, k=k)  # host buffers: the whole superstring comes back (not its length mod 2^32)
    assert rh.length == r.length and rh.ms == ms_bytes
    del rh
    d_in = lctx.kmer_digest(host, k=k)
    del host
    d_out = lctx.kmer_digest(ms, k=k, masked=True)
    assert d_in[0] == r.n_kmers
    assert d_out == d_in


@pytest.mark.parametrize("what", ["digest_z2", "digest_k21", "streaming_k21", "lowerbound_S"])
def test_large_refusals(lctx, inputs, what):
    big, _ = inputs
    reason = {"digest_z2": "-z", "digest_k21": "k is below 26", "streaming_k21": "k is below 26", "lowerbound_S": "-S was asked"}[what]
    with pytest.raises(kb.KcError) as e:
        if what == "digest_z2":
            lctx.kmer_digest(big, k=31, min_frequency=2)
        elif what == "digest_k21":
            lctx.kmer_digest(big, k=21)
        elif what == "streaming_k21":
            lctx.streaming(big, k=21)
        else:
            lctx.lower_bound(big, k=31, assume_simplitigs=True)
    assert e.value.code == -6
    msg = str(e.value)
    assert "2^32 bytes or more" in msg and reason in msg, msg


def _cli(*args):
    return subprocess.run([EXE, *map(str, args)], capture_output=True)


def test_cli_large(lctx, inputs, tmp_path):
    big, small = inputs
    if shutil.disk_usage(tmp_path).free < 10e9:
        pytest.skip("needs 10 GB of free disk for a 4.3 GB FASTA")
    _need_gpu_gb(40)
    if not os.path.exists(EXE):
        subprocess.check_call(["make", "-C", ROOT, "host/kmercamel"], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    k = 31
    lb_small, _ = lctx.lower_bound(small, k=k)
    st_small = lctx.streaming(small, k=k)
    fa = tmp_path / "big.fa"
    with open(fa, "wb") as f:
        f.write(b">big\n")
        f.write(memoryview(big))
    lctx.close()  # the CLI processes need the device memory
    p = _cli("lowerbound", "-k", k, fa)
    assert p.returncode == 0, p.stderr.decode()
    assert int(p.stdout.split()[0]) == lb_small
    p = _cli("compute", "-a", "streaming", "-k", k, fa)
    assert p.returncode == 0, p.stderr.decode()
    assert p.stdout.split(b"\n")[1] == st_small.ms
    out = tmp_path / "big.msfa"
    p = _cli("compute", "-k", k, "-o", out, fa)
    assert p.returncode == 0, p.stderr.decode()
    p = _cli("verify", "-k", k, fa, out)
    err = p.stderr.decode()
    assert p.returncode == 0 and "Verification passed" in err, err
    lines = out.read_bytes().split(b"\n")
    ms = bytearray(lines[1])
    i = next(i for i, c in enumerate(ms) if c < ord("a"))
    ms[i] |= 0x20
    bad = tmp_path / "bad.msfa"
    bad.write_bytes(lines[0] + b"\n" + bytes(ms) + b"\n")
    p = _cli("verify", "-k", k, fa, bad)
    err = p.stderr.decode()
    assert p.returncode == 2 and "Verification FAILED" in err, err
    fa.unlink()


def test_cli_verify_spneumoniae(tmp_path):
    if not os.path.exists(EXE):
        subprocess.check_call(["make", "-C", ROOT, "host/kmercamel"], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    sp = tmp_path / "spneumoniae.fa"
    sp.write_bytes(gzip.open(os.path.join(GOLDEN_DIR, "spneumoniae.fa.gz")).read())
    out = tmp_path / "sp.msfa"
    for flags in ([], ["-u"]):
        p = _cli("compute", "-k", 31, *flags, "-o", out, sp)
        assert p.returncode == 0, p.stderr.decode()
        p = _cli("verify", "-k", 31, *flags, sp, out)
        err = p.stderr.decode()
        assert p.returncode == 0 and "Verification passed" in err, err
    two = tmp_path / "two.msfa"
    two.write_bytes(out.read_bytes() * 2)
    p = _cli("verify", "-k", 31, sp, two)
    assert p.returncode == 1 and "single FASTA record" in p.stderr.decode()
