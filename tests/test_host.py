"""Host-side logic and the C-ABI surface — CPU only (no compute calls).

* libkcgpu.so loads and exports every symbol include/kcgpu.h declares;
* kc_frame_fasta (kseq semantics, host C++) against the oracle's restatement and the reference's outputs;
* the engine/emission control flow, compiled for the host (tests/host_emul, KC_HOST_EMUL), against the oracle.
"""
import ctypes
import functools
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import kmercamel_b200 as kb
from kmercamel_b200 import api
from oracle import orc
from conftest import ROOT, keys_md5, md5


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "kcgpu.h")).read()
    declared = set(re.findall(r"\b(kc_[a-z_0-9]+)\s*\(", header))
    assert declared == set(api.EXPORTED_SYMBOLS)
    lib = ctypes.CDLL(kb.lib_path())
    for name in declared:
        assert hasattr(lib, name), name


def test_error_strings():
    lib = kb.load_library()
    assert lib.kc_strerror(0) == b"ok"
    assert lib.kc_strerror(-8) == b"no CUDA device"
    assert lib.kc_limbs_for_k(31) == 1 and lib.kc_limbs_for_k(32) == 2 and lib.kc_limbs_for_k(64) == 4


def test_no_cpu_fallback_without_device():
    """Without a GPU the product refuses to run instead of falling back to a CPU path."""
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        pytest.skip("a GPU is present")
    with pytest.raises(kb.KcError) as e:
        kb.Context(0)
    assert e.value.code == -8


def test_frame_fasta_matches_oracle_and_reference(golden, test_fa_bytes):
    for name, g in golden["parser_cases"].items():
        data = g["text"].encode()
        seq, off, ln = kb.frame_fasta(data)
        want = orc.frame_fasta(data)
        got = [bytes(seq[int(o):int(o) + int(l)]) for o, l in zip(off, ln)]
        assert got == want, name
        for o, l in zip(off, ln):
            assert seq[int(o) + int(l)] == 10
        keys, _ = orc.count_kmers(seq, off, ln, 3, False)
        assert len(keys) == g["n_kmers_k3u"] and keys_md5(keys) == g["keys_md5"], name
    seq, off, ln = kb.frame_fasta(test_fa_bytes)
    assert bytes(seq) == b"ACCCGAAC\nCGTANATGC\nAcCCGTTTAACG\nA\n"
    assert off.tolist() == [0, 9, 19, 32] and ln.tolist() == [8, 9, 12, 1]


def test_frame_fasta_big_and_empty(spneumoniae_bytes):
    seq, off, ln = kb.frame_fasta(spneumoniae_bytes)
    want = orc.frame_fasta(spneumoniae_bytes)
    assert len(off) == len(want) == 1 and int(ln[0]) == len(want[0])
    assert bytes(seq[:int(ln[0])]) == want[0]
    seq, off, ln = kb.frame_fasta(b"")
    assert len(off) == 0
    seq, off, ln = kb.frame_fasta(b"no header here\n")
    assert len(off) == 0


def _fuzz_fasta(rng, n_rec, max_lines, widths, final_nl):
    out = []
    alphabet = np.frombuffer(b"ACGTacgtN>@+ ", dtype=np.uint8)
    for r in range(n_rec):
        hdr = b">" + (b"r%d" % r if rng.random() < 0.8 else b"") + (b" some comment" if rng.random() < 0.3 else b"") + (b"\tx" if rng.random() < 0.1 else b"")
        out.append(hdr + b"\n")
        for _ in range(int(rng.integers(0, max_lines + 1))):
            line = bytes(rng.choice(alphabet, size=int(rng.choice(widths))))
            if line[:1] in (b">", b"@", b"+"):
                line = b"A" + line[1:]
            out.append(line + b"\n")
            if rng.random() < 0.1:
                out.append(b"\n")
    data = b"".join(out)
    return data if final_nl or not data.endswith(b"\n") else data[:-1]


def test_frame_fasta_parallel_path(golden, monkeypatch):
    """Plain FASTA is framed by several threads (framing.cpp frame_plain_fasta_parallel; default for inputs >= 8 MB): same records
    as the oracle's restatement of kseq_read whatever the thread count; FASTQ / '\\r' / stray-marker inputs are declined and take
    the serial reader."""
    rng = np.random.default_rng(5)
    for it in range(150):
        data = _fuzz_fasta(rng, int(rng.integers(1, 40)), int(rng.integers(0, 6)), [0, 1, 2, 5, 60, 80], bool(rng.random() < 0.7))
        want = orc.frame_fasta(data)
        for threads in ("2", "3", "8", "32"):
            monkeypatch.setenv("KC_FRAME_THREADS", threads)
            seq, off, ln = kb.frame_fasta(data)
            assert [bytes(seq[int(o):int(o) + int(l)]) for o, l in zip(off, ln)] == want, (it, threads)
            assert all(seq[int(o) + int(l)] == 10 for o, l in zip(off, ln)) and len(seq) == int(off[-1]) + int(ln[-1]) + 1
    for name, g in golden["parser_cases"].items():
        data = g["text"].encode()
        for threads in ("2", "8"):
            monkeypatch.setenv("KC_FRAME_THREADS", threads)
            seq, off, ln = kb.frame_fasta(data)
            assert [bytes(seq[int(o):int(o) + int(l)]) for o, l in zip(off, ln)] == orc.frame_fasta(data), name
    # above the size threshold the parallel path is the default: identical bytes to the serial reader
    big = _fuzz_fasta(rng, 60, 400, [80], True) * 10
    assert len(big) > (8 << 20)
    monkeypatch.setenv("KC_FRAME_THREADS", "1")
    a = kb.frame_fasta(big)
    monkeypatch.delenv("KC_FRAME_THREADS")
    b = kb.frame_fasta(big)
    assert all(np.array_equal(x, y) for x, y in zip(a, b)) and len(a[1]) == 600


def test_synth_fasta_roundtrip():
    from kmercamel_b200 import synth
    recs = synth.random_genome_records(3, 205, 7)
    text = synth.fasta_bytes(recs, width=80)
    seq, off, ln = kb.frame_fasta(text)
    s2, o2, l2 = synth.frame_records(recs)
    assert np.array_equal(seq, s2) and np.array_equal(off, o2) and np.array_equal(ln, l2)


# ---- host emulation of the engine ------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def host_emul():
    exe = os.path.join(ROOT, "tests", "host_emul")
    if shutil.which("nvcc") is None and not os.path.exists(exe):
        pytest.skip("nvcc not available to build tests/host_emul")
    if shutil.which("nvcc") is not None:
        subprocess.check_call(["make", "-C", ROOT, "tests/host_emul"], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)

    def run(mode, k, compl, strict, flag, records, poison=None):
        env = dict(os.environ)
        env.pop("KC_ARENA_POISON", None)
        if poison is not None:
            env["KC_ARENA_POISON"] = str(poison)
        p = subprocess.run([exe, mode, str(k), str(int(compl)), str(int(strict)), str(int(flag))],
                           input=b"\n".join(records) + b"\n", capture_output=True, env=env)
        assert p.returncode == 0, p.stderr
        return p.stdout.split(b"\n"), p.stderr.decode()
    return run


def test_host_emul_path_kats(host_emul):
    from test_oracle import PATH_KATS
    for records, k, compl, lb, want_ef, want_ov in PATH_KATS:
        out, _ = host_emul("path", k, compl, True, lb, [r.encode() for r in records])
        rows = [tuple(map(int, ln.split())) for ln in out if ln]
        assert [r[0] for r in rows] == want_ef and [r[1] for r in rows] == want_ov


def test_host_emul_fuzz_S_byte_exact(host_emul, golden):
    for g in golden["fuzz_S"]:
        out, _ = host_emul("ms", g["k"], g["complements"], True, True, [r.encode() for r in g["records"]])
        assert out[0].decode() == g["ms"]
        assert md5(out[1] + b"\n") == g["maxone_md5"]


def test_host_emul_simplitigs_md5(host_emul, golden, simplitigs_bytes):
    g = golden["simplitigs_S"]["k31"]
    out, err = host_emul("ms", 31, True, True, True, orc.frame_fasta(simplitigs_bytes))
    assert md5(out[0] + b"\n") == g["md5"] and md5(out[1] + b"\n") == g["maxone_md5"]


def tie_heavy_node_set(seed):
    """Seeded node set with many equal overlaps: records over a small alphabet, half of them periodic (a motif of 1-6 bases with a
    few substitutions), the rest random; k from 3 to 127 so that all three word widths are covered.  -> (k, complements, records)"""
    rng = np.random.default_rng(seed)
    k = int(rng.choice([3, 4, 5, 6, 7, 8, 8, 12, 31, 32, 40, 63, 64, 100, 127]))
    alpha = [b"AC", b"AT", b"ACG", b"ACGT"][seed % 4]
    letters = np.frombuffer(alpha, dtype=np.uint8)
    motifs = [rng.choice(letters, size=int(rng.integers(1, 7))).tobytes() for _ in range(4)]
    recs = []
    for _ in range(int(rng.integers(30, 401))):
        n = k + int(rng.integers(0, k + 3))
        if rng.random() < 0.5:
            m = motifs[int(rng.integers(0, len(motifs)))]
            ph = int(rng.integers(0, len(m)))
            r = bytearray((m * (n // len(m) + 2))[ph:ph + n])
            for _ in range(int(rng.integers(0, 3))):
                r[int(rng.integers(0, n))] = int(rng.choice(letters))
        else:
            r = bytearray(rng.choice(letters, size=n).tobytes())
        recs.append(bytes(r))
    return k, bool(seed % 3), recs


def test_host_emul_path_matches_oracle_batches(host_emul):
    """The engine's tie order, compiled for the host, is the reference's greedy with the prefix nodes in one batch when it runs
    non-strict (the from-FASTA regime: every prefix in batch 0, all cycle closers of a round banned at once) and with the
    reference's 16 batches when it runs strict (-S).  Byte for byte, on node sets where equal overlaps and cycles abound."""
    from test_oracle import node_ends
    n_cases, banned, widths = 120, 0, set()
    for seed in range(n_cases):
        k, compl, recs = tie_heavy_node_set(seed)
        widths.add(orc.limbs_for_k(k))
        first, last = node_ends([r.decode() for r in recs], k)
        for strict, parts in ((False, 1), (True, 16)):
            out, err = host_emul("path", k, compl, strict, False, recs)
            rows = np.array([list(map(int, ln.split())) for ln in out if ln], dtype=np.int64)
            want_ef, want_ov = orc.overlap_path(first, last, k, compl, parts=parts)
            assert np.array_equal(rows[:, 0], want_ef) and np.array_equal(rows[:, 1], want_ov), (seed, k, compl, strict)
            if not strict and int(re.search(r"\bbans=(\d+)", err).group(1)) > 0:
                banned += 1
    assert widths == {1, 2, 4}
    print(f"non-strict engine banned edges in {banned} of {n_cases} node sets")
    assert 3 * banned >= n_cases  # the ban / replay path of the non-strict engine is covered, not avoided


def test_host_emul_from_kmers_valid(host_emul):
    """From-FASTA regime (k-mer nodes, non-strict): the superstring represents exactly the k-mer set."""
    import random
    rng = random.Random(5)
    for k, compl in [(5, True), (8, False), (12, True), (31, True), (33, False)]:
        genome = "".join(rng.choice("ACGT") for _ in range(3000))
        recs = [genome[i:i + 400].encode() for i in range(0, 2800, 300)] + [b"A" * 60, b"ACACACACACACACACACACACACACACACACACACACACACAC"]
        out, _ = host_emul("kmers", k, compl, False, True, recs)
        seq, off, ln = orc.records_to_arrays(recs)
        exp, _ = orc.count_kmers(seq, off, ln, k, compl)
        assert orc.verify_ms(out[0], k, compl, exp) and orc.verify_ms(out[1], k, compl, exp)
        assert sum(1 for c in out[0] if c <= 90) == len(exp)  # min-one: every k-mer ON exactly once


@pytest.mark.parametrize("poison", [0x00, 0xA5, 0xFF])
def test_host_emul_poisoned_arena(host_emul, golden, simplitigs_bytes, poison):
    """The cases above with every arena block filled with `poison` before it is handed out: the engine and the emission must
    write everything they read.  0x00 looks like a finished zero-fill, 0xFF like KC_NONE."""
    run = functools.partial(host_emul, poison=poison)
    test_host_emul_path_kats(run)
    test_host_emul_fuzz_S_byte_exact(run, golden)
    test_host_emul_simplitigs_md5(run, golden, simplitigs_bytes)
    test_host_emul_path_matches_oracle_batches(run)
    test_host_emul_from_kmers_valid(run)


# ---- plan of the fixed-slot k-mer set construction (csrc/ksf_plan.h) -----------------------------------------------
def _ksf_plan(m, leaf_target=768, sigmas=8):
    exe = os.path.join(ROOT, "tests", "host_emul")
    out = subprocess.run([exe, "plan", str(m), str(leaf_target), str(sigmas), "0"], capture_output=True, check=True).stdout.split(b"\n")
    ok, levels, n_leaf, s0, s1 = map(int, out[0].split())
    return ok, levels, n_leaf, (s0, s1), [tuple(map(int, ln.split())) for ln in out[1:1 + levels]] if ok else []


@pytest.mark.parametrize("m", [1 << 16, 100_000, 210_006, 6_500_007, 50_000_050, 400_000_400, 500_000_050, 3_100_000_024, 4_200_000_000])
@pytest.mark.parametrize("leaf_target", [768, 16, 1])
def test_ksf_plan_invariants(host_emul, m, leaf_target):
    """What the fixed-slot kernels rely on (kmerset_fast.cuh): digits of at most 8 bits (256 counters per tile), slots that are
    multiples of 32 items (16-byte cp.async copies of tiles and leaves stay aligned), all digits inside the top 40 bits of the
    scrambled word (KWord::digit_top; the sharded path puts 8 more bits in front), leaf slots of KSF_LEAF_CAP items with a mean
    fill of at most leaf_target, ping/pong buffers that hold every level they serve."""
    ok, levels, n_leaf, slots, rows = _ksf_plan(m, leaf_target)
    assert ok and 1 <= levels <= 4 and len(rows) == levels      # every size up to 2^32 positions is plannable, down to leaves of 1
    cum = 0
    for i, (bits, c, cap) in enumerate(rows):
        assert 1 <= bits <= 8
        cum += bits
        assert c == cum and cum <= 40
        assert cap % 32 == 0 and 0 < cap < 1 << 32
        mean = m / (1 << cum)
        if i == levels - 1:
            assert cap == 1024 and (m >> cum) <= leaf_target
        else:
            assert cap >= mean + 8 * mean ** 0.5                     # mean + 8 sigma of a Poisson-tight bucket
        assert slots[i & 1] >= (1 << cum) * cap
    assert n_leaf == 1 << cum
    assert max(b for b, _, _ in rows) - min(b for b, _, _ in rows) <= 1  # digits spread evenly over the levels


def test_ksf_plan_small_inputs_take_the_exact_path(host_emul):
    assert _ksf_plan((1 << 16) - 1)[0] == 0 and _ksf_plan(0)[0] == 0
    ok, levels, n_leaf, _, rows = _ksf_plan(50_000_050)              # configs[1]: two 8-bit levels, 65536 leaves of ~763
    assert (ok, levels, n_leaf) == (1, 2, 65536) and [r[0] for r in rows] == [8, 8]
