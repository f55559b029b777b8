"""The oracle (oracle/oracle.cpp, oracle/orc.py) against the reference's golden vectors — CPU only.

Vectors come from (a) the reference's own unit tests, cited per test, and (b) tests/golden/golden.json, generated
by tests/golden/make_golden.py from the unmodified reference compiled into oracle/_ref.
"""
import hashlib

import numpy as np
import pytest

from oracle import orc
from conftest import keys_md5, md5


def K(s, k=None):
    return orc.kmer_from_string(s, k)


def kint(s):
    v = 0
    for ch in s:
        v = (v << 2) | "ACGT".index(ch)
    return v


# ---- k-mer arithmetic: reference tests/kmers_unittest.h:10-24,99-117 ------------------------------------------
@pytest.mark.parametrize("kmer,d,want", [("TACG", 2, "CG"), ("TACG", 0, ""), ("ACGT", 4, "ACGT"), ("G" * 31, 30, "G" * 30)])
def test_bit_suffix(kmer, d, want):
    assert orc.kmer_to_int(orc.bit_suffix(K(kmer), len(kmer), d)) == kint(want)


@pytest.mark.parametrize("kmer,d,want", [("TACG", 2, "TA"), ("TACG", 0, ""), ("ACGT", 4, "ACGT"), ("C" + "G" * 30, 1, "C")])
def test_bit_prefix(kmer, d, want):
    assert orc.kmer_to_int(orc.bit_prefix(K(kmer), len(kmer), d)) == kint(want)


@pytest.mark.parametrize("kmer,want", [("A", "T"), ("ACG", "CGT"), ("TAGCTAGCTAGCTAGCTAGCTAGCTAGCTAG", "CTAGCTAGCTAGCTAGCTAGCTAGCTAGCTA"),
                                       ("ACGT" * 10, "ACGT" * 10), ("A" * 70 + "C", "G" + "T" * 70)])
def test_reverse_complement(kmer, want):
    k = len(kmer)
    assert orc.kmer_to_int(orc.reverse_complement(K(kmer), k)) == kint(want)


# ---- set construction: tests/parser_unittest.h:38-91 on tests/testdata/test.fa -------------------------------
@pytest.mark.parametrize("k,compl,size", [(10, True, 3), (5, True, 11), (5, False, 11), (2, True, 9), (2, False, 11)])
def test_read_kmers_sizes(test_fa_bytes, k, compl, size):
    seq, off, ln = orc.records_to_arrays(orc.frame_fasta(test_fa_bytes))
    keys, _ = orc.count_kmers(seq, off, ln, k, compl)
    assert len(keys) == size


@pytest.mark.parametrize("k,compl,z,size", [(3, True, 2, 6), (3, False, 2, 5), (3, True, 3, 2), (4, True, 2, 3), (1, False, 5, 4),
                                            (1, False, 6, 2), (1, False, 10, 1)])
def test_read_kmers_filtered_sizes(test_fa_bytes, k, compl, z, size):
    seq, off, ln = orc.records_to_arrays(orc.frame_fasta(test_fa_bytes))
    _, vals = orc.count_kmers(seq, off, ln, k, compl)
    assert int((vals.astype(int) + 1 >= z).sum()) == size  # src/khash_utils.h:146


def test_counts_golden_small(test_fa_bytes):
    """SURVEY.md appendix B-3: value = occurrences - 1 for k=3 canonical on test.fa."""
    seq, off, ln = orc.records_to_arrays(orc.frame_fasta(test_fa_bytes))
    keys, vals = orc.count_kmers(seq, off, ln, 3, True)
    got = " ".join("".join("ACGT"[(int(x[0]) >> (2 * (2 - i))) & 3] for i in range(3)) + str(v) for x, v in zip(keys, vals))
    assert got == "AAA0 AAC2 ACC1 ACG2 ATG0 CCC1 CCG1 CGA0 GAA0 GCA0 GTA0 TAA1"


@pytest.mark.parametrize("name", ["k3", "k3u", "k10", "k5", "k5u", "k2", "k2u", "k1u", "k4"])
def test_kmers_vs_reference_test_fa(golden, test_fa_bytes, name):
    g = golden["test_fa_kmers"][name]
    k = int(name[1:].rstrip("u"))
    seq, off, ln = orc.records_to_arrays(orc.frame_fasta(test_fa_bytes))
    keys, vals = orc.count_kmers(seq, off, ln, k, not name.endswith("u"))
    assert len(keys) == g["n"] and keys_md5(keys) == g["keys_md5"] and md5(vals.tobytes()) == g["vals_md5"]


@pytest.mark.parametrize("name", ["k31", "k31u", "k63", "k127u", "k32", "k64", "k5", "k1u"])
def test_kmers_vs_reference_spneumoniae(golden, spneumoniae_bytes, name):
    g = golden["spneumoniae_kmers"][name]
    k = int(name[1:].rstrip("u"))
    seq, off, ln = orc.records_to_arrays(orc.frame_fasta(spneumoniae_bytes))
    keys, vals = orc.count_kmers(seq, off, ln, k, not name.endswith("u"))
    assert len(keys) == g["n"] and keys.shape[1] == g["limbs"]
    assert keys_md5(keys) == g["keys_md5"] and md5(vals.tobytes()) == g["vals_md5"]


# ---- kseq framing: SURVEY.md appendix B-4 cases, outputs from the compiled reference ---------------------------
def test_frame_fasta_cases(golden):
    for name, g in golden["parser_cases"].items():
        recs = orc.frame_fasta(g["text"].encode())
        seq, off, ln = orc.records_to_arrays(recs)
        keys, _ = orc.count_kmers(seq, off, ln, 3, False)
        assert len(keys) == g["n_kmers_k3u"], name
        assert keys_md5(keys) == g["keys_md5"], name


# ---- greedy tie order: tests/global_unittest.h:61-104 and tests/global_sparse_unittest.h:84-103 ---------------
PATH_KATS = [
    (["AT"], 2, True, False, [-1, -1], [255, 255]),
    (["ACG", "TAC", "GGC"], 3, False, False, [2, 0, -1], [1, 2, 255]),
    (["ACAA", "ATTT", "AACA"], 4, True, False, [4, 3, 0, 5, -1, -1], [2, 2, 3, 3, 255, 255]),
    (["ACG", "CGT", "TAA"], 3, False, True, [1, 2, 0], [2, 1, 1]),
    (["ACGT", "TAA"], 3, False, True, [1, 0], [1, 1]),
    (["ACC", "CGG"], 3, True, True, [3, 2, 0, 1], [2, 2, 0, 2]),
]


def node_ends(records, k):
    first = np.stack([orc.kmer_from_string(r[:k], k) for r in records])
    last = np.stack([orc.kmer_from_string(r[len(r) - k:], k) for r in records])
    return first, last


@pytest.mark.parametrize("records,k,compl,lb,want_ef,want_ov", PATH_KATS)
def test_overlap_path_kats(records, k, compl, lb, want_ef, want_ov):
    first, last = node_ends(records, k)
    ef, ov = orc.overlap_path(first, last, k, compl, lb)
    assert ef.tolist() == want_ef and ov.tolist() == want_ov


@pytest.mark.parametrize("records,k,compl,lb,want_ef,want_ov", PATH_KATS)
def test_overlap_path_parts(records, k, compl, lb, want_ef, want_ov):
    """parts = 16 is the reference's batching (the default); one batch agrees with it where no tie spans two batches."""
    first, last = node_ends(records, k)
    for parts in (16, 1):
        ef, ov = orc.overlap_path(first, last, k, compl, lb, parts=parts)
        assert ef.tolist() == want_ef and ov.tolist() == want_ov, parts


# ---- the product's from-FASTA nodes: first-occurrence runs (kmercamel_b200/csrc/runs.cuh) --------------------------
def _messy_records(seed):
    """Records with N bytes, lower-case stretches, records shorter than k and repeated pieces."""
    from kmercamel_b200 import synth
    rng = np.random.default_rng(seed)
    recs = [bytearray(r.tobytes()) for r in synth.random_genome_records(4, 900, seed)]
    recs.append(bytearray(recs[0][200:500]))                                  # repeated piece: later occurrences are not first
    recs[1][100:160] = bytes(recs[1][100:160]).lower()
    recs[2][300:305] = b"NNNNN"
    recs += [bytearray(b"ACGTA"), bytearray(b""), bytearray(b"acgtNacgtacgtt"), bytearray(recs[3][:40]).lower()]
    for _ in range(30):                                                     # short pieces of earlier records
        r = recs[int(rng.integers(0, 4))]
        a = int(rng.integers(0, len(r) - 40))
        recs.append(bytearray(r[a:a + int(rng.integers(1, 40))]))
    return [bytes(r) for r in recs]


@pytest.mark.parametrize("k", [1, 5, 11, 21, 31])
@pytest.mark.parametrize("compl", [True, False])
def test_first_occurrence_runs_vs_flags(k, compl):
    """orc.first_occurrence_runs against the plain numpy first-occurrence flags of the sharded tests: the runs are exactly the
    maximal stretches of flagged window ends, in input order, and the kept counts agree."""
    from test_sharded import first_occurrence_flags, make_input
    inputs = [make_input(3), make_input(4), orc.records_to_arrays(_messy_records(5))[0]]
    for seq in inputs:
        recs = bytes(seq).split(b"\n")[:-1]
        s2, off, ln = orc.records_to_arrays(recs)
        assert np.array_equal(s2, seq)
        for z in (1, 2, 3):
            words, kept = first_occurrence_flags(seq, k, compl, z)
            ro, rl, n_kept = orc.first_occurrence_runs(seq, off, ln, k, compl, z)
            assert n_kept == kept and int((rl - np.uint64(k - 1)).sum()) == kept, (k, compl, z)
            got = np.zeros_like(words)
            ends = np.concatenate([np.arange(int(o) + k - 1, int(o) + int(l)) for o, l in zip(ro, rl)]) if len(ro) else np.zeros(0, np.int64)
            np.bitwise_or.at(got, ends >> 5, np.uint32(1) << (ends & 31).astype(np.uint32))
            assert np.array_equal(got, words), (k, compl, z)
            assert np.all(ro[1:] > ro[:-1] + rl[:-1] - np.uint64(k - 1))       # input order, maximal: no two runs touch


def test_compute_from_fasta_is_a_min_one_superstring():
    """The restated from-FASTA pipeline emits a superstring of exactly the kept k-mers with every k-mer ON once, in both node
    regimes (runs and, past the sparse switch, k-mer nodes), and its lower bound does not exceed it."""
    from kmercamel_b200 import synth
    cases = [(_messy_records(7), 11, True, 1), (_messy_records(8), 31, False, 1), (_messy_records(9), 5, True, 2),
             ([r.tobytes() for r in synth.short_records(300, 9, 11, 19)], 9, False, 1),
             ([r.tobytes() for r in synth.short_records(200, 31, 34, 17)], 31, True, 1)]
    for recs, k, compl, z in cases:
        seq, off, ln = orc.records_to_arrays(recs)
        keys, vals = orc.count_kmers(seq, off, ln, k, compl)
        keys = keys[vals.astype(np.int64) + 1 >= z]
        for sparse in (True, False):
            r = orc.compute_from_fasta(seq, off, ln, k, compl, z, want_maxone=True, sparse_switch=sparse)
            assert r["n_kmers"] == len(keys)
            assert orc.verify_ms(r["ms"], k, compl, keys) and orc.verify_ms(r["maxone"], k, compl, keys)
            assert sum(1 for c in r["ms"] if c <= 90) == len(keys)
            assert r["ms"].upper() == r["maxone"].upper()
            switched = sparse and r["n_simplitigs"] * 5 >= r["n_kmers"]
            assert r["n_nodes"] == (r["n_kmers"] if switched else r["n_simplitigs"])
            assert orc.lower_bound_from_fasta(seq, off, ln, k, compl, z, sparse_switch=sparse) <= len(r["ms"])


# ---- lowerbound: tests/lower_bound_unittest.h:11-41 and the reference CLI on the fuzzed -S inputs -------------
LOWER_BOUND_KATS = [(["ACG", "CGT", "TAA"], 3, False, 5), (["ACGT", "TAA"], 3, False, 5), (["AC", "GG"], 2, True, 3),
                    (["AAACCC", "CCCAAA", "TGGGGT"], 6, False, 11)]


@pytest.mark.parametrize("records,k,compl,want", LOWER_BOUND_KATS)
def test_lower_bound_kats(records, k, compl, want):
    assert orc.lower_bound_from_simplitigs([r.encode() for r in records], k, compl) == want


def test_lower_bound_fuzz_vs_reference_cli(golden):
    for g, want in zip(golden["fuzz_S"], golden["lowerbound"]["fuzz_S"]):
        assert orc.lower_bound_from_simplitigs([r.encode() for r in g["records"]], g["k"], g["complements"]) == want, g


# ---- Global end to end: tests/global_unittest.h:120-129 -----------------------------------------------------
GLOBAL_KATS = [
    ("TACgt", 3, ["CGT", "TAC", "ACG"], False), ("ACGT", 1, ["ACGT"], False), ("ACgTtt", 3, ["CGT", "TTT", "ACG"], False),
    ("ACgTtt", 3, ["ACGT", "TTT"], False), ("TActt", 4, ["TACT", "ACTT"], False),
    ("TActTaaGgac", 4, ["TACT", "ACTT", "GGAC", "TAAG"], False),
    ("TTtcttttttttttttttttttttttttttga", 31, ["TTTCTTTTTTTTTTTTTTTTTTTTTTTTTTG", "TTCTTTTTTTTTTTTTTTTTTTTTTTTTTGA"], False),
    ("AtTTgtt", 4, ["ACAA", "ATTT", "AACA"], True),
]


@pytest.mark.parametrize("want,k,records,compl", GLOBAL_KATS)
def test_global_kats(want, k, records, compl):
    ms, _ = orc.compute_from_simplitigs([r.encode() for r in records], k, compl)
    assert ms.decode() == want


# SuperstringFromPath: tests/global_unittest.h:11-51
@pytest.mark.parametrize("ef,ov,records,k,want,compl", [
    ([2, 0, -1], [1, 2, 255], ["ACG", "TAC", "GGC"], 3, "TAcGgc", False),
    ([4, 3, 1, -1, 5, -1], [1, 2, 1, 255, 2, 255], ["GCC", "ACG", "TAC"], 3, "GcCGta", True),
    ([3, 1, -1, -1], [1, 1, 255, 255], ["GCC", "TACG"], 3, "GcCGta", True),
])
def test_superstring_from_path(ef, ov, records, k, want, compl):
    seq, off, ln = orc.records_to_arrays([r.encode() for r in records])
    ms, _ = orc.superstring(seq, off, ln, k, compl, np.array(ef), np.array(ov, dtype=np.uint8))
    assert ms.decode() == want


# ---- -S regime byte-exact against the compiled reference --------------------------------------------------------
def test_fuzz_S_vs_reference(golden):
    for g in golden["fuzz_S"]:
        ms, mo = orc.compute_from_simplitigs([r.encode() for r in g["records"]], g["k"], g["complements"], True)
        assert ms.decode() == g["ms"]
        assert md5(mo + b"\n") == g["maxone_md5"]


@pytest.mark.parametrize("name", ["k31", "k31u", "k25", "k17u"])
def test_simplitigs_S_md5(golden, simplitigs_bytes, name):
    g = golden["simplitigs_S"][name]
    k = int(name[1:].rstrip("u"))
    recs = orc.frame_fasta(simplitigs_bytes)
    ms, mo = orc.compute_from_simplitigs(recs, k, not name.endswith("u"), True)
    assert len(ms) == g["length"] and md5(ms + b"\n") == g["md5"] and md5(mo + b"\n") == g["maxone_md5"]


# ---- verifier: must accept the reference's output and reject a corrupted one -------------------------------------
def test_verifier_pinned(golden):
    g = golden["fuzz_S"][3]
    recs = [r.encode() for r in g["records"]]
    seq, off, ln = orc.records_to_arrays(recs)
    exp, _ = orc.count_kmers(seq, off, ln, g["k"], g["complements"])
    ms = g["ms"].encode()
    assert orc.verify_ms(ms, g["k"], g["complements"], exp)
    on = [i for i, c in enumerate(ms) if c <= 90]
    bad = bytearray(ms)
    bad[on[0]] += 32  # switch one represented k-mer off
    got, _ = orc.ms_kmers(bytes(bad), g["k"], g["complements"])
    assert len(got) <= len(exp)
    if len(set(map(bytes, got))) != len(exp):
        assert not orc.verify_ms(bytes(bad), g["k"], g["complements"], exp)


def test_synth_human_like_genome_is_seeded_and_has_repeats():
    """Generator of configs[4] (SURVEY.md §8d config 5): deterministic, 24 records in human-like proportions, a few N runs, and
    ~1 % of the 31-mer windows are repeats of earlier ones (5 % of the bases are copies with 1-10 % divergence)."""
    import hashlib
    from kmercamel_b200 import synth
    recs = synth.human_like_genome(2_000_000, seed=3100)
    again = synth.human_like_genome(2_000_000, seed=3100)
    assert len(recs) == 24 and sum(len(r) for r in recs) == 2_000_000
    assert all(np.array_equal(a, b) for a, b in zip(recs, again))
    assert len(recs[0]) > 4 * len(recs[21])                              # chr1 vs chr22
    seq, off, ln = synth.frame_records(recs)
    assert hashlib.md5(seq.tobytes()).hexdigest() == "e72bac7b262774df96c6416fdca95166"
    n_frac = float((seq == ord("N")).mean())
    assert 0.001 < n_frac < 0.03
    keys, vals = orc.count_kmers(seq, off, ln, 31, True)
    repeats = int(vals.astype(np.int64).sum())                           # occurrences beyond the first
    assert 0.003 * len(keys) < repeats < 0.03 * len(keys)
    other = synth.human_like_genome(2_000_000, seed=3101)
    assert not np.array_equal(other[0], recs[0])
