"""TEST INFRASTRUCTURE ONLY — ctypes front end of oracle/liboracle.so plus a pure-Python kseq restatement.

Importers allowed: tests/, __graft_entry__.smoke(), bench.py (cpu_baseline / --impl reference legs).
The product package `kmercamel_b200` never imports this module.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

u8p = C.POINTER(C.c_uint8)
u64p = C.POINTER(C.c_uint64)
i64p = C.POINTER(C.c_int64)


def build(force: bool = False) -> str:
    """Compile liboracle.so (g++ only).  Returns its path."""
    so = os.path.join(_HERE, "liboracle.so")
    src = [os.path.join(_HERE, f) for f in ("oracle.cpp", "oracle.h")]
    if force or not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in src):
        subprocess.check_call(["make", "-C", _HERE, "liboracle.so"], stdout=subprocess.DEVNULL)
    return so


def lib():
    global _LIB
    if _LIB is None:
        L = C.CDLL(build())
        L.orc_limbs_for_k.restype = C.c_int
        L.orc_count_kmers.argtypes = [u8p, u64p, u64p, C.c_uint64, C.c_int, C.c_int, C.POINTER(u64p), C.POINTER(u8p), u64p]
        L.orc_overlap_path.argtypes = [u64p, u64p, C.c_uint64, C.c_int, C.c_int, C.c_int, i64p, u8p]
        L.orc_overlap_path_parts.argtypes = [u64p, u64p, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_int, i64p, u8p]
        L.orc_first_occurrence_runs.argtypes = [u8p, u64p, u64p, C.c_uint64, C.c_int, C.c_int, C.c_int, C.POINTER(u64p),
                                                C.POINTER(u64p), u64p, u64p]
        L.orc_superstring.argtypes = [u8p, u64p, u64p, C.c_uint64, C.c_int, C.c_int, i64p, u8p, u64p, C.c_uint64,
                                      C.POINTER(u8p), C.POINTER(u8p), u64p]
        L.orc_compute_from_simplitigs.argtypes = [u8p, u64p, u64p, C.c_uint64, C.c_int, C.c_int, C.c_int,
                                                  C.POINTER(u8p), C.POINTER(u8p), u64p]
        L.orc_ms_kmers.argtypes = [u8p, C.c_uint64, C.c_int, C.c_int, C.POINTER(u64p), u64p, u64p]
        L.orc_reverse_complement.argtypes = [u64p, C.c_int, u64p]
        L.orc_bit_prefix.argtypes = [u64p, C.c_int, C.c_int, u64p]
        L.orc_bit_suffix.argtypes = [u64p, C.c_int, C.c_int, u64p]
        L.orc_streaming.argtypes = [u8p, u64p, u64p, C.c_uint64, C.c_int, C.c_int, C.c_int, C.POINTER(u8p), u64p]
        L.orc_maskopt.argtypes = [u8p, C.c_uint64, C.c_int, C.c_int, C.c_int, u8p]
        L.orc_free.argtypes = [C.c_void_p]
        _LIB = L
    return _LIB


def limbs_for_k(k: int) -> int:
    return 1 if k < 32 else (2 if k < 64 else 4)


def _ptr(a, t):
    return a.ctypes.data_as(t)


def _take(ptr, n, dtype):
    """Copy n items out of a malloc'ed oracle buffer and free it."""
    if n == 0:
        out = np.zeros(0, dtype=dtype)
    else:
        out = np.ctypeslib.as_array(ptr, shape=(n,)).astype(dtype, copy=True)
    lib().orc_free(C.cast(ptr, C.c_void_p))
    return out


# ----------------------------------------------------------------------------------------------------
# kseq restatement (reference src/kseq.h:182-224 kseq_read, :98-147 ks_getuntil2) — pure Python, small inputs.
def frame_fasta(data: bytes):
    """Return the list of record sequences (bytes) exactly as kseq_read yields them to ReadKMers
    (reference src/parser.h:106-118): reading stops at the first negative return value."""
    n = len(data)
    pos = 0
    last_char = 0
    records = []
    SPACE = b" \t\n\v\f\r"
    GT, AT, PLUS, NL, CR = 0x3E, 0x40, 0x2B, 0x0A, 0x0D

    def getc():
        nonlocal pos
        if pos >= n:
            return -1
        c = data[pos]
        pos += 1
        return c

    def getuntil_line(acc: bytearray) -> int:
        """ks_getuntil2(KS_SEP_LINE, append=1): -1 if already at EOF, else the accumulated length."""
        nonlocal pos
        if pos >= n:
            return -1
        e = data.find(b"\n", pos)
        if e < 0:
            acc += data[pos:n]
            pos = n
        else:
            acc += data[pos:e]
            pos = e + 1
        if len(acc) > 1 and acc[-1] == CR:  # kseq.h:143
            del acc[-1]
        return len(acc)

    while True:
        if last_char == 0:  # kseq.h:187-191 jump to the next header character, wherever it is
            c = getc()
            while c >= 0 and c != GT and c != AT:
                c = getc()
            if c < 0:
                return records
            last_char = c
        if pos >= n:  # kseq.h:193 name: ks_getuntil returns -1 when nothing is left
            return records
        q = pos
        while q < n and data[q] not in SPACE:
            q += 1
        delim = data[q] if q < n else 0
        pos = min(n, q + 1)
        if delim != NL:  # kseq.h:194 comment
            getuntil_line(bytearray())
        seq = bytearray()
        c = getc()
        while c >= 0 and c != GT and c != PLUS and c != AT:  # kseq.h:199-203
            if c != NL:
                seq.append(c)
                getuntil_line(seq)
            c = getc()
        if c == GT or c == AT:
            last_char = c
        if c != PLUS:  # FASTA record
            records.append(bytes(seq))
            continue
        c = getc()  # kseq.h:217 skip the rest of the '+' line
        while c >= 0 and c != NL:
            c = getc()
        if c < 0:
            return records  # -2: no quality string; the record is dropped, ReadKMers stops
        qual = bytearray()
        while getuntil_line(qual) >= 0 and len(qual) < len(seq):  # kseq.h:219
            pass
        last_char = 0
        if len(qual) != len(seq):
            return records  # -2: truncated quality
        records.append(bytes(seq))


def records_to_arrays(records):
    """Concatenate records with a '\\n' separator; return (seq u8 array, rec_off u64, rec_len u64)."""
    off = np.zeros(len(records), dtype=np.uint64)
    ln = np.zeros(len(records), dtype=np.uint64)
    parts = []
    p = 0
    for i, r in enumerate(records):
        off[i] = p
        ln[i] = len(r)
        parts.append(r)
        parts.append(b"\n")
        p += len(r) + 1
    seq = np.frombuffer(b"".join(parts) if parts else b"\n", dtype=np.uint8).copy()
    return seq, off, ln


# ----------------------------------------------------------------------------------------------------
def count_kmers(seq, rec_off, rec_len, k: int, complements: bool):
    """-> (keys [n, limbs] u64, vals [n] u8) sorted by key; vals = min(occurrences-1, 255)."""
    L = limbs_for_k(k)
    seq = np.ascontiguousarray(seq, dtype=np.uint8)
    rec_off = np.ascontiguousarray(rec_off, dtype=np.uint64)
    rec_len = np.ascontiguousarray(rec_len, dtype=np.uint64)
    keys, vals, n = u64p(), u8p(), C.c_uint64()
    rc = lib().orc_count_kmers(_ptr(seq, u8p), _ptr(rec_off, u64p), _ptr(rec_len, u64p), len(rec_off), k,
                               int(complements), C.byref(keys), C.byref(vals), C.byref(n))
    assert rc == 0
    nn = n.value
    return _take(keys, nn * L, np.uint64).reshape(nn, L), _take(vals, nn, np.uint8)


def partial_presort(kmers, k: int):
    """PartialPreSort (reference src/global_sparse.h:14-35): stable counting sort of [n, limbs] u64 k-mers on their top
    min(2k, 8) bits."""
    kmers = np.ascontiguousarray(kmers, dtype=np.uint64).reshape(-1, limbs_for_k(k))
    sfb = min(2 * k, 8)
    pos = 2 * k - sfb
    limb, off = pos >> 6, pos & 63
    v = kmers[:, limb] >> np.uint64(off)
    if off + sfb > 64 and limb + 1 < kmers.shape[1]:
        v = v | (kmers[:, limb + 1] << np.uint64(64 - off))
    digit = (v & np.uint64((1 << sfb) - 1)).astype(np.int64)
    return kmers[np.argsort(digit, kind="stable")]


def _mix64(x):
    x = x ^ (x >> np.uint64(30))
    x = x * np.uint64(0xbf58476d1ce4e5b9)
    x = x ^ (x >> np.uint64(27))
    x = x * np.uint64(0x94d049bb133111eb)
    return x ^ (x >> np.uint64(31))


def kmer_digest(keys, vals, min_frequency: int = 1):
    """[n, sum h, xor h, sum h * c] mod 2^64 over the (key, val) pairs with val + 1 >= min_frequency, c = val + 1 with
    min_frequency > 1 and 1 otherwise (the reference keeps no counts without -z) —
    the digest of oracle/ref_harness.cpp `full` (kmer_digest there) and of the product's kc_kmer_digest.  numpy, wrapping."""
    keys = np.ascontiguousarray(keys, dtype=np.uint64)
    keys = keys.reshape(len(keys), -1)
    vals = np.asarray(vals, dtype=np.uint64)
    keep = vals + np.uint64(1) >= np.uint64(min_frequency)
    keys, vals = keys[keep], vals[keep]
    c = np.uint64(0x9e3779b97f4a7c15)
    with np.errstate(over="ignore"):
        h = _mix64(keys[:, 0] + c)
        for i in range(1, keys.shape[1]):
            h = _mix64(h ^ (keys[:, i] + c * np.uint64(i + 1)))
        return [int(len(h)), int(h.sum(dtype=np.uint64)), int(np.bitwise_xor.reduce(h)) if len(h) else 0,
                int((h * (vals + np.uint64(1)) if min_frequency > 1 else h).sum(dtype=np.uint64))]


def overlap_path(first, last, k: int, complements: bool, lower_bound: bool = False, parts: int = 16):
    """first/last: [n, limbs] u64 -> (edge_from [N] i64, overlaps [N] u8).  parts = number of prefix batches: 16 is the
    reference, 1 the product's from-FASTA engine (engine.cuh with strict = false)."""
    first = np.ascontiguousarray(first, dtype=np.uint64)
    last = np.ascontiguousarray(last, dtype=np.uint64)
    n = first.shape[0]
    N = n * (2 if complements else 1)
    ef = np.zeros(N, dtype=np.int64)
    ov = np.zeros(N, dtype=np.uint8)
    if parts == 16:
        rc = lib().orc_overlap_path(_ptr(first, u64p), _ptr(last, u64p), n, k, int(complements), int(lower_bound),
                                    _ptr(ef, i64p), _ptr(ov, u8p))
    else:
        rc = lib().orc_overlap_path_parts(_ptr(first, u64p), _ptr(last, u64p), n, k, int(complements), int(lower_bound),
                                          int(parts), _ptr(ef, i64p), _ptr(ov, u8p))
    assert rc == 0, rc
    return ef, ov


def superstring(seq, rec_off, rec_len, k, complements, edge_from, overlaps, set_keys=None):
    seq = np.ascontiguousarray(seq, dtype=np.uint8)
    rec_off = np.ascontiguousarray(rec_off, dtype=np.uint64)
    rec_len = np.ascontiguousarray(rec_len, dtype=np.uint64)
    ef = np.ascontiguousarray(edge_from, dtype=np.int64)
    ov = np.ascontiguousarray(overlaps, dtype=np.uint8)
    ms, mo, ln = u8p(), u8p(), C.c_uint64()
    if set_keys is not None:
        sk = np.ascontiguousarray(set_keys, dtype=np.uint64)
        rc = lib().orc_superstring(_ptr(seq, u8p), _ptr(rec_off, u64p), _ptr(rec_len, u64p), len(rec_off), k,
                                   int(complements), _ptr(ef, i64p), _ptr(ov, u8p), _ptr(sk, u64p), sk.shape[0],
                                   C.byref(ms), C.byref(mo), C.byref(ln))
    else:
        rc = lib().orc_superstring(_ptr(seq, u8p), _ptr(rec_off, u64p), _ptr(rec_len, u64p), len(rec_off), k,
                                   int(complements), _ptr(ef, i64p), _ptr(ov, u8p), None, 0, C.byref(ms), None,
                                   C.byref(ln))
    assert rc == 0, rc
    out = _take(ms, ln.value, np.uint8).tobytes()
    if set_keys is not None:
        return out, _take(mo, ln.value, np.uint8).tobytes()
    return out, None


def compute_from_simplitigs(records, k: int, complements: bool, want_maxone: bool = False):
    """`kmercamel compute -S` on a list of record byte strings -> (ms bytes, maxone bytes | None)."""
    seq, off, ln = records_to_arrays(records)
    ms, mo, n = u8p(), u8p(), C.c_uint64()
    rc = lib().orc_compute_from_simplitigs(_ptr(seq, u8p), _ptr(off, u64p), _ptr(ln, u64p), len(records), k,
                                           int(complements), int(want_maxone), C.byref(ms), C.byref(mo), C.byref(n))
    if rc != 0:
        raise ValueError(f"oracle compute_from_simplitigs failed: {rc}")
    out = _take(ms, n.value, np.uint8).tobytes()
    return out, (_take(mo, n.value, np.uint8).tobytes() if want_maxone else None)


def lower_bound_from_simplitigs(records, k: int, complements: bool, parts: int = 16) -> int:
    """`kmercamel lowerbound -S` (reference src/lower_bound.h:9-22 LowerBoundLength): cycle cover of the records as
    nodes, (sum of lengths over the strands - sum of overlaps) / strands."""
    first = np.stack([kmer_from_string(r[:k].decode(), k) for r in records])
    last = np.stack([kmer_from_string(r[len(r) - k:].decode(), k) for r in records])
    _, ov = overlap_path(first, last, k, complements, lower_bound=True, parts=parts)
    strands = 2 if complements else 1
    return (sum(len(r) for r in records) * strands - int(ov.astype(np.int64).sum())) // strands


def first_occurrence_runs(seq, rec_off, rec_len, k: int, complements: bool, min_frequency: int = 1):
    """The from-FASTA nodes of the product (kmercamel_b200/csrc/runs.cuh): maximal runs of consecutive window ends that are the
    first occurrence, in input order, of a kept canonical k-mer -> (run start byte [n] u64, run length [n] u64, kept k-mers)."""
    seq = np.ascontiguousarray(seq, dtype=np.uint8)
    rec_off = np.ascontiguousarray(rec_off, dtype=np.uint64)
    rec_len = np.ascontiguousarray(rec_len, dtype=np.uint64)
    ro, rl, n, kept = u64p(), u64p(), C.c_uint64(), C.c_uint64()
    rc = lib().orc_first_occurrence_runs(_ptr(seq, u8p), _ptr(rec_off, u64p), _ptr(rec_len, u64p), len(rec_off), k,
                                         int(complements), int(min_frequency), C.byref(ro), C.byref(rl), C.byref(n),
                                         C.byref(kept))
    assert rc == 0, rc
    return _take(ro, n.value, np.uint64), _take(rl, n.value, np.uint64), kept.value


_CODES = np.full(256, 4, dtype=np.uint8)
for _i, _c in enumerate(b"ACGT"):
    _CODES[_c] = _CODES[_c + 32] = _i


def window_words(seq, starts, k: int):
    """The k-mer (as read, not canonical) of the k bytes at each start -> [n, limbs] u64; the bytes must be ACGT or acgt."""
    codes = _CODES[np.ascontiguousarray(seq, dtype=np.uint8)]
    starts = np.asarray(starts, dtype=np.int64)
    out = np.zeros((len(starts), limbs_for_k(k)), dtype=np.uint64)
    for i in range(k):
        c = codes[starts + i]
        assert np.all(c < 4), "a node holds a non-ACGT byte"
        bit = 2 * (k - 1 - i)  # base i (0 = leftmost) lies in one limb: 2-bit symbols never straddle a limb boundary
        out[:, bit // 64] |= c.astype(np.uint64) << np.uint64(bit % 64)
    return out


def fasta_nodes(seq, rec_off, rec_len, k: int, complements: bool, min_frequency: int = 1, sparse_switch: bool = True):
    """The nodes the product hands to its overlap stage from FASTA (kcgpu.cu run_tail) -> (node start [n] u64,
    node length [n] u64, kept k-mers, first-occurrence runs).  The runs, unless there are at least U / 5 of them (the sparse
    switch, reference src/main.cpp:94,175-181): then one node per k-mer of the runs, in run order and in the orientation it has
    in the input, stably sorted on its first min(k, 4) bases (PartialPreSort, src/global_sparse.h:14-35)."""
    off, ln, kept = first_occurrence_runs(seq, rec_off, rec_len, k, complements, min_frequency)
    n_runs = len(off)
    if kept == 0:
        raise ValueError("the input contains no k-mers")
    if sparse_switch and n_runs * 5 >= kept:
        cnt = (ln - np.uint64(k - 1)).astype(np.int64)
        base = np.repeat(off.astype(np.int64), cnt)
        within = np.arange(int(cnt.sum())) - np.repeat(np.cumsum(cnt) - cnt, cnt)
        starts = base + within
        nb = min(k, 4)
        codes = _CODES[np.ascontiguousarray(seq, dtype=np.uint8)].astype(np.int64)
        digit = np.zeros(len(starts), dtype=np.int64)
        for j in range(nb):
            digit = (digit << 2) | codes[starts + j]
        starts = starts[np.argsort(digit, kind="stable")]
        off = starts.astype(np.uint64)
        ln = np.full(len(starts), k, dtype=np.uint64)
    return off, ln, kept, n_runs


def compute_from_fasta(seq, rec_off, rec_len, k: int, complements: bool, min_frequency: int = 1, want_maxone: bool = False,
                       sparse_switch: bool = True):
    """The product's `compute` from FASTA, restated: fasta_nodes, then the greedy with one prefix batch (overlap_path
    parts = 1, the engine's non-strict tie order), then the emission of the reference.  seq / rec_off / rec_len: framed
    records (records_to_arrays, synth.frame_records).  -> dict(ms, maxone, n_kmers, n_nodes, n_simplitigs)."""
    seq = np.ascontiguousarray(seq, dtype=np.uint8)
    off, ln, kept, n_runs = fasta_nodes(seq, rec_off, rec_len, k, complements, min_frequency, sparse_switch)
    first = window_words(seq, off, k)
    last = window_words(seq, off + ln - np.uint64(k), k)
    ef, ov = overlap_path(first, last, k, complements, parts=1)
    set_keys = None
    if want_maxone:
        keys, vals = count_kmers(seq, rec_off, rec_len, k, complements)
        set_keys = keys[vals.astype(np.int64) + 1 >= min_frequency]
    ms, mo = superstring(seq, off, ln, k, complements, ef, ov, set_keys)
    return dict(ms=ms, maxone=mo, n_kmers=kept, n_nodes=len(off), n_simplitigs=n_runs)


def lower_bound_from_fasta(seq, rec_off, rec_len, k: int, complements: bool, min_frequency: int = 1,
                           sparse_switch: bool = True) -> int:
    """The product's `lowerbound` from FASTA, restated: the cycle cover (overlap_path lower_bound = True, parts = 1) of the
    nodes of fasta_nodes, (sum of lengths over the strands - sum of overlaps) / strands (src/lower_bound.h:9-22)."""
    seq = np.ascontiguousarray(seq, dtype=np.uint8)
    off, ln, _, _ = fasta_nodes(seq, rec_off, rec_len, k, complements, min_frequency, sparse_switch)
    _, ov = overlap_path(window_words(seq, off, k), window_words(seq, off + ln - np.uint64(k), k), k, complements,
                         lower_bound=True, parts=1)
    assert not np.any(ov == 255)  # a cycle cover: every node has a successor
    strands = 2 if complements else 1
    return (int(ln.astype(np.int64).sum()) * strands - int(ov.astype(np.int64).sum())) // strands


def ms_kmers(ms: bytes, k: int, complements: bool):
    """-> (sorted unique ON k-mers [n, limbs] u64, number of ON positions)."""
    L = limbs_for_k(k)
    a = np.frombuffer(ms, dtype=np.uint8).copy() if len(ms) else np.zeros(1, dtype=np.uint8)
    keys, n, n_on = u64p(), C.c_uint64(), C.c_uint64()
    rc = lib().orc_ms_kmers(_ptr(a, u8p), len(ms), k, int(complements), C.byref(keys), C.byref(n), C.byref(n_on))
    assert rc == 0
    return _take(keys, n.value * L, np.uint64).reshape(n.value, L), n_on.value


def verify_ms(ms: bytes, k: int, complements: bool, expected_keys) -> bool:
    """verify.py's acceptance test: the ON k-mers of `ms` are exactly `expected_keys` (sorted unique)."""
    got, _ = ms_kmers(ms, k, complements)
    exp = np.ascontiguousarray(expected_keys, dtype=np.uint64).reshape(-1, limbs_for_k(k))
    return got.shape == exp.shape and bool(np.array_equal(got, exp))


def streaming(seq, rec_off, rec_len, k: int, complements: bool, min_frequency: int = 1) -> bytes:
    """`kmercamel compute -a streaming [-z]` (reference src/streaming.h:12-107) over framed records -> sequence line."""
    seq = np.ascontiguousarray(seq, dtype=np.uint8)
    rec_off = np.ascontiguousarray(rec_off, dtype=np.uint64)
    rec_len = np.ascontiguousarray(rec_len, dtype=np.uint64)
    out, n = u8p(), C.c_uint64()
    rc = lib().orc_streaming(_ptr(seq, u8p), _ptr(rec_off, u64p), _ptr(rec_len, u64p), len(rec_off), k, int(complements),
                             int(min_frequency), C.byref(out), C.byref(n))
    assert rc == 0, rc
    return _take(out, n.value, np.uint8).tobytes()


def maskopt(ms: bytes, k: int, complements: bool, minimize: bool) -> bytes:
    """`kmercamel maskopt -t min-one|max-one` (reference src/masks.h:40-78,240-261) on the sequence of one record."""
    a = np.frombuffer(ms, dtype=np.uint8).copy() if len(ms) else np.zeros(1, dtype=np.uint8)
    out = np.zeros(max(len(ms), 1), dtype=np.uint8)
    rc = lib().orc_maskopt(_ptr(a, u8p), len(ms), k, int(complements), int(minimize), _ptr(out, u8p))
    if rc != 0:
        raise ValueError("Masked superstring contains invalid characters.")
    return out[:len(ms)].tobytes()


# reference src/conversions.h, restated in pure Python (small inputs)
def _is_upper(c: int) -> bool:  # src/conversions.h:6-8
    return c <= ord("Z")


def _masked(c: int, mask: bool) -> int:  # src/kmers.h:124-127
    return c + (int(c <= ord("Z")) - int(mask)) * 32


def split_ms(ms: bytes):
    """src/conversions.h:16-33 -> (superstring, mask) without the trailing newlines."""
    return bytes(c if _is_upper(c) else c - 32 for c in ms), bytes(ord("1") if _is_upper(c) else ord("0") for c in ms)


def join_ms(superstring: bytes, mask: bytes) -> bytes:
    """src/conversions.h:35-44, the text after the header line."""
    return bytes(_masked(c, i < len(mask) and mask[i] == ord("1")) for i, c in enumerate(superstring))


def ms_to_spss(ms: bytes, k: int) -> bytes:
    """src/conversions.h:46-72, the complete output text."""
    out = bytearray()
    masked, counter, l = False, 0, len(ms)
    for i in range(l):
        if _is_upper(ms[i]):
            if not masked:
                out += b">%d\n" % counter
                counter += 1
            masked = True
            out.append(ms[i])
        else:
            if not masked:
                continue
            masked = False
            for j in range(k - 1):
                if i + j < l:
                    c = ms[i + j]
                    out.append(c if _is_upper(c) else c - 32)
            out += b"\n"
    return bytes(out)


def spss_to_ms(records, k: int) -> bytes:
    """src/conversions.h:74-91, the text after the header line."""
    out = bytearray()
    for r in records:
        l = len(r)
        if l < k:
            continue
        out += bytes(_masked(c, i <= l - k) for i, c in enumerate(r))
    return bytes(out)


def kmer_from_string(s: str, k: int | None = None):
    """ASCII k-mer -> limbs (little-endian u64), the layout of reference src/ac/kmers_ac.h:47-54 KMerToNumber."""
    k = len(s) if k is None else k
    v = 0
    for ch in s:
        v = (v << 2) | "ACGT".index(ch.upper())
    L = limbs_for_k(k)
    return np.array([(v >> (64 * i)) & 0xFFFFFFFFFFFFFFFF for i in range(L)], dtype=np.uint64)


def kmer_to_int(limbs) -> int:
    return sum(int(x) << (64 * i) for i, x in enumerate(limbs))


def reverse_complement(limbs, k):
    a = np.ascontiguousarray(limbs, dtype=np.uint64)
    out = np.zeros_like(a)
    lib().orc_reverse_complement(_ptr(a, u64p), k, _ptr(out, u64p))
    return out


def bit_prefix(limbs, k, d):
    a = np.ascontiguousarray(limbs, dtype=np.uint64)
    out = np.zeros_like(a)
    lib().orc_bit_prefix(_ptr(a, u64p), k, d, _ptr(out, u64p))
    return out


def bit_suffix(limbs, k, d):
    a = np.ascontiguousarray(limbs, dtype=np.uint64)
    out = np.zeros_like(a)
    lib().orc_bit_suffix(_ptr(a, u64p), k, d, _ptr(out, u64p))
    return out
