"""ctypes binding of include/kcgpu.h.

Mirrors the reference's call sequence for `compute` (reference src/main.cpp:122-212): ReadKMers[Filtered] ->
get_simplitigs | simplitigs_from_fasta -> Global/GlobalSparse, exposed as Context.compute(); the stage entry points
Context.count_kmers() and Context.overlap_path() exist so that parity tests can hit each stage.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

u8p = C.POINTER(C.c_uint8)
u64p = C.POINTER(C.c_uint64)
i64p = C.POINTER(C.c_int64)

ERRORS = {0: "KC_OK", -1: "KC_ERR_CUDA", -2: "KC_ERR_ARG", -3: "KC_ERR_OOM", -4: "KC_ERR_EMPTY", -5: "KC_ERR_BAD_SEQ",
          -6: "KC_ERR_TOO_LARGE", -7: "KC_ERR_INTERNAL", -8: "KC_ERR_NO_DEVICE"}


class KcError(RuntimeError):
    def __init__(self, code: int, detail: str = ""):
        self.code = code
        self.name = ERRORS.get(code, str(code))
        super().__init__(f"{self.name}: {detail}" if detail else self.name)


class kc_params(C.Structure):
    _fields_ = [("k", C.c_int), ("complements", C.c_int), ("min_frequency", C.c_int), ("assume_simplitigs", C.c_int),
                ("want_maxone", C.c_int)]


class kc_input(C.Structure):
    _fields_ = [("seq", C.c_void_p), ("n_bytes", C.c_uint64), ("rec_off", C.c_void_p), ("rec_len", C.c_void_p),
                ("n_recs", C.c_uint64)]


class kc_stage_times(C.Structure):
    _fields_ = [("extract_ms", C.c_float), ("count_ms", C.c_float), ("path_ms", C.c_float), ("emit_ms", C.c_float),
                ("total_ms", C.c_float)]


class kc_output(C.Structure):
    _fields_ = [("ms", C.c_void_p), ("ms_maxone", C.c_void_p), ("length", C.c_uint64), ("n_kmers", C.c_uint64),
                ("n_occurrences", C.c_uint64), ("n_nodes", C.c_uint64), ("n_launches", C.c_uint64), ("n_simplitigs", C.c_uint64), ("t", kc_stage_times)]


def lib_path() -> str:
    return os.path.join(_HERE, "csrc", "libkcgpu.so")


def load_library():
    """Load libkcgpu.so.  There is no fallback: a missing library is an error."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if not os.path.exists(path):
        raise ImportError(f"{path} is missing: build it with `make` (or __graft_entry__.build()); "
                          "kmercamel_b200 has no CPU fallback")
    L = C.CDLL(path)
    L.kc_init.argtypes = [C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]
    L.kc_destroy.argtypes = [C.c_void_p]
    L.kc_destroy.restype = None
    L.kc_compute.argtypes = [C.c_void_p, C.POINTER(kc_params), C.POINTER(kc_input), C.POINTER(kc_output)]
    L.kc_compute_device.argtypes = [C.c_void_p, C.POINTER(kc_params), C.POINTER(kc_input), C.POINTER(kc_output)]
    L.kc_lower_bound.argtypes = [C.c_void_p, C.POINTER(kc_params), C.POINTER(kc_input), u64p, C.POINTER(kc_output)]
    L.kc_copy_to_host.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]
    L.kc_streaming.argtypes = [C.c_void_p, C.POINTER(kc_params), C.POINTER(kc_input), C.POINTER(kc_output)]
    L.kc_maskopt.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_int, C.c_int, C.POINTER(kc_output)]
    L.kc_split_ms.argtypes = [C.c_char_p, C.c_uint64, C.POINTER(u8p), C.POINTER(u8p)]
    L.kc_join_ms.argtypes = [C.c_char_p, C.c_uint64, C.c_char_p, C.c_uint64, C.POINTER(u8p), u64p]
    L.kc_ms_to_spss.argtypes = [C.c_char_p, C.c_uint64, C.c_int, C.POINTER(u8p), u64p]
    L.kc_spss_to_ms.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.POINTER(u8p), u64p]
    L.kc_fasta_first_header.argtypes = [C.c_char_p, C.c_uint64, u64p]
    L.kc_count_kmers.argtypes = [C.c_void_p, C.POINTER(kc_params), C.POINTER(kc_input), C.POINTER(u64p), C.POINTER(u8p),
                                 u64p]
    L.kc_partial_presort.argtypes = [C.c_void_p, u64p, C.c_uint64, C.c_int, u64p]
    L.kc_debug_sort.argtypes = [C.c_void_p, u64p, C.c_uint64, C.c_int, C.c_int, u64p, u64p]
    L.kc_kmer_digest.argtypes = [C.c_void_p, C.POINTER(kc_params), C.POINTER(kc_input), C.c_int, u64p]
    L.kc_overlap_path.argtypes = [C.c_void_p, u64p, u64p, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_int, i64p, u8p]
    L.kc_frame_fasta.argtypes = [C.c_char_p, C.c_uint64, C.POINTER(u8p), u64p, C.POINTER(u64p), C.POINTER(u64p), u64p]
    L.kc_shard_granule.argtypes = [C.c_int]
    L.kc_shard_granule.restype = C.c_uint64
    L.kc_init_multi.argtypes = [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_void_p)]
    L.kc_group_destroy.argtypes = [C.c_void_p]
    L.kc_group_destroy.restype = None
    L.kc_group_size.argtypes = [C.c_void_p]
    L.kc_group_ctx.argtypes = [C.c_void_p, C.c_int]
    L.kc_group_ctx.restype = C.c_void_p
    L.kc_group_compute.argtypes = [C.c_void_p, C.POINTER(kc_params), C.POINTER(kc_input), C.POINTER(kc_output)]
    L.kc_group_last_error.argtypes = [C.c_void_p]
    L.kc_group_last_error.restype = C.c_char_p
    L.kc_group_alloc.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_void_p]
    L.kc_group_open.argtypes = [C.c_void_p, C.c_void_p]
    L.kc_group_compute_device.argtypes = [C.c_void_p, C.POINTER(kc_params), C.POINTER(kc_input), C.POINTER(kc_output), u64p, u64p]
    L.kc_group_close.argtypes = [C.c_void_p]
    L.kc_group_plan.argtypes = [C.c_int, C.c_int, C.c_int, C.c_uint64, u64p]
    L.kc_total_launches.argtypes = [C.c_void_p]
    L.kc_total_launches.restype = C.c_uint64
    L.kc_set_option.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
    L.kc_get_stat.argtypes = [C.c_void_p, C.c_char_p, C.POINTER(C.c_uint64)]
    L.kc_get_stat.restype = C.c_int
    L.kc_profile_enable.argtypes = [C.c_void_p, C.c_int]
    L.kc_profile_count.restype = C.c_int
    L.kc_profile_get.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_double), u64p, u64p]
    L.kc_profile_reset.argtypes = [C.c_void_p]
    L.kc_limbs_for_k.argtypes = [C.c_int]
    L.kc_free.argtypes = [C.c_void_p]
    L.kc_free.restype = None
    L.kc_strerror.argtypes = [C.c_int]
    L.kc_strerror.restype = C.c_char_p
    L.kc_last_error.argtypes = [C.c_void_p]
    L.kc_last_error.restype = C.c_char_p
    _LIB = L
    return L


EXPORTED_SYMBOLS = ["kc_kmer_digest", "kc_partial_presort", "kc_debug_sort", "kc_init", "kc_destroy", "kc_compute", "kc_compute_device", "kc_lower_bound",
                    "kc_copy_to_host", "kc_count_kmers", "kc_overlap_path", "kc_total_launches", "kc_shard_granule",
                    "kc_init_multi", "kc_group_destroy", "kc_group_size", "kc_group_ctx", "kc_group_compute", "kc_group_last_error",
                    "kc_group_alloc", "kc_group_open", "kc_group_compute_device", "kc_group_close", "kc_group_plan",
                    "kc_streaming", "kc_maskopt", "kc_split_ms", "kc_join_ms", "kc_ms_to_spss", "kc_spss_to_ms", "kc_fasta_first_header",
                    "kc_frame_fasta", "kc_set_option", "kc_get_stat", "kc_profile_enable", "kc_profile_count", "kc_profile_get", "kc_profile_reset",
                    "kc_limbs_for_k", "kc_free", "kc_strerror", "kc_last_error"]


def limbs_for_k(k: int) -> int:
    return 1 if k < 32 else (2 if k < 64 else 4)


def _take(ptr, n, dtype):
    out = np.ctypeslib.as_array(ptr, shape=(max(n, 1),))[:n].astype(dtype, copy=True)
    load_library().kc_free(C.cast(ptr, C.c_void_p))
    return out


def frame_fasta(data: bytes):
    """FASTA/FASTQ bytes -> (seq u8, rec_off u64, rec_len u64) with kseq semantics (host only, no GPU needed)."""
    L = load_library()
    seq, off, ln = u8p(), u64p(), u64p()
    nb, nr = C.c_uint64(), C.c_uint64()
    rc = L.kc_frame_fasta(data, len(data), C.byref(seq), C.byref(nb), C.byref(off), C.byref(ln), C.byref(nr))
    if rc != 0:
        raise KcError(rc)
    return _take(seq, nb.value, np.uint8), _take(off, nr.value, np.uint64), _take(ln, nr.value, np.uint64)


def frame_fasta_file(path: str):
    import gzip
    with open(path, "rb") as f:
        data = f.read()
    if data[:2] == b"\x1f\x8b":
        data = gzip.decompress(data)
    return frame_fasta(data)


# ---- host-only text conversions (reference src/conversions.h) -------------------------------------------------------
def split_ms(ms: bytes):
    """`ms2mssep` (src/conversions.h:16-33) -> (superstring in upper case, mask as b'0'/b'1' characters)."""
    L = load_library()
    sup, mask = u8p(), u8p()
    rc = L.kc_split_ms(ms, len(ms), C.byref(sup), C.byref(mask))
    if rc != 0:
        raise KcError(rc)
    return _take(sup, len(ms), np.uint8).tobytes(), _take(mask, len(ms), np.uint8).tobytes()


def join_ms(superstring: bytes, mask: bytes) -> bytes:
    """`mssep2ms` (src/conversions.h:35-44): the sequence line."""
    L = load_library()
    out, n = u8p(), C.c_uint64()
    rc = L.kc_join_ms(superstring, len(superstring), mask, len(mask), C.byref(out), C.byref(n))
    if rc != 0:
        raise KcError(rc)
    return _take(out, n.value, np.uint8).tobytes()


def ms_to_spss(ms: bytes, k: int) -> bytes:
    """`ms2spss` (src/conversions.h:46-72): the complete FASTA text."""
    L = load_library()
    out, n = u8p(), C.c_uint64()
    rc = L.kc_ms_to_spss(ms, len(ms), k, C.byref(out), C.byref(n))
    if rc != 0:
        raise KcError(rc)
    return _take(out, n.value, np.uint8).tobytes()


def spss_to_ms(seq, rec_off, rec_len, k: int) -> bytes:
    """`spss2ms` (src/conversions.h:74-91) on framed records: the sequence line."""
    L = load_library()
    seq = np.ascontiguousarray(seq, dtype=np.uint8)
    rec_off = np.ascontiguousarray(rec_off, dtype=np.uint64)
    rec_len = np.ascontiguousarray(rec_len, dtype=np.uint64)
    out, n = u8p(), C.c_uint64()
    rc = L.kc_spss_to_ms(seq.ctypes.data, rec_off.ctypes.data, rec_len.ctypes.data, len(rec_off), k, C.byref(out), C.byref(n))
    if rc != 0:
        raise KcError(rc)
    return _take(out, n.value, np.uint8).tobytes()


def fasta_first_header(data: bytes):
    """-> (name, comment | None) of the first record as kseq parses the header line."""
    L = load_library()
    span = (C.c_uint64 * 5)()
    rc = L.kc_fasta_first_header(data, len(data), span)
    if rc != 0:
        raise KcError(rc)
    name = data[span[0]:span[0] + span[1]]
    return name, (data[span[3]:span[3] + span[4]] if span[2] else None)


@dataclass
class ComputeResult:
    ms: bytes | None
    maxone: bytes | None
    length: int
    n_kmers: int
    n_occurrences: int
    n_nodes: int
    n_launches: int
    n_simplitigs: int = 0
    times_ms: dict = field(default_factory=dict)
    ms_ptr: int = 0        # device pointers for compute_device
    maxone_ptr: int = 0
    slice_begin: int = 0   # compute_from_flags(..., slice=(i, n)): ms_ptr holds bytes [slice_begin, slice_begin + slice_len)
    slice_len: int = 0     # of the superstring (length = the whole superstring)


def _string_at(ptr, n: int) -> bytes:
    """n bytes at host address ptr.  ctypes.string_at passes its length as a C int, which cuts results of 2^31 bytes and more."""
    return bytes((C.c_char * n).from_address(ptr)) if n else b""


class Context:
    """One context per process and GPU (kc_init / kc_destroy)."""

    def __init__(self, device: int = 0, stream: int | None = None):
        """stream: a cudaStream_t handle to run on (e.g. torch.cuda.current_stream().cuda_stream), None = a private
        non-blocking stream.  Handle 0 is the legacy default stream (what torch uses unless told otherwise): it is passed as
        cudaStreamLegacy, so the library's kernels are ordered with the caller's work on that stream (NULL would mean "private")."""
        self._lib = load_library()
        self._h = C.c_void_p()
        self.stream_handle = None if stream is None else int(stream)  # as given by the caller (0 = legacy default stream)
        if stream is not None and int(stream) == 0:
            stream = 1  # cudaStreamLegacy
        rc = self._lib.kc_init(device, C.c_void_p(stream) if stream else None, C.byref(self._h))
        if rc != 0:
            raise KcError(rc, "kc_init")

    def close(self):
        if self._h:
            self._lib.kc_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise KcError(rc, self._lib.kc_last_error(self._h).decode())

    @staticmethod
    def _params(k, complements, min_frequency, assume_simplitigs, want_maxone):
        return kc_params(int(k), int(bool(complements)), int(min_frequency), int(bool(assume_simplitigs)),
                         int(bool(want_maxone)))

    def _result(self, out, copy_host: bool):
        t = out.t
        times = dict(extract=t.extract_ms, count=t.count_ms, path=t.path_ms, emit=t.emit_ms, total=t.total_ms)
        ms = mo = None
        if copy_host:
            ms = _string_at(out.ms, out.length)
            mo = _string_at(out.ms_maxone, out.length) if out.ms_maxone else None
        return ComputeResult(ms, mo, out.length, out.n_kmers, out.n_occurrences, out.n_nodes, out.n_launches, out.n_simplitigs, times,
                             out.ms or 0, out.ms_maxone or 0)

    def compute(self, seq, rec_off=None, rec_len=None, *, k, complements=True, min_frequency=1, assume_simplitigs=False,
                want_maxone=False, copy=True) -> ComputeResult:
        """`kmercamel compute` on framed host buffers (H2D + all stages + D2H)."""
        seq = np.ascontiguousarray(seq, dtype=np.uint8)
        n_recs = 0 if rec_off is None else len(rec_off)
        if rec_off is not None:
            rec_off = np.ascontiguousarray(rec_off, dtype=np.uint64)
            rec_len = np.ascontiguousarray(rec_len, dtype=np.uint64)
        p = self._params(k, complements, min_frequency, assume_simplitigs, want_maxone)
        inp = kc_input(seq.ctypes.data, seq.size, rec_off.ctypes.data if n_recs else None,
                       rec_len.ctypes.data if n_recs else None, n_recs)
        out = kc_output()
        self._check(self._lib.kc_compute(self._h, C.byref(p), C.byref(inp), C.byref(out)))
        return self._result(out, copy)

    def lower_bound(self, seq, rec_off=None, rec_len=None, *, k, complements=True, min_frequency=1, assume_simplitigs=False):
        """`kmercamel lowerbound` (reference src/lower_bound.h:9-22): -> (cycle-cover lower bound, ComputeResult stats)."""
        seq = np.ascontiguousarray(seq, dtype=np.uint8)
        n_recs = 0 if rec_off is None else len(rec_off)
        if rec_off is not None:
            rec_off = np.ascontiguousarray(rec_off, dtype=np.uint64)
            rec_len = np.ascontiguousarray(rec_len, dtype=np.uint64)
        p = self._params(k, complements, min_frequency, assume_simplitigs, False)
        inp = kc_input(seq.ctypes.data, seq.size, rec_off.ctypes.data if n_recs else None,
                       rec_len.ctypes.data if n_recs else None, n_recs)
        out = kc_output()
        lb = C.c_uint64()
        self._check(self._lib.kc_lower_bound(self._h, C.byref(p), C.byref(inp), C.byref(lb), C.byref(out)))
        return lb.value, self._result(out, False)

    def streaming(self, seq, *, k, complements=True, min_frequency=1, copy=True) -> ComputeResult:
        """`kmercamel compute -a streaming [-z]` (reference src/streaming.h:12-107) on framed host buffers."""
        seq = np.ascontiguousarray(seq, dtype=np.uint8)
        p = self._params(k, complements, min_frequency, False, False)
        inp = kc_input(seq.ctypes.data, seq.size, None, None, 0)
        out = kc_output()
        self._check(self._lib.kc_streaming(self._h, C.byref(p), C.byref(inp), C.byref(out)))
        return self._result(out, copy)

    def maskopt(self, ms, *, k, complements=True, minimize=False, copy=True) -> ComputeResult:
        """`kmercamel maskopt -t max-one|min-one` (reference src/masks.h:40-78,240-261) on one record's sequence
        (bytes, or a uint8 numpy array, e.g. a view of pinned memory)."""
        out = kc_output()
        if isinstance(ms, (bytes, bytearray)):
            ptr, n = C.cast(C.c_char_p(bytes(ms)), C.c_void_p), len(ms)
        else:
            ms = np.ascontiguousarray(ms, dtype=np.uint8)
            ptr, n = C.c_void_p(ms.ctypes.data), ms.size
        self._check(self._lib.kc_maskopt(self._h, ptr, n, int(k), int(bool(complements)), int(bool(minimize)), C.byref(out)))
        return self._result(out, copy)

    def compute_device(self, seq_ptr: int, n_bytes: int, rec_off_ptr: int = 0, rec_len_ptr: int = 0, n_recs: int = 0, *, k,
                       complements=True, min_frequency=1, assume_simplitigs=False, want_maxone=False) -> ComputeResult:
        """Same with device pointers in and out (results stay in the context arena until the next call)."""
        p = self._params(k, complements, min_frequency, assume_simplitigs, want_maxone)
        inp = kc_input(seq_ptr, n_bytes, rec_off_ptr or None, rec_len_ptr or None, n_recs)
        out = kc_output()
        self._check(self._lib.kc_compute_device(self._h, C.byref(p), C.byref(inp), C.byref(out)))
        return self._result(out, False)

    def copy_to_host(self, device_ptr: int, n: int) -> bytes:
        buf = C.create_string_buffer(max(n, 1))
        self._check(self._lib.kc_copy_to_host(self._h, buf, C.c_void_p(device_ptr), n))
        return buf.raw[:n]

    def count_kmers(self, seq, *, k, complements=True, min_frequency=1):
        """Stage 1: -> (keys [n, limbs] u64 ascending, counts [n] u8 = min(occurrences-1, 255))."""
        seq = np.ascontiguousarray(seq, dtype=np.uint8)
        p = self._params(k, complements, min_frequency, False, False)
        inp = kc_input(seq.ctypes.data, seq.size, None, None, 0)
        keys, cnt, n = u64p(), u8p(), C.c_uint64()
        self._check(self._lib.kc_count_kmers(self._h, C.byref(p), C.byref(inp), C.byref(keys), C.byref(cnt), C.byref(n)))
        L = limbs_for_k(k)
        return _take(keys, n.value * L, np.uint64).reshape(n.value, L), _take(cnt, n.value, np.uint8)

    def partial_presort(self, kmers, *, k):
        """PartialPreSort (reference src/global_sparse.h:14-35): kmers [n, limbs] u64 -> reordered copy."""
        kmers = np.ascontiguousarray(kmers, dtype=np.uint64).reshape(-1, limbs_for_k(k))
        out = np.zeros_like(kmers)
        self._check(self._lib.kc_partial_presort(self._h, kmers.ctypes.data_as(u64p), kmers.shape[0], int(k), out.ctypes.data_as(u64p)))
        return out

    def debug_sort(self, words, key_bits: int):
        """Test hook kc_debug_sort: the radix sort of sort.cuh on words [n, limbs] u64 (limbs 1, 2, 3 or 5), ascending on their
        low key_bits bits -> (sorted copy, stats).  stats: levels (radix levels run), max_big (most buckets partitioned in one
        level), small (buckets sorted in shared memory), uniform (buckets that ran out of key bits), whole_bitonic (shared-memory
        buckets sorted whole by the bitonic network)."""
        words = np.ascontiguousarray(words, dtype=np.uint64)
        out = np.zeros_like(words)
        st = np.zeros(5, dtype=np.uint64)
        self._check(self._lib.kc_debug_sort(self._h, words.ctypes.data_as(u64p), words.shape[0], words.shape[1], int(key_bits),
                                            out.ctypes.data_as(u64p), st.ctypes.data_as(u64p)))
        return out, dict(zip(("levels", "max_big", "small", "uniform", "whole_bitonic"), (int(x) for x in st)))

    def kmer_digest(self, seq, *, k, complements=True, min_frequency=1, masked=False):
        """Stage 1 as an order-independent digest [n, sum h, xor h, sum h * min(occurrences, 256)] (kc_kmer_digest).
        masked=True: `seq` is one masked superstring; the digest is that of the k-mer set it represents."""
        if isinstance(seq, (bytes, bytearray)):
            seq = np.frombuffer(seq, dtype=np.uint8)
        seq = np.ascontiguousarray(seq, dtype=np.uint8)
        p = self._params(k, complements, min_frequency, False, False)
        inp = kc_input(seq.ctypes.data, seq.size, None, None, 0)
        d = (C.c_uint64 * 4)()
        self._check(self._lib.kc_kmer_digest(self._h, C.byref(p), C.byref(inp), int(bool(masked)), d))
        return [int(x) for x in d]

    def overlap_path(self, first, last, *, k, complements=True, lower_bound=False, strict=True):
        """Overlap stage: first/last [n, limbs] u64 -> (edge_from [N] i64, overlaps [N] u8)."""
        first = np.ascontiguousarray(first, dtype=np.uint64)
        last = np.ascontiguousarray(last, dtype=np.uint64)
        n = first.shape[0]
        N = n * (2 if complements else 1)
        ef = np.zeros(N, dtype=np.int64)
        ov = np.zeros(N, dtype=np.uint8)
        self._check(self._lib.kc_overlap_path(self._h, first.ctypes.data_as(u64p), last.ctypes.data_as(u64p), n, k,
                                              int(complements), int(lower_bound), int(strict), ef.ctypes.data_as(i64p),
                                              ov.ctypes.data_as(u8p)))
        return ef, ov

    # ---- multi-GPU: this context as one rank of a group of processes (include/kcgpu.h "multi-GPU", form 2) ---------------
    def group_alloc(self, n_ranks: int, rank: int, k: int, n_bytes_cap: int) -> np.ndarray:
        """Allocate this rank's heap; -> its 64-byte CUDA IPC handle (to be all-gathered by the caller)."""
        h = np.zeros(64, dtype=np.uint8)
        self._check(self._lib.kc_group_alloc(self._h, n_ranks, rank, int(k), int(n_bytes_cap), h.ctypes.data))
        return h

    def group_open(self, all_handles: np.ndarray):
        all_handles = np.ascontiguousarray(all_handles, dtype=np.uint8)
        self._check(self._lib.kc_group_open(self._h, all_handles.ctypes.data))

    def group_compute_device(self, seq_ptr: int, n_bytes: int, *, k, complements=True, min_frequency=1) -> ComputeResult:
        """One sharded job (every rank makes the same call); ms_ptr holds bytes [slice_begin, slice_begin + slice_len) of the
        superstring on this rank's GPU, length is the whole superstring's."""
        p = self._params(k, complements, min_frequency, False, False)
        inp = kc_input(seq_ptr, n_bytes, None, None, 0)
        out = kc_output()
        sb, sl = C.c_uint64(), C.c_uint64()
        self._check(self._lib.kc_group_compute_device(self._h, C.byref(p), C.byref(inp), C.byref(out), C.byref(sb), C.byref(sl)))
        r = self._result(out, False)
        r.slice_begin, r.slice_len = sb.value, sl.value
        return r

    def group_close(self):
        self._lib.kc_group_close(self._h)

    def total_launches(self) -> int:
        return int(self._lib.kc_total_launches(self._h))

    def set_option(self, name: str, value: int):
        self._check(self._lib.kc_set_option(self._h, name.encode(), int(value)))

    def stat(self, name: str) -> int:
        v = C.c_uint64()
        self._check(self._lib.kc_get_stat(self._h, name.encode(), C.byref(v)))
        return int(v.value)

    # ---- per-kernel-class timers ---------------------------------------------------------------------------
    def profile_enable(self, on: bool = True):
        self._lib.kc_profile_enable(self._h, int(on))

    def profile_reset(self):
        self._lib.kc_profile_reset(self._h)

    def profile(self) -> dict:
        out = {}
        for i in range(self._lib.kc_profile_count()):
            name, ms, n, b = C.c_char_p(), C.c_double(), C.c_uint64(), C.c_uint64()
            self._lib.kc_profile_get(self._h, i, C.byref(name), C.byref(ms), C.byref(n), C.byref(b))
            out[name.value.decode()] = dict(ms=ms.value, launches=n.value, bytes=b.value)
        return out


def group_plan(n_ranks: int, rank: int, k: int, n_bytes: int) -> dict:
    """Host-only geometry of a sharded job (kc_group_plan): no GPU needed."""
    pl = (C.c_uint64 * 8)()
    rc = load_library().kc_group_plan(n_ranks, rank, int(k), int(n_bytes), pl)
    if rc != 0:
        raise KcError(rc)
    return dict(fixed_slots=bool(pl[0]), pos_begin=int(pl[1]), pos_end=int(pl[2]), digit_begin=int(pl[3]), digit_end=int(pl[4]),
                n_digits=int(pl[5]), cap_sub=int(pl[6]), heap_bytes=int(pl[7]))


class _RankView(Context):
    """A rank's context inside a Group: owned by the group, never destroyed on its own."""

    def __init__(self, lib, handle):
        self._lib = lib
        self._h = C.c_void_p(handle)
        self.stream_handle = None

    def close(self):
        self._h = C.c_void_p()


class Group:
    """Several GPUs driven from ONE process (kc_init_multi / kc_group_compute): what `kmercamel compute -g 0,1,...` uses.
    A device ordinal may repeat — the ranks then share a GPU, which exercises the whole peer protocol on a one-GPU box."""

    def __init__(self, device_ids):
        self._lib = load_library()
        self._g = C.c_void_p()
        ids = (C.c_int * len(device_ids))(*[int(d) for d in device_ids])
        rc = self._lib.kc_init_multi(len(device_ids), ids, C.byref(self._g))
        if rc != 0:
            raise KcError(rc, "kc_init_multi")
        self.n = len(device_ids)

    def rank(self, r: int) -> Context:
        return _RankView(self._lib, self._lib.kc_group_ctx(self._g, r))

    def set_option(self, name: str, value: int):
        for r in range(self.n):
            self.rank(r).set_option(name, value)

    def stat(self, name: str):
        return [self.rank(r).stat(name) for r in range(self.n)]

    def compute(self, seq, *, k, complements=True, min_frequency=1, copy=True) -> ComputeResult:
        seq = np.ascontiguousarray(seq, dtype=np.uint8)
        p = Context._params(k, complements, min_frequency, False, False)
        inp = kc_input(seq.ctypes.data, seq.size, None, None, 0)
        out = kc_output()
        rc = self._lib.kc_group_compute(self._g, C.byref(p), C.byref(inp), C.byref(out))
        if rc != 0:
            raise KcError(rc, self._lib.kc_group_last_error(self._g).decode())
        t = out.t
        times = dict(extract=t.extract_ms, count=t.count_ms, path=t.path_ms, emit=t.emit_ms, total=t.total_ms)
        ms = _string_at(out.ms, out.length) if copy else None
        return ComputeResult(ms, None, out.length, out.n_kmers, out.n_occurrences, out.n_nodes, out.n_launches, out.n_simplitigs, times,
                             out.ms or 0, 0, 0, out.length)

    def close(self):
        if self._g:
            self._lib.kc_group_destroy(self._g)
            self._g = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
