// Common definitions for libkcgpu: error handling, device arena, small helpers.
#pragma once
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cuda_runtime.h>

#include "../../include/kcgpu.h"

typedef uint8_t u8;
typedef uint16_t u16;
typedef uint32_t u32;
typedef uint64_t u64;
typedef int64_t i64;

#define KC_HD __host__ __device__ __forceinline__
#define KC_D __device__ __forceinline__
#define KC_HD_LAMBDA __host__ __device__

// Status codes of the C ABI: KC_OK / KC_ERR_* from include/kcgpu.h.

struct KcError {
    int code;
    const char *what;
    const char *file;
    int line;
};

#define KC_THROW(code_, what_) throw KcError{(code_), (what_), __FILE__, __LINE__}

#define KC_CUDA(expr)                                                                         \
    do {                                                                                      \
        cudaError_t kc_e_ = (expr);                                                           \
        if (kc_e_ != cudaSuccess) {                                                           \
            cudaError_t kc_last_ = cudaGetLastError();                                        \
            (void) kc_last_;                                                                  \
            throw KcError{kc_e_ == cudaErrorMemoryAllocation ? KC_ERR_OOM : KC_ERR_CUDA,      \
                          cudaGetErrorString(kc_e_), __FILE__, __LINE__};                     \
        }                                                                                     \
    } while (0)

static const u32 KC_NONE = 0xFFFFFFFFu;
static const int KC_MAX_PEERS = 16;    // GPUs of one group (multi-GPU construction, group.cuh)
static const int KC_MAX_DEVICES = 64;

KC_HD u64 kc_div_up(u64 a, u64 b) { return (a + b - 1) / b; }
KC_HD u64 kc_align_up(u64 a, u64 b) { return (a + b - 1) / b * b; }
inline int kc_ceil_log2(u64 x) {
    int r = 0;
    while ((1ULL << r) < x) ++r;
    return r;
}

// Function attributes (the > 48 KB dynamic shared memory opt-in) and occupancy figures belong to a DEVICE, not to the process:
// a call site keeps one static KcDevOnce and runs its set-up once per device.  The lock also covers two host threads that
// drive the same device (virtual ranks of a group in the tests).
#include <mutex>
struct KcDevOnce {
    std::mutex m;
    bool done[KC_MAX_DEVICES] = {};
    template <class F> int run(F f) {  // -> current device
        int d = 0;
        KC_CUDA(cudaGetDevice(&d));
        if (d < 0 || d >= KC_MAX_DEVICES) KC_THROW(KC_ERR_ARG, "device ordinal out of range");
        std::lock_guard<std::mutex> g(m);
        if (!done[d]) {
            f(d);
            done[d] = true;
        }
        return d;
    }
};
inline int kc_sm_count(int dev) {
    static int n[KC_MAX_DEVICES] = {};
    if (!n[dev]) KC_CUDA(cudaDeviceGetAttribute(&n[dev], cudaDevAttrMultiProcessorCount, dev));
    return n[dev];
}

struct ArenaMark {
    size_t off, top;
};

// Bump allocator over one device (or, in the host-emulation test build, host) slab.  All temporaries of a
// kc_compute call live here so the timed path never calls cudaMalloc.  The slab is never cleared: a block holds whatever an
// earlier call, or an earlier block of the same call, left there, so everything a kernel reads must have been written in this call.
// `poison` (option "arena_poison") makes that testable: every block handed out is first filled with that byte, on `stream`.
struct Arena {
    char *base = nullptr;
    size_t cap = 0;
    size_t off = 0;   // bottom end: temporaries, stack discipline (mark / release)
    size_t top = 0;   // top end: small results that must outlive the temporaries below them
    size_t high = 0;
    int poison = -1;  // 0..255: fill byte of every block handed out; -1 = off
    cudaStream_t stream = nullptr;
    void reset() {
        off = 0;
        top = cap;
    }
    void fill_poison(void *p, size_t bytes) {
#ifdef KC_HOST_EMUL
        std::memset(p, poison, bytes);
#else
        KC_CUDA(cudaMemsetAsync(p, poison, bytes, stream));
#endif
    }
    template <typename T> T *alloc(size_t n) {
        size_t bytes = kc_align_up((n ? n : 1) * sizeof(T), 256);
        if (off + bytes > top) KC_THROW(KC_ERR_OOM, "device arena exhausted");
        T *p = reinterpret_cast<T *>(base + off);
        off += bytes;
        if (off + (cap - top) > high) high = off + (cap - top);
        if (poison >= 0) fill_poison(p, bytes);
        return p;
    }
    template <typename T> T *alloc_top(size_t n) {
        size_t bytes = kc_align_up((n ? n : 1) * sizeof(T), 256);
        if (off + bytes > top) KC_THROW(KC_ERR_OOM, "device arena exhausted");
        top -= bytes;
        if (off + (cap - top) > high) high = off + (cap - top);
        if (poison >= 0) fill_poison(base + top, bytes);
        return reinterpret_cast<T *>(base + top);
    }
    size_t mark() const { return off; }
    void release(size_t m) { off = m; }
    // both ends: restore() frees what either end handed out since checkpoint()
    ArenaMark checkpoint() const { return {off, top}; }
    void restore(const ArenaMark &m) {
        off = m.off;
        top = m.top;
    }
};
