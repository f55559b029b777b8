// Execution policies.
//
// CudaExec is the product: every primitive is a CUDA kernel launched on the context's stream.
// HostExec exists ONLY for tests/host_emul (engine/emission control flow can be debugged in the build
// container, which has no GPU); it is never compiled into libkcgpu.so — kcgpu.cu instantiates CudaExec only and
// the library has no CPU path.
//
// Primitives:
//   for_each(n, f)                 f(u64 i) for i in [0, n)
//   compact_if(n, pred, emit)      order-preserving stream compaction: emit(i, rank) for every i with pred(i)
//   exclusive_scan(in, out, n)     u32 exclusive prefix sum, returns the total
//   fill / copy / read             memset-like helpers and a synchronising scalar read-back
#pragma once
#include <cstring>
#include "kc_common.cuh"
#include <utility>
#include <vector>

#ifdef __CUDA_ARCH__
#define KC_ATOMIC_ADD(ptr, v) atomicAdd((ptr), (v))
#define KC_ATOMIC_MIN(ptr, v) atomicMin((ptr), (v))
#define KC_ATOMIC_MAX(ptr, v) atomicMax((ptr), (v))
#define KC_ATOMIC_OR(ptr, v) atomicOr((ptr), (v))
#else
template <typename T> inline T kc_host_atomic_add(T *p, T v) { T o = *p; *p = o + v; return o; }
template <typename T> inline T kc_host_atomic_min(T *p, T v) { T o = *p; if (v < o) *p = v; return o; }
template <typename T> inline T kc_host_atomic_max(T *p, T v) { T o = *p; if (v > o) *p = v; return o; }
template <typename T> inline T kc_host_atomic_or(T *p, T v) { T o = *p; *p = o | v; return o; }
#define KC_ATOMIC_ADD(ptr, v) kc_host_atomic_add((ptr), (v))
#define KC_ATOMIC_MIN(ptr, v) kc_host_atomic_min((ptr), (v))
#define KC_ATOMIC_MAX(ptr, v) kc_host_atomic_max((ptr), (v))
#define KC_ATOMIC_OR(ptr, v) kc_host_atomic_or((ptr), (v))
#endif

typedef unsigned long long kc_ull;  // CUDA's 64-bit atomic type

// Kernel classes for the per-kernel device timers (kc_profile_* in include/kcgpu.h).
enum KcProfId {
    KP_EXTRACT, KP_SORT_HIST, KP_SORT_SCATTER, KP_SORT_LOCAL, KP_SORT_MISC, KP_COMPACT, KP_SCAN, KP_TUPLES,
    KP_SIMULATE, KP_DOUBLING, KP_COMMIT, KP_SMALL_ENGINE, KP_RANK, KP_EMIT, KP_MAXONE, KP_MISC,
    KP_KS_HIST0, KP_KS_SCATTER0, KP_KS_RESOLVE, KP_RUNS, KP_COUNT
};
static const char *const kc_prof_names[KP_COUNT] = {
    "extract", "sort_hist", "sort_scatter", "sort_local", "sort_misc", "compact", "scan", "tuples",
    "simulate", "doubling", "commit", "small_engine", "rank", "emit", "maxone", "misc",
    "ks_hist0", "ks_scatter0", "ks_resolve", "runs"};

// ---------------------------------------------------------------------------------------------------
#ifdef __CUDACC__

static const int KC_FE_THREADS = 256;

template <typename F> __global__ void __launch_bounds__(KC_FE_THREADS) kc_for_each_kernel(u64 n, F f) {
    kc_pdl_wait();
    u64 i = (u64) blockIdx.x * KC_FE_THREADS + threadIdx.x;
    if (i < n) f(i);
}

// Exclusive scan of one value per thread across a 256-thread block; returns the thread's prefix, *total = block sum.
KC_D u32 kc_block_exclusive_scan_256(u32 v, u32 *total, u32 *smem_warp /*[8]*/) {
    const u32 lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    u32 incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        u32 t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (lane >= (u32) o) incl += t;
    }
    if (lane == 31) smem_warp[warp] = incl;
    __syncthreads();
    u32 warp_prefix = 0, sum = 0;
#pragma unroll
    for (int wi = 0; wi < 8; ++wi) {
        u32 s = smem_warp[wi];
        if ((u32) wi < warp) warp_prefix += s;
        sum += s;
    }
    __syncthreads();
    *total = sum;
    return warp_prefix + incl - v;
}

static const int KC_CP_ITEMS = 4;                         // consecutive items per thread
static const int KC_CP_TILE = KC_FE_THREADS * KC_CP_ITEMS;  // items per block

template <typename Pred>
__global__ void __launch_bounds__(KC_FE_THREADS) kc_compact_count_kernel(u64 n, Pred pred, u32 *block_counts, u32 *grand_total = nullptr) {
    __shared__ u32 sw[8];
    u64 base = (u64) blockIdx.x * KC_CP_TILE + (u64) threadIdx.x * KC_CP_ITEMS;
    u32 c = 0;
#pragma unroll
    for (int j = 0; j < KC_CP_ITEMS; ++j)
        if (base + j < n && pred(base + j)) ++c;
    u32 total;
    kc_block_exclusive_scan_256(c, &total, sw);
    if (threadIdx.x == 0) {
        block_counts[blockIdx.x] = total;
        if (grand_total && total) atomicAdd(grand_total, total);
    }
}

template <typename Pred, typename Emit>
__global__ void __launch_bounds__(KC_FE_THREADS) kc_compact_emit_kernel(u64 n, Pred pred, Emit emit, const u32 *block_offsets) {
    __shared__ u32 sw[8];
    u64 base = (u64) blockIdx.x * KC_CP_TILE + (u64) threadIdx.x * KC_CP_ITEMS;
    bool keep[KC_CP_ITEMS];
    u32 c = 0;
#pragma unroll
    for (int j = 0; j < KC_CP_ITEMS; ++j) {
        keep[j] = base + j < n && pred(base + j);
        c += keep[j];
    }
    u32 total;
    u32 rank = kc_block_exclusive_scan_256(c, &total, sw) + block_offsets[blockIdx.x];
#pragma unroll
    for (int j = 0; j < KC_CP_ITEMS; ++j)
        if (keep[j]) emit(base + j, rank++);
}

// One block scans up to 1024 values (4 per thread) and adds carry-in offsets.
__global__ void __launch_bounds__(KC_FE_THREADS) kc_scan_tile_kernel(const u32 *in, u32 *out, u64 n, u32 *tile_sums) {
    __shared__ u32 sw[8];
    u64 base = (u64) blockIdx.x * 1024 + (u64) threadIdx.x * 4;
    u32 v[4], c = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        v[j] = base + j < n ? in[base + j] : 0;
        c += v[j];
    }
    u32 total;
    u32 p = kc_block_exclusive_scan_256(c, &total, sw);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        if (base + j < n) out[base + j] = p;
        p += v[j];
    }
    if (threadIdx.x == 0 && tile_sums) tile_sums[blockIdx.x] = total;
}

// One block walks up to a few tiles with a running carry: one launch instead of tile scan + scan of the tile sums + add
// (the block counts of a 50 Mbp input are 6104 values: 4 launches, ~11 us, for microseconds of work).
__global__ void __launch_bounds__(KC_FE_THREADS) kc_scan_walk_kernel(const u32 *in, u32 *out, u64 n, u32 *sum) {
    __shared__ u32 sw[8];
    u32 carry = 0;
    for (u64 t0 = 0; t0 < n; t0 += 1024) {
        const u64 base = t0 + (u64) threadIdx.x * 4;
        u32 v[4], c = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            v[j] = base + j < n ? in[base + j] : 0;
            c += v[j];
        }
        u32 total;
        u32 p = kc_block_exclusive_scan_256(c, &total, sw) + carry;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (base + j < n) out[base + j] = p;
            p += v[j];
        }
        carry += total;
        __syncthreads();  // sw is reused by the next tile
    }
    if (threadIdx.x == 0 && sum) *sum = carry;
}

__global__ void __launch_bounds__(KC_FE_THREADS) kc_scan_add_kernel(u32 *out, u64 n, const u32 *tile_offsets) {
    u64 base = (u64) blockIdx.x * 1024 + (u64) threadIdx.x * 4;
    u32 o = tile_offsets[blockIdx.x];
#pragma unroll
    for (int j = 0; j < 4; ++j)
        if (base + j < n) out[base + j] += o;
}

// CUDA-event timers per kernel class; only active after kc_profile_enable (events cost ~1 us per launch).
struct KernelProf {
    bool enabled = false;
    double ms[KP_COUNT] = {0};
    u64 launches[KP_COUNT] = {0};
    u64 bytes[KP_COUNT] = {0};
    struct Rec {
        int id;
        cudaEvent_t a, b;
    };
    std::vector<Rec> pending;
    std::vector<cudaEvent_t> pool;
    cudaEvent_t get() {
        if (!pool.empty()) {
            cudaEvent_t e = pool.back();
            pool.pop_back();
            return e;
        }
        cudaEvent_t e;
        KC_CUDA(cudaEventCreate(&e));
        return e;
    }
    void resolve() {  // call after the stream has been synchronised
        for (Rec &r : pending) {
            float t = 0;
            if (cudaEventElapsedTime(&t, r.a, r.b) == cudaSuccess) ms[r.id] += t;
            ++launches[r.id];
            pool.push_back(r.a);
            pool.push_back(r.b);
        }
        pending.clear();
    }
    void reset() {
        for (int i = 0; i < KP_COUNT; ++i) {
            ms[i] = 0;
            launches[i] = 0;
            bytes[i] = 0;
        }
    }
};

// The kernel nodes of a captured graph whose arguments hold the input pointer `seq`, so that a replay can point them at another input
// of the same size (cudaGraphExecKernelNodeSetParams).  They are found at capture by value: every 8-byte word of an argument that
// equals `seq`.  The input is a caller's buffer or the arena block it was copied to, never an address that another argument holds.
struct SeqPatch {
    const void *seq = nullptr;
    struct Node {
        cudaGraphNode_t node;
        void *func;
        dim3 grid, block;
        size_t smem;
        std::vector<std::vector<u8>> args;  // the captured argument bytes
        std::vector<std::pair<u32, u32>> at;  // (argument, byte offset) of every copy of seq
    };
    std::vector<Node> nodes;

    void set_seq(cudaGraphExec_t exec, const void *s) {
        if (s == seq) return;
        for (Node &n : nodes) {
            std::vector<void *> ptrs;
            for (const auto &[i, off] : n.at) std::memcpy(n.args[i].data() + off, &s, 8);
            for (auto &a : n.args) ptrs.push_back(a.data());
            cudaKernelNodeParams kp{n.func, n.grid, n.block, (unsigned) n.smem, ptrs.data(), nullptr};
            KC_CUDA(cudaGraphExecKernelNodeSetParams(exec, n.node, &kp));
        }
        seq = s;
    }
};

struct CudaExec {
    cudaStream_t stream;
    Arena *arena;
    KernelProf *prof = nullptr;
    bool pdl = false;            // launch with programmatic stream serialization (the kernels wait in kc_pdl_wait)
    SeqPatch *patch = nullptr;   // != nullptr while a graph is captured from this policy's launches
    u64 launches = 0;  // kernels launched through this policy (bench.py reports it as gpu_launches)
    u64 read_backs = 0;  // synchronising read-backs (read_n), i.e. host round trips
    u8 *pinned = nullptr;  // page-locked host scratch of the context for the synchronising read-backs below: a pageable
    size_t pinned_cap = 0;  // destination makes the driver stage the copy, which costs several us per read on an idle stream

    // RAII timer around one kernel launch (or a short fixed group of launches) of class `id`.
    struct Scope {
        CudaExec &ex;
        bool on;
        KernelProf::Rec rec;
        Scope(CudaExec &e, int id, u64 bytes = 0) : ex(e), on(e.prof && e.prof->enabled) {
            if (!on) return;
            rec.id = id;
            rec.a = ex.prof->get();
            rec.b = ex.prof->get();
            ex.prof->bytes[id] += bytes;
            cudaEventRecord(rec.a, ex.stream);
        }
        ~Scope() {
            if (!on) return;
            cudaEventRecord(rec.b, ex.stream);
            ex.prof->pending.push_back(rec);
        }
    };

    static constexpr bool is_device = true;

    template <typename T> T *alloc(size_t n) { return arena->alloc<T>(n); }

    // One kernel launch on the stream; with `pdl`, the kernel may start before the previous one ends (it waits in kc_pdl_wait).
    template <typename... P, typename... A> void launch(void (*kern)(P...), dim3 grid, dim3 block, size_t smem, const A &...a) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = grid;
        cfg.blockDim = block;
        cfg.dynamicSmemBytes = smem;
        cfg.stream = stream;
        cudaLaunchAttribute attr[1];
        if (pdl) {
            attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
            attr[0].val.programmaticStreamSerializationAllowed = 1;
            cfg.attrs = attr;
            cfg.numAttrs = 1;
        }
        KC_CUDA(cudaLaunchKernelEx(&cfg, kern, a...));
        ++launches;
        if (patch) note_seq<P...>(reinterpret_cast<void *>(kern), grid, block, smem, a...);
    }

    // While capturing: the node just added, if any of its arguments holds patch->seq (see SeqPatch).
    template <typename... P> void note_seq(void *func, dim3 grid, dim3 block, size_t smem, const P &...p) {
        SeqPatch::Node n{};
        (n.args.emplace_back(reinterpret_cast<const u8 *>(&p), reinterpret_cast<const u8 *>(&p) + sizeof(P)), ...);
        for (u32 i = 0; i < (u32) n.args.size(); ++i)
            for (u32 off = 0; off + 8 <= n.args[i].size(); off += 8)
                if (std::memcmp(n.args[i].data() + off, &patch->seq, 8) == 0) n.at.emplace_back(i, off);
        if (n.at.empty()) return;
        cudaStreamCaptureStatus cs;
        const cudaGraphNode_t *deps = nullptr;
        size_t n_deps = 0;
        KC_CUDA(cudaStreamGetCaptureInfo(stream, &cs, nullptr, nullptr, &deps, &n_deps));
        if (cs != cudaStreamCaptureStatusActive || n_deps != 1) KC_THROW(KC_ERR_INTERNAL, "graph capture: no kernel node to patch");
        n.node = deps[0];
        n.func = func;
        n.grid = grid;
        n.block = block;
        n.smem = smem;
        patch->nodes.push_back(std::move(n));
    }

    template <typename F> void for_each(u64 n, F f, int id = KP_MISC, u64 bytes = 0) {
        if (n == 0) return;
        Scope sc(*this, id, bytes);
        u64 blocks = kc_div_up(n, KC_FE_THREADS);
        if (blocks > 0x7FFFFFFFULL) KC_THROW(KC_ERR_TOO_LARGE, "for_each grid too large");
        launch(kc_for_each_kernel<F>, (unsigned) blocks, KC_FE_THREADS, 0, n, f);
    }

    void fill_bytes(void *p, int value, size_t bytes) {
        if (bytes) KC_CUDA(cudaMemsetAsync(p, value, bytes, stream));
    }
    void copy_bytes(void *dst, const void *src, size_t bytes) {
        if (bytes) KC_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, stream));
    }
    template <typename T> T read(const T *p) {
        T v;
        read_n(p, &v, 1);
        return v;
    }
    void sync() { KC_CUDA(cudaStreamSynchronize(stream)); }
    template <typename T> void read_n(const T *p, T *host, size_t n) {  // one synchronising read-back of n values
        const size_t bytes = n * sizeof(T);
        ++read_backs;
        if (pinned && bytes <= pinned_cap) {
            KC_CUDA(cudaMemcpyAsync(pinned, p, bytes, cudaMemcpyDeviceToHost, stream));
            KC_CUDA(cudaStreamSynchronize(stream));
            std::memcpy(host, pinned, bytes);
            return;
        }
        KC_CUDA(cudaMemcpyAsync(host, p, bytes, cudaMemcpyDeviceToHost, stream));
        KC_CUDA(cudaStreamSynchronize(stream));
    }

    // out may alias in.  Returns the sum of all inputs.
    u32 exclusive_scan(const u32 *in, u32 *out, u64 n) {
        if (n == 0) return 0;
        size_t m = arena->mark();
        u32 total = scan_rec(in, out, n, true);
        arena->release(m);
        return total;
    }

    // Same without the synchronising read-back of the total (out[n-1] + in[n-1] holds it on the device).
    void exclusive_scan_nosync(const u32 *in, u32 *out, u64 n) {
        if (n == 0) return;
        size_t m = arena->mark();
        scan_rec(in, out, n, false);
        arena->release(m);
    }

    template <typename Pred, typename Emit> u64 compact_if(u64 n, Pred pred, Emit emit, u64 bytes = 0) {
        if (n == 0) return 0;
        if (n >= 0xFFFFFFFFULL) KC_THROW(KC_ERR_TOO_LARGE, "compact_if over more than 2^32-1 items");
        Scope sc(*this, KP_COMPACT, bytes);
        size_t m = arena->mark();
        u64 blocks = kc_div_up(n, KC_CP_TILE);
        u32 *counts = arena->alloc<u32>(blocks);
        kc_compact_count_kernel<<<(unsigned) blocks, KC_FE_THREADS, 0, stream>>>(n, pred, counts);
        ++launches;
        KC_CUDA(cudaGetLastError());
        u32 total = scan_rec(counts, counts, blocks, true);
        kc_compact_emit_kernel<<<(unsigned) blocks, KC_FE_THREADS, 0, stream>>>(n, pred, emit, counts);
        ++launches;
        KC_CUDA(cudaGetLastError());
        arena->release(m);
        return total;
    }

    // The same without the synchronising read-back: the number of kept items is ADDED to *total_dev (device memory, zero on entry).
    template <typename Pred, typename Emit> void compact_if_nosync(u64 n, Pred pred, Emit emit, u32 *total_dev, u64 bytes = 0) {
        if (n == 0) return;
        if (n >= 0xFFFFFFFFULL) KC_THROW(KC_ERR_TOO_LARGE, "compact_if over more than 2^32-1 items");
        Scope sc(*this, KP_COMPACT, bytes);
        size_t m = arena->mark();
        u64 blocks = kc_div_up(n, KC_CP_TILE);
        u32 *counts = arena->alloc<u32>(blocks);
        kc_compact_count_kernel<<<(unsigned) blocks, KC_FE_THREADS, 0, stream>>>(n, pred, counts, total_dev);
        ++launches;
        KC_CUDA(cudaGetLastError());
        scan_rec(counts, counts, blocks, false);
        kc_compact_emit_kernel<<<(unsigned) blocks, KC_FE_THREADS, 0, stream>>>(n, pred, emit, counts);
        ++launches;
        KC_CUDA(cudaGetLastError());
        arena->release(m);
    }

  private:
    u32 scan_rec(const u32 *in, u32 *out, u64 n, bool want_total) {
        u64 tiles = kc_div_up(n, 1024);
        if (tiles <= 8) {
            u32 *sum = arena->alloc<u32>(1);
            kc_scan_walk_kernel<<<1, KC_FE_THREADS, 0, stream>>>(in, out, n, sum);
            ++launches;
            KC_CUDA(cudaGetLastError());
            return want_total ? read(sum) : 0;
        }
        u32 *sums = arena->alloc<u32>(tiles);
        kc_scan_tile_kernel<<<(unsigned) tiles, KC_FE_THREADS, 0, stream>>>(in, out, n, sums);
        ++launches;
        KC_CUDA(cudaGetLastError());
        u32 total = scan_rec(sums, sums, tiles, want_total);
        kc_scan_add_kernel<<<(unsigned) tiles, KC_FE_THREADS, 0, stream>>>(out, n, sums);
        ++launches;
        KC_CUDA(cudaGetLastError());
        return total;
    }
};

#endif  // __CUDACC__

// ---------------------------------------------------------------------------------------------------
#ifdef KC_HOST_EMUL
// Serial stand-in used by tests/host_emul only.
struct HostExec {
    Arena *arena;
    u64 launches = 0;
    static constexpr bool is_device = false;
    template <typename T> T *alloc(size_t n) { return arena->alloc<T>(n); }
    template <typename F> void for_each(u64 n, F f, int = 0, u64 = 0) {
        for (u64 i = 0; i < n; ++i) f(i);
    }
    void fill_bytes(void *p, int value, size_t bytes) { std::memset(p, value, bytes); }
    void copy_bytes(void *dst, const void *src, size_t bytes) { std::memmove(dst, src, bytes); }
    template <typename T> T read(const T *p) { return *p; }
    template <typename T> void read_n(const T *p, T *host, size_t n) { std::memcpy(host, p, n * sizeof(T)); }
    void sync() {}
    u32 exclusive_scan(const u32 *in, u32 *out, u64 n) {
        u32 s = 0;
        for (u64 i = 0; i < n; ++i) {
            u32 v = in[i];
            out[i] = s;
            s += v;
        }
        return s;
    }
    template <typename Pred, typename Emit> u64 compact_if(u64 n, Pred pred, Emit emit, u64 = 0) {
        u64 r = 0;
        for (u64 i = 0; i < n; ++i)
            if (pred(i)) emit(i, (u32) r++);
        return r;
    }
};
#endif
