// libkcgpu: C ABI (include/kcgpu.h) over the CUDA pipeline.  Only CudaExec is instantiated here: the library has
// no CPU path and fails with KC_ERR_NO_DEVICE when no GPU is present.
#include "../../include/kcgpu.h"

#include "digest.cuh"
#include "emit.cuh"
#include "engine.cuh"
#include "exec.cuh"
#include "group.cuh"
#include "kmerset.cuh"
#include "kmerset_fast.cuh"
#include "kmerset_sig.cuh"
#include "kword.cuh"
#include "masks.cuh"
#include "runs.cuh"
#include "set_routes.cuh"
#include "sort.cuh"
#include "stage1.cuh"
#include "tail_spec.cuh"

#include <chrono>
#include <exception>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <type_traits>
#include <vector>

static double kc_now_ms() {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}
static const bool kc_trace = std::getenv("KC_TRACE") != nullptr;
#define KC_TRACE_POINT(label)                                                               \
    do {                                                                                    \
        if (kc_trace) std::fprintf(stderr, "[kc_trace] %-28s %.3f ms\n", (label), kc_now_ms()); \
    } while (0)

// Page-locked host buffer, grown on demand and reused across calls.
struct PinnedBuf {
    u8 *p = nullptr;
    size_t cap = 0;
    unsigned flags = cudaHostAllocDefault;
    void reserve(size_t need) {
        if (cap >= need) return;
        if (p) KC_CUDA(cudaFreeHost(p));
        p = nullptr;
        cap = 0;
        KC_CUDA(cudaHostAlloc(reinterpret_cast<void **>(&p), need + need / 8, flags));
        cap = need + need / 8;
    }
};

// What the host needs of a queued speculative tail once its status block is back (tail_spec_queue -> tail_spec_finish).
struct SpecTail {
    size_t mark = 0;  // arena bottom before the tail
    const u8 *ms = nullptr;
    u64 total_ub = 0;
    u64 n_s = 0, n_p = 0;  // the small engine's sizes (apply_small_status)
    int small_d = 0;
};

// The from-FASTA call of one genome on one GPU (signature construction + speculative tail, up to the copy of the status block into
// pinned memory) captured as a CUDA graph and replayed by later calls of the same shape: the launches of the step cost one
// cudaGraphLaunch.  Everything the key holds fixes the arena layout and the launch shapes; options that change either clear the cache
// (kc_set_option), and so does a new arena.  The input pointer is the one argument that changes between calls (SeqPatch).
struct SpecGraph {
    int limbs = 0, k = 0;
    bool complements = false;
    u64 n_bytes = 0;
    const char *arena_base = nullptr;
    ArenaMark arena_at;  // both arena ends when the call reached the construction
    const u32 *flags = nullptr;
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    SeqPatch patch;
    u64 launches = 0, arena_high = 0;
    ArenaMark arena_after;
    u64 *blk = nullptr;
    SpecTail tail;
    bool same_shape(const SpecGraph &o) const {
        return limbs == o.limbs && k == o.k && complements == o.complements && n_bytes == o.n_bytes && arena_base == o.arena_base &&
               arena_at.off == o.arena_at.off && arena_at.top == o.arena_at.top && flags == o.flags;
    }
    void destroy() {
        if (exec) cudaGraphExecDestroy(exec);
        if (graph) cudaGraphDestroy(graph);
        exec = nullptr;
        graph = nullptr;
    }
};

struct kc_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    Arena arena;
    KernelProf prof;
    PinnedBuf pin_out;  // the host results of kc_compute, kc_streaming and kc_maskopt
    static const size_t KC_PIN_SMALL = 4096;
    u8 *pin_small = nullptr;  // page-locked scratch for the small synchronising read-backs (CudaExec::read_n)
    cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    // kc_compute with host buffers: the input is copied in chunks on its own stream, the first partition pass follows the copy front
    static const int KC_H2D_CHUNKS = 4;
    cudaStream_t copy_stream = nullptr;
    cudaStream_t capture_stream = nullptr;  // SpecGraph captures (the context's stream may be the legacy default stream, which cannot capture)
    cudaEvent_t chunk_ev[KC_H2D_CHUNKS] = {nullptr, nullptr, nullptr, nullptr};
    bool small_engine = true;
    int small_threads = 0;   // 0 = chosen by the number of free ends (option "small_threads": 256 or 512)
    bool sparse_switch = true;  // src/main.cpp:175 (option "sparse_switch" = 0 keeps the runs as nodes whatever their number)
    SetRoutes routes;        // the constructions of the first-occurrence bits, their tuning, counters and memories (set_routes.cuh)
    u64 total_launches = 0;  // kernels launched through this context since kc_init
    u64 read_backs = 0;      // synchronising device -> host reads of this context since kc_init (host round trips)
    bool tail_spec = true;   // option "tail_spec": queue the tail of the from-FASTA path without reading the run count (run_sig_spec)
    u64 tail_spec_runs = 0, tail_spec_fallbacks = 0;
    EngineStats path_stats;   // the overlap stage of the last call that ran it (stats "path_levels", "path_ban_rounds", "path_bans")
    KcGroup grp;             // multi-GPU: this context as one rank of a group (group.cuh)
    bool arena_limited = false;
    u32 arena_estimate_ppm = 1000000;  // option "arena_estimate_ppm": scales the first arena estimate of run_with_arena (tests)
    u64 arena_retries = 0;         // calls repeated by run_with_arena after running out of arena
    std::vector<SpecGraph> spec_graphs;  // cached graphs of the speculative from-FASTA call (SpecGraph), at most KC_SPEC_GRAPHS
    static const size_t KC_SPEC_GRAPHS = 8;
    u64 spec_graph_captures = 0, spec_graph_replays = 0;
    std::string last_error;
    void clear_spec_graphs() {
        for (SpecGraph &g : spec_graphs) g.destroy();
        spec_graphs.clear();
    }
};

namespace {

void set_error(kc_ctx *ctx, const KcError &e) {
    if (!ctx) return;
    char buf[512];
    std::snprintf(buf, sizeof(buf), "%s (%s:%d)", e.what, e.file, e.line);
    ctx->last_error = buf;
}

#define KC_API_BEGIN try {
#define KC_API_END(ctx)                                                \
    }                                                                  \
    catch (const KcError &e) {                                         \
        set_error((ctx), e);                                           \
        return e.code;                                                 \
    }                                                                  \
    catch (const std::bad_alloc &) {                                   \
        if (ctx) (ctx)->last_error = "host allocation failed";         \
        return KC_ERR_OOM;                                             \
    }                                                                  \
    catch (...) {                                                      \
        if (ctx) (ctx)->last_error = "unknown failure";                \
        return KC_ERR_INTERNAL;                                        \
    }

// The state of one call on a context: its device is made current, and `ex` runs on the context's stream, arena, profiler and
// pinned scratch.  The call's launches and read-backs are added to the context's totals when it returns; a failed call (one that
// leaves by an exception) adds nothing.
struct CallFrame {
    kc_ctx *ctx;
    CudaExec ex{ctx->stream, &ctx->arena};
    const int exceptions = std::uncaught_exceptions();
    explicit CallFrame(kc_ctx *c) : ctx(c) {
        KC_CUDA(cudaSetDevice(c->device));
        ex.prof = &c->prof;
        ex.pinned = c->pin_small;
        ex.pinned_cap = c->pin_small ? kc_ctx::KC_PIN_SMALL : 0;
    }
    ~CallFrame() {
        if (std::uncaught_exceptions() > exceptions) return;
        ctx->total_launches += ex.launches;
        ctx->read_backs += ex.read_backs;
    }
};

// f(std::integral_constant<int, L>()) for the k-mer word of `limbs` 64-bit limbs (kc_limbs_for_k: 1, 2 or 4).
template <class F> decltype(auto) with_limbs(int limbs, F &&f) {
    if (limbs == 1) return f(std::integral_constant<int, 1>());
    if (limbs == 2) return f(std::integral_constant<int, 2>());
    return f(std::integral_constant<int, 4>());
}

void check_params(const kc_params *p) {
    if (!p) KC_THROW(KC_ERR_ARG, "params is NULL");
    if (p->k < 1 || p->k > 127) KC_THROW(KC_ERR_ARG, "k must be in 1..127");                          // src/main.cpp:93,285-292
    if (p->min_frequency < 1 || p->min_frequency > 255) KC_THROW(KC_ERR_ARG, "min_frequency must be in 1..255");  // :302-304
    if (p->min_frequency != 1 && p->assume_simplitigs) KC_THROW(KC_ERR_ARG, "-z is not compatible with -S");   // :305-308
}

// Inputs of KC_POS32_BYTES or more need 64-bit window positions, which only the signature construction carries (the fixed-slot
// and exact constructions move 32-bit positions, the -S path and the other entry points keep their 32-bit caps).
void check_large_input(const kc_ctx *ctx, const kc_params *p, u64 n_bytes) {
    if (n_bytes < KC_POS32_BYTES) return;
    if (p->assume_simplitigs) KC_THROW(KC_ERR_TOO_LARGE, KC_LARGE_ONLY "; -S was asked");
    if (p->min_frequency > 1) KC_THROW(KC_ERR_TOO_LARGE, KC_LARGE_ONLY "; -z (min_frequency > 1) was asked");
    if (p->want_maxone) KC_THROW(KC_ERR_TOO_LARGE, KC_LARGE_ONLY "; -M (want_maxone) was asked");
    if (p->k < 26) KC_THROW(KC_ERR_TOO_LARGE, KC_LARGE_ONLY "; k is below 26");
    if (!ctx->routes.sig.enabled) KC_THROW(KC_ERR_TOO_LARGE, KC_LARGE_ONLY "; it is switched off (option sig_set = 0)");
    if (!kc_sig_plan(n_bytes, p->k, ctx->routes.sig).ok) KC_THROW(KC_ERR_TOO_LARGE, KC_LARGE_ONLY "; its bucket plan does not fit this input");
}

// Make sure the arena can hold `need` bytes (bounded by what the device can give).
void ensure_arena(kc_ctx *ctx, size_t need) {
    need = (need + 4095) & ~(size_t) 4095;  // both arena ends stay 256-byte aligned
    if (ctx->arena.cap >= need) return;
    if (ctx->arena.cap && ctx->arena_limited && need >= ctx->arena.cap) return;  // already holds all the device can give
    ctx->clear_spec_graphs();
    if (ctx->arena.base) {
        KC_CUDA(cudaFree(ctx->arena.base));
        ctx->arena.base = nullptr;
        ctx->arena.cap = 0;
    }
    size_t free_b = 0, total_b = 0;
    KC_CUDA(cudaMemGetInfo(&free_b, &total_b));
    size_t limit = (size_t) (free_b * 0.92);
    size_t want = need < limit ? need : (limit & ~(size_t) 4095);
    ctx->arena_limited = want < need;
    KC_CUDA(cudaMalloc(&ctx->arena.base, want));
    ctx->arena.cap = want;
    ctx->arena.reset();
}

// Arena bytes of the overlap stage and the emission for `nodes` nodes per strand (the part of estimate_arena after stage 1).
double overlap_emit_bytes(double nodes, int limbs, bool complements, u64 n_bytes) {
    const double wb = 8.0 * limbs;
    const double N = (complements ? 2.0 : 1.0) * nodes;
    return N * (60.0 + 2.0 * 2.0 * (wb + 8.0) + 12.0 + 40.0) + N * 32.0 + 3.0 * n_bytes;
}

// Arena bytes one kc_compute needs (see DESIGN.md "Data layout in HBM").  Stage 1 is an exact upper bound; the overlap
// stage depends on the number of nodes, which for a FASTA input (first-occurrence runs) is only known after stage 1:
// `pessimistic = false` assumes one run per 64 sequence bytes (reads with 1 % errors give one per ~650), and a call that
// runs out of arena is repeated once with the worst case (one run per 2 bytes), see run_with_arena.
// Inputs of KC_POS32_BYTES or more take the signature construction alone (`sig`: its plan at this size): sequence, flags, code
// words and record rows.
size_t estimate_arena(u64 n_bytes, u64 n_recs, int limbs, bool complements, bool simplitigs, bool pessimistic = false,
                      const KsfTuning *fast = nullptr, const SigPlan *sig = nullptr) {
    const double wb = 8.0 * limbs;
    double stage1 = n_bytes * (1.0 + 2.0 * (wb + 4.0) + 1.0 + 1.0 + 0.2);  // sequence, keys + positions x2, counts, control, flags
    if (n_bytes >= KC_POS32_BYTES && sig && sig->ok) {
        stage1 = n_bytes * (1.0 + 0.125) + (double) kc_sig_arena_bytes(*sig, n_bytes);
    } else if (fast) {  // fixed-slot buckets of the histogram-free construction (tried first, released before the exact one runs)
        const KsfPlan pl = kc_ksf_plan(n_bytes, *fast);
        if (pl.ok) {
            const double f = n_bytes * 1.2 + (double) (pl.slots[0] + pl.slots[1]) * (wb + 4.0) + (double) pl.n_leaf * 28.0 + 65536.0;
            if (f > stage1) stage1 = f;
        }
    }
    double nodes = simplitigs ? (double) n_recs : (pessimistic ? n_bytes * 0.85 : n_bytes / 64.0 + 1e6);  // sparse switch: up to 5 k-mer nodes per 6 bytes
    double total = (stage1 + overlap_emit_bytes(nodes, limbs, complements, n_bytes)) * 1.1 + (256u << 20);
    return (size_t) total;
}

// Runs body() with an arena of estimate_arena's bytes for this input; if the arena is exhausted (more nodes than the estimate
// assumed) the call is repeated once with the pessimistic estimate.
template <class F> void run_with_arena(kc_ctx *ctx, const kc_params &p, const kc_input &in, F body) {
    const SigPlan sig = kc_sig_plan(in.n_bytes, p.k, ctx->routes.sig);
    auto estimate = [&](bool pessimistic) {
        return estimate_arena(in.n_bytes, in.n_recs, kc_limbs_for_k(p.k), p.complements != 0, p.assume_simplitigs != 0, pessimistic,
                              &ctx->routes.fast, &sig);
    };
    const size_t need = estimate(false), need_max = estimate(true);
    ensure_arena(ctx, (size_t) ((double) need * ctx->arena_estimate_ppm / 1e6));
    try {
        ctx->arena.reset();
        body();
    } catch (const KcError &e) {
        if (e.code != KC_ERR_OOM || need_max <= ctx->arena.cap || ctx->arena_limited) throw;
        ++ctx->arena_retries;
        KC_CUDA(cudaStreamSynchronize(ctx->stream));
        ensure_arena(ctx, need_max);
        ctx->arena.reset();
        body();
    }
}

struct DevInput {
    const u8 *seq;
    u64 n_bytes;
    const u64 *rec_off, *rec_len;
    u64 n_recs;
    InputChunks *chunks = nullptr;  // != nullptr: seq is still being copied in (see InputChunks); wait before reading it
};

struct DevResult {
    const u8 *ms = nullptr, *maxone = nullptr;
    u64 length = 0, n_kmers = 0, n_occ = 0, n_nodes = 0, n_simplitigs = 0;
    u64 lower_bound = 0;  // only with run_tail(..., lower_bound = true)
    u64 slice_begin = 0, slice_len = 0;
};

// Host -> device: the sequence and, with `records` (-S), the records.  The 64 bytes past n_bytes are never written: every loader
// of the from-FASTA path is bounded by n_bytes (kc_compute_device gets a caller's buffer without them).  With `chunks`, a large
// from-FASTA input goes in chunks on the copy stream: the level-0 partition pass of chunk c starts as soon as chunk c has landed
// (InputChunks), instead of after the whole copy.  The returned input carries `chunks` when it was used.
DevInput upload_input(kc_ctx *ctx, CudaExec &ex, const kc_input *in, bool records, InputChunks *chunks) {
    u8 *d_seq = ex.alloc<u8>(in->n_bytes + 64);
    if (records || in->n_bytes < (8u << 20)) chunks = nullptr;
    if (chunks) {
        if (!ctx->copy_stream) {
            KC_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
            for (int c = 0; c < kc_ctx::KC_H2D_CHUNKS; ++c) KC_CUDA(cudaEventCreateWithFlags(&ctx->chunk_ev[c], cudaEventDisableTiming));
        }
        const u64 granule = 32768;  // whole level-0 tiles for every word width
        chunks->chunk_bytes = (in->n_bytes / kc_ctx::KC_H2D_CHUNKS + granule) / granule * granule;
        chunks->ev = ctx->chunk_ev;
        if (ctx->arena.poison >= 0) {  // the copy must land after the poison fill of d_seq on the context stream
            KC_CUDA(cudaEventRecord(ctx->ev[5], ctx->stream));
            KC_CUDA(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev[5], 0));
        }
        for (u64 off = 0; off < in->n_bytes; off += chunks->chunk_bytes) {
            const u64 len = std::min<u64>(chunks->chunk_bytes, in->n_bytes - off);
            KC_CUDA(cudaMemcpyAsync(d_seq + off, in->seq + off, len, cudaMemcpyHostToDevice, ctx->copy_stream));
            KC_CUDA(cudaEventRecord(ctx->chunk_ev[chunks->n++], ctx->copy_stream));
        }
    } else {
        KC_CUDA(cudaMemcpyAsync(d_seq, in->seq, in->n_bytes, cudaMemcpyHostToDevice, ctx->stream));
    }
    u64 *d_off = nullptr, *d_len = nullptr;
    if (records) {
        d_off = ex.alloc<u64>(in->n_recs);
        d_len = ex.alloc<u64>(in->n_recs);
        KC_CUDA(cudaMemcpyAsync(d_off, in->rec_off, in->n_recs * 8, cudaMemcpyHostToDevice, ctx->stream));
        KC_CUDA(cudaMemcpyAsync(d_len, in->rec_len, in->n_recs * 8, cudaMemcpyHostToDevice, ctx->stream));
    }
    return DevInput{d_seq, in->n_bytes, d_off, d_len, in->n_recs, chunks};
}

// Host -> device for the mask passes: n bytes, then '\n' from the last whole 32-byte word on through 64 bytes past the end.
u8 *upload_padded(CudaExec &ex, const u8 *src, u64 n) {
    const u64 padded = (n + 31) / 32 * 32 + 64;
    u8 *d = ex.alloc<u8>(padded);
    ex.fill_bytes(d + (n & ~(u64) 31), '\n', padded - (n & ~(u64) 31));
    if (n) KC_CUDA(cudaMemcpyAsync(d, src, n, cudaMemcpyHostToDevice, ex.stream));
    return d;
}

// What stage 1 hands to run_tail: the nodes (first-occurrence runs, or with -S the records), the kept distinct k-mers U, the k-mer
// occurrences and, for -M, the sorted k-mer set (kMersDict of src/global.h:165-167).
template <int L> struct Stage1 {
    RunNodes nodes;
    u64 U = 0, n_occ = 0;
    KWord<L> *uniq = nullptr;
};

// Stage 1 alone.  Leaves the sorted distinct k-mers (and their counts) at the current arena top and returns them.
template <int L> u64 run_stage1(kc_ctx *ctx, CudaExec &ex, const DevInput &in, const kc_params &p, KWord<L> **uniq_out, u8 **cnt_out,
                               u64 *n_occ) {
    KC_CUDA(cudaEventRecord(ctx->ev[0], ex.stream));
    KC_CUDA(cudaEventRecord(ctx->ev[1], ex.stream));  // extraction is fused into the partition passes
    if (in.chunks) in.chunks->wait_all(ex.stream);
    KmerSet<L> set = kc_kmerset_build<L>(ex, in.seq, in.n_bytes, p.k, p.complements != 0, p.min_frequency, nullptr, true);
    KC_CUDA(cudaEventRecord(ctx->ev[2], ex.stream));
    *n_occ = set.n_occ;
    *uniq_out = set.keys;
    *cnt_out = set.cnt;
    return set.n_kept;
}

// The speculative tail (tail_spec.cuh): from the first-occurrence flags to the last emission kernel, sized for KC_SPEC_RUNS runs, and
// the copy of the status block `blk` (cells4 of the signature construction first, KC_SPEC_BLOCK_WORDS words, zeroed) into the pinned
// scratch behind them.  tail_spec_finish reads it.
template <int L>
SpecTail tail_spec_queue(kc_ctx *ctx, CudaExec &ex, const DevInput &in, const kc_params &p, const u32 *flags, u64 *blk) {
    SpecTail t;
    const u64 nb = in.n_bytes;
    const int k = p.k;
    const bool complements = p.complements != 0;
    t.mark = ex.arena->mark();
    const u32 C = KC_SPEC_RUNS, N_cap = complements ? 2 * C : C;
    const u64 n_words = kc_div_up(nb, 32);
    const u32 blocks = (u32) kc_div_up(nb, (u64) KC_RUN_TILE);
    u32 *counts = ex.alloc<u32>(blocks);
    u64 *rec_off = ex.alloc<u64>(C), *rec_len = ex.alloc<u64>(C);
    kc_ull *n_runs = reinterpret_cast<kc_ull *>(blk + 1);
    auto stage_event = [&](int i) {  // a captured graph is timed as a whole (run_sig_spec)
        if (!ex.patch) KC_CUDA(cudaEventRecord(ctx->ev[i], ex.stream));
    };
    {
        CudaExec::Scope sc(ex, KP_RUNS, nb / 8);
        ex.launch(kc_runs_count_kernel, blocks, 256, 0, flags, n_words, counts, n_runs);
        ex.launch(kc_runs_emit_kernel, blocks, 256, 0, flags, n_words, (const u32 *) counts, rec_off, rec_len, (const kc_ull *) n_runs, (u64) C);
    }
    stage_event(2);
    NodeView<L> nv;
    nv.k = k;
    nv.complements = complements;
    nv.n = C;
    nv.N = N_cap;
    KWord<L> *first = ex.alloc<KWord<L>>(C), *last = ex.alloc<KWord<L>>(C);
    nv.first = first;
    nv.last = last;
    Engine<CudaExec, L> eng(ex, nv, /*strict=*/false, /*lower_bound=*/false);
    eng.small_threads_opt = ctx->small_threads;
    eng.alloc_state();
    u32 *spec = reinterpret_cast<u32 *>(blk + KC_SPEC_SPEC);
    eng.n_dev = spec + 1;
    eng.small_status = reinterpret_cast<u32 *>(blk + KC_SPEC_SMALL);
    const u64 mask_words = kc_small_mask_words(N_cap, N_cap);
    eng.small_masks = ex.alloc<u32>(mask_words + 4 * (u64) (2 * N_cap));  // + the second copies of the end masks
    eng.live_s = ex.alloc<u32>(N_cap);
    eng.live_p = ex.alloc<u32>(N_cap);
    eng.n_s = eng.n_p = N_cap;
    {
        CudaExec::Scope sc(ex, KP_RUNS, 32 * (u64) C);
        ex.launch(kc_spec_nodes_kernel<L>, 1, 1024, 0, (const u64 *) blk, spec, ctx->sparse_switch, complements, in.seq, k, rec_off, rec_len, first, last,
                  eng.st, eng.ban_flag, eng.ban_ctr, eng.live_s, eng.live_p, eng.small_masks, (u32) mask_words);
    }
    static_assert(4 * KC_SPEC_RUNS <= SmallCfg<L>::T && 2 * KC_SPEC_RUNS <= SmallCfg<L>::NS && 2 * KC_SPEC_RUNS <= KC_RANK_SMALL,
                  "the speculative tail runs on the one-CTA kernels");
    eng.run();  // all levels in the single-CTA engine
    stage_event(3);
    NodeSeq<L> ns;
    ns.k = k;
    ns.kmers = nullptr;
    ns.seq = in.seq;
    ns.rec_off = rec_off;
    ns.rec_len = rec_len;
    ns.n = C;
    const EmitSpec es{spec + 1, blk + KC_SPEC_EMIT};
    // every character of the superstring is a character of some node: nodes are pieces of the input that overlap by < k
    t.total_ub = nb + (u64) C * k + 16;
    t.ms = kc_emit_superstring<CudaExec, L>(ex, ns, nv, eng.st, nullptr, 0, false, 0, 1, t.total_ub, &es).ms;
    stage_event(4);
    if (!ex.pinned || ex.pinned_cap < KC_SPEC_BLOCK_WORDS * 8) KC_THROW(KC_ERR_INTERNAL, "no pinned scratch for the status block");
    KC_CUDA(cudaMemcpyAsync(ex.pinned, blk, KC_SPEC_BLOCK_WORDS * 8, cudaMemcpyDeviceToHost, ex.stream));
    t.n_s = eng.n_s;
    t.n_p = eng.n_p;
    t.small_d = eng.small_d;
    KC_TRACE_POINT("tail_spec: queued");
    return t;
}

// The one read-back of the speculative tail.  Returns the status: KC_SPEC_OK = `res` holds the result; otherwise nothing was done and
// the arena bottom is as it was before the tail.
template <int L> u32 tail_spec_finish(kc_ctx *ctx, CudaExec &ex, const SpecTail &t, DevResult &res) {
    u64 h[KC_SPEC_BLOCK_WORDS];
    ex.sync();
    std::memcpy(h, ex.pinned, sizeof(h));
    ++ex.read_backs;
    const u32 *hs = reinterpret_cast<const u32 *>(h + KC_SPEC_SPEC);
    if (hs[0] != KC_SPEC_OK) {
        ex.arena->release(t.mark);
        return hs[0];
    }
    Engine<CudaExec, L> eng(ex, NodeView<L>(), false, false);
    eng.n_s = t.n_s;
    eng.n_p = t.n_p;
    eng.small_d = t.small_d;
    eng.apply_small_status(reinterpret_cast<const u32 *>(h + KC_SPEC_SMALL));  // a failed small-engine run is the cause, report that one
    ctx->path_stats = eng.stats;
    kc_emit_check(h + KC_SPEC_EMIT, hs[2], t.total_ub);
    res.ms = t.ms;
    res.maxone = nullptr;
    res.length = h[KC_SPEC_EMIT + 2];
    res.slice_begin = 0;
    res.slice_len = res.length;
    res.n_kmers = h[0];
    res.n_occ = h[2];
    res.n_nodes = hs[1];
    res.n_simplitigs = hs[1];
    return KC_SPEC_OK;
}

// The signature construction into `flags` and the speculative tail behind it, with programmatic dependent launches: directly while
// the kernel-class timers are on (they bracket every launch with events) or the input is still being copied in, otherwise as a cached
// graph (SpecGraph) that the first call of a shape captures from the same launches.  Returns false (nothing queued) when the
// signature plan does not apply.
template <int L>
bool run_sig_spec(kc_ctx *ctx, CudaExec &ex, const DevInput &in, const kc_params &p, u32 *flags, u64 **blk, SpecTail &t) {
    if (!kc_sig_plan(in.n_bytes, p.k, ctx->routes.sig).ok) {
        ex.arena->alloc_top<u64>(KC_SPEC_BLOCK_WORDS);  // as every rung, the block stays allocated when the plan does not apply
        return false;
    }
    auto queue = [&] {
        *blk = ex.arena->alloc_top<u64>(KC_SPEC_BLOCK_WORDS);
        kc_kmerset_build_sig<L>(ex, in.seq, in.n_bytes, p.k, p.complements != 0, flags, *blk, ctx->routes.sig, in.chunks, nullptr, nullptr,
                                KC_SPEC_BLOCK_WORDS);
        t = tail_spec_queue<L>(ctx, ex, in, p, flags, *blk);
    };
    ex.pdl = true;
    if ((ex.prof && ex.prof->enabled) || in.chunks) {
        queue();
        ex.pdl = false;
        return true;
    }
    Arena &A = *ex.arena;
    SpecGraph key;
    key.limbs = L;
    key.k = p.k;
    key.complements = p.complements != 0;
    key.n_bytes = in.n_bytes;
    key.arena_base = A.base;
    key.arena_at = A.checkpoint();
    key.flags = flags;
    SpecGraph *g = nullptr;
    for (SpecGraph &c : ctx->spec_graphs)
        if (c.same_shape(key)) g = &c;
    if (g) {
        A.restore(g->arena_after);
        if (g->arena_high > A.high) A.high = g->arena_high;
        *blk = g->blk;
        t = g->tail;
        ++ctx->spec_graph_replays;
    } else {
        if (ctx->spec_graphs.size() >= kc_ctx::KC_SPEC_GRAPHS) ctx->clear_spec_graphs();
        if (!ctx->capture_stream) KC_CUDA(cudaStreamCreateWithFlags(&ctx->capture_stream, cudaStreamNonBlocking));
        key.patch.seq = in.seq;
        const u64 launches0 = ex.launches;
        cudaStream_t run_stream = ex.stream;
        auto end_capture = [&](cudaGraph_t *graph) {  // the capture stream only records: nothing runs until the graph is launched
            ex.patch = nullptr;
            ex.stream = A.stream = run_stream;
            return cudaStreamEndCapture(ctx->capture_stream, graph);
        };
        KC_CUDA(cudaStreamBeginCapture(ctx->capture_stream, cudaStreamCaptureModeRelaxed));
        ex.stream = A.stream = ctx->capture_stream;
        ex.patch = &key.patch;
        try {
            queue();
        } catch (...) {
            ex.pdl = false;
            cudaGraph_t partial = nullptr;
            end_capture(&partial);
            if (partial) cudaGraphDestroy(partial);
            (void) cudaGetLastError();
            throw;
        }
        KC_CUDA(end_capture(&key.graph));
        if (cudaGraphInstantiate(&key.exec, key.graph, 0) != cudaSuccess) {
            key.destroy();
            ex.pdl = false;
            KC_THROW(KC_ERR_CUDA, "cudaGraphInstantiate failed");
        }
        key.launches = ex.launches - launches0;
        ex.launches = launches0;
        key.arena_after = A.checkpoint();
        key.arena_high = A.high;
        key.blk = *blk;
        key.tail = t;
        ctx->spec_graphs.push_back(std::move(key));
        g = &ctx->spec_graphs.back();
        ++ctx->spec_graph_captures;
    }
    ex.pdl = false;
    g->patch.set_seq(g->exec, in.seq);
    KC_CUDA(cudaGraphLaunch(g->exec, ex.stream));
    ex.launches += g->launches;
    for (int i = 2; i <= 4; ++i) KC_CUDA(cudaEventRecord(ctx->ev[i], ex.stream));  // the stage timers see the graph as one piece
    return true;
}

// From-FASTA regime: the nodes handed to the overlap stage are FIRST-OCCURRENCE RUNS.
//
// The reference turns the k-mer set into simplitigs by walking a hash table (src/simplitigs.h:105-205); which
// simplitigs come out depends on khash iteration order and is unspecified (its tests sort them before comparing).
// Here every k-mer occurrence carries the position of its window through the partition passes, the distinct k-mer
// keeps its smallest position, and those positions are flagged in the input.  A maximal run of consecutive flagged
// positions is a path of distinct k-mers whose neighbours overlap by k-1 (adjacent windows of one record): a
// simplitig read directly off the input, with no hash walk and no per-k-mer pointer chasing.  Runs are numbered
// in input order and go through the same overlap levels d = k-1..0 as `-S` records, so run ends that overlap by
// k-1 are still joined first, exactly as BIGREEDY requires.
//
// The first-occurrence flags come from kc_set_ladder (set_routes.cuh), or else from the exact construction.
// spec_res != nullptr: after the signature construction, try the speculative tail (run_sig_spec).  When it holds, *spec_res is the whole
// result and *spec_done is set; otherwise the runs are counted as if it had not been tried, on the same flags.
template <int L>
Stage1<L> run_stage1_runs(kc_ctx *ctx, CudaExec &ex, const DevInput &in, const kc_params &p, DevResult *spec_res, bool *spec_done) {
    Stage1<L> s;
    KC_CUDA(cudaEventRecord(ctx->ev[0], ex.stream));
    KC_CUDA(cudaEventRecord(ctx->ev[1], ex.stream));  // extraction is fused into the partition passes
    KC_TRACE_POINT("stage1: begin");
    const u64 nb = in.n_bytes;
    const size_t fwords = kc_runs_flag_words(nb);
    u32 *flags = ex.arena->alloc_top<u32>(fwords);  // zeroed by the construction that fills it (the signature scan writes every word)
    u64 *cells = ex.arena->alloc_top<u64>(2);  // {kept distinct k-mers, runs}
    u64 *cells4 = nullptr, hc[4];
    KsfPlan plan;
    SpecTail tail;
    auto launch = [&](KcRoute r) {
        if (r == KC_ROUTE_SIG && spec_res) return run_sig_spec<L>(ctx, ex, in, p, flags, &cells4, tail);
        cells4 = ex.arena->alloc_top<u64>(4);  // {kept, runs, M, overflow status}
        if (r == KC_ROUTE_SIG) return kc_kmerset_build_sig<L>(ex, in.seq, nb, p.k, p.complements != 0, flags, cells4, ctx->routes.sig, in.chunks, nullptr, nullptr, 4);
        ex.fill_bytes(flags, 0, fwords * 4);
        ex.fill_bytes(cells4, 0, 32);
        return kc_kmerset_build_fast<L>(ex, in.seq, nb, p.k, p.complements != 0, p.min_frequency, flags, cells4, ctx->routes.fast, &plan, in.chunks);
    };
    auto consume = [&](KcRoute r) {
        KC_TRACE_POINT(r == KC_ROUTE_SIG ? "stage1: signature set launched" : "stage1: fast set launched");
        bool aborted = false;
        if (r == KC_ROUTE_SIG && spec_res) {
            const u32 st = tail_spec_finish<L>(ctx, ex, tail, *spec_res);
            if (st == KC_SPEC_OK) {
                ++ctx->tail_spec_runs;
                *spec_done = true;
                return true;
            }
            ++ctx->tail_spec_fallbacks;
            aborted = st == KC_SPEC_SIG_OVERFLOW;
            if (!aborted) {  // the flags stand: the ordinary tail counts the runs again
                if (st != KC_SPEC_EMPTY) ctx->routes.tail.remember(nb);
                ex.fill_bytes(cells4 + 1, 0, 8);
            }
        }
        if (!aborted) s.nodes = kc_runs_from_flags(ex, flags, nb, p.k, cells4, hc, 4, &aborted);
        return !aborted;  // incomplete flags: the next construction clears them first
    };
    const KcRoute route = kc_set_ladder(ctx->routes, ctx->routes.compute_policy(p, nb), nb, *ex.arena, launch, consume);
    if (route != KC_ROUTE_NONE) {
        if (*spec_done) return s;
        // the timers charged the fixed-slot partition passes with M = n_bytes; now that M is known, correct the byte counts
        if (route == KC_ROUTE_FAST && ex.prof && ex.prof->enabled && nb > hc[2]) {
            const u64 d = (nb - hc[2]) * (sizeof(KWord<L>) + 4);
            ex.prof->bytes[KP_KS_SCATTER0] -= d;
            ex.prof->bytes[KP_SORT_SCATTER] -= 2 * d * (u64) (plan.n_levels - 1);
            ex.prof->bytes[KP_KS_RESOLVE] -= d;
        }
        s.n_occ = hc[2];
        s.U = hc[2] ? hc[0] : 0;
        return s;
    }
    // with -M the sorted k-mer set doubles as kMersDict of src/global.h:165-167; it stays at the arena bottom
    if (in.chunks) in.chunks->wait_all(ex.stream);
    ex.fill_bytes(flags, 0, fwords * 4);
    ex.fill_bytes(cells, 0, 16);
    KmerSet<L> set = kc_kmerset_build<L>(ex, in.seq, nb, p.k, p.complements != 0, p.min_frequency, flags, p.want_maxone != 0, cells);
    KC_TRACE_POINT("stage1: set built");
    s.n_occ = set.n_occ;
    s.uniq = set.keys;
    if (set.n_occ == 0 || set.n_kept == 0) return s;
    if (p.want_maxone) {  // the KEYS path has read the count back already
        const u64 kept = set.n_kept;
        KC_CUDA(cudaMemcpyAsync(cells, &kept, 8, cudaMemcpyHostToDevice, ex.stream));
    }
    u64 host_cells[2];
    s.nodes = kc_runs_from_flags(ex, flags, nb, p.k, cells, host_cells);
    s.U = p.want_maxone ? set.n_kept : host_cells[0];
    KC_TRACE_POINT("stage1: runs built");
    return s;
}

// From stage 1's outcome to the result: the sparse switch, the node ends, the overlap stage, then the lower bound or the emission
// (of slice `slice_index` of `n_slices`).  Stage 1 ends here, at event 2.
template <int L>
void run_tail(kc_ctx *ctx, CudaExec &ex, const DevInput &in, const kc_params &p, Stage1<L> s, DevResult &res, bool lower_bound,
              u32 slice_index = 0, u32 n_slices = 1) {
    const bool complements = p.complements != 0;
    KC_CUDA(cudaEventRecord(ctx->ev[2], ex.stream));
    res.n_simplitigs = s.nodes.n_runs;
    if (!p.assume_simplitigs) {
        if (s.U == 0) KC_THROW(KC_ERR_EMPTY, "the input contains no k-mers");  // src/main.cpp:155-158
        // src/main.cpp:94,175-181: simplitigs barely longer than k-mers -> the greedy runs on the k-mers themselves (PartialPreSort order)
        if (ctx->sparse_switch && s.nodes.n_runs * 5 >= s.U) {
            // one node per k-mer; kc_kmer_nodes_from_runs numbers them with 32-bit offsets (inputs of 2^32 bytes or more can have that many)
            if (s.U * (complements ? 2 : 1) >= 0xFFFFFFF0ULL) KC_THROW(KC_ERR_TOO_LARGE, "too many nodes for one GPU");
            s.nodes = kc_kmer_nodes_from_runs(ex, in.seq, s.nodes, p.k);
        }
        if (s.nodes.n_runs * (complements ? 2 : 1) >= 0xFFFFFFF0ULL) KC_THROW(KC_ERR_TOO_LARGE, "too many nodes for one GPU");
    }
    const u64 n_nodes = s.nodes.n_runs;
    const u64 *node_off = s.nodes.rec_off, *node_len = s.nodes.rec_len;
    NodeView<L> nv;
    nv.k = p.k;
    nv.complements = complements;
    {
        KWord<L> *first = ex.alloc<KWord<L>>(n_nodes), *last = ex.alloc<KWord<L>>(n_nodes);
        u32 *err = ex.alloc<u32>(1);
        ex.fill_bytes(err, 0, 4);
        kc_extract_node_ends<L>(ex, in.seq, in.n_bytes, node_off, node_len, n_nodes, p.k, first, last, err,
                                /*validate_bytes=*/p.assume_simplitigs != 0);
        // first-occurrence runs are valid by construction; only -S records need the check (and its read-back)
        if (p.assume_simplitigs && ex.read(err)) KC_THROW(KC_ERR_BAD_SEQ, "-S input must hold only ACGT records of at least k bases");
        nv.first = first;
        nv.last = last;
        nv.n = (u32) n_nodes;
    }
    nv.N = nv.n * (complements ? 2u : 1u);
    NodeSeq<L> ns;
    ns.k = p.k;
    ns.kmers = nullptr;
    ns.seq = in.seq;
    ns.rec_off = node_off;
    ns.rec_len = node_len;
    ns.n = nv.n;
    KC_TRACE_POINT("pipeline: nodes ready");
    Engine<CudaExec, L> eng(ex, nv, /*strict=*/p.assume_simplitigs != 0, lower_bound);
    eng.use_small = ctx->small_engine;
    eng.small_threads_opt = ctx->small_threads;
    eng.init_state();
    eng.run();
    KC_TRACE_POINT("pipeline: engine done");
    KC_CUDA(cudaEventRecord(ctx->ev[3], ex.stream));
    if (lower_bound) {
        // src/lower_bound.h:10-22: (sum of node lengths over both strands - sum of the cycle cover's overlaps) / strands.
        // In this mode every virtual node has an out-edge after d = 0, so no 255 is left among the overlaps.
        kc_ull *acc = reinterpret_cast<kc_ull *>(ex.alloc<u64>(2));
        ex.fill_bytes(acc, 0, 16);
        const u64 *len = node_len;
        const u8 *ovl = eng.st.ovl;
        const u32 n = nv.n;
        ex.for_each(nv.N, [=] __device__(u64 i) {
            if (i < n) atomicAdd(&acc[0], (kc_ull) len[i]);
            if (ovl[i]) atomicAdd(&acc[1], (kc_ull) ovl[i]);
        });
        u64 h[2];
        ex.read_n(reinterpret_cast<const u64 *>(acc), h, 2);
        eng.check_small();
        ctx->path_stats = eng.stats;
        const u64 strands = complements ? 2 : 1;
        res.lower_bound = (h[0] * strands - h[1]) / strands;
        KC_CUDA(cudaEventRecord(ctx->ev[4], ex.stream));
        res.n_kmers = s.U;
        res.n_occ = s.n_occ;
        res.n_nodes = nv.n;
        return;
    }
    EmitResult er;
    try {
        // every character of the superstring is a character of some node: nodes are pieces of the input that overlap by < k
        er = kc_emit_superstring<CudaExec, L>(ex, ns, nv, eng.st, s.uniq, s.U, p.want_maxone != 0, slice_index, n_slices, in.n_bytes + n_nodes * (u64) p.k + 16);
    } catch (const KcError &) {
        eng.check_small();  // a failed small-engine run is the cause, report that one
        throw;
    }
    KC_CUDA(cudaEventRecord(ctx->ev[4], ex.stream));
    eng.check_small();  // deferred status of the single-CTA engine kernel: everything above is queued already
    ctx->path_stats = eng.stats;
    res.ms = er.ms;
    res.maxone = er.maxone;
    res.length = er.length;
    res.slice_begin = er.slice_begin;
    res.slice_len = er.slice_len;
    res.n_kmers = s.U;
    res.n_occ = s.n_occ;
    res.n_nodes = nv.n;
}

// One GPU: stage 1 (the -S records, or the first-occurrence runs, behind which the speculative tail may finish the call), then
// run_tail.
template <int L> void run_pipeline(kc_ctx *ctx, CudaExec &ex, const DevInput &in, const kc_params &p, DevResult &res, bool lower_bound) {
    Stage1<L> s;
    if (p.assume_simplitigs) {
        if (in.n_recs == 0) KC_THROW(KC_ERR_EMPTY, "input cannot be empty");  // src/global.h:219-221
        if (in.n_recs * (p.complements ? 2 : 1) >= 0xFFFFFFF0ULL) KC_THROW(KC_ERR_TOO_LARGE, "too many records for one GPU");
        KC_CUDA(cudaEventRecord(ctx->ev[0], ex.stream));
        if (p.want_maxone) {  // kMersDict of src/global.h:165-167 = every k-mer of the records
            u8 *cnt = nullptr;
            s.U = run_stage1<L>(ctx, ex, in, p, &s.uniq, &cnt, &s.n_occ);
        } else {
            KC_CUDA(cudaEventRecord(ctx->ev[1], ex.stream));
        }
        s.nodes = RunNodes{in.rec_off, in.rec_len, in.n_recs};
    } else {
        // the speculative tail: a FASTA input with few runs (a genome) is computed behind one read-back (run_sig_spec)
        const u64 nb = in.n_bytes;
        const bool spec_failed = ctx->routes.heuristics && ctx->routes.tail.near(nb);
        const bool spec = ctx->tail_spec && !spec_failed && !lower_bound && ctx->small_engine && nb > 0 && nb < KC_POS32_BYTES;
        bool spec_done = false;
        s = run_stage1_runs<L>(ctx, ex, in, p, spec ? &res : nullptr, &spec_done);
        if (spec_done) return;
    }
    run_tail<L>(ctx, ex, in, p, s, res, lower_bound);
}

void fill_times(kc_ctx *ctx, kc_output *out) {
    float t = 0;
    out->t = kc_stage_times{0, 0, 0, 0, 0};
    if (cudaEventElapsedTime(&t, ctx->ev[0], ctx->ev[1]) == cudaSuccess) out->t.extract_ms = t;
    if (cudaEventElapsedTime(&t, ctx->ev[1], ctx->ev[2]) == cudaSuccess) out->t.count_ms = t;
    if (cudaEventElapsedTime(&t, ctx->ev[2], ctx->ev[3]) == cudaSuccess) out->t.path_ms = t;
    if (cudaEventElapsedTime(&t, ctx->ev[3], ctx->ev[4]) == cudaSuccess) out->t.emit_ms = t;
    if (cudaEventElapsedTime(&t, ctx->ev[0], ctx->ev[4]) == cudaSuccess) out->t.total_ms = t;
    (void) cudaGetLastError();
}

// A call's result in the ABI's form, with the device pointers of `res` (kc_compute points them at its pinned copy).
void fill_output(kc_ctx *ctx, const DevResult &res, u64 launches, kc_output *out) {
    out->ms = const_cast<u8 *>(res.ms);
    out->ms_maxone = const_cast<u8 *>(res.maxone);
    out->length = res.length;
    out->n_kmers = res.n_kmers;
    out->n_occurrences = res.n_occ;
    out->n_nodes = res.n_nodes;
    out->n_simplitigs = res.n_simplitigs;
    out->n_launches = launches;
    fill_times(ctx, out);
}

// Device result -> the context's pinned host buffer; with -M the max-one mask follows the superstring there.
u8 *copy_to_pinned(kc_ctx *ctx, const u8 *ms, const u8 *maxone, u64 n) {
    ctx->pin_out.reserve((size_t) n * (maxone ? 2 : 1) + 64);
    if (n) KC_CUDA(cudaMemcpyAsync(ctx->pin_out.p, ms, n, cudaMemcpyDeviceToHost, ctx->stream));
    if (maxone) KC_CUDA(cudaMemcpyAsync(ctx->pin_out.p + n, maxone, n, cudaMemcpyDeviceToHost, ctx->stream));
    KC_CUDA(cudaStreamSynchronize(ctx->stream));
    return ctx->pin_out.p;
}

template <int L>
void count_only(kc_ctx *ctx, CudaExec &ex, const DevInput &in, const kc_params &p, uint64_t **keys, uint8_t **counts, uint64_t *n) {
    KWord<L> *uniq = nullptr;
    u8 *cnt = nullptr;
    u64 n_occ = 0;
    u64 U = run_stage1<L>(ctx, ex, in, p, &uniq, &cnt, &n_occ);
    *n = U;
    *keys = (uint64_t *) std::malloc(U ? U * sizeof(KWord<L>) : 8);
    *counts = (uint8_t *) std::malloc(U ? U : 1);
    if (!*keys || !*counts) KC_THROW(KC_ERR_OOM, "host allocation failed");
    if (U) {
        KC_CUDA(cudaMemcpyAsync(*keys, uniq, U * sizeof(KWord<L>), cudaMemcpyDeviceToHost, ex.stream));
        KC_CUDA(cudaMemcpyAsync(*counts, cnt, U, cudaMemcpyDeviceToHost, ex.stream));
    }
    KC_CUDA(cudaStreamSynchronize(ex.stream));
}

// kc_kmer_digest: (n, sum h, xor h, sum h * c) over the kept (k-mer, c = min(occurrences, 256), or 1 without -z) pairs, h = the splitmix64 fold of
// the limbs (kc_kmer_hash).  The same four numbers come out of oracle/ref_harness `full` for the reference's own hash table.
// Without -z the set is first tried as first-occurrence flags (kc_set_ladder), hashed window by window (digest.cuh); the sorted keys
// of kc_kmerset_build are the other route.  The digest is a function of the set: both give the same four words.  win_mask: optional
// window filter over END positions, sized for the signature scan's tiles of 256 * 32 positions.
template <int L>
void digest_only(kc_ctx *ctx, CudaExec &ex, const DevInput &in, const kc_params &p, const u32 *win_mask, uint64_t *digest) {
    KC_CUDA(cudaEventRecord(ctx->ev[0], ex.stream));
    if (p.min_frequency == 1) {  // c = 1: digest[3] = digest[1]
        const ArenaMark mark = ex.arena->checkpoint();
        const size_t fwords = kc_runs_flag_words(in.n_bytes);
        u32 *flags = ex.arena->alloc_top<u32>(fwords);
        ex.fill_bytes(flags, 0, fwords * 4);
        u64 *cells = ex.arena->alloc_top<u64>(8);  // {kept, -, M, status, n, sum h, xor h, -}
        ex.fill_bytes(cells, 0, 64);
        kc_ull *acc = reinterpret_cast<kc_ull *>(cells + 4);
        u64 hc[7];
        RoutePolicy pol;
        pol.sig = true;
        const KcRoute route = kc_set_ladder(ctx->routes, pol, in.n_bytes, *ex.arena, [&](KcRoute) {
            return kc_kmerset_build_sig<L>(ex, in.seq, in.n_bytes, p.k, p.complements != 0, flags, cells, ctx->routes.sig, nullptr, win_mask);
        }, [&](KcRoute) {
            kc_flag_digest<L>(ex, in.seq, in.n_bytes, flags, fwords, p.k, p.complements != 0, acc);
            ex.read_n(cells, hc, 7);
            return hc[3] == 0;
        });
        if (route == KC_ROUTE_SIG) {
            digest[0] = hc[4];
            digest[1] = hc[5];
            digest[2] = hc[6];
            digest[3] = hc[5];
            return;
        }
        ex.arena->restore(mark);
    }
    KmerSet<L> set = kc_kmerset_build<L>(ex, in.seq, in.n_bytes, p.k, p.complements != 0, p.min_frequency, nullptr, true, nullptr, win_mask);
    const u64 U = set.n_kept;
    kc_ull *acc = reinterpret_cast<kc_ull *>(ex.alloc<u64>(4));
    ex.fill_bytes(acc, 0, 32);
    const KWord<L> *keys = set.keys;
    const u8 *cnt = set.cnt;
    const bool counted = p.min_frequency > 1;  // ReadKMers (-z 1) keeps no counts: c = 1
    ex.for_each(kc_div_up(U, 32) * 32, [=] __device__(u64 i) {
        u64 h = 0, wv = 0;
        if (i < U) {
            h = kc_kmer_hash<L>(keys[i]);
            wv = counted ? h * ((u64) cnt[i] + 1) : h;
        }
        u64 s = h, x = h;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            s += __shfl_xor_sync(0xFFFFFFFFu, s, o);
            x ^= __shfl_xor_sync(0xFFFFFFFFu, x, o);
            wv += __shfl_xor_sync(0xFFFFFFFFu, wv, o);
        }
        if ((threadIdx.x & 31) == 0) {
            atomicAdd(&acc[1], (kc_ull) s);
            atomicXor(&acc[2], (kc_ull) x);
            atomicAdd(&acc[3], (kc_ull) wv);
        }
    }, KP_MISC, U * (sizeof(KWord<L>) + 1));
    u64 h4[4];
    ex.read_n(reinterpret_cast<const u64 *>(acc), h4, 4);
    digest[0] = U;
    digest[1] = h4[1];
    digest[2] = h4[2];
    digest[3] = h4[3];
}

template <int L>
void overlap_only(kc_ctx *ctx, CudaExec &ex, const uint64_t *first, const uint64_t *last, u64 n, int k, bool complements, bool lower_bound,
                  bool strict, int64_t *edge_from, uint8_t *overlaps) {
    KWord<L> *df = ex.alloc<KWord<L>>(n), *dl = ex.alloc<KWord<L>>(n);
    KC_CUDA(cudaMemcpyAsync(df, first, n * sizeof(KWord<L>), cudaMemcpyHostToDevice, ex.stream));
    KC_CUDA(cudaMemcpyAsync(dl, last, n * sizeof(KWord<L>), cudaMemcpyHostToDevice, ex.stream));
    NodeView<L> nv;
    nv.first = df;
    nv.last = dl;
    nv.n = (u32) n;
    nv.N = nv.n * (complements ? 2u : 1u);
    nv.k = k;
    nv.complements = complements;
    Engine<CudaExec, L> eng(ex, nv, strict, lower_bound);
    eng.use_small = ctx->small_engine;
    eng.small_threads_opt = ctx->small_threads;
    eng.init_state();
    eng.run();
    eng.check_small();
    ctx->path_stats = eng.stats;
    std::vector<u32> ef(nv.N);
    KC_CUDA(cudaMemcpyAsync(ef.data(), eng.st.edge_from, (size_t) nv.N * 4, cudaMemcpyDeviceToHost, ex.stream));
    KC_CUDA(cudaMemcpyAsync(overlaps, eng.st.ovl, nv.N, cudaMemcpyDeviceToHost, ex.stream));
    KC_CUDA(cudaStreamSynchronize(ex.stream));
    for (u32 i = 0; i < nv.N; ++i) edge_from[i] = ef[i] == KC_NONE ? -1 : (int64_t) ef[i];
}

// ---- multi-GPU: one context = one rank of a group (group.cuh) ---------------------------------------------------------------------
void group_alloc_common(kc_ctx *ctx, int n_ranks, int rank, int k, uint64_t n_bytes_cap, bool with_seq) {
    if (n_ranks < 1 || n_ranks > KC_MAX_PEERS || rank < 0 || rank >= n_ranks) KC_THROW(KC_ERR_ARG, "bad rank / group size");
    if (k < 1 || k > 127) KC_THROW(KC_ERR_ARG, "k must be in 1..127");
    if (n_bytes_cap >= KC_POS32_BYTES)
        if (const char *why = kc_grp_large_bound(n_bytes_cap, n_ranks)) KC_THROW(KC_ERR_TOO_LARGE, why);
    KcGroup &G = ctx->grp;
    if (G.heap) KC_THROW(KC_ERR_ARG, "this context already belongs to a group");
    KC_CUDA(cudaSetDevice(ctx->device));
    G.n = n_ranks;
    G.rank = rank;
    G.lay = kc_grp_layout(n_bytes_cap, kc_limbs_for_k(k), n_ranks, with_seq, kc_shard_granule(k), ctx->routes.fast);
    KC_CUDA(cudaMalloc(reinterpret_cast<void **>(&G.heap), G.lay.total));
    KC_CUDA(cudaMemset(G.heap, 0, G.lay.off_flags));  // sync words, cells, counts
    KC_CUDA(cudaMalloc(reinterpret_cast<void **>(&G.cnt0), 256 * 4));
    KC_CUDA(cudaMalloc(reinterpret_cast<void **>(&G.cells_local), 64));
    KC_CUDA(cudaMalloc(reinterpret_cast<void **>(&G.dst_k), 256 * sizeof(void *)));
    KC_CUDA(cudaMalloc(reinterpret_cast<void **>(&G.dst_p), 256 * sizeof(void *)));
    KC_CUDA(cudaHostAlloc(reinterpret_cast<void **>(&G.h_dst), 512 * sizeof(void *), cudaHostAllocDefault));
    KC_CUDA(cudaDeviceSynchronize());
    for (int r = 0; r < KC_MAX_PEERS; ++r) G.peer[r] = nullptr;
    G.peer[rank] = G.heap;
    G.seq = 0;
    G.done_pending = false;
    G.failed = false;
    G.refused = false;
    G.tab_n_bytes = ~0ull;
    if (const char *e = std::getenv("KC_GROUP_TIMEOUT_MS")) G.timeout_ns = (u64) std::atoll(e) * 1000000ull;
}

void group_detach(kc_ctx *ctx) {
    KcGroup &G = ctx->grp;
    if (!G.heap) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    for (int r = 0; r < G.n && r < KC_MAX_PEERS; ++r)
        if (G.ipc_opened[r]) {
            cudaIpcCloseMemHandle(G.peer[r]);
            G.ipc_opened[r] = false;
        }
    cudaFree(G.heap);
    if (G.cnt0) cudaFree(G.cnt0);
    if (G.cells_local) cudaFree(G.cells_local);
    if (G.dst_k) cudaFree(G.dst_k);
    if (G.dst_p) cudaFree(G.dst_p);
    if (G.h_dst) cudaFreeHost(G.h_dst);
    if (G.tile_hist) cudaFree(G.tile_hist);
    G = KcGroup();
    (void) cudaGetLastError();
}

// Arena of one rank for a job of n_bytes: the owner-side levels over its hash range (two ping-pong generations of fixed slots, or
// the exact construction's buffers), the node-dependent part of the overlap stage and the emission scratch.
// Inputs of KC_POS32_BYTES or more take the signature construction alone (`sig`: its plan at this size).  Its scratch is released
// before the runs are counted (kc_grp_sig_flags), so a rank needs the larger of it and the overlap stage + emission of one GPU
// (estimate_arena): the sequence, the flags and the code words live in the heap.  Ranks that share a device need this once each.
size_t group_arena_need(u64 n_bytes, int n_ranks, int limbs, bool complements, bool pessimistic, const SigPlan *sig = nullptr) {
    if (n_bytes >= KC_POS32_BYTES && sig && sig->ok) {
        const double tail = overlap_emit_bytes(pessimistic ? n_bytes * 0.85 : n_bytes / 64.0 + 1e6, limbs, complements, n_bytes);
        return (size_t) (std::max(tail, (double) kc_sig_group_arena_bytes(*sig, n_bytes, n_ranks)) * 1.1) + (256u << 20);
    }
    const double owned = (double) n_bytes / n_ranks * 1.3 + (1u << 20);
    const double stage1 = owned * (8.0 * limbs + 4.0 + 2.0) * 4.0;
    const double c = complements ? 2.0 : 1.0;
    const double nodes = pessimistic ? n_bytes * 0.85 : n_bytes / 64.0 + 1e6;
    return (size_t) ((stage1 + c * nodes * (240.0 + 32.0 * limbs) + 3.0 * n_bytes) * 1.1) + (256u << 20);
}

// One job of this rank.  `in.seq` is the WHOLE framed sequence, resident on this GPU.  Every rank of the group must make the
// same call (same input, same parameters, same options) at about the same time.
template <int L> void group_compute_rank(kc_ctx *ctx, CudaExec &ex, const DevInput &in, const kc_params &p, DevResult &res) {
    KcGroup &G = ctx->grp;
    const u64 nb = in.n_bytes;
    KC_CUDA(cudaEventRecord(ctx->ev[0], ex.stream));
    KC_CUDA(cudaEventRecord(ctx->ev[1], ex.stream));
    if (G.done_pending) {  // every rank has finished the previous job: its heaps may be written again
        u32 *ws = reinterpret_cast<u32 *>(ex.arena->alloc_top<u64>(1));
        ex.fill_bytes(ws, 0, 8);
        kc_grp_wait(G, ex, G.done_seq, ws);
        G.done_pending = false;
    }
    // every rank takes the same decisions from values it sees identically: a rung that overflowed on one rank sets the status
    // word every rank reads
    RoutePolicy pol = ctx->routes.compute_policy(p, nb);
    const KsfGroupPlan gp = kc_ksf_group_plan(nb, G.n, KsCfg<L>::EX_TILE, ctx->routes.fast);
    pol.fast = pol.fast && gp.ok && gp.recv_items() <= G.lay.recv_items;
    const u32 *flags = reinterpret_cast<const u32 *>(G.heap + G.lay.off_flags);
    u64 *cells4 = nullptr;  // device words {kept, 0, M, status}, read back together with the run count
    auto ladder = [&] {
        return kc_set_ladder(ctx->routes, pol, nb, *ex.arena, [&](KcRoute r) {
            cells4 = r == KC_ROUTE_SIG ? kc_grp_sig_flags<L>(G, ex, in.seq, nb, p.k, p.complements != 0, ctx->routes.sig)
                                       : kc_grp_fast_flags<L>(G, ex, in.seq, nb, p.k, p.complements != 0, p.min_frequency, gp, ctx->routes.fast);
            return cells4 != nullptr;
        }, [&](KcRoute) {
            Stage1<L> s;
            u64 hc[4];
            bool aborted = false;  // the status word was set (a slot overflowed somewhere): nothing was done
            s.nodes = kc_runs_from_flags(ex, flags, nb, p.k, cells4, hc, 4, &aborted);
            if (aborted && (hc[3] & 2u)) {
                G.failed = true;
                KC_THROW(KC_ERR_INTERNAL, "a rank of the group did not arrive (wait timed out)");
            }
            if (aborted) return false;
            s.U = hc[2] ? hc[0] : 0;
            s.n_occ = hc[2];
            run_tail<L>(ctx, ex, in, p, s, res, false, (u32) G.rank, (u32) G.n);
            return true;
        });
    };
    KcRoute route = KC_ROUTE_NONE;
    if (nb < KC_POS32_BYTES) {
        route = ladder();
    } else {
        // The signature rung alone.  Its refusals (a bucket overflow, seen by every rank through the shared status word; too many
        // runs or nodes, from totals every rank reads) come on every rank at the same point: the job is closed like a finished one,
        // so that the sync numbers stay aligned and the next job waits for every rank's DONE as usual.
        try {
            route = ladder();
        } catch (const KcError &e) {
            if (e.code != KC_ERR_TOO_LARGE || G.failed) throw;
            G.done_seq = ++G.seq;
            kc_grp_signal(G, ex, G.done_seq);
            G.done_pending = true;
            G.refused = true;
            throw;
        }
    }
    if (route == KC_ROUTE_NONE) {  // the exact construction: its totals are on the host already
        Stage1<L> s;
        u64 kept = 0;
        const u32 *xflags = kc_grp_exact_flags<L>(G, ex, in.seq, nb, p.k, p.complements != 0, p.min_frequency, &kept, &s.n_occ);
        u64 *cells = ex.arena->alloc_top<u64>(2);
        ex.fill_bytes(cells, 0, 16);
        u64 host_cells[2];
        s.nodes = kc_runs_from_flags(ex, xflags, nb, p.k, cells, host_cells);
        s.U = s.nodes.n_runs ? kept : 0;
        run_tail<L>(ctx, ex, in, p, s, res, false, (u32) G.rank, (u32) G.n);
    }
    G.done_seq = ++G.seq;
    kc_grp_signal(G, ex, G.done_seq);
    G.done_pending = true;
}

// A group takes an input of KC_POS32_BYTES or more wherever one GPU does (check_large_input), through the same construction with
// 64-bit positions, within the 32-bit bounds of its exchange (kc_grp_large_bound).  Every rank refuses from the same values, before
// anything of the job is queued, so a refusal leaves the group in step.
void group_check_large(const kc_ctx *ctx, const kc_params *p, u64 n_bytes, int n_ranks) {
    if (n_bytes < KC_POS32_BYTES) return;
    check_large_input(ctx, p, n_bytes);
    if (const char *why = kc_grp_large_bound(n_bytes, n_ranks)) KC_THROW(KC_ERR_TOO_LARGE, why);
}

void group_check_job(kc_ctx *ctx, const kc_params *p, u64 n_bytes) {
    check_params(p);
    KcGroup &G = ctx->grp;
    if (!G.attached()) KC_THROW(KC_ERR_ARG, "this context is not part of a group");
    for (int r = 0; r < G.n; ++r)
        if (!G.peer[r]) KC_THROW(KC_ERR_ARG, "the group's heaps have not been opened");
    if (G.failed) KC_THROW(KC_ERR_INTERNAL, "the group lost its synchronisation in an earlier call; create a new one");
    if (p->assume_simplitigs || p->want_maxone) KC_THROW(KC_ERR_ARG, "the multi-GPU construction supports neither -S nor -M");
    if (kc_limbs_for_k(p->k) > G.lay.limbs) KC_THROW(KC_ERR_ARG, "the group heap was sized for a narrower k-mer word");
    if (n_bytes > G.lay.n_bytes_cap) KC_THROW(KC_ERR_TOO_LARGE, "the input exceeds the capacity the group heap was sized for");
    if (G.lay.pos64() && n_bytes < KC_POS32_BYTES)
        KC_THROW(KC_ERR_ARG, "the group heap was sized for inputs of 2^32 bytes or more (signature construction only); smaller inputs need a heap with a cap below 2^32");
    group_check_large(ctx, p, n_bytes, G.n);
}

// Readies this rank's arena for a job (group_arena_need).  There is no retry with a larger arena: a rank that repeated its job alone
// would leave the group's sync numbers behind.  A rank that ran out of arena half way would strand the others, so an input of
// KC_POS32_BYTES or more whose arena the device cannot hold is refused with `refusal` before anything is queued.
void group_prepare_arena(kc_ctx *ctx, const kc_params &p, u64 n_bytes, const char *refusal) {
    const SigPlan sig = kc_sig_plan(n_bytes, p.k, ctx->routes.sig);
    const size_t need = group_arena_need(n_bytes, ctx->grp.n, kc_limbs_for_k(p.k), p.complements != 0, false, &sig);
    ensure_arena(ctx, need);
    if (n_bytes >= KC_POS32_BYTES && ctx->arena.cap < need) KC_THROW(KC_ERR_OOM, refusal);
}

// Marks the group failed unless error `code` leaves it in step: "no k-mers" and the refusals of group_compute_rank are found by
// every rank at the same point, anything else strands the other ranks.  Returns whether it did.
bool group_fail(kc_ctx *ctx, int code) {
    if (code == KC_ERR_EMPTY || ctx->grp.refused) return false;
    ctx->grp.failed = true;
    return true;
}

// This rank's job (group_compute_rank), at the word width of k.
void group_run_job(kc_ctx *ctx, CudaExec &ex, const DevInput &in, const kc_params &p, DevResult &res) {
    try {
        with_limbs(kc_limbs_for_k(p.k), [&](auto l) { group_compute_rank<decltype(l)::value>(ctx, ex, in, p, res); });
    } catch (const KcError &e) {
        group_fail(ctx, e.code);
        throw;
    }
}

}  // namespace

extern "C" {

int kc_limbs_for_k(int k) { return k < 32 ? 1 : (k < 64 ? 2 : 4); }

int kc_init(int device, void *stream, kc_ctx **out) {
    if (!out) return KC_ERR_ARG;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0 || device < 0 || device >= count) {
        (void) cudaGetLastError();
        return KC_ERR_NO_DEVICE;
    }
    kc_ctx *ctx = new (std::nothrow) kc_ctx();
    if (!ctx) return KC_ERR_OOM;
    try {
        ctx->device = device;
        KC_CUDA(cudaSetDevice(device));
        if (stream) {
            ctx->stream = (cudaStream_t) stream;
        } else {
            KC_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
            ctx->own_stream = true;
        }
        ctx->arena.stream = ctx->stream;
        for (int i = 0; i < 6; ++i) KC_CUDA(cudaEventCreate(&ctx->ev[i]));
        KC_CUDA(cudaHostAlloc(reinterpret_cast<void **>(&ctx->pin_small), kc_ctx::KC_PIN_SMALL, cudaHostAllocDefault));
        if (const char *e = std::getenv("KC_FAST_SET")) ctx->routes.fast.enabled = std::atoi(e) != 0;
        if (const char *e = std::getenv("KC_SIG_SET")) ctx->routes.sig.enabled = std::atoi(e) != 0;
        if (const char *e = std::getenv("KC_FAST_MAX_CTAS")) ctx->routes.fast.max_ctas = std::atoi(e);
        if (const char *e = std::getenv("KC_SMALL_THREADS")) ctx->small_threads = std::atoi(e);
    } catch (const KcError &e) {
        int code = e.code;
        kc_destroy(ctx);
        return code;
    }
    *out = ctx;
    return KC_OK;
}

void kc_destroy(kc_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    ctx->clear_spec_graphs();
    if (ctx->arena.base) cudaFree(ctx->arena.base);
    if (ctx->pin_out.p) cudaFreeHost(ctx->pin_out.p);
    if (ctx->pin_small) cudaFreeHost(ctx->pin_small);
    group_detach(ctx);
    for (int i = 0; i < 6; ++i)
        if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
    for (int i = 0; i < kc_ctx::KC_H2D_CHUNKS; ++i)
        if (ctx->chunk_ev[i]) cudaEventDestroy(ctx->chunk_ev[i]);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->capture_stream) cudaStreamDestroy(ctx->capture_stream);
    for (cudaEvent_t e : ctx->prof.pool) cudaEventDestroy(e);
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

int kc_compute_device(kc_ctx *ctx, const kc_params *p, const kc_input *in, kc_output *out) {
    if (!ctx || !in || !out) return KC_ERR_ARG;
    KC_API_BEGIN
    check_params(p);
    check_large_input(ctx, p, in->n_bytes);
    if ((reinterpret_cast<uintptr_t>(in->seq) & 15) != 0) KC_THROW(KC_ERR_ARG, "device sequence pointer must be 16-byte aligned");
    CallFrame f(ctx);
    DevInput di{in->seq, in->n_bytes, in->rec_off, in->rec_len, in->n_recs};
    DevResult res;
    KC_TRACE_POINT("compute_device: start");
    run_with_arena(ctx, *p, *in, [&] {
        with_limbs(kc_limbs_for_k(p->k), [&](auto l) { run_pipeline<decltype(l)::value>(ctx, f.ex, di, *p, res, false); });
    });
    KC_TRACE_POINT("compute_device: launched");
    KC_CUDA(cudaStreamSynchronize(ctx->stream));
    KC_TRACE_POINT("compute_device: synced");
    fill_output(ctx, res, f.ex.launches, out);
    return KC_OK;
    KC_API_END(ctx)
}

int kc_compute(kc_ctx *ctx, const kc_params *p, const kc_input *in, kc_output *out) {
    if (!ctx || !in || !out) return KC_ERR_ARG;
    KC_API_BEGIN
    check_params(p);
    check_large_input(ctx, p, in->n_bytes);
    CallFrame f(ctx);
    DevResult res;
    run_with_arena(ctx, *p, *in, [&] {
        InputChunks chunks;
        const DevInput di = upload_input(ctx, f.ex, in, p->assume_simplitigs != 0, &chunks);
        try {
            with_limbs(kc_limbs_for_k(p->k), [&](auto l) { run_pipeline<decltype(l)::value>(ctx, f.ex, di, *p, res, false); });
        } catch (...) {
            if (di.chunks) cudaStreamSynchronize(ctx->copy_stream);  // `chunks` and the caller's buffer must outlive the copy
            throw;
        }
        if (di.chunks) chunks.wait_all(ctx->stream);
    });
    u8 *host = copy_to_pinned(ctx, res.ms, res.maxone, res.length);
    fill_output(ctx, res, f.ex.launches, out);
    out->ms = host;
    out->ms_maxone = res.maxone ? host + res.length : nullptr;
    return KC_OK;
    KC_API_END(ctx)
}

int kc_lower_bound(kc_ctx *ctx, const kc_params *p, const kc_input *in, uint64_t *lower_bound, kc_output *stats) {
    if (!ctx || !in || !lower_bound) return KC_ERR_ARG;
    KC_API_BEGIN
    check_params(p);
    if (p->want_maxone) KC_THROW(KC_ERR_ARG, "lowerbound has no mask output");
    check_large_input(ctx, p, in->n_bytes);
    CallFrame f(ctx);
    DevResult res;
    run_with_arena(ctx, *p, *in, [&] {
        const DevInput di = upload_input(ctx, f.ex, in, p->assume_simplitigs != 0, nullptr);
        with_limbs(kc_limbs_for_k(p->k), [&](auto l) { run_pipeline<decltype(l)::value>(ctx, f.ex, di, *p, res, true); });
    });
    KC_CUDA(cudaStreamSynchronize(ctx->stream));
    *lower_bound = res.lower_bound;
    if (stats) fill_output(ctx, res, f.ex.launches, stats);
    return KC_OK;
    KC_API_END(ctx)
}

int kc_streaming(kc_ctx *ctx, const kc_params *p, const kc_input *in, kc_output *out) {
    if (!ctx || !in || !out) return KC_ERR_ARG;
    KC_API_BEGIN
    check_params(p);
    if (p->assume_simplitigs || p->want_maxone) KC_THROW(KC_ERR_ARG, "-S and -M belong to the greedy algorithm");  // src/main.cpp:296-301
    {   // -z Z is Z first-occurrence passes, each of which the signature construction takes (kc_streaming_run)
        kc_params q = *p;
        q.min_frequency = 1;
        check_large_input(ctx, &q, in->n_bytes);
    }
    CallFrame f(ctx);
    const int limbs = kc_limbs_for_k(p->k);
    const SigPlan sig = kc_sig_plan(in->n_bytes, p->k, ctx->routes.sig);
    ensure_arena(ctx, estimate_arena(in->n_bytes, 0, limbs, false, true, false, &ctx->routes.fast, &sig));
    ctx->arena.reset();
    std::memset(out, 0, sizeof(*out));
    KC_CUDA(cudaEventRecord(ctx->ev[0], ctx->stream));
    const u8 *d_seq = upload_padded(f.ex, in->seq, in->n_bytes);
    KC_CUDA(cudaEventRecord(ctx->ev[1], ctx->stream));
    const StreamingResult r = with_limbs(limbs, [&](auto l) {
        return kc_streaming_run<decltype(l)::value>(f.ex, d_seq, in->n_bytes, p->k, p->complements != 0, p->min_frequency, ctx->routes);
    });
    for (int i = 2; i <= 4; ++i) KC_CUDA(cudaEventRecord(ctx->ev[i], ctx->stream));
    out->ms = copy_to_pinned(ctx, r.ms, nullptr, r.length);
    out->length = r.length;
    out->n_kmers = r.n_kept;
    out->n_occurrences = r.n_occ;
    out->n_launches = f.ex.launches;
    fill_times(ctx, out);
    return KC_OK;
    KC_API_END(ctx)
}

int kc_maskopt(kc_ctx *ctx, const uint8_t *ms, uint64_t n, int k, int complements, int minimize, kc_output *out) {
    if (!ctx || (!ms && n) || !out) return KC_ERR_ARG;
    KC_API_BEGIN
    if (k < 1 || k > 127) KC_THROW(KC_ERR_ARG, "k must be in 1..127");
    if (n + 1 >= 0xFFFFFFF0ULL) KC_THROW(KC_ERR_TOO_LARGE, "more than 2^32 sequence bytes on one GPU");
    CallFrame f(ctx);
    const int limbs = kc_limbs_for_k(k);
    // min-one keeps the sorted key set of the first construction (n * (8 limbs + 1) bytes) at the arena bottom while a second,
    // flags-only construction runs above it
    ensure_arena(ctx, estimate_arena(n + 1, 0, limbs, false, true) + 2 * n + (minimize ? (size_t) n * (8 * limbs + 1) + n / 4 : 0));
    ctx->arena.reset();
    std::memset(out, 0, sizeof(*out));
    KC_CUDA(cudaEventRecord(ctx->ev[0], ctx->stream));
    const u8 *d_seq = upload_padded(f.ex, ms, n);
    KC_CUDA(cudaEventRecord(ctx->ev[1], ctx->stream));
    const MaskoptResult r = with_limbs(limbs, [&](auto l) {
        return kc_maskopt_run<decltype(l)::value>(f.ex, d_seq, n, k, complements != 0, minimize != 0);
    });
    for (int i = 2; i <= 4; ++i) KC_CUDA(cudaEventRecord(ctx->ev[i], ctx->stream));
    out->ms = copy_to_pinned(ctx, r.ms, nullptr, r.length);
    out->length = r.length;
    out->n_kmers = r.n_kmers;
    out->n_launches = f.ex.launches;
    fill_times(ctx, out);
    return KC_OK;
    KC_API_END(ctx)
}

int kc_copy_to_host(kc_ctx *ctx, void *dst_host, const void *src_device, uint64_t n) {
    if (!ctx || (!dst_host && n) || (!src_device && n)) return KC_ERR_ARG;
    KC_API_BEGIN
    KC_CUDA(cudaSetDevice(ctx->device));
    if (n) KC_CUDA(cudaMemcpyAsync(dst_host, src_device, n, cudaMemcpyDeviceToHost, ctx->stream));
    KC_CUDA(cudaStreamSynchronize(ctx->stream));
    return KC_OK;
    KC_API_END(ctx)
}

int kc_count_kmers(kc_ctx *ctx, const kc_params *p, const kc_input *in, uint64_t **keys, uint8_t **counts, uint64_t *n) {
    if (!ctx || !in || !keys || !counts || !n) return KC_ERR_ARG;
    KC_API_BEGIN
    check_params(p);
    if (in->n_bytes >= 0xFFFFFFF0ULL) KC_THROW(KC_ERR_TOO_LARGE, "more than 2^32 sequence bytes on one GPU");
    CallFrame f(ctx);
    const int limbs = kc_limbs_for_k(p->k);
    size_t need = (size_t) ((double) in->n_bytes * (1.0 + 2.0 * 8 * limbs + 4.0) * 1.15) + (256u << 20);
    ensure_arena(ctx, need);
    ctx->arena.reset();
    const DevInput di = upload_input(ctx, f.ex, in, false, nullptr);
    with_limbs(limbs, [&](auto l) { count_only<decltype(l)::value>(ctx, f.ex, di, *p, keys, counts, n); });
    return KC_OK;
    KC_API_END(ctx)
}

int kc_partial_presort(kc_ctx *ctx, const uint64_t *kmers, uint64_t n, int k, uint64_t *out) {
    if (!ctx || (n && (!kmers || !out))) return KC_ERR_ARG;
    KC_API_BEGIN
    if (k < 1 || k > 127) KC_THROW(KC_ERR_ARG, "k must be in 1..127");
    if (n >= 0xFFFFFFF0ULL) KC_THROW(KC_ERR_TOO_LARGE, "too many k-mers");
    if (n == 0) return KC_OK;
    CallFrame f(ctx);
    CudaExec &ex = f.ex;
    const int limbs = kc_limbs_for_k(k);
    ensure_arena(ctx, (size_t) (n * (16.0 * limbs + 64.0)) + (64u << 20));
    ctx->arena.reset();
    u64 *src = ex.alloc<u64>(n * limbs), *dst = ex.alloc<u64>(n * limbs);
    KC_CUDA(cudaMemcpyAsync(src, kmers, n * limbs * 8, cudaMemcpyHostToDevice, ctx->stream));
    const int sfb = 2 * k < 8 ? 2 * k : 8;  // SORT_FIRST_BITS, src/global_sparse.h:16
    const int pos = 2 * k - sfb, limb = pos >> 6, off = pos & 63;
    const u64 *perm = kc_partial_presort_perm(ex, n, [=] __device__(u64 i) {
        u64 v = src[i * limbs + limb] >> off;
        if (off + sfb > 64 && limb + 1 < limbs) v |= src[i * limbs + limb + 1] << (64 - off);
        return (u32) (v & ((1u << sfb) - 1u));
    });
    ex.for_each(n * limbs, [=] __device__(u64 t) { dst[t] = src[(perm[t / limbs] & 0xFFFFFFFFULL) * limbs + t % limbs]; });
    KC_CUDA(cudaMemcpyAsync(out, dst, n * limbs * 8, cudaMemcpyDeviceToHost, ctx->stream));
    KC_CUDA(cudaStreamSynchronize(ctx->stream));
    return KC_OK;
    KC_API_END(ctx)
}

int kc_debug_sort(kc_ctx *ctx, const uint64_t *words, uint64_t n, int limbs, int key_bits, uint64_t *out, uint64_t *stats) {
    if (!ctx || (n && (!words || !out))) return KC_ERR_ARG;
    KC_API_BEGIN
    if (limbs != 1 && limbs != 2 && limbs != 3 && limbs != 5) KC_THROW(KC_ERR_ARG, "limbs must be 1, 2, 3 or 5");
    if (key_bits < 0 || key_bits > 64 * limbs) KC_THROW(KC_ERR_ARG, "key_bits must be in 0..64 limbs");
    for (u64 i = 0; i < n; ++i)
        for (int j = 0; j < limbs; ++j) {
            const int rem = key_bits - 64 * j;
            const u64 high = rem >= 64 ? 0 : (rem <= 0 ? ~0ULL : ~0ULL << rem);
            if (words[i * limbs + j] & high) KC_THROW(KC_ERR_ARG, "a word has a bit set at or above key_bits");
        }
    CallFrame f(ctx);
    CudaExec &ex = f.ex;
    ensure_arena(ctx, (size_t) n * (16 * limbs + 8) + (64u << 20));
    ctx->arena.reset();
    u64 *a = ex.alloc<u64>(n * limbs), *b = ex.alloc<u64>(n * limbs);
    if (n) KC_CUDA(cudaMemcpyAsync(a, words, n * limbs * 8, cudaMemcpyHostToDevice, ctx->stream));
    KcSortStats st;
    switch (limbs) {
    case 1: kc_sort<1>(ex, (KWord<1> *) a, (KWord<1> *) b, n, key_bits, &st); break;
    case 2: kc_sort<2>(ex, (KWord<2> *) a, (KWord<2> *) b, n, key_bits, &st); break;
    case 3: kc_sort<3>(ex, (KWord<3> *) a, (KWord<3> *) b, n, key_bits, &st); break;
    default: kc_sort<5>(ex, (KWord<5> *) a, (KWord<5> *) b, n, key_bits, &st); break;
    }
    if (n) KC_CUDA(cudaMemcpyAsync(out, a, n * limbs * 8, cudaMemcpyDeviceToHost, ctx->stream));
    KC_CUDA(cudaStreamSynchronize(ctx->stream));
    if (stats) {
        // the local kernel's path, from its rule (kc_sort_local_kernel): digit width about two sub-buckets per item, and a
        // bucket with more than 64 sub-buckets of more than KC_SUB_SMALL items is sorted whole; a digit count does not depend
        // on the order of the items, so the sorted words give the same counts
        u64 whole = 0;
        std::vector<u32> cnt(1u << KC_SUB_BITS_MAX);
        for (const SortBucket &d : st.small) {
            if (d.size < 2) continue;
            int bits = 1;
            while ((1u << bits) < 2 * d.size && bits < KC_SUB_BITS_MAX) ++bits;
            if (bits > (int) d.rem) bits = d.rem;
            const int shift = d.rem - bits;
            std::fill(cnt.begin(), cnt.begin() + (1u << bits), 0u);
            for (u64 i = d.off; i < d.off + d.size; ++i) {
                u32 dg = 0;
                for (int j = bits - 1; j >= 0; --j) {
                    const int p = shift + j;
                    dg = dg << 1 | (u32) ((out[i * limbs + (p >> 6)] >> (p & 63)) & 1);
                }
                ++cnt[dg];
            }
            u32 over = 0;
            for (u32 s = 0; s < (1u << bits); ++s) over += cnt[s] > KC_SUB_SMALL;
            whole += over > 64;
        }
        stats[0] = st.levels;
        stats[1] = st.max_big;
        stats[2] = st.small.size();
        stats[3] = st.n_uniform;
        stats[4] = whole;
    }
    return KC_OK;
    KC_API_END(ctx)
}

int kc_kmer_digest(kc_ctx *ctx, const kc_params *p, const kc_input *in, int masked, uint64_t *digest) {
    if (!ctx || !in || !digest) return KC_ERR_ARG;
    KC_API_BEGIN
    check_params(p);
    if (masked && p->min_frequency != 1) KC_THROW(KC_ERR_ARG, "a masked superstring has no counts");
    // masked: the bytes are ONE masked superstring (no framing); a '\n' is appended so that it is a framed record
    const u64 nb = masked ? in->n_bytes + 1 : in->n_bytes;
    {   // the digest ignores -S and -M: only -z and k decide whether an input of 2^32 bytes or more can be taken
        kc_params q = *p;
        q.assume_simplitigs = 0;
        q.want_maxone = 0;
        check_large_input(ctx, &q, nb);
    }
    CallFrame f(ctx);
    CudaExec &ex = f.ex;
    const int limbs = kc_limbs_for_k(p->k);
    // the sorted-keys route, or at 2^32 bytes and more the signature construction alone: sequence, flags, window mask, its buffers
    size_t need = (size_t) ((double) nb * (1.0 + 2.0 * 8 * limbs + 4.0 + 0.2) * 1.15) + (256u << 20);
    if (nb >= KC_POS32_BYTES)
        need = (size_t) (((double) nb * 1.25 + (double) kc_sig_arena_bytes(kc_sig_plan(nb, p->k, ctx->routes.sig), nb)) * 1.05) + (256u << 20);
    ensure_arena(ctx, need);
    ctx->arena.reset();
    u8 *d_seq = ex.alloc<u8>(nb + 64);
    if (in->n_bytes) KC_CUDA(cudaMemcpyAsync(d_seq, in->seq, in->n_bytes, cudaMemcpyHostToDevice, ctx->stream));
    u32 *win_mask = nullptr;
    if (masked) {  // the windows whose first letter is upper case are the represented k-mers (reference verify.py / src/parser.h:41-42)
        ex.fill_bytes(d_seq + in->n_bytes, '\n', 64);
        // whole tiles of the signature scan (256 strips); the extraction tiles of the sorted-keys route divide them
        const u64 mwords = kc_div_up(nb, (u64) 256 * KC_EX_STRIP) * 256 + 1;
        win_mask = ex.arena->alloc_top<u32>(mwords);
        const u64 len = in->n_bytes;
        const int k = p->k;
        u32 *wm = win_mask;
        const u8 *sq = d_seq;
        ex.for_each(mwords, [=] __device__(u64 w) {
            u32 m = 0;
            for (int i = 0; i < 32; ++i) {
                const u64 q = w * 32 + i;
                if (q + 1 >= (u64) k && q < len && sq[q + 1 - k] <= 'Z') m |= 1u << i;
            }
            wm[w] = m;
        }, KP_MISC, len + len / 8);
    }
    DevInput di{d_seq, nb, nullptr, nullptr, in->n_recs};
    with_limbs(limbs, [&](auto l) { digest_only<decltype(l)::value>(ctx, ex, di, *p, win_mask, digest); });
    return KC_OK;
    KC_API_END(ctx)
}

int kc_overlap_path(kc_ctx *ctx, const uint64_t *first, const uint64_t *last, uint64_t n, int k, int complements,
                    int lower_bound, int strict, int64_t *edge_from, uint8_t *overlaps) {
    if (!ctx || !first || !last || !edge_from || !overlaps) return KC_ERR_ARG;
    KC_API_BEGIN
    if (k < 1 || k > 127) KC_THROW(KC_ERR_ARG, "k must be in 1..127");
    if (n == 0) KC_THROW(KC_ERR_EMPTY, "input cannot be empty");
    if (n * (complements ? 2 : 1) >= 0xFFFFFFF0ULL) KC_THROW(KC_ERR_TOO_LARGE, "too many nodes for one GPU");
    CallFrame f(ctx);
    const int limbs = kc_limbs_for_k(k);
    ensure_arena(ctx, estimate_arena(0, n, limbs, complements != 0, true) + n * 16 * limbs);
    ctx->arena.reset();
    with_limbs(limbs, [&](auto l) {
        overlap_only<decltype(l)::value>(ctx, f.ex, first, last, n, k, complements != 0, lower_bound != 0, strict != 0, edge_from, overlaps);
    });
    return KC_OK;
    KC_API_END(ctx)
}

uint64_t kc_shard_granule(int k) {
    return with_limbs(kc_limbs_for_k(k), [](auto l) -> uint64_t { return KsCfg<decltype(l)::value>::EX_TILE; });
}

int kc_group_alloc(kc_ctx *ctx, int n_ranks, int rank, int k, uint64_t n_bytes_cap, uint8_t *handle_out) {
    if (!ctx || !handle_out) return KC_ERR_ARG;
    KC_API_BEGIN
    group_alloc_common(ctx, n_ranks, rank, k, n_bytes_cap, false);
    cudaIpcMemHandle_t h;
    KC_CUDA(cudaIpcGetMemHandle(&h, ctx->grp.heap));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    std::memcpy(handle_out, &h, 64);
    return KC_OK;
    KC_API_END(ctx)
}

int kc_group_open(kc_ctx *ctx, const uint8_t *all_handles) {
    if (!ctx || !all_handles) return KC_ERR_ARG;
    KC_API_BEGIN
    KcGroup &G = ctx->grp;
    if (!G.heap) KC_THROW(KC_ERR_ARG, "kc_group_alloc first");
    KC_CUDA(cudaSetDevice(ctx->device));
    for (int r = 0; r < G.n; ++r) {
        if (r == G.rank || G.peer[r]) continue;
        cudaIpcMemHandle_t h;
        std::memcpy(&h, all_handles + (size_t) r * 64, 64);
        void *pp = nullptr;
        KC_CUDA(cudaIpcOpenMemHandle(&pp, h, cudaIpcMemLazyEnablePeerAccess));
        G.peer[r] = reinterpret_cast<char *>(pp);
        G.ipc_opened[r] = true;
    }
    return KC_OK;
    KC_API_END(ctx)
}

int kc_group_compute_device(kc_ctx *ctx, const kc_params *p, const kc_input *in, kc_output *out, uint64_t *slice_begin, uint64_t *slice_len) {
    if (!ctx || !in || !out) return KC_ERR_ARG;
    KC_API_BEGIN
    group_check_job(ctx, p, in->n_bytes);
    if ((reinterpret_cast<uintptr_t>(in->seq) & 15) != 0) KC_THROW(KC_ERR_ARG, "device sequence pointer must be 16-byte aligned");
    CallFrame f(ctx);
    DevInput di{in->seq, in->n_bytes, nullptr, nullptr, 0};
    DevResult res;
    group_prepare_arena(ctx, *p, in->n_bytes, "the device cannot hold this rank's arena for an input of 2^32 bytes or more");
    ctx->arena.reset();
    ctx->grp.refused = false;
    group_run_job(ctx, f.ex, di, *p, res);
    KC_CUDA(cudaStreamSynchronize(ctx->stream));
    if (slice_begin) *slice_begin = res.slice_begin;
    if (slice_len) *slice_len = res.slice_len;
    fill_output(ctx, res, f.ex.launches, out);
    return KC_OK;
    KC_API_END(ctx)
}

int kc_group_close(kc_ctx *ctx) {
    if (!ctx) return KC_ERR_ARG;
    group_detach(ctx);
    return KC_OK;
}

int kc_group_plan(int n_ranks, int rank, int k, uint64_t n_bytes, uint64_t *plan) {
    if (!plan || n_ranks < 1 || n_ranks > KC_MAX_PEERS || rank < 0 || rank >= n_ranks || k < 1 || k > 127) return KC_ERR_ARG;
    const u64 tile = kc_shard_granule(k);
    KsfTuning tune;
    if (n_bytes >= KC_POS32_BYTES) {  // the signature construction alone (default options), within the group's 32-bit bounds
        const SigTuning sig;
        if (k < 26 || !kc_sig_plan(n_bytes, k, sig).ok || kc_grp_large_bound(n_bytes, n_ranks)) return KC_ERR_TOO_LARGE;
    }
    const KsfGroupPlan gp = kc_ksf_group_plan(n_bytes, n_ranks, tile, tune);
    const bool fixed = gp.ok && n_bytes < KC_POS32_BYTES;  // the fixed slots move 32-bit positions
    const GrpLayout lay = kc_grp_layout(n_bytes, kc_limbs_for_k(k), n_ranks, false, tile, tune);
    const u64 tiles = kc_div_up(n_bytes, tile);
    plan[0] = fixed ? 1 : 0;
    plan[1] = std::min<u64>(n_bytes, tiles * (u64) rank / (u64) n_ranks * tile);
    plan[2] = std::min<u64>(n_bytes, tiles * (u64) (rank + 1) / (u64) n_ranks * tile);
    plan[3] = fixed ? gp.dig_begin(rank) : (u64) ((rank * 256 + n_ranks - 1) / n_ranks);
    plan[4] = fixed ? gp.dig_begin(rank + 1) : (u64) (((rank + 1) * 256 + n_ranks - 1) / n_ranks);
    plan[5] = fixed ? gp.n_digits : 256;
    plan[6] = n_bytes < KC_POS32_BYTES ? gp.cap_sub : 0;
    plan[7] = lay.total;
    return KC_OK;
}

// ---- multi-GPU inside one process: SURVEY.md §8(b) `kc_init(n_gpus, device_ids)` ----------------------------------------------
// One host thread per GPU for the duration of a call, peer access between the devices (no IPC handles), the same rank-level
// code as the multi-process form above.  The host side of `kmercamel compute -g 0,1,...` (host/main.cpp).
struct kc_group {
    int n = 0;
    kc_ctx *ctx[KC_MAX_PEERS] = {};
    GrpHostSync hs;
    PinnedBuf pin_out{nullptr, 0, cudaHostAllocPortable};  // every rank copies its slice in
    std::mutex out_mutex;
    std::string last_error;
};

static void group_release_heaps(kc_group *g) {
    for (int r = 0; r < g->n; ++r)
        if (g->ctx[r]) {
            cudaSetDevice(g->ctx[r]->device);
            cudaStreamSynchronize(g->ctx[r]->stream);
        }
    for (int r = 0; r < g->n; ++r)
        if (g->ctx[r]) group_detach(g->ctx[r]);
}

int kc_init_multi(int n_gpus, const int *device_ids, kc_group **out) {
    if (!out || !device_ids || n_gpus < 1 || n_gpus > KC_MAX_PEERS) return KC_ERR_ARG;
    *out = nullptr;
    kc_group *g = new (std::nothrow) kc_group();
    if (!g) return KC_ERR_OOM;
    g->n = n_gpus;
    int rc = KC_OK;
    {   // one thread per rank: creating a primary context costs ~1 s per GPU and the devices do not wait for each other
        int rcs[KC_MAX_PEERS];
        std::vector<std::thread> th;
        for (int r = 0; r < n_gpus; ++r) th.emplace_back([&, r] { rcs[r] = kc_init(device_ids[r], nullptr, &g->ctx[r]); });
        for (auto &t : th) t.join();
        for (int r = 0; r < n_gpus; ++r)
            if (rcs[r] != KC_OK && rc == KC_OK) rc = rcs[r];
    }
    for (int a = 0; a < n_gpus && rc == KC_OK; ++a)
        for (int b = 0; b < n_gpus && rc == KC_OK; ++b) {
            const int da = device_ids[a], db = device_ids[b];
            if (da == db) continue;
            int can = 0;
            if (cudaSetDevice(da) != cudaSuccess || cudaDeviceCanAccessPeer(&can, da, db) != cudaSuccess || !can) {
                rc = KC_ERR_ARG;
                break;
            }
            const cudaError_t e = cudaDeviceEnablePeerAccess(db, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) rc = KC_ERR_CUDA;
            (void) cudaGetLastError();
        }
    g->hs.n = n_gpus;
    for (int r = 0; r < n_gpus && rc == KC_OK; ++r) {
        if (cudaSetDevice(device_ids[r]) != cudaSuccess) rc = KC_ERR_CUDA;
        for (int i = 0; i < 2 && rc == KC_OK; ++i)
            if (cudaEventCreateWithFlags(&g->hs.ev[r][i], cudaEventDisableTiming) != cudaSuccess) rc = KC_ERR_CUDA;
    }
    if (rc != KC_OK) {
        kc_group_destroy(g);
        return rc;
    }
    *out = g;
    return KC_OK;
}

void kc_group_destroy(kc_group *g) {
    if (!g) return;
    group_release_heaps(g);
    for (int r = 0; r < g->n; ++r)
        if (g->ctx[r]) kc_destroy(g->ctx[r]);
    for (int r = 0; r < g->n; ++r)
        for (int i = 0; i < 2; ++i)
            if (g->hs.ev[r][i]) cudaEventDestroy(g->hs.ev[r][i]);
    if (g->pin_out.p) cudaFreeHost(g->pin_out.p);
    delete g;
}

int kc_group_size(const kc_group *g) { return g ? g->n : 0; }
kc_ctx *kc_group_ctx(kc_group *g, int rank) { return g && rank >= 0 && rank < g->n ? g->ctx[rank] : nullptr; }
const char *kc_group_last_error(const kc_group *g) { return g ? g->last_error.c_str() : ""; }

int kc_group_compute(kc_group *g, const kc_params *p, const kc_input *in, kc_output *out) {
    if (!g || !p || !in || !out) return KC_ERR_ARG;
    kc_ctx *c0 = g->ctx[0];
    try {
        check_params(p);
        if (p->assume_simplitigs || p->want_maxone) KC_THROW(KC_ERR_ARG, "the multi-GPU construction supports neither -S nor -M");
        const bool large = in->n_bytes >= KC_POS32_BYTES;
        for (int r = 0; r < g->n; ++r) group_check_large(g->ctx[r], p, in->n_bytes, g->n);  // options are per rank
        const int limbs = kc_limbs_for_k(p->k);
        // (re)build the heaps when the job does not fit the ones in place; a heap for inputs of 2^32 bytes or more takes no smaller job
        const KcGroup &G0 = c0->grp;
        if (!G0.attached() || in->n_bytes > G0.lay.n_bytes_cap || limbs > G0.lay.limbs || G0.failed || (G0.lay.pos64() && !large)) {
            group_release_heaps(g);
            const u64 want = in->n_bytes + in->n_bytes / 16 + (1u << 20);
            const u64 cap = large ? want : std::min<u64>(0xFFFFFFE0ULL, want);
            for (int r = 0; r < g->n; ++r) {
                g->ctx[r]->routes.fast = c0->routes.fast;  // one plan for the whole group
                g->ctx[r]->routes.heuristics = c0->routes.heuristics;
                g->ctx[r]->routes.fast_rung.overflow = c0->routes.fast_rung.overflow;
                group_alloc_common(g->ctx[r], g->n, r, 32 * limbs - 1, cap, true);  // the largest k of this word width
            }
            for (int r = 0; r < g->n; ++r) {
                for (int s = 0; s < g->n; ++s) g->ctx[r]->grp.peer[s] = g->ctx[s]->grp.heap;
                g->ctx[r]->grp.hs = &g->hs;
            }
        }
        {   // a failed call may have left the barrier half way
            std::lock_guard<std::mutex> lk(g->hs.m);
            g->hs.arrived = 0;
            g->hs.aborted = false;
        }
        // every allocation happens BEFORE the first kernel of the job is queued anywhere: cudaMalloc / cudaFree wait for the whole
        // device, which would include a peer rank's wait kernel when two ranks share a GPU (tests)
        {   // (one thread per rank: cudaMalloc of tens of GB takes ~0.1 s per device; ranks that share a device take turns, so that
            //  each one sees what the others took)
            KcError errs[KC_MAX_PEERS];
            bool bad[KC_MAX_PEERS] = {};
            std::mutex dev_mutex[KC_MAX_DEVICES];
            std::vector<std::thread> th;
            for (int r = 0; r < g->n; ++r)
                th.emplace_back([&, r] {
                    try {
                        kc_ctx *ctx = g->ctx[r];
                        std::lock_guard<std::mutex> lk(dev_mutex[ctx->device % KC_MAX_DEVICES]);
                        KC_CUDA(cudaSetDevice(ctx->device));
                        group_prepare_arena(ctx, *p, in->n_bytes,
                                            "the device cannot hold every rank's arena for an input of 2^32 bytes or more (ranks sharing a device need it once each)");
                    } catch (const KcError &e) {
                        errs[r] = e;
                        bad[r] = true;
                    }
                });
            for (auto &t : th) t.join();
            for (int r = 0; r < g->n; ++r)
                if (bad[r]) throw errs[r];
        }
    } catch (const KcError &e) {
        set_error(c0, e);
        g->last_error = c0->last_error;
        return e.code;
    }
    struct RankOut {
        int code = KC_OK;
        std::string what;
        DevResult res;
        kc_output o;
    } ro[KC_MAX_PEERS];
    auto worker = [&](int r) {
        kc_ctx *ctx = g->ctx[r];
        RankOut &R = ro[r];
        try {
            CallFrame f(ctx);
            CudaExec &ex = f.ex;
            KcGroup &G = ctx->grp;
            ctx->arena.reset();
            G.refused = false;
            // the sequence: this rank brings in its share over its own PCIe link and hands it to every peer over NVLink
            u8 *seq = reinterpret_cast<u8 *>(G.heap + G.lay.off_seq);
            const u64 nb = in->n_bytes;
            const u64 b = (nb * (u64) r / (u64) g->n) & ~(u64) 255, e = r == g->n - 1 ? nb : ((nb * (u64) (r + 1) / (u64) g->n) & ~(u64) 255);
            if (G.done_pending) {  // the peers may still read the previous job's sequence
                u32 *ws = reinterpret_cast<u32 *>(ex.arena->alloc_top<u64>(1));
                ex.fill_bytes(ws, 0, 8);
                kc_grp_wait(G, ex, G.done_seq, ws);
                G.done_pending = false;
            }
            if (e > b) {
                KC_CUDA(cudaMemcpyAsync(seq + b, in->seq + b, e - b, cudaMemcpyHostToDevice, ctx->stream));
                for (int s = 0; s < g->n; ++s)
                    if (s != r) KC_CUDA(cudaMemcpyAsync(G.peer[s] + G.lay.off_seq + b, seq + b, e - b, cudaMemcpyDefault, ctx->stream));
            }
            u32 *ws = reinterpret_cast<u32 *>(ex.arena->alloc_top<u64>(1));
            ex.fill_bytes(ws, 0, 8);
            const u32 s0 = ++G.seq;
            kc_grp_signal(G, ex, s0);
            kc_grp_wait(G, ex, s0, ws);
            DevInput di{seq, nb, nullptr, nullptr, 0};
            group_run_job(ctx, ex, di, *p, R.res);
            {   // the first rank to get here sizes the common result buffer
                std::lock_guard<std::mutex> lk(g->out_mutex);
                g->pin_out.reserve((size_t) R.res.length + 64);
            }
            if (R.res.slice_len)
                KC_CUDA(cudaMemcpyAsync(g->pin_out.p + R.res.slice_begin, R.res.ms, R.res.slice_len, cudaMemcpyDeviceToHost, ctx->stream));
            KC_CUDA(cudaStreamSynchronize(ctx->stream));
            if (ex.read(ws) & 2u) KC_THROW(KC_ERR_INTERNAL, "a rank of the group did not arrive (wait timed out)");
            fill_output(ctx, R.res, ex.launches, &R.o);
        } catch (const KcError &e) {
            R.code = e.code;
            char buf[512];
            std::snprintf(buf, sizeof(buf), "rank %d: %s (%s:%d)", r, e.what, e.file, e.line);
            R.what = buf;
            if (group_fail(ctx, e.code)) g->hs.abort();
        } catch (...) {
            R.code = KC_ERR_INTERNAL;
            R.what = "rank " + std::to_string(r) + ": unknown failure";
            ctx->grp.failed = true;
            g->hs.abort();
        }
    };
    std::vector<std::thread> th;
    for (int r = 1; r < g->n; ++r) th.emplace_back(worker, r);
    worker(0);
    for (auto &t : th) t.join();
    bool all_refused = true;
    for (int r = 0; r < g->n; ++r) all_refused = all_refused && g->ctx[r]->grp.refused;
    for (int r = 0; r < g->n; ++r)
        if (ro[r].code != KC_OK) {
            if (ro[r].code != KC_ERR_EMPTY && !all_refused)
                for (int s = 0; s < g->n; ++s) g->ctx[s]->grp.failed = true;
            g->last_error = ro[r].what;
            c0->last_error = ro[r].what;
            return ro[r].code;
        }
    for (int r = 1; r < g->n; ++r)
        if (ro[r].res.length != ro[0].res.length || ro[r].res.n_kmers != ro[0].res.n_kmers) {
            g->last_error = "the ranks disagree on the result";
            return KC_ERR_INTERNAL;
        }
    *out = ro[0].o;
    out->ms = g->pin_out.p;
    out->n_launches = 0;
    for (int r = 0; r < g->n; ++r) {
        out->n_launches += ro[r].o.n_launches;
        if (ro[r].o.t.total_ms > out->t.total_ms) out->t = ro[r].o.t;  // the slowest rank's stage times
    }
    return KC_OK;
}

uint64_t kc_total_launches(const kc_ctx *ctx) { return ctx ? ctx->total_launches : 0; }

int kc_get_stat(const kc_ctx *ctx, const char *name, uint64_t *value) {
    if (!ctx || !name || !value) return KC_ERR_ARG;
    if (std::strcmp(name, "fast_runs") == 0) *value = ctx->routes.fast_rung.runs;
    else if (std::strcmp(name, "fast_fallbacks") == 0) *value = ctx->routes.fast_rung.fallbacks;
    else if (std::strcmp(name, "sig_runs") == 0) *value = ctx->routes.sig_rung.runs;
    else if (std::strcmp(name, "sig_fallbacks") == 0) *value = ctx->routes.sig_rung.fallbacks;
    else if (std::strcmp(name, "total_launches") == 0) *value = ctx->total_launches;
    else if (std::strcmp(name, "read_backs") == 0) *value = ctx->read_backs;
    else if (std::strcmp(name, "tail_spec_runs") == 0) *value = ctx->tail_spec_runs;
    else if (std::strcmp(name, "tail_spec_fallbacks") == 0) *value = ctx->tail_spec_fallbacks;
    else if (std::strcmp(name, "spec_graph_captures") == 0) *value = ctx->spec_graph_captures;
    else if (std::strcmp(name, "spec_graph_replays") == 0) *value = ctx->spec_graph_replays;
    else if (std::strcmp(name, "arena_bytes") == 0) *value = ctx->arena.cap;
    else if (std::strcmp(name, "arena_high") == 0) *value = ctx->arena.high;
    else if (std::strcmp(name, "arena_retries") == 0) *value = ctx->arena_retries;
    else if (std::strcmp(name, "fast_max_ctas") == 0) *value = (uint64_t) ctx->routes.fast.max_ctas;
    else if (std::strcmp(name, "path_levels") == 0) *value = ctx->path_stats.levels_run;
    else if (std::strcmp(name, "path_ban_rounds") == 0) *value = ctx->path_stats.ban_rounds;
    else if (std::strcmp(name, "path_bans") == 0) *value = ctx->path_stats.bans;
    else return KC_ERR_ARG;
    return KC_OK;
}

int kc_set_option(kc_ctx *ctx, const char *name, int value) {
    if (!ctx || !name) return KC_ERR_ARG;
    cudaSetDevice(ctx->device);
    ctx->clear_spec_graphs();  // an option may change the launch shapes or the arena layout of the cached calls
    if (std::strcmp(name, "sparse_switch") == 0) {
        ctx->sparse_switch = value != 0;
        return KC_OK;
    }
    if (std::strcmp(name, "small_threads") == 0 && (value == 0 || value == 256 || value == 512)) {
        ctx->small_threads = value;
        return KC_OK;
    }
    if (std::strcmp(name, "small_engine") == 0) {
        ctx->small_engine = value != 0;
        return KC_OK;
    }
    if (std::strcmp(name, "tail_spec") == 0 && (value == 0 || value == 1)) {
        ctx->tail_spec = value != 0;
        ctx->routes.tail = SizeMemo();
        return KC_OK;
    }
    // histogram-free set construction (kmerset_fast.cuh); the last three exist so that tests can reach the multi-level
    // plan and the overflow fallback with small inputs
    if (std::strcmp(name, "fast_set") == 0) {
        ctx->routes.fast.enabled = value != 0;
        return KC_OK;
    }
    if (std::strcmp(name, "fast_leaf_target") == 0 && value >= 1 && value <= 1024) {
        ctx->routes.fast.leaf_target = (u32) value;
        return KC_OK;
    }
    if (std::strcmp(name, "fast_sigmas") == 0 && value >= 0) {
        ctx->routes.fast.sigmas = (double) value;
        return KC_OK;
    }
    if (std::strcmp(name, "fast_heuristics") == 0 && (value == 0 || value == 1)) {
        ctx->routes.heuristics = value != 0;
        ctx->routes.sig_rung.overflow = ctx->routes.fast_rung.overflow = ctx->routes.tail = SizeMemo();
        return KC_OK;
    }
    if (std::strcmp(name, "fast_max_ctas") == 0 && value >= 0 && value <= (1 << 20)) {
        ctx->routes.fast.max_ctas = value;
        return KC_OK;
    }
    if (std::strcmp(name, "fast_min_items") == 0 && value >= 0) {
        ctx->routes.fast.min_items = (u64) value;
        return KC_OK;
    }
    // signature-bucket set construction (kmerset_sig.cuh)
    if (std::strcmp(name, "sig_set") == 0) {
        ctx->routes.sig.enabled = value != 0;
        return KC_OK;
    }
    if (std::strcmp(name, "sig_load_pct") == 0 && value >= 0 && value <= 400) {  // > 100 forces overflows (tests)
        ctx->routes.sig.load_pct = (u32) value;  // 0 = planned from the input size
        return KC_OK;
    }
    if (std::strcmp(name, "sig_min_items") == 0 && value >= 0) {
        ctx->routes.sig.min_items = (u64) value;
        return KC_OK;
    }
    // device arena (tests): fill every block it hands out with this byte (-1 = off), and scale the first estimate of a call (in
    // parts per million: 1 % of an estimate is megabytes, more than a stage of a small input allocates) so that a small input runs
    // out of arena at a chosen point and takes the retry with the worst-case estimate
    if (std::strcmp(name, "arena_poison") == 0 && value >= -1 && value <= 255) {
        ctx->arena.poison = value;
        return KC_OK;
    }
    if (std::strcmp(name, "arena_estimate_ppm") == 0 && value >= 1 && value <= 1000000) {
        ctx->arena_estimate_ppm = (u32) value;
        return KC_OK;
    }
    return KC_ERR_ARG;
}

int kc_profile_enable(kc_ctx *ctx, int on) {
    if (!ctx) return KC_ERR_ARG;
    ctx->prof.enabled = on != 0;
    return KC_OK;
}
int kc_profile_count(void) { return KP_COUNT; }
int kc_profile_get(kc_ctx *ctx, int i, const char **name, double *ms, uint64_t *launches, uint64_t *bytes) {
    if (!ctx || i < 0 || i >= KP_COUNT) return KC_ERR_ARG;
    if (!ctx->prof.pending.empty()) {
        cudaStreamSynchronize(ctx->stream);
        ctx->prof.resolve();
    }
    if (name) *name = kc_prof_names[i];
    if (ms) *ms = ctx->prof.ms[i];
    if (launches) *launches = ctx->prof.launches[i];
    if (bytes) *bytes = ctx->prof.bytes[i];
    return KC_OK;
}
int kc_profile_reset(kc_ctx *ctx) {
    if (!ctx) return KC_ERR_ARG;
    cudaStreamSynchronize(ctx->stream);
    ctx->prof.resolve();
    ctx->prof.reset();
    return KC_OK;
}

void kc_free(void *p) { std::free(p); }

const char *kc_strerror(int code) {
    switch (code) {
        case KC_OK: return "ok";
        case KC_ERR_CUDA: return "CUDA error";
        case KC_ERR_ARG: return "invalid argument";
        case KC_ERR_OOM: return "out of memory";
        case KC_ERR_EMPTY: return "input contains no k-mers";
        case KC_ERR_BAD_SEQ: return "invalid sequence for -S";
        case KC_ERR_TOO_LARGE: return "input too large for one GPU";
        case KC_ERR_INTERNAL: return "internal error";
        case KC_ERR_NO_DEVICE: return "no CUDA device";
        default: return "unknown error";
    }
}

const char *kc_last_error(const kc_ctx *ctx) { return ctx ? ctx->last_error.c_str() : ""; }

}  // extern "C"
