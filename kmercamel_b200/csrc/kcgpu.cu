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
#include "sort.cuh"
#include "stage1.cuh"
#include "tail_spec.cuh"

#include <chrono>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

static double kc_now_ms() {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}
static const bool kc_trace = std::getenv("KC_TRACE") != nullptr;
#define KC_TRACE_POINT(label)                                                               \
    do {                                                                                    \
        if (kc_trace) std::fprintf(stderr, "[kc_trace] %-28s %.3f ms\n", (label), kc_now_ms()); \
    } while (0)

struct kc_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    Arena arena;
    KernelProf prof;
    // pinned host staging for kc_compute (grown on demand, reused across calls)
    u8 *pin_in = nullptr;
    size_t pin_in_cap = 0;
    u8 *pin_out = nullptr;
    size_t pin_out_cap = 0;
    static const size_t KC_PIN_SMALL = 4096;
    u8 *pin_small = nullptr;  // page-locked scratch for the small synchronising read-backs (CudaExec::read_n)
    cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    // kc_compute with host buffers: the input is copied in chunks on its own stream, the first partition pass follows the copy front
    static const int KC_H2D_CHUNKS = 4;
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t chunk_ev[KC_H2D_CHUNKS] = {nullptr, nullptr, nullptr, nullptr};
    bool small_engine = true;
    int small_threads = 0;   // 0 = chosen by the number of free ends (option "small_threads": 256 or 512)
    bool sparse_switch = true;  // src/main.cpp:175 (option "sparse_switch" = 0 keeps the runs as nodes whatever their number)
    KsfTuning fast;          // histogram-free set construction (kmerset_fast.cuh); KC_FAST_* environment knobs for tests
    u64 fast_runs = 0, fast_fallbacks = 0;
    SigTuning sig;           // signature-bucket set construction (kmerset_sig.cuh), tried first in the FLAGS regime
    u64 sig_runs = 0, sig_fallbacks = 0;
    u64 sig_overflow_bytes = 0;   // input size of the last call whose signature buckets overflowed (0 = none)
    bool fast_heuristics = true;  // skip the fixed-slot attempt when duplicates are expected (see run_stage1_runs)
    u64 fast_overflow_bytes = 0;  // input size of the last call whose fixed-slot attempt overflowed (0 = none)
    u64 total_launches = 0;  // kernels launched through this context since kc_init
    u64 read_backs = 0;      // synchronising device -> host reads of this context since kc_init (host round trips)
    bool tail_spec = true;   // option "tail_spec": queue the tail of the from-FASTA path without reading the run count (run_tail_spec)
    u64 tail_spec_runs = 0, tail_spec_fallbacks = 0;
    u64 spec_fail_bytes = 0;  // input size of the last call whose speculative tail did not hold (0 = none)
    EngineStats path_stats;   // the overlap stage of the last call that ran it (stats "path_levels", "path_ban_rounds", "path_bans")
    KcGroup grp;             // multi-GPU: this context as one rank of a group (group.cuh)
    bool arena_limited = false;
    std::string last_error;
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

void check_params(const kc_params *p) {
    if (!p) KC_THROW(KC_ERR_ARG, "params is NULL");
    if (p->k < 1 || p->k > 127) KC_THROW(KC_ERR_ARG, "k must be in 1..127");                          // src/main.cpp:93,285-292
    if (p->min_frequency < 1 || p->min_frequency > 255) KC_THROW(KC_ERR_ARG, "min_frequency must be in 1..255");  // :302-304
    if (p->min_frequency != 1 && p->assume_simplitigs) KC_THROW(KC_ERR_ARG, "-z is not compatible with -S");   // :305-308
}

// Inputs of KC_POS32_BYTES or more need 64-bit window positions, which only the signature construction carries (the fixed-slot
// and exact constructions move 32-bit positions, the -S path and the other entry points keep their 32-bit caps).
#define KC_LARGE_ONLY "inputs of 2^32 bytes or more are built by the signature construction only (k >= 26, no -z, no -M, no -S)"
void check_large_input(const kc_ctx *ctx, const kc_params *p, u64 n_bytes) {
    if (n_bytes < KC_POS32_BYTES) return;
    if (p->assume_simplitigs) KC_THROW(KC_ERR_TOO_LARGE, KC_LARGE_ONLY "; -S was asked");
    if (p->min_frequency > 1) KC_THROW(KC_ERR_TOO_LARGE, KC_LARGE_ONLY "; -z (min_frequency > 1) was asked");
    if (p->want_maxone) KC_THROW(KC_ERR_TOO_LARGE, KC_LARGE_ONLY "; -M (want_maxone) was asked");
    if (p->k < 26) KC_THROW(KC_ERR_TOO_LARGE, KC_LARGE_ONLY "; k is below 26");
    if (!ctx->sig.enabled) KC_THROW(KC_ERR_TOO_LARGE, KC_LARGE_ONLY "; it is switched off (option sig_set = 0)");
    if (!kc_sig_plan(n_bytes, p->k, ctx->sig).ok) KC_THROW(KC_ERR_TOO_LARGE, KC_LARGE_ONLY "; its bucket plan does not fit this input");
}

// Make sure the arena can hold `need` bytes (bounded by what the device can give).
void ensure_arena(kc_ctx *ctx, size_t need) {
    need = (need + 4095) & ~(size_t) 4095;  // both arena ends stay 256-byte aligned
    if (ctx->arena.cap >= need) return;
    if (ctx->arena.cap && ctx->arena_limited && need >= ctx->arena.cap) return;  // already holds all the device can give
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

// Arena bytes one kc_compute needs (see DESIGN.md "Data layout in HBM").  Stage 1 is an exact upper bound; the overlap
// stage depends on the number of nodes, which for a FASTA input (first-occurrence runs) is only known after stage 1:
// `pessimistic = false` assumes one run per 64 sequence bytes (reads with 1 % errors give one per ~650), and a call that
// runs out of arena is repeated once with the worst case (one run per 2 bytes), see run_with_arena.
// Inputs of KC_POS32_BYTES or more take the signature construction alone (`sig`: its plan at this size): sequence, flags, code
// words and record rows.
size_t estimate_arena(u64 n_bytes, u64 n_recs, int limbs, bool complements, bool simplitigs, bool pessimistic = false,
                      const KsfTuning *fast = nullptr, const SigPlan *sig = nullptr) {
    const double wb = 8.0 * limbs;
    const double c = complements ? 2.0 : 1.0;
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
    double N = c * nodes;
    double engine = N * (60.0 + 2.0 * 2.0 * (wb + 8.0) + 12.0 + 40.0);
    double emit = N * 32.0 + 3.0 * n_bytes;
    double total = (stage1 + engine + emit) * 1.1 + (256u << 20);
    return (size_t) total;
}

// Runs body() with an arena of `need` bytes; if the arena is exhausted (more nodes than the estimate assumed) the call is
// repeated once with `need_max`.
template <class F> void run_with_arena(kc_ctx *ctx, size_t need, size_t need_max, F body) {
    ensure_arena(ctx, need);
    try {
        ctx->arena.reset();
        body();
    } catch (const KcError &e) {
        if (e.code != KC_ERR_OOM || need_max <= ctx->arena.cap || ctx->arena_limited) throw;
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
    u64 lower_bound = 0;  // only with run_pipeline(..., lower_bound = true)
    u64 slice_begin = 0, slice_len = 0;
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

// The speculative tail (tail_spec.cuh): from the first-occurrence flags to the last emission kernel, sized for KC_SPEC_RUNS runs, with
// ONE read-back of the status block `blk` (cells4 of the signature construction first, KC_SPEC_BLOCK_WORDS words, zeroed) at the end.
// Returns the status: KC_SPEC_OK = `res` holds the result; otherwise nothing was done and the arena is as it was on entry.
template <int L>
u32 run_tail_spec(kc_ctx *ctx, CudaExec &ex, const DevInput &in, const kc_params &p, const u32 *flags, u64 *blk, DevResult &res) {
    const u64 nb = in.n_bytes;
    const int k = p.k;
    const bool complements = p.complements != 0;
    const size_t mark = ex.arena->mark();
    const u32 C = KC_SPEC_RUNS, N_cap = complements ? 2 * C : C;
    const u64 n_words = kc_div_up(nb, 32);
    const u32 blocks = (u32) kc_div_up(nb, (u64) KC_RUN_TILE);
    u32 *counts = ex.alloc<u32>(blocks);
    u64 *rec_off = ex.alloc<u64>(C), *rec_len = ex.alloc<u64>(C);
    kc_ull *n_runs = reinterpret_cast<kc_ull *>(blk + 1);
    {
        CudaExec::Scope sc(ex, KP_RUNS, nb / 8);
        kc_runs_count_kernel<<<blocks, 256, 0, ex.stream>>>(flags, n_words, counts, n_runs);
        kc_runs_emit_kernel<<<blocks, 256, 0, ex.stream>>>(flags, n_words, counts, rec_off, rec_len, n_runs, C);
    }
    ex.launches += 2;
    KC_CUDA(cudaGetLastError());
    KC_CUDA(cudaEventRecord(ctx->ev[2], ex.stream));
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
        kc_spec_nodes_kernel<L><<<1, 1024, 0, ex.stream>>>(blk, spec, ctx->sparse_switch, complements, in.seq, k, rec_off, rec_len, first, last,
                                                            eng.st, eng.ban_flag, eng.ban_ctr, eng.live_s, eng.live_p, eng.small_masks, (u32) mask_words);
    }
    ++ex.launches;
    KC_CUDA(cudaGetLastError());
    static_assert(4 * KC_SPEC_RUNS <= SmallCfg<L>::T && 2 * KC_SPEC_RUNS <= SmallCfg<L>::NS && 2 * KC_SPEC_RUNS <= KC_RANK_SMALL,
                  "the speculative tail runs on the one-CTA kernels");
    eng.run();  // all levels in the single-CTA engine
    KC_CUDA(cudaEventRecord(ctx->ev[3], ex.stream));
    NodeSeq<L> ns;
    ns.k = k;
    ns.kmers = nullptr;
    ns.seq = in.seq;
    ns.rec_off = rec_off;
    ns.rec_len = rec_len;
    ns.n = C;
    const EmitSpec es{spec + 1, blk + KC_SPEC_EMIT};
    // every character of the superstring is a character of some node: nodes are pieces of the input that overlap by < k
    const u64 total_ub = nb + (u64) C * k + 16;
    const EmitResult er = kc_emit_superstring<CudaExec, L>(ex, ns, nv, eng.st, nullptr, 0, false, 0, 1, total_ub, &es);
    KC_CUDA(cudaEventRecord(ctx->ev[4], ex.stream));
    KC_TRACE_POINT("tail_spec: queued");
    u64 h[KC_SPEC_BLOCK_WORDS];
    ex.read_n(blk, h, KC_SPEC_BLOCK_WORDS);
    const u32 *hs = reinterpret_cast<const u32 *>(h + KC_SPEC_SPEC);
    if (hs[0] != KC_SPEC_OK) {
        ex.arena->release(mark);
        return hs[0];
    }
    eng.apply_small_status(reinterpret_cast<const u32 *>(h + KC_SPEC_SMALL));  // a failed small-engine run is the cause, report that one
    ctx->path_stats = eng.stats;
    kc_emit_check(h + KC_SPEC_EMIT, hs[2], total_ub);
    res.ms = er.ms;
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
// spec_res != nullptr: after the signature construction, try the speculative tail (run_tail_spec).  When it holds, *spec_res is the whole
// result and *spec_done is set; otherwise the code below continues as if it had not been tried, on the same flags.
template <int L>
u64 run_stage1_runs(kc_ctx *ctx, CudaExec &ex, const DevInput &in, const kc_params &p, RunNodes *runs, KWord<L> **set_out, u64 *n_occ,
                    DevResult *spec_res = nullptr, bool *spec_done = nullptr) {
    KC_CUDA(cudaEventRecord(ctx->ev[0], ex.stream));
    KC_CUDA(cudaEventRecord(ctx->ev[1], ex.stream));  // extraction is fused into the partition passes
    KC_TRACE_POINT("stage1: begin");
    const u64 nb = in.n_bytes;
    const size_t fwords = kc_runs_flag_words(nb);
    u32 *flags = ex.arena->alloc_top<u32>(fwords);
    ex.fill_bytes(flags, 0, fwords * 4);
    u64 *cells = ex.arena->alloc_top<u64>(2);  // {kept distinct k-mers, runs}
    ex.fill_bytes(cells, 0, 16);
    // FLAGS-only: try the histogram-free construction first (no host synchronisation until the runs are counted).  Its
    // fixed slots assume mostly distinct k-mers; `-z Z > 1` announces a read set with coverage (every k-mer ~coverage times:
    // the leaf slots overflow and the attempt is wasted — configs[3] at full size lost 70 ms to it), and so does an
    // overflow in the previous call of this context on an input of similar size.
    const bool expect_duplicates = ctx->fast_heuristics && (p.min_frequency > 1 || (ctx->fast_overflow_bytes && nb >= ctx->fast_overflow_bytes / 2 && nb <= ctx->fast_overflow_bytes * 2));
    // Signature buckets first (kmerset_sig.cuh): records of ~7 windows instead of 12-byte items.  Read sets with coverage overflow
    // its buckets (every run of windows comes c times: sigma grows by sqrt(c)) and are remembered like a fixed-slot overflow.
    // Inputs of KC_POS32_BYTES or more have no other construction (check_large_input): they always try it, and an overflow ends the call.
    const bool large = nb >= KC_POS32_BYTES;
    const bool sig_overflowed = ctx->fast_heuristics && ctx->sig_overflow_bytes && nb >= ctx->sig_overflow_bytes / 2 && nb <= ctx->sig_overflow_bytes * 2;
    if (!p.want_maxone && p.min_frequency == 1 && (large || !sig_overflowed)) {
        const size_t n_cells = spec_res ? KC_SPEC_BLOCK_WORDS : 4;
        u64 *cells4 = ex.arena->alloc_top<u64>(n_cells);  // {kept, runs, M, overflow status} (+ the rest of the speculative tail's status block)
        ex.fill_bytes(cells4, 0, n_cells * 8);
        if (kc_kmerset_build_sig<L>(ex, in.seq, nb, p.k, p.complements != 0, flags, cells4, ctx->sig, in.chunks)) {
            KC_TRACE_POINT("stage1: signature set launched");
            u64 hc[4];
            bool aborted = false;
            if (spec_res) {
                const u32 st = run_tail_spec<L>(ctx, ex, in, p, flags, cells4, *spec_res);
                if (st == KC_SPEC_OK) {
                    ++ctx->sig_runs;
                    ++ctx->tail_spec_runs;
                    *spec_done = true;
                    return spec_res->n_kmers;
                }
                ++ctx->tail_spec_fallbacks;
                if (st == KC_SPEC_SIG_OVERFLOW) {
                    aborted = true;
                } else {  // the flags stand: the ordinary tail counts the runs again
                    if (st != KC_SPEC_EMPTY) ctx->spec_fail_bytes = nb;
                    ex.fill_bytes(cells4 + 1, 0, 8);
                }
            }
            if (!aborted) *runs = kc_runs_from_flags(ex, flags, nb, p.k, cells4, hc, 4, &aborted);
            if (!aborted) {
                ++ctx->sig_runs;
                *n_occ = hc[2];
                *set_out = nullptr;
                KC_CUDA(cudaEventRecord(ctx->ev[2], ex.stream));
                return hc[2] ? hc[0] : 0;
            }
            ++ctx->sig_fallbacks;  // a bucket overflowed: discard the flags, fall through to the other constructions
            ctx->sig_overflow_bytes = nb;
            if (large) KC_THROW(KC_ERR_TOO_LARGE, KC_LARGE_ONLY "; it overflowed on this input (too repetitive)");
            ex.fill_bytes(flags, 0, fwords * 4);
        }
    }
    if (large) KC_THROW(KC_ERR_INTERNAL, "an input of 2^32 bytes or more reached the 32-bit set constructions");
    if (!p.want_maxone && !expect_duplicates) {
        KsfPlan plan;
        u64 *cells4 = ex.arena->alloc_top<u64>(4);  // {kept, runs, M, overflow status}
        ex.fill_bytes(cells4, 0, 32);
        if (kc_kmerset_build_fast<L>(ex, in.seq, nb, p.k, p.complements != 0, p.min_frequency, flags, cells4, ctx->fast, &plan, in.chunks)) {
            KC_TRACE_POINT("stage1: fast set launched");
            u64 hc[4];
            bool aborted = false;
            *runs = kc_runs_from_flags(ex, flags, nb, p.k, cells4, hc, 4, &aborted);
            if (!aborted) {
                ++ctx->fast_runs;
                // the timers charged the partition passes with M = n_bytes; now that M is known, correct the byte counts
                if (ex.prof && ex.prof->enabled && nb > hc[2]) {
                    const u64 d = (nb - hc[2]) * (sizeof(KWord<L>) + 4);
                    ex.prof->bytes[KP_KS_SCATTER0] -= d;
                    ex.prof->bytes[KP_SORT_SCATTER] -= 2 * d * (u64) (plan.n_levels - 1);
                    ex.prof->bytes[KP_KS_RESOLVE] -= d;
                }
                *n_occ = hc[2];
                *set_out = nullptr;
                KC_CUDA(cudaEventRecord(ctx->ev[2], ex.stream));
                return hc[2] ? hc[0] : 0;
            }
            ++ctx->fast_fallbacks;  // a slot overflowed: discard the flags, fall through to the exact construction
            ctx->fast_overflow_bytes = nb;
            ex.fill_bytes(flags, 0, fwords * 4);
        }
    }
    // with -M the sorted k-mer set doubles as kMersDict of src/global.h:165-167; it stays at the arena bottom
    if (in.chunks) in.chunks->wait_all(ex.stream);
    KmerSet<L> set = kc_kmerset_build<L>(ex, in.seq, nb, p.k, p.complements != 0, p.min_frequency, flags, p.want_maxone != 0, cells);
    KC_TRACE_POINT("stage1: set built");
    *n_occ = set.n_occ;
    *set_out = set.keys;
    if (set.n_occ == 0 || set.n_kept == 0) {
        KC_CUDA(cudaEventRecord(ctx->ev[2], ex.stream));
        return 0;
    }
    if (p.want_maxone) {  // the KEYS path has read the count back already
        const u64 kept = set.n_kept;
        KC_CUDA(cudaMemcpyAsync(cells, &kept, 8, cudaMemcpyHostToDevice, ex.stream));
    }
    u64 host_cells[2];
    *runs = kc_runs_from_flags(ex, flags, nb, p.k, cells, host_cells);
    const u64 n_kept = p.want_maxone ? set.n_kept : host_cells[0];
    KC_TRACE_POINT("stage1: runs built");
    KC_CUDA(cudaEventRecord(ctx->ev[2], ex.stream));
    return n_kept;
}

// First-occurrence flags that were built outside run_pipeline (multi-GPU construction, group.cuh).
struct ExtFlags {
    const u32 *flags = nullptr;
    u64 kept = 0, n_occ = 0;   // totals, when they are known on the host already (exact path)
    u64 *cells4 = nullptr;     // fast path: device words {kept, 0, M, status}, read back together with the run count
    bool aborted = false;      // out: the status word was set (a slot overflowed somewhere): nothing was done
};

template <int L>
void run_pipeline(kc_ctx *ctx, CudaExec &ex, const DevInput &in, const kc_params &p, DevResult &res, ExtFlags *ext = nullptr,
                  bool lower_bound = false, u32 slice_index = 0, u32 n_slices = 1) {
    const bool complements = p.complements != 0;
    KWord<L> *uniq = nullptr;
    u8 *cnt = nullptr;
    u64 U = 0, n_occ = 0;
    NodeView<L> nv;
    NodeSeq<L> ns;
    nv.k = p.k;
    nv.complements = complements;
    ns.k = p.k;
    ns.kmers = nullptr;
    ns.seq = in.seq;
    ns.rec_off = in.rec_off;
    ns.rec_len = in.rec_len;
    u64 n_nodes = 0;
    const u64 *node_off = in.rec_off, *node_len = in.rec_len;
    if (in.chunks && (p.assume_simplitigs || ext)) in.chunks->wait_all(ex.stream);
    if (!p.assume_simplitigs) {
        RunNodes runs;
        if (ext && ext->cells4) {  // multi-GPU fast path: totals and status arrive with the run count, in ONE read-back
            u64 hc[4];
            runs = kc_runs_from_flags(ex, ext->flags, in.n_bytes, p.k, ext->cells4, hc, 4, &ext->aborted);
            if (ext->aborted) {
                ext->kept = hc[3];  // the status word, for the caller's diagnosis
                return;
            }
            U = hc[2] ? hc[0] : 0;
            n_occ = hc[2];
            KC_CUDA(cudaEventRecord(ctx->ev[2], ex.stream));
        } else if (ext) {          // multi-GPU exact path
            u64 *cells = ex.arena->alloc_top<u64>(2);
            ex.fill_bytes(cells, 0, 16);
            u64 host_cells[2];
            runs = kc_runs_from_flags(ex, ext->flags, in.n_bytes, p.k, cells, host_cells);
            U = runs.n_runs ? ext->kept : 0;
            n_occ = ext->n_occ;
            KC_CUDA(cudaEventRecord(ctx->ev[2], ex.stream));
        } else {
            // the speculative tail: a FASTA input with few runs (a genome) is computed behind one read-back (run_tail_spec)
            const u64 nb = in.n_bytes;
            const bool spec_failed = ctx->fast_heuristics && ctx->spec_fail_bytes && nb >= ctx->spec_fail_bytes / 2 && nb <= ctx->spec_fail_bytes * 2;
            const bool spec = ctx->tail_spec && !spec_failed && !lower_bound && ctx->small_engine && nb > 0 && nb < KC_POS32_BYTES;
            bool spec_done = false;
            U = run_stage1_runs<L>(ctx, ex, in, p, &runs, &uniq, &n_occ, spec ? &res : nullptr, &spec_done);
            if (spec_done) return;
        }
        if (U == 0) KC_THROW(KC_ERR_EMPTY, "the input contains no k-mers");  // src/main.cpp:155-158
        res.n_simplitigs = runs.n_runs;
        // src/main.cpp:94,175-181: simplitigs barely longer than k-mers -> the greedy runs on the k-mers themselves (PartialPreSort order)
        if (ctx->sparse_switch && runs.n_runs * 5 >= U) {
            // one node per k-mer; kc_kmer_nodes_from_runs numbers them with 32-bit offsets (inputs of 2^32 bytes or more can have that many)
            if (U * (complements ? 2 : 1) >= 0xFFFFFFF0ULL) KC_THROW(KC_ERR_TOO_LARGE, "too many nodes for one GPU");
            runs = kc_kmer_nodes_from_runs(ex, in.seq, runs, p.k);
        }
        n_nodes = runs.n_runs;
        node_off = runs.rec_off;
        node_len = runs.rec_len;
        if (n_nodes * (complements ? 2 : 1) >= 0xFFFFFFF0ULL) KC_THROW(KC_ERR_TOO_LARGE, "too many nodes for one GPU");
    } else {
        if (in.n_recs == 0) KC_THROW(KC_ERR_EMPTY, "input cannot be empty");  // src/global.h:219-221
        if (in.n_recs * (complements ? 2 : 1) >= 0xFFFFFFF0ULL) KC_THROW(KC_ERR_TOO_LARGE, "too many records for one GPU");
        KC_CUDA(cudaEventRecord(ctx->ev[0], ex.stream));
        if (p.want_maxone) {  // kMersDict of src/global.h:165-167 = every k-mer of the records
            U = run_stage1<L>(ctx, ex, in, p, &uniq, &cnt, &n_occ);
        } else {
            KC_CUDA(cudaEventRecord(ctx->ev[1], ex.stream));
            KC_CUDA(cudaEventRecord(ctx->ev[2], ex.stream));
        }
        n_nodes = in.n_recs;
        res.n_simplitigs = in.n_recs;
    }
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
        ns.rec_off = node_off;
        ns.rec_len = node_len;
    }
    nv.N = nv.n * (complements ? 2u : 1u);
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
        const u64 *len = node_off == in.rec_off ? in.rec_len : node_len;
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
        res.n_kmers = U;
        res.n_occ = n_occ;
        res.n_nodes = nv.n;
        return;
    }
    EmitResult er;
    try {
        // every character of the superstring is a character of some node: nodes are pieces of the input that overlap by < k
        er = kc_emit_superstring<CudaExec, L>(ex, ns, nv, eng.st, uniq, U, p.want_maxone != 0, slice_index, n_slices, in.n_bytes + n_nodes * (u64) p.k + 16);
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
    res.n_kmers = U;
    res.n_occ = n_occ;
    res.n_nodes = nv.n;
}

void dispatch_pipeline(kc_ctx *ctx, CudaExec &ex, const DevInput &in, const kc_params &p, DevResult &res, bool lower_bound = false) {
    if (p.k < 32) run_pipeline<1>(ctx, ex, in, p, res, nullptr, lower_bound);
    else if (p.k < 64) run_pipeline<2>(ctx, ex, in, p, res, nullptr, lower_bound);
    else run_pipeline<4>(ctx, ex, in, p, res, nullptr, lower_bound);
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

// The first-occurrence flags of a from-FASTA input built by the signature construction (kmerset_sig.cuh) alone, for the entry
// points that need the k-mer set but not its runs: kc_kmer_digest and kc_streaming.  win_mask: optional window filter over END
// positions, sized for the signature scan's tiles of 256 * 32 positions.  flags (fwords words) and cells {kept, -, M, status, ...}
// arrive zeroed; after() queues the work that reads the flags before the one read-back of cells[0, n_cells) into hc.
// Returns true when the flags stand.  Returns false when the construction does not apply, or when a bucket overflowed: then the overflow
// is counted in sig_fallbacks, flags and cells are zeroed again, and the caller takes the other constructions.  Unlike run_stage1_runs
// it leaves sig_overflow_bytes alone, so a digest or a streaming call does not change which construction a later compute tries.
// Inputs of KC_POS32_BYTES or more have no other construction (check_large_input): there the call fails instead.
template <int L, class After>
bool sig_flags(kc_ctx *ctx, CudaExec &ex, const u8 *seq, u64 nb, const kc_params &p, u32 *flags, size_t fwords, const u32 *win_mask, u64 *cells,
               u64 *hc, int n_cells, After after) {
    const bool large = nb >= KC_POS32_BYTES;
    if (!kc_kmerset_build_sig<L>(ex, seq, nb, p.k, p.complements != 0, flags, cells, ctx->sig, nullptr, win_mask)) {
        if (large) KC_THROW(KC_ERR_TOO_LARGE, KC_LARGE_ONLY "; its bucket plan does not fit this input");
        return false;
    }
    after();
    ex.read_n(cells, hc, (size_t) n_cells);
    if (hc[3] == 0) {
        ++ctx->sig_runs;
        return true;
    }
    ++ctx->sig_fallbacks;
    if (large) KC_THROW(KC_ERR_TOO_LARGE, KC_LARGE_ONLY "; it overflowed on this input (too repetitive)");
    ex.fill_bytes(flags, 0, fwords * 4);
    ex.fill_bytes(cells, 0, (size_t) n_cells * 8);
    return false;
}

// kc_kmer_digest: (n, sum h, xor h, sum h * c) over the kept (k-mer, c = min(occurrences, 256), or 1 without -z) pairs, h = the splitmix64 fold of
// the limbs (kc_kmer_hash).  The same four numbers come out of oracle/ref_harness `full` for the reference's own hash table.
// Without -z the set is first tried as first-occurrence flags of the signature construction, hashed window by window (digest.cuh); the
// sorted keys of kc_kmerset_build are the other route.  The digest is a function of the set: both give the same four words.

template <int L>
void digest_only(kc_ctx *ctx, CudaExec &ex, const DevInput &in, const kc_params &p, const u32 *win_mask, uint64_t *digest) {
    KC_CUDA(cudaEventRecord(ctx->ev[0], ex.stream));
    if (p.min_frequency == 1) {  // c = 1: digest[3] = digest[1]
        const size_t top = ex.arena->top, mark = ex.arena->mark();
        const size_t fwords = kc_runs_flag_words(in.n_bytes);
        u32 *flags = ex.arena->alloc_top<u32>(fwords);
        ex.fill_bytes(flags, 0, fwords * 4);
        u64 *cells = ex.arena->alloc_top<u64>(8);  // {kept, -, M, status, n, sum h, xor h, -}
        ex.fill_bytes(cells, 0, 64);
        kc_ull *acc = reinterpret_cast<kc_ull *>(cells + 4);
        u64 hc[7];
        if (sig_flags<L>(ctx, ex, in.seq, in.n_bytes, p, flags, fwords, win_mask, cells, hc, 7,
                         [&] { kc_flag_digest<L>(ex, in.seq, in.n_bytes, flags, fwords, p.k, p.complements != 0, acc); })) {
            digest[0] = hc[4];
            digest[1] = hc[5];
            digest[2] = hc[6];
            digest[3] = hc[5];
            return;
        }
        ex.arena->release(mark);
        ex.arena->top = top;
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

// kc_streaming: every pass of the first-occurrence construction tries the signature buckets first (sig_flags)
template <int L> StreamingResult streaming_only(kc_ctx *ctx, CudaExec &ex, const u8 *seq, u64 nb, const kc_params &p) {
    auto sig = [&](u32 *flags, size_t fwords, const u32 *win_mask, u64 *cells4, u64 *hc) {
        return sig_flags<L>(ctx, ex, seq, nb, p, flags, fwords, win_mask, cells4, hc, 4, [] {});
    };
    return kc_streaming_run<L>(ex, seq, nb, p.k, p.complements != 0, p.min_frequency, ctx->fast, &ctx->fast_runs, &ctx->fast_fallbacks, sig);
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
    if (n_bytes_cap >= 0xFFFFFFF0ULL) KC_THROW(KC_ERR_TOO_LARGE, "more than 2^32 sequence bytes");
    KcGroup &G = ctx->grp;
    if (G.heap) KC_THROW(KC_ERR_ARG, "this context already belongs to a group");
    KC_CUDA(cudaSetDevice(ctx->device));
    G.n = n_ranks;
    G.rank = rank;
    G.lay = kc_grp_layout(n_bytes_cap, kc_limbs_for_k(k), n_ranks, with_seq, kc_shard_granule(k), ctx->fast);
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
size_t group_arena_need(u64 n_bytes, int n_ranks, int limbs, bool complements, bool pessimistic) {
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
    auto finish = [&]() {
        G.done_seq = ++G.seq;
        kc_grp_signal(G, ex, G.done_seq);
        G.done_pending = true;
    };
    // signature buckets first (kmerset_sig.cuh): every rank takes the same decision from values it sees identically
    const bool sig_overflowed = ctx->fast_heuristics && ctx->sig_overflow_bytes && nb >= ctx->sig_overflow_bytes / 2 && nb <= ctx->sig_overflow_bytes * 2;
    if (p.min_frequency == 1 && !sig_overflowed) {
        const size_t top_mark = ex.arena->top, mark = ex.arena->mark();
        ExtFlags ext;
        ext.flags = reinterpret_cast<const u32 *>(G.heap + G.lay.off_flags);
        ext.cells4 = kc_grp_sig_flags<L>(G, ex, in.seq, nb, p.k, p.complements != 0, ctx->sig);
        if (ext.cells4) {
            run_pipeline<L>(ctx, ex, in, p, res, &ext, false, (u32) G.rank, (u32) G.n);
            if (!ext.aborted) {
                ++ctx->sig_runs;
                finish();
                return;
            }
            if (ext.kept & 2u) {
                G.failed = true;
                KC_THROW(KC_ERR_INTERNAL, "a rank of the group did not arrive (wait timed out)");
            }
            ++ctx->sig_fallbacks;  // a bucket overflowed on some rank: every rank sees the same status word and falls back
            ctx->sig_overflow_bytes = nb;
        }
        ex.arena->release(mark);
        ex.arena->top = top_mark;
    }
    const KsfGroupPlan gp = kc_ksf_group_plan(nb, G.n, KsCfg<L>::EX_TILE, ctx->fast);
    const bool expect_duplicates = ctx->fast_heuristics && (p.min_frequency > 1 || (ctx->fast_overflow_bytes && nb >= ctx->fast_overflow_bytes / 2 && nb <= ctx->fast_overflow_bytes * 2));
    if (gp.ok && !expect_duplicates && gp.recv_items() <= G.lay.recv_items) {
        const size_t top_mark = ex.arena->top, mark = ex.arena->mark();
        ExtFlags ext;
        ext.flags = reinterpret_cast<const u32 *>(G.heap + G.lay.off_flags);
        ext.cells4 = kc_grp_fast_flags<L>(G, ex, in.seq, nb, p.k, p.complements != 0, p.min_frequency, gp, ctx->fast);
        run_pipeline<L>(ctx, ex, in, p, res, &ext, false, (u32) G.rank, (u32) G.n);
        if (!ext.aborted) {
            ++ctx->fast_runs;
            finish();
            return;
        }
        if (ext.kept & 2u) {
            G.failed = true;
            KC_THROW(KC_ERR_INTERNAL, "a rank of the group did not arrive (wait timed out)");
        }
        ++ctx->fast_fallbacks;  // a slot overflowed on some rank: every rank sees the same status word and falls back
        ctx->fast_overflow_bytes = nb;
        ex.arena->release(mark);
        ex.arena->top = top_mark;
    }
    ExtFlags ext;
    ext.flags = kc_grp_exact_flags<L>(G, ex, in.seq, nb, p.k, p.complements != 0, p.min_frequency, &ext.kept, &ext.n_occ);
    run_pipeline<L>(ctx, ex, in, p, res, &ext, false, (u32) G.rank, (u32) G.n);
    finish();
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
        for (int i = 0; i < 6; ++i) KC_CUDA(cudaEventCreate(&ctx->ev[i]));
        KC_CUDA(cudaHostAlloc(reinterpret_cast<void **>(&ctx->pin_small), kc_ctx::KC_PIN_SMALL, cudaHostAllocDefault));
        if (const char *e = std::getenv("KC_FAST_SET")) ctx->fast.enabled = std::atoi(e) != 0;
        if (const char *e = std::getenv("KC_SIG_SET")) ctx->sig.enabled = std::atoi(e) != 0;
        if (const char *e = std::getenv("KC_FAST_MAX_CTAS")) ctx->fast.max_ctas = std::atoi(e);
        if (const char *e = std::getenv("KC_FAST_TMA")) ctx->fast.tma = std::atoi(e) != 0;
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
    if (ctx->arena.base) cudaFree(ctx->arena.base);
    if (ctx->pin_in) cudaFreeHost(ctx->pin_in);
    if (ctx->pin_out) cudaFreeHost(ctx->pin_out);
    if (ctx->pin_small) cudaFreeHost(ctx->pin_small);
    group_detach(ctx);
    for (int i = 0; i < 6; ++i)
        if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
    for (int i = 0; i < kc_ctx::KC_H2D_CHUNKS; ++i)
        if (ctx->chunk_ev[i]) cudaEventDestroy(ctx->chunk_ev[i]);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
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
    KC_CUDA(cudaSetDevice(ctx->device));
    const int limbs = kc_limbs_for_k(p->k);
    CudaExec ex{ctx->stream, &ctx->arena};
    ex.prof = &ctx->prof;
    ex.pinned = ctx->pin_small;
    ex.pinned_cap = ctx->pin_small ? kc_ctx::KC_PIN_SMALL : 0;
    DevInput di{in->seq, in->n_bytes, in->rec_off, in->rec_len, in->n_recs};
    DevResult res;
    KC_TRACE_POINT("compute_device: start");
    const SigPlan sig = kc_sig_plan(in->n_bytes, p->k, ctx->sig);
    run_with_arena(ctx, estimate_arena(in->n_bytes, in->n_recs, limbs, p->complements != 0, p->assume_simplitigs != 0, false, &ctx->fast, &sig),
                   estimate_arena(in->n_bytes, in->n_recs, limbs, p->complements != 0, p->assume_simplitigs != 0, true, &ctx->fast, &sig),
                   [&] { dispatch_pipeline(ctx, ex, di, *p, res); });
    KC_TRACE_POINT("compute_device: launched");
    KC_CUDA(cudaStreamSynchronize(ctx->stream));
    KC_TRACE_POINT("compute_device: synced");
    out->ms = const_cast<u8 *>(res.ms);
    out->ms_maxone = const_cast<u8 *>(res.maxone);
    out->length = res.length;
    out->n_kmers = res.n_kmers;
    out->n_occurrences = res.n_occ;
    out->n_nodes = res.n_nodes;
    out->n_simplitigs = res.n_simplitigs;
    out->n_launches = ex.launches;
    fill_times(ctx, out);
    ctx->total_launches += ex.launches;
    ctx->read_backs += ex.read_backs;
    return KC_OK;
    KC_API_END(ctx)
}

int kc_compute(kc_ctx *ctx, const kc_params *p, const kc_input *in, kc_output *out) {
    if (!ctx || !in || !out) return KC_ERR_ARG;
    KC_API_BEGIN
    check_params(p);
    check_large_input(ctx, p, in->n_bytes);
    KC_CUDA(cudaSetDevice(ctx->device));
    const int limbs = kc_limbs_for_k(p->k);
    const bool simplitigs = p->assume_simplitigs != 0;
    CudaExec ex{ctx->stream, &ctx->arena};
    ex.prof = &ctx->prof;
    ex.pinned = ctx->pin_small;
    ex.pinned_cap = ctx->pin_small ? kc_ctx::KC_PIN_SMALL : 0;
    DevResult res;
    const SigPlan sig = kc_sig_plan(in->n_bytes, p->k, ctx->sig);
    run_with_arena(ctx, estimate_arena(in->n_bytes, in->n_recs, limbs, p->complements != 0, simplitigs, false, &ctx->fast, &sig),
                   estimate_arena(in->n_bytes, in->n_recs, limbs, p->complements != 0, simplitigs, true, &ctx->fast, &sig), [&] {
        // host -> device.  Large from-FASTA inputs go in chunks on the copy stream: the level-0 partition pass of chunk c starts
        // as soon as chunk c has landed (InputChunks), instead of after the whole copy.
        u8 *d_seq = ex.alloc<u8>(in->n_bytes + 64);
        InputChunks chunks;
        const bool chunked = !simplitigs && in->n_bytes >= (8u << 20);
        if (chunked) {
            if (!ctx->copy_stream) {
                KC_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
                for (int c = 0; c < kc_ctx::KC_H2D_CHUNKS; ++c) KC_CUDA(cudaEventCreateWithFlags(&ctx->chunk_ev[c], cudaEventDisableTiming));
            }
            const u64 granule = 32768;  // whole level-0 tiles for every word width
            chunks.chunk_bytes = (in->n_bytes / kc_ctx::KC_H2D_CHUNKS + granule) / granule * granule;
            chunks.ev = ctx->chunk_ev;
            for (u64 off = 0; off < in->n_bytes; off += chunks.chunk_bytes) {
                const u64 len = std::min<u64>(chunks.chunk_bytes, in->n_bytes - off);
                KC_CUDA(cudaMemcpyAsync(d_seq + off, in->seq + off, len, cudaMemcpyHostToDevice, ctx->copy_stream));
                KC_CUDA(cudaEventRecord(ctx->chunk_ev[chunks.n++], ctx->copy_stream));
            }
        } else {
            KC_CUDA(cudaMemcpyAsync(d_seq, in->seq, in->n_bytes, cudaMemcpyHostToDevice, ctx->stream));
        }
        u64 *d_off = nullptr, *d_len = nullptr;
        if (simplitigs) {
            d_off = ex.alloc<u64>(in->n_recs);
            d_len = ex.alloc<u64>(in->n_recs);
            KC_CUDA(cudaMemcpyAsync(d_off, in->rec_off, in->n_recs * 8, cudaMemcpyHostToDevice, ctx->stream));
            KC_CUDA(cudaMemcpyAsync(d_len, in->rec_len, in->n_recs * 8, cudaMemcpyHostToDevice, ctx->stream));
        }
        DevInput di{d_seq, in->n_bytes, d_off, d_len, in->n_recs, chunked ? &chunks : nullptr};
        try {
            dispatch_pipeline(ctx, ex, di, *p, res);
        } catch (...) {
            if (chunked) cudaStreamSynchronize(ctx->copy_stream);  // `chunks` and the caller's buffer must outlive the copy
            throw;
        }
        if (chunked) chunks.wait_all(ctx->stream);
    });
    // device -> pinned host
    const size_t need = (size_t) res.length * (res.maxone ? 2 : 1) + 64;
    if (ctx->pin_out_cap < need) {
        if (ctx->pin_out) KC_CUDA(cudaFreeHost(ctx->pin_out));
        ctx->pin_out = nullptr;
        ctx->pin_out_cap = 0;
        KC_CUDA(cudaMallocHost(&ctx->pin_out, need + need / 8));
        ctx->pin_out_cap = need + need / 8;
    }
    KC_CUDA(cudaMemcpyAsync(ctx->pin_out, res.ms, res.length, cudaMemcpyDeviceToHost, ctx->stream));
    if (res.maxone)
        KC_CUDA(cudaMemcpyAsync(ctx->pin_out + res.length, res.maxone, res.length, cudaMemcpyDeviceToHost, ctx->stream));
    KC_CUDA(cudaStreamSynchronize(ctx->stream));
    out->ms = ctx->pin_out;
    out->ms_maxone = res.maxone ? ctx->pin_out + res.length : nullptr;
    out->length = res.length;
    out->n_kmers = res.n_kmers;
    out->n_occurrences = res.n_occ;
    out->n_nodes = res.n_nodes;
    out->n_simplitigs = res.n_simplitigs;
    out->n_launches = ex.launches;
    fill_times(ctx, out);
    ctx->total_launches += ex.launches;
    ctx->read_backs += ex.read_backs;
    return KC_OK;
    KC_API_END(ctx)
}

int kc_lower_bound(kc_ctx *ctx, const kc_params *p, const kc_input *in, uint64_t *lower_bound, kc_output *stats) {
    if (!ctx || !in || !lower_bound) return KC_ERR_ARG;
    KC_API_BEGIN
    check_params(p);
    if (p->want_maxone) KC_THROW(KC_ERR_ARG, "lowerbound has no mask output");
    check_large_input(ctx, p, in->n_bytes);
    KC_CUDA(cudaSetDevice(ctx->device));
    const int limbs = kc_limbs_for_k(p->k);
    const bool simplitigs = p->assume_simplitigs != 0;
    CudaExec ex{ctx->stream, &ctx->arena};
    ex.prof = &ctx->prof;
    ex.pinned = ctx->pin_small;
    ex.pinned_cap = ctx->pin_small ? kc_ctx::KC_PIN_SMALL : 0;
    DevResult res;
    const SigPlan sig = kc_sig_plan(in->n_bytes, p->k, ctx->sig);
    run_with_arena(ctx, estimate_arena(in->n_bytes, in->n_recs, limbs, p->complements != 0, simplitigs, false, &ctx->fast, &sig),
                   estimate_arena(in->n_bytes, in->n_recs, limbs, p->complements != 0, simplitigs, true, &ctx->fast, &sig), [&] {
        u8 *d_seq = ex.alloc<u8>(in->n_bytes + 64);
        KC_CUDA(cudaMemcpyAsync(d_seq, in->seq, in->n_bytes, cudaMemcpyHostToDevice, ctx->stream));
        u64 *d_off = nullptr, *d_len = nullptr;
        if (simplitigs) {
            d_off = ex.alloc<u64>(in->n_recs);
            d_len = ex.alloc<u64>(in->n_recs);
            KC_CUDA(cudaMemcpyAsync(d_off, in->rec_off, in->n_recs * 8, cudaMemcpyHostToDevice, ctx->stream));
            KC_CUDA(cudaMemcpyAsync(d_len, in->rec_len, in->n_recs * 8, cudaMemcpyHostToDevice, ctx->stream));
        }
        DevInput di{d_seq, in->n_bytes, d_off, d_len, in->n_recs};
        dispatch_pipeline(ctx, ex, di, *p, res, /*lower_bound=*/true);
    });
    KC_CUDA(cudaStreamSynchronize(ctx->stream));
    *lower_bound = res.lower_bound;
    if (stats) {
        std::memset(stats, 0, sizeof(*stats));
        stats->n_kmers = res.n_kmers;
        stats->n_occurrences = res.n_occ;
        stats->n_nodes = res.n_nodes;
        stats->n_simplitigs = res.n_simplitigs;
        stats->n_launches = ex.launches;
        fill_times(ctx, stats);
    }
    ctx->total_launches += ex.launches;
    ctx->read_backs += ex.read_backs;
    return KC_OK;
    KC_API_END(ctx)
}

// device result -> the context's pinned host buffer
static u8 *copy_result_to_pinned(kc_ctx *ctx, const u8 *dev, u64 n) {
    const size_t need = (size_t) n + 64;
    if (ctx->pin_out_cap < need) {
        if (ctx->pin_out) KC_CUDA(cudaFreeHost(ctx->pin_out));
        ctx->pin_out = nullptr;
        ctx->pin_out_cap = 0;
        KC_CUDA(cudaMallocHost(&ctx->pin_out, need + need / 8));
        ctx->pin_out_cap = need + need / 8;
    }
    if (n) KC_CUDA(cudaMemcpyAsync(ctx->pin_out, dev, n, cudaMemcpyDeviceToHost, ctx->stream));
    KC_CUDA(cudaStreamSynchronize(ctx->stream));
    return ctx->pin_out;
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
    KC_CUDA(cudaSetDevice(ctx->device));
    const int limbs = kc_limbs_for_k(p->k);
    const SigPlan sig = kc_sig_plan(in->n_bytes, p->k, ctx->sig);
    ensure_arena(ctx, estimate_arena(in->n_bytes, 0, limbs, false, true, false, &ctx->fast, &sig));
    ctx->arena.reset();
    CudaExec ex{ctx->stream, &ctx->arena};
    ex.prof = &ctx->prof;
    ex.pinned = ctx->pin_small;
    ex.pinned_cap = ctx->pin_small ? kc_ctx::KC_PIN_SMALL : 0;
    std::memset(out, 0, sizeof(*out));
    KC_CUDA(cudaEventRecord(ctx->ev[0], ctx->stream));
    const u64 padded = (in->n_bytes + 31) / 32 * 32 + 64;
    u8 *d_seq = ex.alloc<u8>(padded);
    ex.fill_bytes(d_seq + (in->n_bytes & ~(u64) 31), '\n', padded - (in->n_bytes & ~(u64) 31));
    KC_CUDA(cudaMemcpyAsync(d_seq, in->seq, in->n_bytes, cudaMemcpyHostToDevice, ctx->stream));
    KC_CUDA(cudaEventRecord(ctx->ev[1], ctx->stream));
    StreamingResult r;
    if (limbs == 1) r = streaming_only<1>(ctx, ex, d_seq, in->n_bytes, *p);
    else if (limbs == 2) r = streaming_only<2>(ctx, ex, d_seq, in->n_bytes, *p);
    else r = streaming_only<4>(ctx, ex, d_seq, in->n_bytes, *p);
    for (int i = 2; i <= 4; ++i) KC_CUDA(cudaEventRecord(ctx->ev[i], ctx->stream));
    out->ms = copy_result_to_pinned(ctx, r.ms, r.length);
    out->length = r.length;
    out->n_kmers = r.n_kept;
    out->n_occurrences = r.n_occ;
    out->n_launches = ex.launches;
    fill_times(ctx, out);
    ctx->total_launches += ex.launches;
    ctx->read_backs += ex.read_backs;
    return KC_OK;
    KC_API_END(ctx)
}

int kc_maskopt(kc_ctx *ctx, const uint8_t *ms, uint64_t n, int k, int complements, int minimize, kc_output *out) {
    if (!ctx || (!ms && n) || !out) return KC_ERR_ARG;
    KC_API_BEGIN
    if (k < 1 || k > 127) KC_THROW(KC_ERR_ARG, "k must be in 1..127");
    if (n + 1 >= 0xFFFFFFF0ULL) KC_THROW(KC_ERR_TOO_LARGE, "more than 2^32 sequence bytes on one GPU");
    KC_CUDA(cudaSetDevice(ctx->device));
    const int limbs = kc_limbs_for_k(k);
    // min-one keeps the sorted key set of the first construction (n * (8 limbs + 1) bytes) at the arena bottom while a second,
    // flags-only construction runs above it
    ensure_arena(ctx, estimate_arena(n + 1, 0, limbs, false, true) + 2 * n + (minimize ? (size_t) n * (8 * limbs + 1) + n / 4 : 0));
    ctx->arena.reset();
    CudaExec ex{ctx->stream, &ctx->arena};
    ex.prof = &ctx->prof;
    ex.pinned = ctx->pin_small;
    ex.pinned_cap = ctx->pin_small ? kc_ctx::KC_PIN_SMALL : 0;
    std::memset(out, 0, sizeof(*out));
    KC_CUDA(cudaEventRecord(ctx->ev[0], ctx->stream));
    u8 *d_seq = ex.alloc<u8>(n + 64);
    ex.fill_bytes(d_seq + (n & ~(u64) 31), '\n', n + 64 - (n & ~(u64) 31));
    if (n) KC_CUDA(cudaMemcpyAsync(d_seq, ms, n, cudaMemcpyHostToDevice, ctx->stream));
    KC_CUDA(cudaEventRecord(ctx->ev[1], ctx->stream));
    MaskoptResult r;
    if (limbs == 1) r = kc_maskopt_run<1>(ex, d_seq, n, k, complements != 0, minimize != 0);
    else if (limbs == 2) r = kc_maskopt_run<2>(ex, d_seq, n, k, complements != 0, minimize != 0);
    else r = kc_maskopt_run<4>(ex, d_seq, n, k, complements != 0, minimize != 0);
    for (int i = 2; i <= 4; ++i) KC_CUDA(cudaEventRecord(ctx->ev[i], ctx->stream));
    out->ms = copy_result_to_pinned(ctx, r.ms, r.length);
    out->length = r.length;
    out->n_kmers = r.n_kmers;
    out->n_launches = ex.launches;
    fill_times(ctx, out);
    ctx->total_launches += ex.launches;
    ctx->read_backs += ex.read_backs;
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
    KC_CUDA(cudaSetDevice(ctx->device));
    const int limbs = kc_limbs_for_k(p->k);
    size_t need = (size_t) ((double) in->n_bytes * (1.0 + 2.0 * 8 * limbs + 4.0) * 1.15) + (256u << 20);
    ensure_arena(ctx, need);
    ctx->arena.reset();
    CudaExec ex{ctx->stream, &ctx->arena};
    ex.prof = &ctx->prof;
    ex.pinned = ctx->pin_small;
    ex.pinned_cap = ctx->pin_small ? kc_ctx::KC_PIN_SMALL : 0;
    u8 *d_seq = ex.alloc<u8>(in->n_bytes + 64);
    KC_CUDA(cudaMemcpyAsync(d_seq, in->seq, in->n_bytes, cudaMemcpyHostToDevice, ctx->stream));
    DevInput di{d_seq, in->n_bytes, nullptr, nullptr, in->n_recs};
    if (p->k < 32) count_only<1>(ctx, ex, di, *p, keys, counts, n);
    else if (p->k < 64) count_only<2>(ctx, ex, di, *p, keys, counts, n);
    else count_only<4>(ctx, ex, di, *p, keys, counts, n);
    ctx->total_launches += ex.launches;
    ctx->read_backs += ex.read_backs;
    return KC_OK;
    KC_API_END(ctx)
}

int kc_partial_presort(kc_ctx *ctx, const uint64_t *kmers, uint64_t n, int k, uint64_t *out) {
    if (!ctx || (n && (!kmers || !out))) return KC_ERR_ARG;
    KC_API_BEGIN
    if (k < 1 || k > 127) KC_THROW(KC_ERR_ARG, "k must be in 1..127");
    if (n >= 0xFFFFFFF0ULL) KC_THROW(KC_ERR_TOO_LARGE, "too many k-mers");
    if (n == 0) return KC_OK;
    KC_CUDA(cudaSetDevice(ctx->device));
    const int limbs = kc_limbs_for_k(k);
    ensure_arena(ctx, (size_t) (n * (16.0 * limbs + 64.0)) + (64u << 20));
    ctx->arena.reset();
    CudaExec ex{ctx->stream, &ctx->arena};
    ex.prof = &ctx->prof;
    ex.pinned = ctx->pin_small;
    ex.pinned_cap = ctx->pin_small ? kc_ctx::KC_PIN_SMALL : 0;
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
    ctx->total_launches += ex.launches;
    ctx->read_backs += ex.read_backs;
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
    KC_CUDA(cudaSetDevice(ctx->device));
    const int limbs = kc_limbs_for_k(p->k);
    // the sorted-keys route, or at 2^32 bytes and more the signature construction alone: sequence, flags, window mask, its buffers
    size_t need = (size_t) ((double) nb * (1.0 + 2.0 * 8 * limbs + 4.0 + 0.2) * 1.15) + (256u << 20);
    if (nb >= KC_POS32_BYTES) need = (size_t) (((double) nb * 1.25 + (double) kc_sig_arena_bytes(kc_sig_plan(nb, p->k, ctx->sig), nb)) * 1.05) + (256u << 20);
    ensure_arena(ctx, need);
    ctx->arena.reset();
    CudaExec ex{ctx->stream, &ctx->arena};
    ex.prof = &ctx->prof;
    ex.pinned = ctx->pin_small;
    ex.pinned_cap = ctx->pin_small ? kc_ctx::KC_PIN_SMALL : 0;
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
    if (limbs == 1) digest_only<1>(ctx, ex, di, *p, win_mask, digest);
    else if (limbs == 2) digest_only<2>(ctx, ex, di, *p, win_mask, digest);
    else digest_only<4>(ctx, ex, di, *p, win_mask, digest);
    ctx->total_launches += ex.launches;
    ctx->read_backs += ex.read_backs;
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
    KC_CUDA(cudaSetDevice(ctx->device));
    const int limbs = kc_limbs_for_k(k);
    ensure_arena(ctx, estimate_arena(0, n, limbs, complements != 0, true) + n * 16 * limbs);
    ctx->arena.reset();
    CudaExec ex{ctx->stream, &ctx->arena};
    ex.prof = &ctx->prof;
    ex.pinned = ctx->pin_small;
    ex.pinned_cap = ctx->pin_small ? kc_ctx::KC_PIN_SMALL : 0;
    if (k < 32) overlap_only<1>(ctx, ex, first, last, n, k, complements != 0, lower_bound != 0, strict != 0, edge_from, overlaps);
    else if (k < 64) overlap_only<2>(ctx, ex, first, last, n, k, complements != 0, lower_bound != 0, strict != 0, edge_from, overlaps);
    else overlap_only<4>(ctx, ex, first, last, n, k, complements != 0, lower_bound != 0, strict != 0, edge_from, overlaps);
    ctx->total_launches += ex.launches;
    ctx->read_backs += ex.read_backs;
    return KC_OK;
    KC_API_END(ctx)
}

uint64_t kc_shard_granule(int k) {
    const int limbs = kc_limbs_for_k(k);
    return limbs == 1 ? KsCfg<1>::EX_TILE : (limbs == 2 ? KsCfg<2>::EX_TILE : KsCfg<4>::EX_TILE);
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
    KC_CUDA(cudaSetDevice(ctx->device));
    const int limbs = kc_limbs_for_k(p->k);
    CudaExec ex{ctx->stream, &ctx->arena};
    ex.prof = &ctx->prof;
    ex.pinned = ctx->pin_small;
    ex.pinned_cap = ctx->pin_small ? kc_ctx::KC_PIN_SMALL : 0;
    DevInput di{in->seq, in->n_bytes, nullptr, nullptr, 0};
    DevResult res;
    // no retry with a larger arena here: a rank that repeated its job alone would leave the group's sync numbers behind
    ensure_arena(ctx, group_arena_need(in->n_bytes, ctx->grp.n, limbs, p->complements != 0, false));
    ctx->arena.reset();
    try {
        if (limbs == 1) group_compute_rank<1>(ctx, ex, di, *p, res);
        else if (limbs == 2) group_compute_rank<2>(ctx, ex, di, *p, res);
        else group_compute_rank<4>(ctx, ex, di, *p, res);
    } catch (const KcError &e) {
        if (e.code != KC_ERR_EMPTY) ctx->grp.failed = true;  // "no k-mers" is found by every rank at the same point
        throw;
    }
    KC_CUDA(cudaStreamSynchronize(ctx->stream));
    if (slice_begin) *slice_begin = res.slice_begin;
    if (slice_len) *slice_len = res.slice_len;
    out->ms = const_cast<u8 *>(res.ms);
    out->ms_maxone = nullptr;
    out->length = res.length;
    out->n_kmers = res.n_kmers;
    out->n_occurrences = res.n_occ;
    out->n_nodes = res.n_nodes;
    out->n_simplitigs = res.n_simplitigs;
    out->n_launches = ex.launches;
    fill_times(ctx, out);
    ctx->total_launches += ex.launches;
    ctx->read_backs += ex.read_backs;
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
    const KsfGroupPlan gp = kc_ksf_group_plan(n_bytes, n_ranks, tile, tune);
    const GrpLayout lay = kc_grp_layout(n_bytes, kc_limbs_for_k(k), n_ranks, false, tile, tune);
    const u64 tiles = kc_div_up(n_bytes, tile);
    plan[0] = gp.ok ? 1 : 0;
    plan[1] = std::min<u64>(n_bytes, tiles * (u64) rank / (u64) n_ranks * tile);
    plan[2] = std::min<u64>(n_bytes, tiles * (u64) (rank + 1) / (u64) n_ranks * tile);
    plan[3] = gp.ok ? gp.dig_begin(rank) : (u64) ((rank * 256 + n_ranks - 1) / n_ranks);
    plan[4] = gp.ok ? gp.dig_begin(rank + 1) : (u64) (((rank + 1) * 256 + n_ranks - 1) / n_ranks);
    plan[5] = gp.ok ? gp.n_digits : 256;
    plan[6] = gp.cap_sub;
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
    u8 *pin_out = nullptr;
    size_t pin_out_cap = 0;
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
    if (g->pin_out) cudaFreeHost(g->pin_out);
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
        if (in->n_bytes >= 0xFFFFFFF0ULL) KC_THROW(KC_ERR_TOO_LARGE, "more than 2^32 sequence bytes");
        const int limbs = kc_limbs_for_k(p->k);
        // (re)build the heaps when the job does not fit the ones in place
        const KcGroup &G0 = c0->grp;
        if (!G0.attached() || in->n_bytes > G0.lay.n_bytes_cap || limbs > G0.lay.limbs || G0.failed) {
            group_release_heaps(g);
            const u64 cap = std::min<u64>(0xFFFFFFE0ULL, in->n_bytes + in->n_bytes / 16 + (1u << 20));
            for (int r = 0; r < g->n; ++r) {
                g->ctx[r]->fast = c0->fast;  // one plan for the whole group
                g->ctx[r]->fast_heuristics = c0->fast_heuristics;
                g->ctx[r]->fast_overflow_bytes = c0->fast_overflow_bytes;
                group_alloc_common(g->ctx[r], g->n, r, limbs == 1 ? 31 : (limbs == 2 ? 63 : 127), cap, true);
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
        {   // (one thread per rank: cudaMalloc of tens of GB takes ~0.1 s per device)
            KcError errs[KC_MAX_PEERS];
            bool bad[KC_MAX_PEERS] = {};
            std::vector<std::thread> th;
            for (int r = 0; r < g->n; ++r)
                th.emplace_back([&, r] {
                    try {
                        KC_CUDA(cudaSetDevice(g->ctx[r]->device));
                        ensure_arena(g->ctx[r], group_arena_need(in->n_bytes, g->n, limbs, p->complements != 0, false));
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
        u64 launches = 0;
        kc_output o;
    } ro[KC_MAX_PEERS];
    auto worker = [&](int r) {
        kc_ctx *ctx = g->ctx[r];
        RankOut &R = ro[r];
        try {
            KC_CUDA(cudaSetDevice(ctx->device));
            KcGroup &G = ctx->grp;
            ctx->arena.reset();
            CudaExec ex{ctx->stream, &ctx->arena};
            ex.prof = &ctx->prof;
            ex.pinned = ctx->pin_small;
            ex.pinned_cap = ctx->pin_small ? kc_ctx::KC_PIN_SMALL : 0;
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
            const int limbs = kc_limbs_for_k(p->k);
            if (limbs == 1) group_compute_rank<1>(ctx, ex, di, *p, R.res);
            else if (limbs == 2) group_compute_rank<2>(ctx, ex, di, *p, R.res);
            else group_compute_rank<4>(ctx, ex, di, *p, R.res);
            {   // the first rank to get here sizes the common result buffer
                std::lock_guard<std::mutex> lk(g->out_mutex);
                const size_t need = (size_t) R.res.length + 64;
                if (g->pin_out_cap < need) {
                    if (g->pin_out) KC_CUDA(cudaFreeHost(g->pin_out));
                    g->pin_out = nullptr;
                    g->pin_out_cap = 0;
                    KC_CUDA(cudaHostAlloc(reinterpret_cast<void **>(&g->pin_out), need + need / 8, cudaHostAllocPortable));
                    g->pin_out_cap = need + need / 8;
                }
            }
            if (R.res.slice_len)
                KC_CUDA(cudaMemcpyAsync(g->pin_out + R.res.slice_begin, R.res.ms, R.res.slice_len, cudaMemcpyDeviceToHost, ctx->stream));
            KC_CUDA(cudaStreamSynchronize(ctx->stream));
            if (ex.read(ws) & 2u) KC_THROW(KC_ERR_INTERNAL, "a rank of the group did not arrive (wait timed out)");
            R.launches = ex.launches;
            fill_times(ctx, &R.o);
            ctx->total_launches += ex.launches;
            ctx->read_backs += ex.read_backs;
        } catch (const KcError &e) {
            R.code = e.code;
            char buf[512];
            std::snprintf(buf, sizeof(buf), "rank %d: %s (%s:%d)", r, e.what, e.file, e.line);
            R.what = buf;
            if (e.code != KC_ERR_EMPTY) {  // "no k-mers" is found by every rank at the same point; anything else strands the others
                ctx->grp.failed = true;
                g->hs.abort();
            }
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
    for (int r = 0; r < g->n; ++r)
        if (ro[r].code != KC_OK) {
            if (ro[r].code != KC_ERR_EMPTY)
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
    std::memset(out, 0, sizeof(*out));
    out->ms = g->pin_out;
    out->length = ro[0].res.length;
    out->n_kmers = ro[0].res.n_kmers;
    out->n_occurrences = ro[0].res.n_occ;
    out->n_nodes = ro[0].res.n_nodes;
    out->n_simplitigs = ro[0].res.n_simplitigs;
    out->t = ro[0].o.t;
    for (int r = 0; r < g->n; ++r) {
        out->n_launches += ro[r].launches;
        if (ro[r].o.t.total_ms > out->t.total_ms) out->t = ro[r].o.t;  // the slowest rank's stage times
    }
    return KC_OK;
}

uint64_t kc_total_launches(const kc_ctx *ctx) { return ctx ? ctx->total_launches : 0; }

int kc_get_stat(const kc_ctx *ctx, const char *name, uint64_t *value) {
    if (!ctx || !name || !value) return KC_ERR_ARG;
    if (std::strcmp(name, "fast_runs") == 0) *value = ctx->fast_runs;
    else if (std::strcmp(name, "fast_fallbacks") == 0) *value = ctx->fast_fallbacks;
    else if (std::strcmp(name, "sig_runs") == 0) *value = ctx->sig_runs;
    else if (std::strcmp(name, "sig_fallbacks") == 0) *value = ctx->sig_fallbacks;
    else if (std::strcmp(name, "total_launches") == 0) *value = ctx->total_launches;
    else if (std::strcmp(name, "read_backs") == 0) *value = ctx->read_backs;
    else if (std::strcmp(name, "tail_spec_runs") == 0) *value = ctx->tail_spec_runs;
    else if (std::strcmp(name, "tail_spec_fallbacks") == 0) *value = ctx->tail_spec_fallbacks;
    else if (std::strcmp(name, "arena_bytes") == 0) *value = ctx->arena.cap;
    else if (std::strcmp(name, "arena_high") == 0) *value = ctx->arena.high;
    else if (std::strcmp(name, "fast_max_ctas") == 0) *value = (uint64_t) ctx->fast.max_ctas;
    else if (std::strcmp(name, "path_levels") == 0) *value = ctx->path_stats.levels_run;
    else if (std::strcmp(name, "path_ban_rounds") == 0) *value = ctx->path_stats.ban_rounds;
    else if (std::strcmp(name, "path_bans") == 0) *value = ctx->path_stats.bans;
    else return KC_ERR_ARG;
    return KC_OK;
}

int kc_set_option(kc_ctx *ctx, const char *name, int value) {
    if (!ctx || !name) return KC_ERR_ARG;
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
        ctx->spec_fail_bytes = 0;
        return KC_OK;
    }
    // histogram-free set construction (kmerset_fast.cuh); the last three exist so that tests can reach the multi-level
    // plan and the overflow fallback with small inputs
    if (std::strcmp(name, "fast_set") == 0) {
        ctx->fast.enabled = value != 0;
        return KC_OK;
    }
    if (std::strcmp(name, "fast_leaf_target") == 0 && value >= 1 && value <= 1024) {
        ctx->fast.leaf_target = (u32) value;
        return KC_OK;
    }
    if (std::strcmp(name, "fast_sigmas") == 0 && value >= 0) {
        ctx->fast.sigmas = (double) value;
        return KC_OK;
    }
    if (std::strcmp(name, "fast_tma") == 0 && (value == 0 || value == 1)) {
        ctx->fast.tma = value != 0;
        return KC_OK;
    }
    if (std::strcmp(name, "fast_heuristics") == 0 && (value == 0 || value == 1)) {
        ctx->fast_heuristics = value != 0;
        ctx->fast_overflow_bytes = 0;
        ctx->sig_overflow_bytes = 0;
        ctx->spec_fail_bytes = 0;
        return KC_OK;
    }
    if (std::strcmp(name, "fast_max_ctas") == 0 && value >= 0 && value <= (1 << 20)) {
        ctx->fast.max_ctas = value;
        return KC_OK;
    }
    if (std::strcmp(name, "fast_min_items") == 0 && value >= 0) {
        ctx->fast.min_items = (u64) value;
        return KC_OK;
    }
    // signature-bucket set construction (kmerset_sig.cuh)
    if (std::strcmp(name, "sig_set") == 0) {
        ctx->sig.enabled = value != 0;
        return KC_OK;
    }
    if (std::strcmp(name, "sig_load_pct") == 0 && value >= 0 && value <= 400) {  // > 100 forces overflows (tests)
        ctx->sig.load_pct = (u32) value;  // 0 = planned from the input size
        return KC_OK;
    }
    if (std::strcmp(name, "sig_min_items") == 0 && value >= 0) {
        ctx->sig.min_items = (u64) value;
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
