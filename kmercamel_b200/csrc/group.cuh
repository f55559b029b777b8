// Multi-GPU k-mer set construction: hash-range sharding across the GPUs of one box (SURVEY.md §8e; the reference,
// src/parser.h:22-141 + khash, is single-threaded).
//
// Every rank (one GPU; one host thread of a single process, or one process under torchrun) owns a symmetric HEAP in its HBM
// that every other rank can address: peer access inside one process, CUDA IPC between processes — either way plain pointers
// over NVLink / NVSwitch.  All data exchange is device-side stores into a peer's heap, all synchronisation is device-side
// too: a rank announces "my stores for sync number s are done" by writing s into one word of every peer's heap after a
// system-scope fence, and a one-warp wait kernel on the peer's stream spins on those words.  No NCCL, no host round trip and
// no host-side barrier sits on the data path, so the host threads run ahead of their GPUs exactly as on one GPU.
//
// One job (from-FASTA compute, the whole framed sequence resident on every GPU):
//   fast path (fixed slots, kmerset_fast.cuh; what a genome takes)
//     level 0   rank r decodes its slice of the level-0 tiles and stores every (scrambled k-mer, position) straight into the
//               sub-slot (digit, r) of the digit's owner — the partition pass IS the all-to-all; the valid-window words of
//               the slice go to every rank's flag array
//     signal A  fill counts of r's sub-slots -> every owner                  wait A
//     levels 1.., leaf resolve on the owner; a duplicate clears its bit in EVERY rank's flags (remote RED, ~0 on a genome)
//     signal B  (kept, M, overflow status) -> every rank                       wait B
//     every rank now holds the complete first-occurrence bits and the totals: runs -> greedy (deterministic, repeated on
//     every rank) -> the rank's own slice of the superstring
//     signal DONE; the NEXT job waits for it before it touches a peer's heap again
//   exact path (histograms; read sets with coverage, -z > 1, tiny inputs, or after a slot overflow — decided from values every
//   rank sees identically, so all ranks switch together)
//     level-0 histogram of the slice -> counts to every rank -> signal / wait -> exact offsets -> level-0 scatter into the
//     owners' buckets -> signal / wait -> exact levels + resolve into the owner's private bits -> signal / wait -> OR of all
//     ranks' bits read over NVLink.
#pragma once
#include "kmerset_fast.cuh"
#include "kmerset_sig.cuh"
#include "runs.cuh"

struct GrpLayout {
    u64 n_bytes_cap = 0;
    int limbs = 0, n_ranks = 0;
    u64 recv_items = 0, flag_words = 0;
    size_t off_sig = 0, off_cells = 0, off_cnt = 0, off_flags = 0, off_flags2 = 0, off_recv_k = 0, off_recv_p = 0, off_packed = 0, off_seq = 0, total = 0;
};

// Heap of a rank for jobs of up to n_bytes_cap sequence bytes (identical on every rank).
inline GrpLayout kc_grp_layout(u64 n_bytes_cap, int limbs, int n_ranks, bool with_seq, u64 ex_tile, const KsfTuning &tune) {
    GrpLayout y;
    y.n_bytes_cap = n_bytes_cap;
    y.limbs = limbs;
    y.n_ranks = n_ranks;
    const KsfGroupPlan gp = kc_ksf_group_plan(n_bytes_cap, n_ranks, ex_tile, tune);
    const u64 by_plan = gp.ok ? gp.recv_items() + gp.recv_items() / 20 : 0;
    const u64 by_share = (u64) ((double) n_bytes_cap / n_ranks * 1.25) + (1u << 20);  // exact path: a rank's hash range, back to back
    y.recv_items = (by_plan > by_share ? by_plan : by_share) + 65536;
    y.flag_words = n_bytes_cap / 32 + 66;
    size_t o = 0;
    auto take = [&](size_t bytes) {
        const size_t at = o;
        o += (bytes + 255) / 256 * 256;
        return at;
    };
    y.off_sig = take(KC_MAX_PEERS * 4);
    y.off_cells = take(KC_MAX_PEERS * 4 * 8);
    y.off_cnt = take((size_t) KC_MAX_PEERS * 256 * 4);
    y.off_flags = take(y.flag_words * 4);
    y.off_flags2 = take(y.flag_words * 4);
    y.off_recv_k = take(y.recv_items * 8 * (u64) limbs);
    y.off_recv_p = take(y.recv_items * 4);
    y.off_packed = take(n_bytes_cap / 4 + 4096);  // 2-bit code words of the whole sequence (signature construction, kmerset_sig.cuh)
    y.off_seq = take(with_seq ? n_bytes_cap + 256 : 0);
    y.total = o;
    return y;
}

struct GrpDev {  // the group as a kernel sees it (by-value kernel parameter)
    char *base[KC_MAX_PEERS];
    int n, rank;
    u32 off_sig, off_cells, off_cnt;
};

// Ranks that live in ONE process (kc_init_multi) do not spin on the device: a wait is "every rank has queued its signal (host
// barrier between the rank threads), then my stream waits for the events the others recorded behind theirs".  Nothing busy-
// waits on a GPU, so ranks may share a device (tests on a one-GPU box; a spinning kernel there would starve the very rank it
// waits for whenever that rank's host thread needs the device to go idle — lazy module loading, cudaMalloc).  The host threads
// still never wait for a GPU, only for each other.
#include <condition_variable>
struct GrpHostSync {
    std::mutex m;
    std::condition_variable cv;
    int n = 0, arrived = 0;
    u64 generation = 0;
    bool aborted = false;
    cudaEvent_t ev[KC_MAX_PEERS][2] = {};
    bool arrive_and_wait() {  // false: some rank left the job (abort())
        std::unique_lock<std::mutex> lk(m);
        if (aborted) return false;
        const u64 gen = generation;
        if (++arrived == n) {
            arrived = 0;
            ++generation;
            cv.notify_all();
            return true;
        }
        cv.wait(lk, [&] { return generation != gen || aborted; });
        return !aborted;
    }
    void abort() {
        std::lock_guard<std::mutex> lk(m);
        aborted = true;
        cv.notify_all();
    }
};

struct KcGroup {
    int n = 0, rank = 0;
    GrpHostSync *hs = nullptr;            // != nullptr: in-process group (events + host barrier instead of the wait kernel)
    GrpLayout lay;
    char *heap = nullptr;                 // own heap (cudaMalloc by the library)
    char *peer[KC_MAX_PEERS] = {};        // every rank's heap as mapped here (peer[rank] = heap)
    bool ipc_opened[KC_MAX_PEERS] = {};
    u32 seq = 0;                          // sync numbers used so far (identical on every rank)
    bool done_pending = false;            // a DONE signal (number done_seq) is out; the next job waits for it
    u32 done_seq = 0;
    bool failed = false;                  // a wait timed out or a rank left a job half way: the sync numbers no longer agree
    // per-rank scratch outside the heap
    u32 *cnt0 = nullptr;                  // [256] level-0 fill counts of this rank's sub-slots
    u64 *cells_local = nullptr;           // [4]
    void **dst_k = nullptr;               // [256] device tables for the level-0 pass
    u32 **dst_p = nullptr;
    void **h_dst = nullptr;               // pinned host staging of both tables: [512]
    u16 *tile_hist = nullptr;             // exact path: level-0 tile histograms of the slice
    size_t tile_hist_cap = 0;
    u64 tab_n_bytes = ~0ull;              // the job geometry the device tables dst_k / dst_p were built for (fast path)
    int tab_limbs = 0;
    u32 tab_n_digits = 0;                 // ... and the plan they encode (KsfGroupPlan n_digits, cap_sub)
    u64 tab_cap_sub = 0;
    u64 timeout_ns = 30ull * 1000000000ull;
    bool attached() const { return n > 0 && heap != nullptr; }
    GrpDev dev() const {
        GrpDev d;
        for (int i = 0; i < KC_MAX_PEERS; ++i) d.base[i] = i < n ? peer[i] : nullptr;
        d.n = n;
        d.rank = rank;
        d.off_sig = (u32) lay.off_sig;
        d.off_cells = (u32) lay.off_cells;
        d.off_cnt = (u32) lay.off_cnt;
        return d;
    }
    KsfFlagPeers all_flags(size_t off) const {
        KsfFlagPeers fp;
        for (int i = 0; i < KC_MAX_PEERS; ++i) fp.f[i] = i < n ? reinterpret_cast<u32 *>(peer[i] + off) : nullptr;
        fp.n = n;
        return fp;
    }
};

#ifdef __CUDACC__

// One block.  Optional payloads travel in front of the signal:
//   cnt0 != nullptr : min(cnt0[d], cap) for d < n_digits  -> recv_cnt[this rank][d] of EVERY rank
//   cells != nullptr: cells[0..4)                          -> cells[this rank][0..4) of every rank
// then a system-scope fence and sig[this rank] = seq on every rank.
__global__ void __launch_bounds__(256) kc_grp_signal_kernel(GrpDev g, u32 seq, const u32 *cnt0, u32 n_digits, u32 cap, const u64 *cells) {
    if (cnt0) {
        for (u32 d = threadIdx.x; d < n_digits; d += 256) {
            const u32 c = cnt0[d] < cap ? cnt0[d] : cap;
            for (int r = 0; r < g.n; ++r) reinterpret_cast<u32 *>(g.base[r] + g.off_cnt)[g.rank * 256 + d] = c;
        }
    }
    if (cells && threadIdx.x < 4) {
        const u64 v = cells[threadIdx.x];
        for (int r = 0; r < g.n; ++r) reinterpret_cast<u64 *>(g.base[r] + g.off_cells)[g.rank * 4 + threadIdx.x] = v;
    }
    __threadfence_system();
    __syncthreads();
    if ((int) threadIdx.x < g.n) {
        __threadfence_system();
        *reinterpret_cast<volatile u32 *>(g.base[threadIdx.x] + g.off_sig + 4 * g.rank) = seq;
    }
}

// One warp: lane s waits until rank s has announced sync number seq (or a later one).  A rank that never arrives must not
// hang the GPU: after timeout_ns the kernel gives up and raises bit 1 of *status, which every later host read-back checks.
__global__ void __launch_bounds__(32) kc_grp_wait_kernel(GrpDev g, u32 seq, u32 *status, u64 timeout_ns) {
    if ((int) threadIdx.x < g.n) {
        const volatile u32 *sig = reinterpret_cast<const volatile u32 *>(g.base[g.rank] + g.off_sig + 4 * threadIdx.x);
        u64 t0;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
        while ((int) (*sig - seq) < 0) {
            __nanosleep(200);
            u64 t1;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
            if (t1 - t0 > timeout_ns) {
                atomicOr(status, 2u);
                break;
            }
        }
    }
    __threadfence_system();
}

// flags2[w] = OR over the ranks of their private bit arrays (exact path; read over NVLink).
__global__ void __launch_bounds__(256) kc_grp_or_flags_kernel(KsfFlagPeers src, u32 *dst, u64 n_words) {
    const u64 w = (u64) blockIdx.x * 256 + threadIdx.x;
    if (w >= n_words) return;
    u32 v = 0;
    for (int r = 0; r < src.n; ++r) v |= src.f[r][w];
    dst[w] = v;
}

inline void kc_grp_signal(KcGroup &G, CudaExec &ex, u32 seq, const u32 *cnt0 = nullptr, u32 n_digits = 0, u32 cap = 0xFFFFFFFFu, const u64 *cells = nullptr) {
    kc_grp_signal_kernel<<<1, 256, 0, ex.stream>>>(G.dev(), seq, cnt0, n_digits, cap, cells);
    ++ex.launches;
    KC_CUDA(cudaGetLastError());
    if (G.hs) KC_CUDA(cudaEventRecord(G.hs->ev[G.rank][seq & 1], ex.stream));
}
// Signals and waits strictly alternate on every rank (signal s, wait s, signal s + 1, ...), which is what lets two events per
// rank do: nobody re-records event s & 1 before every rank has queued its wait on it (it passed the barrier of wait s + 1).
inline void kc_grp_wait(KcGroup &G, CudaExec &ex, u32 seq, u32 *status) {
    if (G.hs) {
        if (!G.hs->arrive_and_wait()) {
            G.failed = true;
            KC_THROW(KC_ERR_INTERNAL, "another rank of the group failed");
        }
        for (int s = 0; s < G.n; ++s)
            if (s != G.rank) KC_CUDA(cudaStreamWaitEvent(ex.stream, G.hs->ev[s][seq & 1], 0));
        return;
    }
    kc_grp_wait_kernel<<<1, 32, 0, ex.stream>>>(G.dev(), seq, status, G.timeout_ns);
    ++ex.launches;
    KC_CUDA(cudaGetLastError());
}

// cells4 = {sum kept, 0, sum M, OR status} over the cells every rank announced (after the wait that follows signal B).
inline void kc_grp_sum_cells(KcGroup &G, CudaExec &ex, u64 *cells4, const u32 *wait_status) {
    const u64 *hc = reinterpret_cast<const u64 *>(G.heap + G.lay.off_cells);
    const int n = G.n;
    ex.for_each(1, [=] __device__(u64) {
        u64 kept = 0, m = 0, st = wait_status ? (u64) *wait_status : 0;
        for (int r = 0; r < n; ++r) {
            kept += hc[r * 4 + 0];
            m += hc[r * 4 + 2];
            st |= hc[r * 4 + 3] & 0xFFFFFFFFull;
        }
        cells4[0] = kept;
        cells4[1] = 0;
        cells4[2] = m;
        cells4[3] = st;
    });
}

// ---- fast path ---------------------------------------------------------------------------------------------------------------
// Returns cells4 (device, arena top): {kept, 0, M, status}; the first-occurrence bits are in the rank's own heap (off_flags)
// once the kernels queued here have run.  Nothing is read back: the caller's run count read-back brings the status along.
template <int L>
u64 *kc_grp_fast_flags(KcGroup &G, CudaExec &ex, const u8 *seq, u64 n_bytes, int k, bool complements, int min_freq, const KsfGroupPlan &gp, const KsfTuning &tune) {
    typedef KsCfg<L> Cfg;
    u32 *flags = reinterpret_cast<u32 *>(G.heap + G.lay.off_flags);
    const u64 body_words = kc_div_up(n_bytes, (u64) 32);
    ex.fill_bytes(flags + body_words, 0, 8);  // the padding words nobody writes (kc_runs_load reads one past the end)
    // destination tables of this rank's sub-slots: digit d -> (owner's heap, slot (d - dig_begin(owner)) * n + rank)
    // kept from the previous job only if it had the same geometry AND the same plan: the digit count and the sub-slot stride also
    // follow the options fast_leaf_target / fast_sigmas, and stale ones would scatter items where no owner reads them
    if (G.tab_n_bytes != n_bytes || G.tab_limbs != L || G.tab_n_digits != gp.n_digits || G.tab_cap_sub != gp.cap_sub) {
        KC_CUDA(cudaStreamSynchronize(ex.stream));  // the staging table may still feed an earlier copy
        G.tab_n_bytes = n_bytes;
        G.tab_limbs = L;
        G.tab_n_digits = gp.n_digits;
        G.tab_cap_sub = gp.cap_sub;
        for (u32 d = 0; d < 256; ++d) {
            char *kp = nullptr, *pp = nullptr;
            if (d < gp.n_digits) {
                const u32 o = gp.owner(d);
                const u64 slot = (u64) (d - gp.dig_begin((int) o)) * (u64) G.n + (u64) G.rank;
                kp = G.peer[o] + G.lay.off_recv_k + slot * gp.cap_sub * sizeof(KWord<L>);
                pp = G.peer[o] + G.lay.off_recv_p + slot * gp.cap_sub * 4;
            }
            G.h_dst[d] = kp;
            G.h_dst[256 + d] = pp;
        }
        KC_CUDA(cudaMemcpyAsync(G.dst_k, G.h_dst, 256 * sizeof(void *), cudaMemcpyHostToDevice, ex.stream));
        KC_CUDA(cudaMemcpyAsync(G.dst_p, G.h_dst + 256, 256 * sizeof(void *), cudaMemcpyHostToDevice, ex.stream));
    }
    u64 *cells4 = ex.arena->alloc_top<u64>(4);
    u32 *wait_status = reinterpret_cast<u32 *>(ex.arena->alloc_top<u64>(1));
    ex.fill_bytes(G.cells_local, 0, 32);
    ex.fill_bytes(wait_status, 0, 8);
    u32 *status = reinterpret_cast<u32 *>(G.cells_local + 3);
    kc_ksf_group_scatter0<L>(ex, seq, n_bytes, k, complements, gp, G.rank, G.cnt0, status, reinterpret_cast<KWord<L> *const *>(G.dst_k), G.dst_p,
                             G.all_flags(G.lay.off_flags));
    const u32 sa = ++G.seq;
    kc_grp_signal(G, ex, sa, G.cnt0, gp.n_digits, (u32) gp.cap_sub);
    kc_grp_wait(G, ex, sa, wait_status);
    // the fill counts of my digits' sub-slots, in slot order
    const u32 dig_lo = gp.dig_begin(G.rank), dig_n = gp.dig_begin(G.rank + 1) - dig_lo;
    const size_t mark = ex.arena->mark();
    u32 *sub_cnt = ex.alloc<u32>((u64) (dig_n ? dig_n : 1) * G.n);
    {
        const u32 *rc = reinterpret_cast<const u32 *>(G.heap + G.lay.off_cnt);
        const int n = G.n;
        ex.for_each((u64) dig_n * n, [=] __device__(u64 i) {
            const u32 lb = (u32) (i / n), s = (u32) (i % n);
            sub_cnt[i] = rc[s * 256 + dig_lo + lb];
        });
    }
    kc_ksf_group_resolve<L>(ex, min_freq, gp, G.rank, reinterpret_cast<const KWord<L> *>(G.heap + G.lay.off_recv_k),
                            reinterpret_cast<const u32 *>(G.heap + G.lay.off_recv_p), sub_cnt, G.all_flags(G.lay.off_flags), G.cells_local, tune);
    ex.arena->release(mark);
    const u32 sb = ++G.seq;
    kc_grp_signal(G, ex, sb, nullptr, 0, 0, G.cells_local);
    kc_grp_wait(G, ex, sb, wait_status);
    kc_grp_sum_cells(G, ex, cells4, wait_status);
    return cells4;
}

// ---- signature buckets (kmerset_sig.cuh) ---------------------------------------------------------------------------------------------
// What travels is a RECORD (8 bytes for ~5 windows) instead of a 12-byte item per window, so the exchange over NVLink shrinks
// ~7 x and the owner needs no further partition level: the bucket a record lands in is already the unit the resolve works on.
//   scan      rank r scans its slice of the tiles: records staged per bucket in its own HBM (slots reserved with a LOCAL counter);
//             code words + valid-window words of the slice -> every rank
//   ship      the staged records, compacted into one dense stream per owner (bucket % n), -> the owner's receive array, and the
//             offsets of the owner's buckets inside the stream -> its offset table: few, long, coalesced NVLink writes
//   signal A / wait A
//   resolve   the owner walks its buckets (the sub-slots of all senders back to back), clears a duplicate's bit in EVERY rank's flags
//   signal B  (kept, M, overflow status) -> every rank / wait B
// The receive array (one stream per sender) lives in the key receive region of the heap, the offset tables in the position receive region.
// Returns nullptr when the plan does not apply to this job (too small, k < 26, heap regions too small).
template <int L>
u64 *kc_grp_sig_flags(KcGroup &G, CudaExec &ex, const u8 *seq, u64 n_bytes, int k, bool complements, const SigTuning &tune) {
    const SigPlan pl = kc_sig_plan(n_bytes, k, tune);
    if (!pl.ok || G.n < 1 || pl.n_buckets >= (1u << 28)) return nullptr;
    const u32 sub_cap = kc_sig_sub_cap(pl, G.n);
    const u32 nbr = kc_sig_owned_buckets(pl.n_buckets, G.n, 0);
    const u32 region_cap = kc_sig_region_cap(n_bytes, G.n);
    if ((u64) G.n * region_cap * 8 > G.lay.recv_items * 8 * (u64) G.lay.limbs) return nullptr;
    if ((u64) G.n * ((u64) nbr + 1) * 4 > G.lay.recv_items * 4) return nullptr;
    u32 *flags = reinterpret_cast<u32 *>(G.heap + G.lay.off_flags);
    const u64 body_words = kc_div_up(n_bytes, (u64) 32);
    ex.fill_bytes(flags + body_words, 0, 8);  // the padding words nobody writes (kc_runs_load reads one past the end)
    SigPeers sp;
    for (int i = 0; i < KC_MAX_PEERS; ++i) {
        sp.recs[i] = i < G.n ? reinterpret_cast<u64 *>(G.peer[i] + G.lay.off_recv_k) : nullptr;
        sp.packed[i] = i < G.n ? reinterpret_cast<u64 *>(G.peer[i] + G.lay.off_packed) : nullptr;
        sp.flags[i] = i < G.n ? reinterpret_cast<u32 *>(G.peer[i] + G.lay.off_flags) : nullptr;
        sp.cnt[i] = i < G.n ? reinterpret_cast<u32 *>(G.peer[i] + G.lay.off_recv_p) : nullptr;
    }
    sp.n = G.n;
    sp.rank = G.rank;
    sp.magic = (u32) (0x100000000ULL / (u64) G.n) + 1u;
    sp.sub_cap = sub_cap;
    u64 *cells4 = ex.arena->alloc_top<u64>(4);
    u32 *wait_status = reinterpret_cast<u32 *>(ex.arena->alloc_top<u64>(1));
    ex.fill_bytes(G.cells_local, 0, 32);
    ex.fill_bytes(wait_status, 0, 8);
    const size_t mark = ex.arena->mark();
    kc_sig_group_scan(ex, seq, n_bytes, k, pl, sp, region_cap, G.cells_local);
    const u32 sa = ++G.seq;
    kc_grp_signal(G, ex, sa);
    kc_grp_wait(G, ex, sa, wait_status);
    kc_sig_group_resolve<L>(ex, reinterpret_cast<const u64 *>(G.heap + G.lay.off_packed), k, complements, kc_sig_owned_buckets(pl.n_buckets, G.n, G.rank),
                            reinterpret_cast<const u32 *>(G.heap + G.lay.off_recv_p), nbr + 1, reinterpret_cast<const u64 *>(G.heap + G.lay.off_recv_k), G.n, region_cap,
                            G.all_flags(G.lay.off_flags), G.cells_local, n_bytes);
    ex.arena->release(mark);
    const u32 sb = ++G.seq;
    kc_grp_signal(G, ex, sb, nullptr, 0, 0, G.cells_local);
    kc_grp_wait(G, ex, sb, wait_status);
    kc_grp_sum_cells(G, ex, cells4, wait_status);
    return cells4;
}

// ---- exact path ----------------------------------------------------------------------------------------------------------------
// -> the complete first-occurrence bits in the rank's own heap (off_flags2); *kept, *n_occ = totals over all ranks.
template <int L>
const u32 *kc_grp_exact_flags(KcGroup &G, CudaExec &ex, const u8 *seq, u64 n_bytes, int k, bool complements, int min_freq, u64 *kept_out, u64 *n_occ_out) {
    typedef KsCfg<L> Cfg;
    u32 *flags_own = reinterpret_cast<u32 *>(G.heap + G.lay.off_flags);
    u32 *flags_all = reinterpret_cast<u32 *>(G.heap + G.lay.off_flags2);
    const size_t fwords = kc_runs_flag_words(n_bytes);
    ex.fill_bytes(flags_own, 0, fwords * 4);
    u32 *wait_status = reinterpret_cast<u32 *>(ex.arena->alloc_top<u64>(1));
    ex.fill_bytes(wait_status, 0, 8);
    auto check_wait = [&](u32 st) {
        if (st & 2u) {
            G.failed = true;
            KC_THROW(KC_ERR_INTERNAL, "a rank of the group did not arrive (wait timed out)");
        }
    };
    // slice of this rank
    const u32 tiles = (u32) kc_div_up(n_bytes, (u64) Cfg::EX_TILE);
    const u32 t0 = (u32) ((u64) tiles * G.rank / G.n), t1 = (u32) ((u64) tiles * (G.rank + 1) / G.n);
    KsShard sh;
    sh.pos_begin = (u64) t0 * Cfg::EX_TILE;
    sh.pos_end = std::min<u64>(n_bytes, (u64) t1 * Cfg::EX_TILE);
    const size_t th_need = ((size_t) (t1 - t0) + 1) * 256 * sizeof(u16);
    if (G.tile_hist_cap < th_need) {
        if (G.tile_hist) KC_CUDA(cudaFree(G.tile_hist));
        G.tile_hist = nullptr;
        G.tile_hist_cap = 0;
        KC_CUDA(cudaMalloc(&G.tile_hist, th_need));
        G.tile_hist_cap = th_need;
    }
    sh.tile_hist_keep = G.tile_hist;
    const u64 n_mine = kc_kmerset_hist_only<L>(ex, seq, n_bytes, k, complements, &sh);  // host_hist[256], synchronises
    // the 256 counts of every rank -> every rank
    KC_CUDA(cudaMemcpyAsync(G.cnt0, sh.host_hist, 1024, cudaMemcpyHostToDevice, ex.stream));
    const u32 sa = ++G.seq;
    kc_grp_signal(G, ex, sa, G.cnt0, 256);
    kc_grp_wait(G, ex, sa, wait_status);
    std::vector<u32> all_counts((size_t) G.n * 256);
    KC_CUDA(cudaMemcpyAsync(all_counts.data(), G.heap + G.lay.off_cnt, all_counts.size() * 4, cudaMemcpyDeviceToHost, ex.stream));
    check_wait(ex.read(wait_status));
    // layout of every owner's receive buffer: its digits ascending, inside a digit the ranks ascending
    u64 off[256], size[256], owned[KC_MAX_PEERS], cursor0[256];
    for (int r = 0; r < G.n; ++r) owned[r] = 0;
    for (int g = 0; g < 256; ++g) {
        const int o = g * G.n / 256;
        u64 sz = 0;
        for (int s = 0; s < G.n; ++s) sz += all_counts[(size_t) s * 256 + g];
        off[g] = owned[o];
        size[g] = sz;
        owned[o] += sz;
    }
    for (int r = 0; r < G.n; ++r)
        if (owned[r] > G.lay.recv_items) KC_THROW(KC_ERR_TOO_LARGE, "a rank's hash range exceeds the receive buffer of the group heap");
    KC_CUDA(cudaStreamSynchronize(ex.stream));  // staging table free
    G.tab_n_bytes = ~0ull;
    for (int g = 0; g < 256; ++g) {
        const int o = g * G.n / 256;
        u64 before = 0;
        for (int s = 0; s < G.rank; ++s) before += all_counts[(size_t) s * 256 + g];
        cursor0[g] = off[g] + before;
        G.h_dst[g] = G.peer[o] + G.lay.off_recv_k;
        G.h_dst[256 + g] = G.peer[o] + G.lay.off_recv_p;
    }
    KC_CUDA(cudaMemcpyAsync(G.dst_k, G.h_dst, 256 * sizeof(void *), cudaMemcpyHostToDevice, ex.stream));
    KC_CUDA(cudaMemcpyAsync(G.dst_p, G.h_dst + 256, 256 * sizeof(void *), cudaMemcpyHostToDevice, ex.stream));
    sh.cursor0 = cursor0;
    sh.dst_k = G.dst_k;
    sh.dst_p = G.dst_p;
    kc_kmerset_scatter_p2p<L>(ex, seq, n_bytes, k, complements, n_mine, &sh);  // synchronises
    const u32 sb = ++G.seq;
    kc_grp_signal(G, ex, sb);
    kc_grp_wait(G, ex, sb, wait_status);
    // exact levels + resolve over this rank's hash range
    u64 kept = 0;
    if (owned[G.rank]) {
        u64 my_off[256], my_size[256];
        u32 n_pre = 0;
        for (int g = 0; g < 256; ++g)
            if (g * G.n / 256 == G.rank) {
                my_off[n_pre] = off[g];
                my_size[n_pre] = size[g];
                ++n_pre;
            }
        KsShard rs;
        rs.keys = G.heap + G.lay.off_recv_k;
        rs.pos = reinterpret_cast<u32 *>(G.heap + G.lay.off_recv_p);
        rs.n_items = owned[G.rank];
        rs.n_pre = n_pre;
        rs.pre_off = my_off;
        rs.pre_size = my_size;
        kept = kc_kmerset_resolve<L>(ex, k, min_freq, flags_own, &rs);
    }
    const u64 hc[4] = {kept, 0, n_mine, 0};
    KC_CUDA(cudaMemcpyAsync(G.cells_local, hc, 32, cudaMemcpyHostToDevice, ex.stream));
    KC_CUDA(cudaStreamSynchronize(ex.stream));  // hc is a stack array
    const u32 sc = ++G.seq;
    kc_grp_signal(G, ex, sc, nullptr, 0, 0, G.cells_local);
    kc_grp_wait(G, ex, sc, wait_status);
    {
        CudaExec::Scope scope(ex, KP_MISC, fwords * 4 * (u64) (G.n + 1));
        kc_grp_or_flags_kernel<<<(unsigned) kc_div_up((u64) fwords, 256), 256, 0, ex.stream>>>(G.all_flags(G.lay.off_flags), flags_all, fwords);
        ++ex.launches;
        KC_CUDA(cudaGetLastError());
    }
    u64 *cells4 = ex.arena->alloc_top<u64>(4);
    kc_grp_sum_cells(G, ex, cells4, wait_status);
    u64 h4[4];
    ex.read_n(cells4, h4, 4);
    check_wait((u32) h4[3]);
    *kept_out = h4[0];
    *n_occ_out = h4[2];
    return flags_all;
}

#endif  // __CUDACC__
