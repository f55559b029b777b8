// Histogram-free k-mer set construction for the FLAGS-only regime (from-FASTA `compute` without -M): the same
// decode -> canonical k-mer -> MSD partition -> shared-memory hash resolve as kmerset.cuh (reference src/parser.h:22-141
// AddKMers / AddKMersWithFrequencies + khash), but planned from the input size alone so that NO counting pass and NO
// host synchronisation sits between the kernels.
//
// Why this is possible: FLAGS-only buckets by a bijective multiplicative hash of the k-mer word (kmer_scramble), so for
// any input made of mostly distinct k-mers the bucket sizes are Poisson-tight around M / ways.  Every bucket of every
// level therefore gets a FIXED slot of  mean + 8 sigma  items (the leaves: 1024, the capacity of the hash resolve) and
// a tile reserves its place inside a slot with one atomicAdd per digit.  What disappears against kmerset.cuh:
//   * kc_ks_hist0_kernel   — the sequence is decoded and the canonical k-mers are computed ONCE (they wait in shared
//                            memory while the tile's digit counts are scanned), not twice;
//   * kc_kv_hist_kernel    — no second read of the level-0 output (8L bytes per k-mer);
//   * two host read-backs (bucket lists / tile counts) and six scan / bookkeeping launches.
// Algorithmic HBM bytes per k-mer (L = 1): 1 + 12 (level 0) + 12 + 12 (level 1) + 12 (resolve) = 49 instead of 58.
//
// Flags are "clear the losers": level 0 writes the bit of every valid window (one coalesced word per strip), and every
// atomicMin that folds a duplicate in the leaf resolve clears exactly one bit — the larger of the two positions it compared.
// A genome has ~0 duplicates, so the resolve writes almost nothing.
//
// Multi-GPU (group.cuh): the same kernels with P2P = true.  Level 0 runs over the rank's slice of the input and stores every
// item straight into the (digit, sender) sub-slot of the digit's OWNER GPU through peer pointers (NVLink), and the valid-window
// words into every rank's flag array; the owner's level 1 reads the sub-slots of all senders as parents of one bucket, and
// the resolve clears losers in every rank's flags.
//
// Inputs that break the assumption (30x read sets: every k-mer ~30 times, so sigma grows by sqrt(30); low-complexity
// sequence) overflow a slot.  Overflow is detected on the device (items beyond the slot are dropped, a status word is
// set) and reported with the same read-back that returns the counts; the caller then discards the flags and runs the
// exact histogram-based construction of kmerset.cuh.  Results never depend on which of the two ran.
#pragma once
#include "kmerset.cuh"

#include "ksf_plan.h"  // KSF_LEAF_CAP, KsfTuning, KsfPlan, kc_ksf_plan

// Host-to-device copy of the sequence in flight on another stream, cut into chunks of whole level-0 tiles: event c is recorded
// once bytes [0, (c + 1) * chunk_bytes) have landed.  The level-0 scatter of the fixed-slot construction waits per chunk, so
// the first partition pass runs behind the copy front instead of after the whole copy (kc_compute with host buffers).
struct InputChunks {
    int n = 0;
    u64 chunk_bytes = 0;     // a multiple of every KsCfg<L>::EX_TILE
    cudaEvent_t *ev = nullptr;
    bool waited = false;     // every chunk has been waited for on the compute stream
    void wait_all(cudaStream_t st) {
        if (n && !waited) KC_CUDA(cudaStreamWaitEvent(st, ev[n - 1], 0));
        waited = true;
    }
};

// The first-occurrence bit arrays a loser is cleared in / the valid-window words are written to: this GPU's own array, or
// the arrays of every rank of the group (peer pointers).
struct KsfFlagPeers {
    u32 *f[KC_MAX_PEERS];
    int n;
};
inline KsfFlagPeers kc_ksf_own_flags(u32 *flags) {
    KsfFlagPeers fp;
    for (int i = 0; i < KC_MAX_PEERS; ++i) fp.f[i] = nullptr;
    fp.f[0] = flags;
    fp.n = 1;
    return fp;
}

#ifdef __CUDACC__

// MULTI = false is the single-GPU instance: one RED on the GPU's own array, nothing else in the instruction stream (the loop over
// the ranks cost the leaf resolve 9 % on one GPU although it almost never runs).
template <bool MULTI, class Pos> KC_D void kc_flag_clear_all(const KsfFlagPeers &fp, Pos pos) {  // Pos: u32, or u64 past 2^32 bytes
    const u32 m = ~(1u << (pos & 31));
    if (MULTI) {
        for (int r = 0; r < fp.n; ++r) atomicAnd(&fp.f[r][pos >> 5], m);
    } else {
        atomicAnd(&fp.f[0][pos >> 5], m);
    }
}

// status[0] = 1: some slot overflowed (the flags are incomplete and must be discarded)
// ---- level 0: sequence -> fixed-slot buckets, one compute pass ----------------------------------------------------------
// P2P = false: bucket i is the slot keys[i * cap0 ..), the valid-window word goes to vf.f[0] (only words with a window: the
//              array arrives zeroed).
// P2P = true : bucket i is the sub-slot dst_k[i] / dst_p[i] (cap0 items, somewhere in the heap of the digit's owner), the
//              valid-window word of EVERY strip goes to all vf.n arrays (they do not arrive zeroed).
template <int L, bool P2P>
__global__ void __launch_bounds__(KsCfg<L>::EX_THREADS) kc_ksf_scatter0_kernel(const u8 *__restrict__ seq, u64 n_bytes, int k, int complements,
                                                                                int shift, int bits, u32 *bucket_cnt, u32 cap0,
                                                                                KWord<L> *__restrict__ keys, u32 *__restrict__ pos, u32 *status, u32 tile0,
                                                                                KsfFlagPeers vf, u32 n_flag_words,
                                                                                KWord<L> *const *__restrict__ dst_k = nullptr,
                                                                                u32 *const *__restrict__ dst_p = nullptr) {
    constexpr int T = KsCfg<L>::EX_THREADS;
    constexpr int LOG_T = T == 256 ? 8 : (T == 128 ? 7 : 6);
    constexpr int R = 256 / T;
    constexpr int TILE = KsCfg<L>::EX_TILE;
    extern __shared__ __align__(16) unsigned char kc_smem_raw[];
    KWord<L> *stash = reinterpret_cast<KWord<L> *>(kc_smem_raw);  // slot j * T + t = window j of thread t (conflict-free)
    u16 *rk = reinterpret_cast<u16 *>(stash + TILE);               // rank of the slot's k-mer inside its digit, 0xFFFF = no k-mer
    u16 *perm = rk + TILE;                                         // digit-ordered position -> slot
    __shared__ u64 pk[KC_EX_HALO + T];
    __shared__ u32 vm[KC_EX_HALO + T];
    __shared__ u32 cnt[256];
    __shared__ u32 loff[256];
    __shared__ u64 dbase[256];  // slot index of the digit's first item of this tile, minus its staged position: at = dbase + q
                                // (P2P: the address of the key with staged position 0, pbase the same for the positions)
    __shared__ u64 pbase[P2P ? 256 : 1];
    __shared__ u32 qlim[256];   // staged positions below this still fit into the digit's slot
    __shared__ u32 sw[T / 32];
    const i64 block_pos0 = (i64) (tile0 + blockIdx.x) * TILE;
    kc_tile_load<T>(seq, n_bytes, block_pos0, pk, vm);
    for (int i = threadIdx.x; i < 256; i += T) cnt[i] = 0;
#pragma unroll
    for (int j = 0; j < KC_EX_STRIP; ++j) rk[j * T + threadIdx.x] = 0xFFFFu;
    __syncthreads();
    const int widx = KC_EX_HALO + threadIdx.x;
    const u32 em = kc_strip_emit_mask(vm, widx, k);
    {   // clear-the-losers flags: every window starts as "first occurrence" (bit p & 31 of word p >> 5 = window END p)
        const u64 w = (u64) (block_pos0 >> 5) + threadIdx.x;
        if (P2P) {
            if (w < n_flag_words)
                for (int r = 0; r < vf.n; ++r) vf.f[r][w] = __brev(em);
        } else if (em && w < n_flag_words) {
            vf.f[0][w] = __brev(em);
        }
    }
    kc_strip_windows<L>(pk, widx, em, k, complements, [&](int j, const KWord<L> &c0) {
        const KWord<L> c = kmer_scramble(c0);
        const u32 slot = (u32) j * T + threadIdx.x;
        stash[slot] = c;
        rk[slot] = (u16) atomicAdd(&cnt[c.digit_top(shift, bits)], 1u);
    });
    __syncthreads();
    u32 total;
    {
        u32 v[R], c = 0;
#pragma unroll
        for (int r = 0; r < R; ++r) {
            v[r] = cnt[threadIdx.x * R + r];
            c += v[r];
        }
        u32 p = kc_block_exclusive_scan<T>(c, &total, sw);
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int i = threadIdx.x * R + r;
            loff[i] = p;
            u32 gb = 0;
            if (v[r]) gb = atomicAdd(&bucket_cnt[i], v[r]);  // reserve the tile's place inside the slot of bucket i
            const u32 room = gb < cap0 ? cap0 - gb : 0u;
            if (P2P) {
                const i64 d = (i64) gb - (i64) p;
                dbase[i] = (u64) (reinterpret_cast<i64>(dst_k[i]) + d * (i64) sizeof(KWord<L>));
                pbase[i] = (u64) (reinterpret_cast<i64>(dst_p[i]) + d * 4);
            } else {
                dbase[i] = (u64) i * cap0 + gb - p;
            }
            qlim[i] = p + (v[r] < room ? v[r] : room);
            p += v[r];
        }
    }
    __syncthreads();
    if (total == 0) return;
    // perm[] shares the dynamic array with rk[] / stash[], so the compiler must keep every store behind the loads of the same
    // iteration and in front of the next one's (ncu r01h: 16 % of the kernel's samples on this one line).  Batches of 8 slots:
    // all ranks, all top limbs, all offsets, then the stores — the shared-memory round trips overlap.
#pragma unroll
    for (int j0 = 0; j0 < KC_EX_STRIP; j0 += 8) {
        u32 r[8], o[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) r[u] = rk[(u32) (j0 + u) * T + threadIdx.x];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            KWord<L> t = KWord<L>::zero();
            t.w[L - 1] = stash[(u32) (j0 + u) * T + threadIdx.x].w[L - 1];  // the digit lives in the top limb
            o[u] = t.digit_top(shift, bits);
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) o[u] = loff[o[u]];
#pragma unroll
        for (int u = 0; u < 8; ++u)
            if (r[u] != 0xFFFFu) perm[o[u] + r[u]] = (u16) ((u32) (j0 + u) * T + threadIdx.x);
    }
    __syncthreads();
    bool over = false;
    if constexpr (P2P) {
        // Most of these stores cross NVLink, where a partially written 128-byte line travels as several small packets.  A warp
        // therefore takes whole digit runs and lines its lanes up with the DESTINATION: lane l writes the items whose index in the
        // owner's sub-slot is l mod 32, so that every warp-wide store covers one aligned 256-byte block of keys (128 bytes of
        // positions) and only the two ends of a run are partial lines.
        const u32 lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        const u32 n_dig = 1u << bits;
        for (u32 dg = warp; dg < n_dig; dg += T / 32) {
            const u32 q0 = loff[dg], n_all = cnt[dg], n_ok = qlim[dg] - q0;
            if (n_ok < n_all) over = true;
            if (n_ok == 0) continue;
            KWord<L> *kd = reinterpret_cast<KWord<L> *>(dbase[dg]);
            u32 *pd = reinterpret_cast<u32 *>(pbase[dg]);
            const u32 mis = (u32) ((dbase[dg] / sizeof(KWord<L>) + q0) & 31u);
            for (i64 i = (i64) lane - (i64) mis; i < (i64) n_ok; i += 32) {
                if (i < 0) continue;
                const u32 q = q0 + (u32) i;
                const u32 slot = perm[q];
                kd[q] = stash[slot];
                pd[q] = (u32) block_pos0 + (slot & (T - 1)) * KC_EX_STRIP + (slot >> LOG_T);
            }
        }
    } else {
#pragma unroll 4
        for (u32 q = threadIdx.x; q < total; q += T) {
            const u32 slot = perm[q];
            const KWord<L> v = stash[slot];
            const u32 dg = v.digit_top(shift, bits);
            if (q < qlim[dg]) {
                const u64 at = dbase[dg] + q;
                keys[at] = v;
                pos[at] = (u32) block_pos0 + (slot & (T - 1)) * KC_EX_STRIP + (slot >> LOG_T);
            } else {
                over = true;
            }
        }
    }
    if (over) status[0] = 1;
}

// Between two levels: clamp the fill counts of the nP parent slots, count their tiles (tile_count[nP] = 0 for the scan
// that follows) and, after level 0, add up M.
__global__ void __launch_bounds__(256) kc_ksf_prep_kernel(const u32 *cnt, u32 nP, u32 capP, u32 tile, u32 *size_out, u32 *tile_count, u32 *status,
                                                          kc_ull *m_cell) {
    const u32 p = blockIdx.x * 256 + threadIdx.x;
    if (p > nP) return;
    if (p == nP) {
        tile_count[p] = 0;
        return;
    }
    u32 c = cnt[p];
    if (m_cell && c) atomicAdd(m_cell, (kc_ull) (c < capP ? c : capP));
    if (c > capP) {
        status[0] = 1;
        c = capP;
    }
    size_out[p] = c;
    tile_count[p] = (c + tile - 1) / tile;
}

// ---- leaf resolve: exact dedup of one fixed slot through shared-memory tables, two barriers per bucket ------------------------
// Persistent CTAs walk the leaf slots with stride gridDim.x.  The slot of bucket n + 1 streams into the second staging
// buffer with cp.async while bucket n is resolved, so no thread ever waits on HBM between the barriers.
//   A  every item writes its index into T1[h1(key)] with a plain store (some writer wins);
//   -- barrier --
//   B  the winner of a slot represents its key.  An item that finds an EQUAL key there is a duplicate: it folds its
//      position into the winner's with atomicMin (and bumps the occurrence count for -z).  An item that finds a
//      DIFFERENT key (~16 % at load 0.37) inserts itself into T2 with atomicCAS + linear probing, folding into an
//      equal key if it meets one.  All copies of a key take the same route, so they always meet;
//   -- barrier --
//   C  every representative with >= min_count occurrences sets the bit of its smallest position.
// Against kc_ks_resolve_hash_kernel (up to six write-then-verify rounds, each ending in a barrier + vote): 2 barriers
// instead of ~5 per bucket, no register staging (64 -> 40 registers), twice the resident CTAs.
KC_D void kc_cp_async16(void *smem_dst, const void *gmem_src) {
    const u32 d = (u32) __cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(gmem_src) : "memory");
}
KC_D void kc_cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }

// ---- 1-D bulk copies (TMA) completing on an mbarrier: one elected thread arms the barrier with the byte count and issues the
// copy; the copy engine streams the bytes into shared memory without any thread issuing per-chunk loads, and every thread that
// needs the data waits on the barrier's phase.  Addresses and sizes are multiples of 16 bytes (slots are 128-byte aligned,
// ksf_plan.h).  SASS: UBLKCP (the copy) and SYNCS (mbarrier arrive / try_wait).
KC_D u32 kc_smem_u32(const void *p) { return (u32) __cvta_generic_to_shared(p); }
KC_D void kc_mbar_init(u64 *bar, u32 count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(kc_smem_u32(bar)), "r"(count) : "memory");
}
KC_D void kc_mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory"); }
KC_D void kc_mbar_expect_tx(u64 *bar, u32 bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(kc_smem_u32(bar)), "r"(bytes) : "memory");
}
KC_D void kc_bulk_g2s(void *smem_dst, const void *gmem_src, u32 bytes, u64 *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(kc_smem_u32(smem_dst)), "l"(gmem_src),
                 "r"(bytes), "r"(kc_smem_u32(bar))
                 : "memory");
}
KC_D void kc_mbar_wait(u64 *bar, u32 parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred P1;\n\t"
        "KC_WAIT:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1, 0x989680;\n\t"
        "@P1 bra KC_DONE;\n\t"
        "bra KC_WAIT;\n\t"
        "KC_DONE:\n\t"
        "}" ::"r"(kc_smem_u32(bar)),
        "r"(parity)
        : "memory");
}
KC_D void kc_cp_async_wait_all() { asm volatile("cp.async.wait_group 0;\n" ::: "memory"); }


// The flags arrive with the bit of every valid window set (written by level 0); every atomicMin that folds a duplicate knocks
// out exactly one position — the larger of the two it compared — so only the DUPLICATES cost a scattered RED and the kept
// bits are never touched.  This kernel serves -z Z > 1 (COUNTED); -z 1 takes kc_ksf_resolve2_kernel.
template <int L, bool COUNTED, bool MULTI>
__global__ void __launch_bounds__(256) kc_ksf_resolve_kernel(const KWord<L> *__restrict__ keys, const u32 *__restrict__ pos, const u32 *__restrict__ cnt,
                                                             u32 n_leaf, KsfFlagPeers fl, u32 min_count, kc_ull *n_unique, u32 *status) {
    constexpr u32 CAP = KSF_LEAF_CAP;
    constexpr u32 T1N = 2 * CAP, T2N = CAP;
    constexpr int KPC = 16 / (int) sizeof(KWord<L>) > 0 ? 16 / (int) sizeof(KWord<L>) : 1;  // keys per 16-byte chunk (L = 1: 2)
    constexpr int CPK = (int) sizeof(KWord<L>) / 16 > 0 ? (int) sizeof(KWord<L>) / 16 : 1;  // 16-byte chunks per key (L = 4: 2)
    extern __shared__ __align__(16) unsigned char kc_smem_raw[];
    KWord<L> *sk0 = reinterpret_cast<KWord<L> *>(kc_smem_raw);
    u32 *sp0 = reinterpret_cast<u32 *>(sk0 + 2 * CAP);
    u32 *T1 = sp0 + 2 * CAP;
    u32 *T2 = T1 + T1N;
    u32 *occ = T2 + T2N;  // COUNTED only
    const u32 stride = gridDim.x;
    u32 c = blockIdx.x;
    if (c >= n_leaf) return;
    auto fetch = [&](u32 bucket, u32 size, int buf) {
        const char *gk = reinterpret_cast<const char *>(keys + (u64) bucket * CAP);
        const char *gp = reinterpret_cast<const char *>(pos + (u64) bucket * CAP);
        char *dk = reinterpret_cast<char *>(sk0 + (u32) buf * CAP);
        char *dp = reinterpret_cast<char *>(sp0 + (u32) buf * CAP);
        // a thread copies whole units (L = 1: a pair of keys, otherwise one key), so the keys it hashes in phase A are
        // the ones it fetched itself
        const u32 n_units = (size + KPC - 1) / KPC, pchunks = (size * 4 + 15) / 16;
        for (u32 u = threadIdx.x; u < n_units; u += 256) {
#pragma unroll
            for (int cc = 0; cc < CPK; ++cc) kc_cp_async16(dk + 16 * (u * CPK + cc), gk + 16 * (u * CPK + cc));
        }
        for (u32 q = threadIdx.x; q < pchunks; q += 256) kc_cp_async16(dp + 16 * q, gp + 16 * q);
        kc_cp_async_commit();
    };
    u32 size = cnt[c];
    if (size > CAP) {
        size = CAP;
        if (threadIdx.x == 0) status[0] = 1;
    }
    fetch(c, size, 0);
    int buf = 0;
    u32 kept = 0;
    while (true) {
        const u32 cn = c + stride;
        u32 size_n = 0;
        if (cn < n_leaf) {
            size_n = cnt[cn];
            if (size_n > CAP) {
                size_n = CAP;
                if (threadIdx.x == 0) status[0] = 1;
            }
        }
        KWord<L> *sk = sk0 + (u32) buf * CAP;
        u32 *sp = sp0 + (u32) buf * CAP;
        kc_cp_async_wait_all();  // the thread's own chunks of bucket c have landed
        // A: own items = the keys of the chunks this thread copied itself (visible without a barrier)
        const u32 n_chunk_items = (size + KPC - 1) / KPC;  // L = 1: pairs of keys; L >= 2: single keys
        {
            const uint4 e = make_uint4(KC_NONE, KC_NONE, KC_NONE, KC_NONE);
            reinterpret_cast<uint4 *>(T2)[threadIdx.x] = e;  // T2N = 1024 slots = 256 x 16 bytes
        }
        for (u32 q = threadIdx.x; q < n_chunk_items; q += 256) {
#pragma unroll
            for (int e = 0; e < KPC; ++e) {
                const u32 i = q * KPC + e;
                if (i < size) {
                    u64 h = 0;
#pragma unroll
                    for (int w = 0; w < L; ++w) h = (h ^ sk[i].w[w]) * 0xD6E8FEB86659FD93ULL;
                    T1[h >> 53] = i;
                    if (COUNTED) occ[i] = 1;
                }
            }
        }
        __syncthreads();
        if (cn < n_leaf) fetch(cn, size_n, buf ^ 1);  // every thread is past phase C of the bucket that used that buffer
        // B
        u32 rep = 0;  // bit (2 m + e): item e of the thread's m-th chunk represents its key
        {
            u32 m = 0;
            for (u32 q = threadIdx.x; q < n_chunk_items; q += 256, ++m) {
#pragma unroll
                for (int e = 0; e < KPC; ++e) {
                    const u32 i = q * KPC + e;
                    if (i >= size) continue;
                    const KWord<L> key = sk[i];
                    u64 h = 0;
#pragma unroll
                    for (int w = 0; w < L; ++w) h = (h ^ key.w[w]) * 0xD6E8FEB86659FD93ULL;
                    const u32 o = T1[h >> 53];
                    if (o == i) {
                        rep |= 1u << (m * KPC + e);
                    } else if (sk[o] == key) {
                        const u32 mine = sp[i];
                        const u32 was = atomicMin(&sp[o], mine);
                        kc_flag_clear_all<MULTI>(fl, was > mine ? was : mine);
                        if (COUNTED) atomicAdd(&occ[o], 1u);
                    } else {
                        u32 s = (u32) (h >> 43) & (T2N - 1);
                        while (true) {
                            const u32 old = atomicCAS(&T2[s], KC_NONE, i);
                            if (old == KC_NONE) {
                                rep |= 1u << (m * KPC + e);
                                break;
                            }
                            if (sk[old] == key) {
                                const u32 mine = sp[i];
                                const u32 was = atomicMin(&sp[old], mine);
                                kc_flag_clear_all<MULTI>(fl, was > mine ? was : mine);
                                if (COUNTED) atomicAdd(&occ[old], 1u);
                                break;
                            }
                            s = (s + 1) & (T2N - 1);
                        }
                    }
                }
            }
        }
        __syncthreads();
        // C
        {
            u32 m = 0;
            for (u32 q = threadIdx.x; q < n_chunk_items; q += 256, ++m) {
#pragma unroll
                for (int e = 0; e < KPC; ++e) {
                    const u32 i = q * KPC + e;
                    if (!((rep >> (m * KPC + e)) & 1u)) continue;
                    if (!COUNTED || occ[i] >= min_count) {
                        ++kept;
                    } else {
                        kc_flag_clear_all<MULTI>(fl, sp[i]);  // too few occurrences: the surviving (smallest) position goes as well
                    }
                }
            }
        }
        if (cn >= n_leaf) break;
        c = cn;
        size = size_n;
        buf ^= 1;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) kept += __shfl_down_sync(0xFFFFFFFFu, kept, o);
    if ((threadIdx.x & 31) == 0 && kept) atomicAdd(n_unique, (kc_ull) kept);
}

// ---- one-barrier leaf resolve with the thread's items staged in registers ------------------------------------------------------
// The stage sweep of the round-1 leaf resolve (profiles/r01h_variant_sweep2.json) showed its time going with 1 / (CTAs per SM):
// 0.235 ms at 5 CTAs (2 stages), 0.270 at 4 (3 stages), 0.324 at 3 (4 stages) — the kernel is bound by the latency of one
// leaf's dependent chain (LDS key -> hash -> STS/LDS table -> compare, item after item), not by DRAM.  Here a thread loads
// ALL its keys first, hashes them together, then issues the table accesses together, so the chain is paid once per phase
// instead of once per item; key and hash stay in registers between the phases.  THREADS = 512 halves the items per thread.
// The leaf arrives by two bulk copies (keys, positions) that one thread issues and that complete on an mbarrier; the items are
// then dealt out to the threads round-robin (any thread may read any item once the barrier's phase has flipped).
template <int L, int THREADS, bool MULTI>
__global__ void __launch_bounds__(THREADS) kc_ksf_resolve2_kernel(const KWord<L> *__restrict__ keys, const u32 *__restrict__ pos, const u32 *__restrict__ cnt,
                                                                  u32 n_leaf, KsfFlagPeers fl, kc_ull *n_unique, u32 *status) {
    constexpr u32 CAP = KSF_LEAF_CAP;
    constexpr u32 T1N = 2 * CAP, T2N = CAP;
    constexpr int NI = (int) CAP / THREADS;  // items per thread
    static_assert(NI >= 1 && NI * THREADS == (int) CAP, "CAP must be a whole number of items per thread");
    extern __shared__ __align__(16) unsigned char kc_smem_raw[];
    KWord<L> *sk0 = reinterpret_cast<KWord<L> *>(kc_smem_raw);
    u32 *sp0 = reinterpret_cast<u32 *>(sk0 + 2 * CAP);
    u32 *T2a = sp0 + 2 * CAP;                                  // [2][T2N]
    u16 *T1a = reinterpret_cast<u16 *>(T2a + 2 * T2N);         // [2][T1N]
    __shared__ __align__(8) u64 full[2];  // "leaf in staging buffer b has landed"
    const u64 stride = gridDim.x;
    u64 c = blockIdx.x;
    if (c >= n_leaf) return;
    if (threadIdx.x == 0) {
        kc_mbar_init(&full[0], 1);
        kc_mbar_init(&full[1], 1);
        kc_mbar_fence_init();
    }
    __syncthreads();
    u32 full_phase = 0;  // bit b: parity to wait for on full[b]
    auto leaf_size = [&](u64 leaf) -> u32 {
        if (leaf >= n_leaf) return 0u;
        u32 sz = cnt[leaf];
        if (sz > CAP) {
            sz = CAP;
            if (threadIdx.x == 0) status[0] = 1;
        }
        return sz;
    };
    auto fetch = [&](u64 bucket, u32 size, int buf) {
        if (bucket < n_leaf && threadIdx.x == 0) {
            const u32 kb = (size * (u32) sizeof(KWord<L>) + 15u) & ~15u, pb = (size * 4u + 15u) & ~15u;
            kc_mbar_expect_tx(&full[buf], kb + pb);
            if (kb) kc_bulk_g2s(sk0 + (u32) buf * CAP, keys + bucket * CAP, kb, &full[buf]);
            if (pb) kc_bulk_g2s(sp0 + (u32) buf * CAP, pos + bucket * CAP, pb, &full[buf]);
        }
    };
    u32 size = leaf_size(c);
    u32 size_n = leaf_size(c + stride);
    fetch(c, size, 0);
    int buf = 0;
    u32 kept = 0;
    while (true) {
        const u64 cn = c + stride;
        KWord<L> *sk = sk0 + (u32) buf * CAP;
        u32 *sp = sp0 + (u32) buf * CAP;
        u32 *T2 = T2a + (u32) buf * T2N;
        u16 *T1 = T1a + (u32) buf * T1N;
        kc_mbar_wait(&full[buf], (full_phase >> buf) & 1u);  // leaf c has landed (all of it, for every thread)
        full_phase ^= 1u << buf;
        if (threadIdx.x < 256) reinterpret_cast<uint4 *>(T2)[threadIdx.x] = make_uint4(KC_NONE, KC_NONE, KC_NONE, KC_NONE);  // T2N = 256 x 4 slots
        // A: all keys, then all hashes, then all table stores
        KWord<L> key[NI];
        u32 h1[NI], h2[NI];
#pragma unroll
        for (int m = 0; m < NI; ++m) {
            const u32 i = threadIdx.x + (u32) m * THREADS;
            if (i < size) key[m] = sk[i];
        }
#pragma unroll
        for (int m = 0; m < NI; ++m) {
            u64 h = 0;
#pragma unroll
            for (int w = 0; w < L; ++w) h = (h ^ key[m].w[w]) * 0xD6E8FEB86659FD93ULL;
            h1[m] = (u32) (h >> 53);
            h2[m] = (u32) (h >> 43) & (T2N - 1);
        }
#pragma unroll
        for (int m = 0; m < NI; ++m) {
            const u32 i = threadIdx.x + (u32) m * THREADS;
            if (i < size) T1[h1[m]] = (u16) i;
        }
        __syncthreads();
        fetch(cn, size_n, buf ^ 1);  // every thread is past phase B of the leaf that used that buffer
        // B: all table reads first; winners are done, the others compare against their slot's winner
        u32 o[NI];
#pragma unroll
        for (int m = 0; m < NI; ++m) {
            const u32 i = threadIdx.x + (u32) m * THREADS;
            o[m] = i < size ? (u32) T1[h1[m]] : i;
        }
#pragma unroll
        for (int m = 0; m < NI; ++m) {
            const u32 i = threadIdx.x + (u32) m * THREADS;
            if (i >= size) continue;
            if (o[m] == i) {
                ++kept;
            } else if (sk[o[m]] == key[m]) {
                const u32 mine = sp[i];
                const u32 was = atomicMin(&sp[o[m]], mine);
                kc_flag_clear_all<MULTI>(fl, was > mine ? was : mine);
            } else {
                u32 s = h2[m];
                while (true) {
                    const u32 old = atomicCAS(&T2[s], KC_NONE, i);
                    if (old == KC_NONE) {
                        ++kept;
                        break;
                    }
                    if (sk[old] == key[m]) {
                        const u32 mine = sp[i];
                        const u32 was = atomicMin(&sp[old], mine);
                        kc_flag_clear_all<MULTI>(fl, was > mine ? was : mine);
                        break;
                    }
                    s = (s + 1) & (T2N - 1);
                }
            }
        }
        if (cn >= n_leaf) break;
        c = cn;
        size = size_n;
        size_n = leaf_size(c + stride);
        buf ^= 1;
    }
#pragma unroll
    for (int o2 = 16; o2 > 0; o2 >>= 1) kept += __shfl_down_sync(0xFFFFFFFFu, kept, o2);
    if ((threadIdx.x & 31) == 0 && kept) atomicAdd(n_unique, (kc_ull) kept);
}

// ---- levels >= 1 with the next tile in flight ---------------------------------------------------------------------------------
// A scatter that issues a tile's loads and then waits for them (round 1, ncu: long scoreboard, 47 % of the HBM peak) is bound
// by that wait.  Here the tile after the current one streams into a shared-memory input buffer by two bulk copies (issued by
// one thread, completing on an mbarrier) while the current tile is ranked, staged and written out: a thread takes its items
// out of the input buffer into registers, and the barrier that ends the ranking phase frees the buffer for the next copy.
// Tiles are contiguous in their parent slot, slots are 128-byte aligned.
template <int L, int TILE, int MINB, int THREADS>
__global__ void __launch_bounds__(THREADS, MINB) kc_ksf_scatter_pf_kernel(const KWord<L> *__restrict__ ksrc, const u32 *__restrict__ psrc, KWord<L> *__restrict__ kdst,
                                                                u32 *__restrict__ pdst, const u32 *__restrict__ P_size, const u32 *__restrict__ tile_prefix,
                                                                u32 nP, u64 capP, u32 tiles_per_cta, int shift, int bits, u32 *C_cnt, u32 capC, u32 *status,
                                                                u32 pdiv = 1) {
    constexpr int ITEMS = TILE / THREADS;
    extern __shared__ __align__(16) unsigned char kc_smem_raw[];
    KWord<L> *in_k = reinterpret_cast<KWord<L> *>(kc_smem_raw);
    KWord<L> *stage_k = in_k + TILE;
    u32 *in_p = reinterpret_cast<u32 *>(stage_k + TILE);
    u32 *stage_p = in_p + TILE;
    u16 *rk = reinterpret_cast<u16 *>(stage_p + TILE);
    __shared__ u32 cnt[256];
    __shared__ u32 loff[256];
    __shared__ u64 dbase[256];  // slot index of the digit's first item of this tile, minus its staged position: at = dbase + q
    __shared__ u32 qlim[256];   // staged positions below this still fit into the child's slot
    __shared__ u32 sw[THREADS / 32];
    __shared__ __align__(8) u64 full;  // "the tile in the input buffer has landed"
    const u32 n_tiles = tile_prefix[nP];
    const u32 t0 = blockIdx.x * tiles_per_cta;
    const u32 t1 = min(n_tiles, t0 + tiles_per_cta);
    if (t0 >= t1) return;
    u32 b = kc_upper_bound_u32(tile_prefix, nP + 1, t0) - 1;
    if (threadIdx.x < 256) cnt[threadIdx.x] = 0;
    if (threadIdx.x == 0) {
        kc_mbar_init(&full, 1);
        kc_mbar_fence_init();
    }
    __syncthreads();
    u32 full_phase = 0;
    bool over = false;
    // tile t of the CTA -> (parent bucket, first item inside the source arrays, items)
    auto describe = [&](u32 t, u32 &bb, u64 &first, u32 &n_here) {
        while (t >= tile_prefix[bb + 1]) ++bb;
        const u32 start = (t - tile_prefix[bb]) * TILE;
        n_here = min((u32) TILE, P_size[bb] - start);
        first = (u64) bb * capP + start;
    };
    auto prefetch = [&](u64 first, u32 n_here) {  // tiles start on 128-byte boundaries of their slot
        if (threadIdx.x == 0) {
            const u32 kb = (n_here * (u32) sizeof(KWord<L>) + 15u) & ~15u, pb = (n_here * 4u + 15u) & ~15u;
            kc_mbar_expect_tx(&full, kb + pb);
            if (kb) kc_bulk_g2s(in_k, ksrc + first, kb, &full);
            if (pb) kc_bulk_g2s(in_p, psrc + first, pb, &full);
        }
    };
    u64 first;
    u32 n_here;
    describe(t0, b, first, n_here);
    prefetch(first, n_here);
    for (u32 t = t0; t < t1; ++t) {
        kc_mbar_wait(&full, full_phase);
        full_phase ^= 1u;
        __syncthreads();  // tile t is complete in the input buffer; the write-out of tile t - 1 has left the staging buffers
        KWord<L> item[ITEMS];
        u32 pay[ITEMS];
#pragma unroll
        for (int j = 0; j < ITEMS; ++j) {
            const u32 i = threadIdx.x + j * THREADS;
            if (i < n_here) {
                item[j] = in_k[i];
                pay[j] = in_p[i];
            }
        }
        // all atomics first, then the rank stores (a store behind every atomic would wait for its result before the next
        // atomic is issued: one shared-memory round trip per item instead of one per tile)
        {
            u32 rr[ITEMS];
#pragma unroll
            for (int j = 0; j < ITEMS; ++j) {
                const u32 i = threadIdx.x + j * THREADS;
                rr[j] = i < n_here ? atomicAdd(&cnt[item[j].digit_top(shift, bits)], 1u) : 0u;
            }
#pragma unroll
            for (int j = 0; j < ITEMS; ++j) {
                const u32 i = threadIdx.x + j * THREADS;
                if (i < n_here) rk[i] = (u16) rr[j];
            }
        }
        __syncthreads();  // counts complete, input buffer free
        u32 b_next = b, n_next = 0;
        u64 first_next = 0;
        if (t + 1 < t1) {
            describe(t + 1, b_next, first_next, n_next);
            prefetch(first_next, n_next);
        }
        const u32 c = threadIdx.x < 256 ? cnt[threadIdx.x] : 0u;
        u32 total;
        const u32 p = kc_block_exclusive_scan<THREADS>(c, &total, sw);
        if (threadIdx.x < 256) {
            loff[threadIdx.x] = p;
            u32 gb = 0;
            const u64 child = ((u64) (b / pdiv) << bits) + threadIdx.x;  // pdiv parents (one per sender) share a bucket's children
            if (c) gb = atomicAdd(&C_cnt[child], c);
            const u32 room = gb < capC ? capC - gb : 0u;
            dbase[threadIdx.x] = child * capC + gb - p;
            qlim[threadIdx.x] = p + (c < room ? c : room);
            cnt[threadIdx.x] = 0;
        }
        __syncthreads();
        {   // staged positions of all items first (rk[] shares the dynamic array with the staging buffers: no load may pass a store)
            u32 qq[ITEMS];
#pragma unroll
            for (int j = 0; j < ITEMS; ++j) {
                const u32 i = threadIdx.x + j * THREADS;
                qq[j] = i < n_here ? (u32) rk[i] : 0u;
            }
#pragma unroll
            for (int j = 0; j < ITEMS; ++j) qq[j] += loff[item[j].digit_top(shift, bits)];
#pragma unroll
            for (int j = 0; j < ITEMS; ++j) {
                const u32 i = threadIdx.x + j * THREADS;
                if (i < n_here) {
                    stage_k[qq[j]] = item[j];
                    stage_p[qq[j]] = pay[j];
                }
            }
        }
        __syncthreads();
#pragma unroll 4
        for (u32 q = threadIdx.x; q < n_here; q += THREADS) {
            const KWord<L> v = stage_k[q];
            const u32 dg = v.digit_top(shift, bits);
            if (q < qlim[dg]) {
                const u64 at = dbase[dg] + q;
                kdst[at] = v;
                pdst[at] = stage_p[q];
            } else {
                over = true;
            }
        }
        b = b_next;
        n_here = n_next;
    }
    if (over) status[0] = 1;
}

// ---- host side -----------------------------------------------------------------------------------------------------------------
template <int L> struct KsfKernels {  // the kernel instances this construction launches, their shared memory, the per-device opt-in
    typedef KsCfg<L> Cfg;
    static constexpr int TILE1 = Cfg::TILE;
    static constexpr int THREADS1 = 512;
    static int smem0() { return Cfg::EX_TILE * ((int) sizeof(KWord<L>) + 4); }
    static int smem1() { return TILE1 * (2 * ((int) sizeof(KWord<L>) + 4) + 2); }
    static int smem_r(bool counted) {
        return counted ? (int) KSF_LEAF_CAP * (16 * L + 24) : (int) KSF_LEAF_CAP * (2 * (8 * L + 4) + 16);
    }
    struct Dev {
        int n_sm = 0, occ_r[2] = {0, 0};
    };
    static const Dev &prepare() {
        static KcDevOnce once;
        static Dev dev[KC_MAX_DEVICES];
        const int d = once.run([&](int dv) {
            KC_CUDA(cudaFuncSetAttribute(kc_ksf_scatter0_kernel<L, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem0()));
            KC_CUDA(cudaFuncSetAttribute(kc_ksf_scatter0_kernel<L, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem0()));
            KC_CUDA(cudaFuncSetAttribute(kc_ksf_scatter_pf_kernel<L, TILE1, 2, THREADS1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem1()));
            KC_CUDA(cudaFuncSetAttribute(kc_ksf_resolve2_kernel<L, 256, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_r(false)));
            KC_CUDA(cudaFuncSetAttribute(kc_ksf_resolve2_kernel<L, 256, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_r(false)));
            KC_CUDA(cudaFuncSetAttribute(kc_ksf_resolve_kernel<L, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_r(true)));
            KC_CUDA(cudaFuncSetAttribute(kc_ksf_resolve_kernel<L, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_r(true)));
            dev[dv].n_sm = kc_sm_count(dv);
            KC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&dev[dv].occ_r[0], kc_ksf_resolve2_kernel<L, 256, false>, 256, smem_r(false)));
            KC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&dev[dv].occ_r[1], kc_ksf_resolve_kernel<L, true, false>, 256, smem_r(true)));
        });
        return dev[d];
    }
};

// One level >= 1: the nP parent slots (capP items each, fill counts cnt_par) -> children of capC items (counters cnt_next).
// pdiv > 1: pdiv consecutive parents are the per-sender sub-slots of ONE bucket and share its children (multi-GPU level 1).
template <int L>
void kc_ksf_level(CudaExec &ex, const KWord<L> *ksrc, const u32 *psrc, KWord<L> *kdst, u32 *pdst, const u32 *cnt_par, u32 nP, u64 capP, u32 *cnt_next,
                  u64 capC, int shift, int bits, u64 items_ub, u32 *status, kc_ull *m_cell, const KsfTuning &tune, u32 pdiv = 1) {
    typedef KsfKernels<L> KK;
    cudaStream_t st = ex.stream;
    const size_t mark = ex.arena->mark();
    u32 *P_size = ex.alloc<u32>(nP);
    u32 *tile_prefix = ex.alloc<u32>((u64) nP + 1);
    kc_ksf_prep_kernel<<<(unsigned) kc_div_up((u64) nP + 1, 256), 256, 0, st>>>(cnt_par, nP, (u32) capP, (u32) KK::TILE1, P_size, tile_prefix, status, m_cell);
    ++ex.launches;
    ex.exclusive_scan_nosync(tile_prefix, tile_prefix, (u64) nP + 1);
    const u32 max_ctas = tune.max_ctas > 0 ? (u32) tune.max_ctas : 148 * 16;
    const u64 tiles_ub = items_ub / KK::TILE1 + nP + 1;
    const u32 tiles_per_cta = (u32) kc_div_up(tiles_ub, max_ctas);
    const u32 ctas = (u32) kc_div_up(tiles_ub, tiles_per_cta);
    {
        CudaExec::Scope sc(ex, KP_SORT_SCATTER, 2 * items_ub * (sizeof(KWord<L>) + 4));
        kc_ksf_scatter_pf_kernel<L, KK::TILE1, 2, KK::THREADS1><<<ctas, KK::THREADS1, KK::smem1(), st>>>(ksrc, psrc, kdst, pdst, P_size, tile_prefix, nP, capP,
                                                                                                      tiles_per_cta, shift, bits, cnt_next, (u32) capC, status,
                                                                                                      pdiv);
        ++ex.launches;
        KC_CUDA(cudaGetLastError());
    }
    ex.arena->release(mark);  // stream order keeps P_size / tile_prefix alive until the scatter has run
}

// Leaf slots (KSF_LEAF_CAP items each) -> losers cleared in fl, *n_unique += kept k-mers.
template <int L>
void kc_ksf_resolve(CudaExec &ex, const KWord<L> *keys, const u32 *pos, const u32 *cnt, u64 n_leaf, const KsfFlagPeers &fl, int min_freq, kc_ull *n_unique,
                    u32 *status, u64 items_ub) {
    typedef KsfKernels<L> KK;
    if (n_leaf >= 0xFFFFFFFFULL) KC_THROW(KC_ERR_TOO_LARGE, "too many leaf buckets");
    const typename KK::Dev &dv = KK::prepare();
    const bool counted = min_freq > 1;
    const u32 fit = (u32) (dv.n_sm * (dv.occ_r[counted] > 0 ? dv.occ_r[counted] : 1));
    const u32 grid = (u32) n_leaf < fit ? (u32) n_leaf : fit;
    CudaExec::Scope sc(ex, KP_KS_RESOLVE, items_ub * (sizeof(KWord<L>) + 4));
    const bool multi = fl.n > 1;
    if (counted && multi) kc_ksf_resolve_kernel<L, true, true><<<grid, 256, KK::smem_r(true), ex.stream>>>(keys, pos, cnt, (u32) n_leaf, fl, (u32) min_freq, n_unique, status);
    else if (counted) kc_ksf_resolve_kernel<L, true, false><<<grid, 256, KK::smem_r(true), ex.stream>>>(keys, pos, cnt, (u32) n_leaf, fl, (u32) min_freq, n_unique, status);
    else if (multi) kc_ksf_resolve2_kernel<L, 256, true><<<grid, 256, KK::smem_r(false), ex.stream>>>(keys, pos, cnt, (u32) n_leaf, fl, n_unique, status);
    else kc_ksf_resolve2_kernel<L, 256, false><<<grid, 256, KK::smem_r(false), ex.stream>>>(keys, pos, cnt, (u32) n_leaf, fl, n_unique, status);
    ++ex.launches;
    KC_CUDA(cudaGetLastError());
}

// Launches the whole construction on ex.stream and returns without synchronising.
//   cells[0] += distinct k-mers with >= min_freq occurrences, cells[2] = M (k-mer windows), low word of cells[3] = overflow status;
//   flags: zeroed bit array over the n_bytes positions (see kc_kmerset_build).
// Returns false (nothing launched) when the plan does not apply; the caller then uses kc_kmerset_build.
template <int L>
bool kc_kmerset_build_fast(CudaExec &ex, const u8 *seq, u64 n_bytes, int k, bool complements, int min_freq, u32 *flags, u64 *cells,
                           const KsfTuning &tune, KsfPlan *plan_out = nullptr, InputChunks *chunks = nullptr) {
    typedef KsCfg<L> Cfg;
    typedef KsfKernels<L> KK;
    const KsfPlan pl = kc_ksf_plan(n_bytes, tune);
    if (plan_out) *plan_out = pl;
    if (!pl.ok) return false;
    KK::prepare();
    cudaStream_t st = ex.stream;
    const size_t base_mark = ex.arena->mark();
    const u64 item_bytes = sizeof(KWord<L>) + 4;
    KWord<L> *kb[2];
    u32 *pb[2];
    for (int i = 0; i < 2; ++i) {
        kb[i] = ex.alloc<KWord<L>>(pl.slots[i] ? pl.slots[i] : 1);
        pb[i] = ex.alloc<u32>(pl.slots[i] ? pl.slots[i] : 1);
    }
    u64 n_cnt = 0;
    for (int i = 0; i < pl.n_levels; ++i) n_cnt += 1ULL << pl.cum[i];
    u32 *cnt_all = ex.alloc<u32>(n_cnt);
    ex.fill_bytes(cnt_all, 0, n_cnt * 4);
    u32 *status = reinterpret_cast<u32 *>(cells + 3);
    kc_ull *m_cell = reinterpret_cast<kc_ull *>(cells + 2);
    const KsfFlagPeers fl = kc_ksf_own_flags(flags);

    // ---- level 0 ----
    u32 *cnt_cur = cnt_all;
    {
        const u32 blocks = (u32) kc_div_up(n_bytes, (u64) Cfg::EX_TILE);
        // one launch, or one launch per chunk of an input that is still being copied in (each waits for its own chunk only)
        const int n_parts = chunks && chunks->n > 1 && !chunks->waited ? chunks->n : 1;
        if (chunks && n_parts == 1) chunks->wait_all(st);
        for (int c = 0; c < n_parts; ++c) {
            u32 t0 = 0, t1 = blocks;
            if (n_parts > 1) {
                KC_CUDA(cudaStreamWaitEvent(st, chunks->ev[c], 0));
                t0 = (u32) std::min<u64>(blocks, (u64) c * (chunks->chunk_bytes / Cfg::EX_TILE));
                t1 = c == n_parts - 1 ? blocks : (u32) std::min<u64>(blocks, (u64) (c + 1) * (chunks->chunk_bytes / Cfg::EX_TILE));
            }
            if (t1 <= t0) continue;
            const u64 part_bytes = std::min<u64>(n_bytes, (u64) t1 * Cfg::EX_TILE) - (u64) t0 * Cfg::EX_TILE;
            CudaExec::Scope sc(ex, KP_KS_SCATTER0, part_bytes + part_bytes * item_bytes);
            kc_ksf_scatter0_kernel<L, false><<<t1 - t0, Cfg::EX_THREADS, KK::smem0(), st>>>(seq, n_bytes, k, complements ? 1 : 0, 64 * L - pl.cum[0], pl.bits[0],
                                                                                         cnt_cur, (u32) pl.cap[0], kb[0], pb[0], status, t0, fl,
                                                                                         (u32) (kc_div_up(n_bytes, (u64) 32) + 1));  // = kc_runs_flag_words(n_bytes)
            ++ex.launches;
            KC_CUDA(cudaGetLastError());
        }
        if (chunks) chunks->waited = true;
    }
    // ---- levels >= 1 ----
    for (int lv = 1; lv < pl.n_levels; ++lv) {
        const u32 nP = (u32) (1ULL << pl.cum[lv - 1]);
        u32 *cnt_next = cnt_cur + nP;
        kc_ksf_level<L>(ex, kb[(lv - 1) & 1], pb[(lv - 1) & 1], kb[lv & 1], pb[lv & 1], cnt_cur, nP, pl.cap[lv - 1], cnt_next, pl.cap[lv], 64 * L - pl.cum[lv],
                        pl.bits[lv], n_bytes, status, lv == 1 ? m_cell : nullptr, tune);
        cnt_cur = cnt_next;
    }
    // ---- leaves -> hash resolve ----
    const int last = pl.n_levels - 1;
    if (pl.n_levels == 1) {  // M has not been added up by a prep kernel
        const u32 *cc = cnt_cur;
        ex.for_each(pl.n_leaf, [=] __device__(u64 i) {
            const u32 c = cc[i] < KSF_LEAF_CAP ? cc[i] : KSF_LEAF_CAP;
            if (c) atomicAdd(m_cell, (kc_ull) c);
        });
    }
    kc_ksf_resolve<L>(ex, kb[last & 1], pb[last & 1], cnt_cur, pl.n_leaf, fl, min_freq, reinterpret_cast<kc_ull *>(cells), status, n_bytes);
    ex.arena->release(base_mark);
    return true;
}

// Level 0 of rank `rank` over its tile slice: items into the owners' sub-slots (dst tables), valid-window words into every
// rank's flags, fill counts into cnt0[n_digits] (this rank's own counters, zeroed here).
template <int L>
void kc_ksf_group_scatter0(CudaExec &ex, const u8 *seq, u64 n_bytes, int k, bool complements, const KsfGroupPlan &g, int rank, u32 *cnt0, u32 *status,
                           KWord<L> *const *dst_k, u32 *const *dst_p, const KsfFlagPeers &all_flags) {
    typedef KsCfg<L> Cfg;
    typedef KsfKernels<L> KK;
    KK::prepare();
    ex.fill_bytes(cnt0, 0, (size_t) g.n_digits * 4);
    const u32 t0 = g.tile_begin(rank), t1 = g.tile_begin(rank + 1);
    if (t1 <= t0) return;
    const u64 part_bytes = std::min<u64>(n_bytes, (u64) t1 * Cfg::EX_TILE) - (u64) t0 * Cfg::EX_TILE;
    CudaExec::Scope sc(ex, KP_KS_SCATTER0, part_bytes + part_bytes * (sizeof(KWord<L>) + 4));
    kc_ksf_scatter0_kernel<L, true><<<t1 - t0, Cfg::EX_THREADS, KK::smem0(), ex.stream>>>(seq, n_bytes, k, complements ? 1 : 0, 64 * L - g.pl.cum[0], g.pl.bits[0], cnt0,
                                                                                       (u32) g.cap_sub, nullptr, nullptr, status, t0, all_flags,
                                                                                       (u32) kc_div_up(n_bytes, (u64) 32), dst_k, dst_p);
    ++ex.launches;
    KC_CUDA(cudaGetLastError());
}

// Owner side: the sub-slots of this rank's digits (recv_k / recv_p: [digit - dig_begin][sender] x cap_sub items, fill counts
// sub_cnt in the same order, already clamped to cap_sub) -> levels 1.. -> leaf resolve, losers cleared in every rank's flags.
// cells: {kept (+=), -, M of this rank's digits (+=), status (low word)}.
template <int L>
void kc_ksf_group_resolve(CudaExec &ex, int min_freq, const KsfGroupPlan &g, int rank, const KWord<L> *recv_k, const u32 *recv_p, const u32 *sub_cnt,
                          const KsfFlagPeers &all_flags, u64 *cells, const KsfTuning &tune) {
    const KsfPlan &pl = g.pl;
    const u32 dig_n = g.dig_begin(rank + 1) - g.dig_begin(rank);
    if (dig_n == 0) return;
    const size_t base_mark = ex.arena->mark();
    u32 *status = reinterpret_cast<u32 *>(cells + 3);
    kc_ull *m_cell = reinterpret_cast<kc_ull *>(cells + 2);
    u64 slots[2] = {1, 1}, n_cnt = 0;
    for (int lv = 1; lv < pl.n_levels; ++lv) {
        const u64 nb = (u64) dig_n << (pl.cum[lv] - pl.cum[0]);
        slots[lv & 1] = std::max<u64>(slots[lv & 1], nb * pl.cap[lv]);
        n_cnt += nb;
    }
    KWord<L> *kb[2];
    u32 *pb[2];
    for (int i = 0; i < 2; ++i) {
        kb[i] = ex.alloc<KWord<L>>(slots[i]);
        pb[i] = ex.alloc<u32>(slots[i]);
    }
    u32 *cnt_all = ex.alloc<u32>(n_cnt);
    ex.fill_bytes(cnt_all, 0, n_cnt * 4);
    const u64 items_ub = (u64) dig_n * (u64) g.n_ranks * g.cap_sub;
    const KWord<L> *ksrc = recv_k;
    const u32 *psrc = recv_p;
    const u32 *cnt_par = sub_cnt;
    u32 *cnt_cur = cnt_all;
    for (int lv = 1; lv < pl.n_levels; ++lv) {
        const u32 nP = lv == 1 ? dig_n * (u32) g.n_ranks : (u32) ((u64) dig_n << (pl.cum[lv - 1] - pl.cum[0]));
        kc_ksf_level<L>(ex, ksrc, psrc, kb[lv & 1], pb[lv & 1], cnt_par, nP, lv == 1 ? g.cap_sub : pl.cap[lv - 1], cnt_cur, pl.cap[lv], 64 * L - pl.cum[lv], pl.bits[lv],
                        items_ub, status, lv == 1 ? m_cell : nullptr, tune, lv == 1 ? (u32) g.n_ranks : 1u);
        ksrc = kb[lv & 1];
        psrc = pb[lv & 1];
        cnt_par = cnt_cur;
        cnt_cur += (u64) dig_n << (pl.cum[lv] - pl.cum[0]);
    }
    const u64 n_leaf = (u64) dig_n << (pl.cum[pl.n_levels - 1] - pl.cum[0]);
    kc_ksf_resolve<L>(ex, ksrc, psrc, cnt_par, n_leaf, all_flags, min_freq, reinterpret_cast<kc_ull *>(cells), status, items_ub);
    ex.arena->release(base_mark);
}

#endif  // __CUDACC__
