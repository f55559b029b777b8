// K-mer set construction (reference src/parser.h:22-141 AddKMers / AddKMersWithFrequencies / ReadKMers[Filtered],
// src/khash_utils.h:143-159) as a fused  decode -> canonical k-mer -> radix partition -> shared-memory resolve.
//
// Items are kept as structure-of-arrays: the k-mer word (KWord<L>, 8L bytes) and, when the caller needs to know
// WHERE a k-mer first occurs (the from-FASTA regime, see set_routes.cuh), a 32-bit payload = END position
// of the window in the framed sequence.  Nothing else is ever materialised:
//
//   level 0   kc_ks_hist0_kernel      sequence bytes -> k-mers in registers -> 256-bin histogram of the top key bits
//             kc_ks_scatter0_kernel   sequence bytes -> k-mers in registers -> partitioned (key, pos) arrays
//             (the 1 byte/base input is decoded twice instead of writing + re-reading 8L+4 bytes per k-mer)
//   level 1.. kc_kv_hist_kernel / kc_kv_scatter_kernel   MSD radix partitioning of every bucket still larger than
//             CAP items, digit width adapted to the bucket size (as sort.cuh, but SoA and payload-aware)
//   resolve   kc_ks_resolve_kernel    one CTA per bucket (<= CAP items): counting sort on the next <= 11 key bits in
//             shared memory, per-thread insertion sort of the (tiny) sub-buckets, run-length encode;  then, per
//             distinct key with >= min_count occurrences:   flags[min position] = 1   (FLAGS mode, nothing is written
//             back to HBM except those bytes)   and/or   unique key + min(occurrences-1, 255) to the bucket's slice
//             (KEYS mode, followed by one compaction).
//
// Algorithmic HBM bytes per k-mer occurrence (L = 1, with positions): 1 (hist0) + 1 + 12 (scatter0) + 8 (hist1)
// + 12 + 12 (scatter1) + 12 (resolve) = 58; without the fusion and with 16-byte AoS items the same work moved 146.
#pragma once
#include "exec.cuh"
#include "kword.cuh"
#include "sort.cuh"
#include "stage1.cuh"
#include <vector>

template <int L> struct KsCfg {
    static constexpr int EX_THREADS = L == 1 ? 256 : (L == 2 ? 128 : 64);  // level 0: one 32-base strip per thread
    static constexpr int EX_TILE = EX_THREADS * KC_EX_STRIP;               // window END positions per CTA
    static constexpr int CAP = L <= 2 ? 2048 : 1024;                       // resolve capacity (items per CTA)
    static constexpr int CAP_A = 1024;                                     // size class A of the hash resolve (most buckets)
    static constexpr int TILE = L == 1 ? 4096 : (L == 2 ? 2048 : 1024);    // level >= 1 scatter tile
    static constexpr int D0 = 8;                                           // level-0 digit width
};

#ifdef __CUDACC__

// First-occurrence flags are a BIT array (bit p of word p / 32 = position p): 50 M scattered atomicOr's (RED, no return
// value) cost ~0.14 ms on a B200 where 50 M scattered byte stores cost ~0.5 ms, and every later pass reads 8x less.
KC_D void kc_flag_set(u32 *flags, u32 pos) { atomicOr(&flags[pos >> 5], 1u << (pos & 31)); }

// ---- block helpers -----------------------------------------------------------------------------------------------
template <int THREADS> KC_D u32 kc_block_exclusive_scan(u32 v, u32 *total, u32 *smem_warp /*[THREADS/32]*/) {
    constexpr int W = THREADS / 32;
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
    for (int wi = 0; wi < W; ++wi) {
        u32 s = smem_warp[wi];
        if ((u32) wi < warp) warp_prefix += s;
        sum += s;
    }
    __syncthreads();
    *total = sum;
    return warp_prefix + incl - v;
}

// ---- sequence tile -> k-mers in registers --------------------------------------------------------------------------
// Decode the CTA's 32-base strips (plus KC_EX_HALO strips to the left) into packed 2-bit codes + validity bits.
template <int THREADS> KC_D void kc_tile_load(const u8 *__restrict__ seq, u64 n_bytes, i64 block_pos0, u64 *pk, u32 *vm) {
    for (int wi = threadIdx.x; wi < KC_EX_HALO + THREADS; wi += THREADS) {
        i64 p = block_pos0 + (i64) (wi - KC_EX_HALO) * KC_EX_STRIP;
        u64 codes = 0;
        u32 valid = 0;
        if (p >= 0 && (u64) p + KC_EX_STRIP <= n_bytes) {
            const uint4 *src = reinterpret_cast<const uint4 *>(seq + p);
            uint4 a = src[0], b = src[1];
            u32 w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                u32 c4, v4;
                kc_pack4(w[j], c4, v4);
                codes = (codes << 8) | c4;
                valid = (valid << 4) | v4;
            }
        } else if (p + KC_EX_STRIP > 0 && (u64) (p < 0 ? 0 : p) < n_bytes) {
            for (int j = 0; j < KC_EX_STRIP; ++j) {
                i64 q = p + j;
                u32 code = 4;
                if (q >= 0 && (u64) q < n_bytes) code = kc_nucleotide_code(seq[q]);
                codes = (codes << 2) | (code & 3);
                valid = (valid << 1) | (code < 4 ? 1u : 0u);
            }
        }
        pk[wi] = codes;
        vm[wi] = valid;
    }
}

// Bit (31 - j) set  <=>  a valid k-mer window ENDS at base j of strip widx (all k bases ACGT, src/parser.h:32-37).
KC_D u32 kc_strip_emit_mask(const u32 *vm, int widx, int k) {
    const u32 myv = vm[widx];
    int run = 0;
#pragma unroll
    for (int w = 1; w <= KC_EX_HALO; ++w) {
        u32 pv = vm[widx - w];
        if (pv == 0xFFFFFFFFu) {
            run += 32;
        } else {
            run += __ffs(~pv) - 1;  // trailing ones: bit 0 is the last base of that word
            break;
        }
    }
    u32 em = 0;
#pragma unroll
    for (int j = 0; j < KC_EX_STRIP; ++j) {
        run = ((myv >> (31 - j)) & 1) ? run + 1 : 0;
        if (run >= k) em |= 1u << (31 - j);
    }
    return em;
}

// Optional window filter (maskopt, src/parser.h:41-42 case_sensitive): win_mask is a bit array over window END positions
// (bit p & 31 of word p >> 5, padded to whole extraction tiles); only windows whose bit is set are emitted.
KC_D u32 kc_strip_window_filter(const u32 *__restrict__ win_mask, i64 block_pos0) {
    if (!win_mask) return 0xFFFFFFFFu;
    return __brev(win_mask[(block_pos0 >> 5) + threadIdx.x]);  // strip base j <-> em bit 31 - j
}

// f(j, canonical k-mer) for every valid window ending at base j of the strip (src/parser.h:38-46).
template <int L, class F> KC_D void kc_strip_windows(const u64 *pk, int widx, u32 em, int k, int complements, F &&f) {
    if (!em) return;
    const u64 mine = pk[widx];
    if constexpr (L == 1) {
        // k < 32: every window is a funnel shift of (previous word : own word); the reverse complement rolls
        const u64 prev = pk[widx - 1];
        const u64 mask = (1ULL << (2 * k)) - 1;
        const int top = 2 * (k - 1);
        KWord<1> pw;
        pw.w[0] = prev & ((1ULL << top) - 1);
        u64 rcs = k > 1 ? kmer_reverse_complement(pw, k - 1).w[0] : 0;  // rc of the k-1 bases before the strip
#pragma unroll
        for (int j = 0; j < KC_EX_STRIP; ++j) {
            const int sh = 2 * (31 - j);
            u64 fwd = (mine >> sh);
            if (j < 31) fwd |= prev << (2 * (j + 1));
            fwd &= mask;
            const u64 c = (mine >> sh) & 3;
            const u64 rcf = rcs | ((3 ^ c) << top);
            rcs = rcf >> 2;
            if ((em >> (31 - j)) & 1) {
                KWord<1> canon;
                canon.w[0] = (!complements || fwd < rcf) ? fwd : rcf;
                f(j, canon);
            }
        }
    } else {
        const KWord<L> mask = KWord<L>::low_mask(2 * k);
        const int top = 2 * (k - 1);
        const int top_limb = top >> 6, top_off = top & 63;
        KWord<L> fwd = KWord<L>::zero(), rcs = KWord<L>::zero();
        for (int h = k - 1; h >= 1; --h) {
            int gp = widx * 32 - h;
            u64 c = (pk[gp >> 5] >> (2 * (31 - (gp & 31)))) & 3;
            fwd = fwd.shl(2);
            fwd.w[0] |= c;
            KWord<L> rcf = rcs;
#pragma unroll
            for (int i = 0; i < L; ++i)
                if (i == top_limb) rcf.w[i] |= (3 ^ c) << top_off;
            rcs = rcf.shr(2);
        }
#pragma unroll 4
        for (int j = 0; j < KC_EX_STRIP; ++j) {
            u64 c = (mine >> (2 * (31 - j))) & 3;
            fwd = fwd.shl(2);
            fwd.w[0] |= c;
            fwd = fwd & mask;
            KWord<L> rcf = rcs;
#pragma unroll
            for (int i = 0; i < L; ++i)
                if (i == top_limb) rcf.w[i] |= (3 ^ c) << top_off;
            rcs = rcf.shr(2);
            if ((em >> (31 - j)) & 1) {
                const KWord<L> canon = (!complements || fwd < rcf) ? fwd : rcf;
                f(j, canon);
            }
        }
    }
}

// Bijective scrambling of a k-mer word for the FLAGS-only mode, where no sorted output is needed: the top limb (the one
// MSD digits are taken from) is replaced by a multiplicative hash of all limbs.  Equal words stay equal, different
// words stay different, and bucket sizes no longer depend on the k-mer composition of the input (canonical k-mers
// alone are skewed towards small values: half of them begin with A).
template <int L> KC_D KWord<L> kmer_scramble(const KWord<L> &x) {
    KWord<L> r = x;
    u64 t = 0;
#pragma unroll
    for (int i = 0; i < L; ++i) t = (t ^ x.w[i]) * 0x9E3779B97F4A7C15ULL;
    r.w[L - 1] = t;  // x.w[L-1] -> t is a bijection for fixed lower limbs (xor, then multiplication by an odd constant)
    return r;
}

// ---- level 0 -------------------------------------------------------------------------------------------------------
template <int L, bool SCR>
__global__ void __launch_bounds__(KsCfg<L>::EX_THREADS) kc_ks_hist0_kernel(const u8 *__restrict__ seq, u64 n_bytes, int k, int complements,
                                                                            int shift, int bits, u32 *hist, u16 *tile_hist, u32 tile0,
                                                                            const u32 *__restrict__ win_mask = nullptr) {
    constexpr int T = KsCfg<L>::EX_THREADS;
    __shared__ u64 pk[KC_EX_HALO + T];
    __shared__ u32 vm[KC_EX_HALO + T];
    __shared__ u32 sh[256];
    const i64 block_pos0 = (i64) (tile0 + blockIdx.x) * KsCfg<L>::EX_TILE;
    kc_tile_load<T>(seq, n_bytes, block_pos0, pk, vm);
    for (int i = threadIdx.x; i < 256; i += T) sh[i] = 0;
    __syncthreads();
    const int widx = KC_EX_HALO + threadIdx.x;
    const u32 em = kc_strip_emit_mask(vm, widx, k) & kc_strip_window_filter(win_mask, block_pos0);
    kc_strip_windows<L>(pk, widx, em, k, complements, [&](int, const KWord<L> &c0) {
        const KWord<L> c = SCR ? kmer_scramble(c0) : c0;
        atomicAdd(&sh[c.digit(shift, bits)], 1u);
    });
    __syncthreads();
    // the tile's digit counts are kept (512 bytes per 8L KB of k-mers) so that the scatter pass needs no counting pass
    for (int i = threadIdx.x; i < 256; i += T) {
        const u32 c = sh[i];
        tile_hist[(u64) blockIdx.x * 256 + i] = (u16) c;
        if (c) atomicAdd(&hist[i], c);
    }
}

// One CTA: level-0 digit counts -> bucket offsets (cursor) and the classified child buckets.
// ctr[0] = big, ctr[1] = small, ctr[2] = uniform, ctr[3] = overflow flag, ctr[4] = tiles of the big children,
// ctr[5] = small buckets of more than 1024 items (size class B of the hash resolve).
__global__ void __launch_bounds__(256) kc_ks_scan0_kernel(const u32 *hist, u64 *cursor, SortBucket *next_big, u32 next_cap, SortBucket *small,
                                                          u32 small_cap, SortBucket *uniform, u32 uniform_cap, u32 *ctr, u64 *total_out, u32 cap,
                                                          u32 tile, int rem_after) {
    __shared__ u32 sw[8];
    const u32 c = hist[threadIdx.x];
    u32 total;
    const u32 p = kc_block_exclusive_scan<256>(c, &total, sw);
    cursor[threadIdx.x] = p;
    if (threadIdx.x == 0) *total_out = total;
    if (c == 0) return;
    SortBucket ch;
    ch.off = p;
    ch.size = c;
    ch.rem = (u16) rem_after;
    ch.parity = 0;
    ch.bits = 0;
    if (c <= cap) {
        u32 s = atomicAdd(&ctr[1], 1u);
        if (s < small_cap) small[s] = ch;
        else ctr[3] = 1;
        if (c > 1024u) atomicAdd(&ctr[5], 1u);
    } else if (ch.rem == 0) {
        u32 s = atomicAdd(&ctr[2], 1u);
        if (s < uniform_cap) uniform[s] = ch;
        else ctr[3] = 1;
    } else {
        u32 s = atomicAdd(&ctr[0], 1u);
        if (s < next_cap) next_big[s] = ch;
        else ctr[3] = 1;
        atomicAdd(&ctr[4], (c + tile - 1) / tile);
    }
}

// P2P = true (multi-GPU): bucket g is stored through dst_k[g] / dst_p[g], which point into the receive buffers of the
// bucket's OWNER GPU (peer memory mapped over NVLink); cursor[g] then starts at this rank's segment of that bucket, so
// the partition pass IS the all-to-all: no intermediate send buffer, no separate collective, and the owner finds its
// level-0 buckets complete and contiguous.
template <int L, bool PAY, bool SCR, bool P2P = false>
__global__ void __launch_bounds__(KsCfg<L>::EX_THREADS) kc_ks_scatter0_kernel(const u8 *__restrict__ seq, u64 n_bytes, int k, int complements,
                                                                               int shift, int bits, u64 *cursor, const u16 *__restrict__ tile_hist,
                                                                               KWord<L> *__restrict__ keys, u32 *__restrict__ pos, u32 tile0,
                                                                               KWord<L> *const *__restrict__ dst_k = nullptr,
                                                                               u32 *const *__restrict__ dst_p = nullptr,
                                                                               const u32 *__restrict__ win_mask = nullptr) {
    constexpr int T = KsCfg<L>::EX_THREADS;
    constexpr int R = 256 / T;
    constexpr int TILE = KsCfg<L>::EX_TILE;
    extern __shared__ __align__(16) unsigned char kc_smem_raw[];
    KWord<L> *stage_k = reinterpret_cast<KWord<L> *>(kc_smem_raw);
    u16 *stage_s = reinterpret_cast<u16 *>(stage_k + TILE);
    __shared__ u64 pk[KC_EX_HALO + T];
    __shared__ u32 vm[KC_EX_HALO + T];
    __shared__ u32 cnt[256];
    __shared__ u32 loff[256];
    __shared__ u64 gbase[256];
    __shared__ u32 sw[T / 32];
    const i64 block_pos0 = (i64) (tile0 + blockIdx.x) * TILE;
    kc_tile_load<T>(seq, n_bytes, block_pos0, pk, vm);
    for (int i = threadIdx.x; i < 256; i += T) cnt[i] = 0;
    __syncthreads();
    const int widx = KC_EX_HALO + threadIdx.x;
    const u32 em = kc_strip_emit_mask(vm, widx, k) & kc_strip_window_filter(win_mask, block_pos0);
    // digit counts of the tile, left behind by kc_ks_hist0_kernel
    u32 total;
    {
        u32 v[R], c = 0;
#pragma unroll
        for (int r = 0; r < R; ++r) {
            v[r] = tile_hist[(u64) blockIdx.x * 256 + threadIdx.x * R + r];
            c += v[r];
        }
        u32 p = kc_block_exclusive_scan<T>(c, &total, sw);
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int i = threadIdx.x * R + r;
            loff[i] = p;
            if (v[r]) gbase[i] = atomicAdd((kc_ull *) &cursor[i], (kc_ull) v[r]);  // reserve the tile's slots of bucket i
            p += v[r];
        }
    }
    __syncthreads();
    if (total == 0) return;
    // the k-mers again, now into their slot of the staged (digit-ordered) tile
    kc_strip_windows<L>(pk, widx, em, k, complements, [&](int j, const KWord<L> &c0) {
        const KWord<L> c = SCR ? kmer_scramble(c0) : c0;
        const u32 dg = c.digit(shift, bits);
        const u32 q = loff[dg] + atomicAdd(&cnt[dg], 1u);
        stage_k[q] = c;
        if (PAY) stage_s[q] = (u16) (threadIdx.x * KC_EX_STRIP + j);
    });
    __syncthreads();
    for (u32 q = threadIdx.x; q < total; q += T) {
        const KWord<L> v = stage_k[q];
        const u32 dg = v.digit(shift, bits);
        const u64 idx = gbase[dg] + (q - loff[dg]);
        KWord<L> *kb = keys;
        u32 *pb = pos;
        if (P2P) {
            kb = dst_k[dg];
            pb = dst_p[dg];
        }
        kb[idx] = v;
        if (PAY) pb[idx] = (u32) ((u64) block_pos0 + stage_s[q]);
    }
}

// ---- levels >= 1 (SoA twins of kc_sort_hist_kernel / kc_sort_scan_kernel / kc_sort_scatter_kernel) ----------------------
template <int L>
__global__ void __launch_bounds__(256) kc_kv_hist_kernel(const KWord<L> *k0, const KWord<L> *k1, const SortBucket *big, const u32 *tile_prefix,
                                                         u32 nb, u32 tiles_per_cta, u32 *hist) {
    constexpr int TILE = KsCfg<L>::TILE;
    __shared__ u32 sh[256];
    const u32 n_tiles = tile_prefix[nb];
    u32 t0 = blockIdx.x * tiles_per_cta;
    u32 t1 = min(n_tiles, t0 + tiles_per_cta);
    if (t0 >= t1) return;
    sh[threadIdx.x] = 0;
    u32 b = kc_upper_bound_u32(tile_prefix, nb + 1, t0) - 1;
    u32 cur = b;
    __syncthreads();
    for (u32 t = t0; t < t1; ++t) {
        while (t >= tile_prefix[b + 1]) ++b;
        if (b != cur) {
            __syncthreads();
            if (sh[threadIdx.x]) atomicAdd(&hist[(u64) cur * 256 + threadIdx.x], sh[threadIdx.x]);
            sh[threadIdx.x] = 0;
            cur = b;
            __syncthreads();
        }
        const SortBucket d = big[b];
        const KWord<L> *src = (d.parity ? k1 : k0) + d.off;
        const u32 start = (t - tile_prefix[b]) * TILE;
        const u32 cnt = min((u32) TILE, d.size - start);
        const int shift = d.rem - d.bits;
        for (u32 i = threadIdx.x; i < cnt; i += 256) atomicAdd(&sh[src[start + i].digit(shift, d.bits)], 1u);
    }
    __syncthreads();
    if (sh[threadIdx.x]) atomicAdd(&hist[(u64) cur * 256 + threadIdx.x], sh[threadIdx.x]);
}

// As kc_sort_scan_kernel, plus ctr[4] += tiles of the children that stay big (so the host learns the next level's
// tile count with the same read-back as the bucket counts).
__global__ void __launch_bounds__(256) kc_kv_scan_kernel(const SortBucket *big, const u32 *hist, u64 *cursor, u8 *skip, SortBucket *next_big,
                                                         u32 next_cap, SortBucket *small, u32 small_cap, SortBucket *uniform, u32 uniform_cap,
                                                         u32 *ctr, u32 cap, u32 tile) {
    __shared__ u32 sw[8];
    const u32 b = blockIdx.x;
    const SortBucket d = big[b];
    const u32 c = hist[(u64) b * 256 + threadIdx.x];
    u32 total;
    const u32 p = kc_block_exclusive_scan<256>(c, &total, sw);
    cursor[(u64) b * 256 + threadIdx.x] = d.off + p;
    const bool single = (c == d.size);  // every item has this digit: nothing needs to move
    if (threadIdx.x == 0) skip[b] = 0;
    __syncthreads();
    if (single) skip[b] = 1;
    if (c == 0) return;
    SortBucket ch;
    ch.off = d.off + p;
    ch.size = c;
    ch.rem = (u16) (d.rem - d.bits);
    ch.parity = single ? d.parity : (u8) (d.parity ^ 1);
    ch.bits = 0;
    if (c <= cap) {
        u32 s = atomicAdd(&ctr[1], 1u);
        if (s < small_cap) small[s] = ch;
        else ctr[3] = 1;
        if (c > 1024u) atomicAdd(&ctr[5], 1u);
    } else if (ch.rem == 0) {
        u32 s = atomicAdd(&ctr[2], 1u);
        if (s < uniform_cap) uniform[s] = ch;
        else ctr[3] = 1;
    } else {
        u32 s = atomicAdd(&ctr[0], 1u);
        if (s < next_cap) next_big[s] = ch;
        else ctr[3] = 1;
        atomicAdd(&ctr[4], (c + tile - 1) / tile);
    }
}

template <int L, bool PAY>
__global__ void __launch_bounds__(256) kc_kv_scatter_kernel(KWord<L> *k0, KWord<L> *k1, u32 *p0, u32 *p1, const SortBucket *big,
                                                            const u32 *tile_prefix, u32 nb, u32 tiles_per_cta, u64 *cursor, const u8 *skip) {
    constexpr int TILE = KsCfg<L>::TILE;
    constexpr int ITEMS = TILE / 256;
    extern __shared__ __align__(16) unsigned char kc_smem_raw[];
    KWord<L> *stage_k = reinterpret_cast<KWord<L> *>(kc_smem_raw);
    u32 *stage_p = reinterpret_cast<u32 *>(stage_k + TILE);
    u16 *rk = reinterpret_cast<u16 *>(stage_p + (PAY ? TILE : 0));  // rank of every item inside its digit (one shared atomic per item)
    __shared__ u32 cnt[256];
    __shared__ u32 loff[256];
    __shared__ u64 gbase[256];
    __shared__ u32 sw[8];
    const u32 n_tiles = tile_prefix[nb];
    u32 t0 = blockIdx.x * tiles_per_cta;
    u32 t1 = min(n_tiles, t0 + tiles_per_cta);
    if (t0 >= t1) return;
    u32 b = kc_upper_bound_u32(tile_prefix, nb + 1, t0) - 1;
    cnt[threadIdx.x] = 0;
    __syncthreads();
    for (u32 t = t0; t < t1; ++t) {
        while (t >= tile_prefix[b + 1]) ++b;
        if (skip[b]) continue;
        const SortBucket d = big[b];
        const KWord<L> *src = (d.parity ? k1 : k0) + d.off;
        const u32 *psrc = (d.parity ? p1 : p0) + d.off;
        KWord<L> *dst = d.parity ? k0 : k1;
        u32 *pdst = d.parity ? p0 : p1;
        const u32 start = (t - tile_prefix[b]) * TILE;
        const u32 n_here = min((u32) TILE, d.size - start);
        const int shift = d.rem - d.bits;
        // all loads of the tile are issued before the first use, so one DRAM latency is exposed per tile
        KWord<L> item[ITEMS];
        u32 pay[ITEMS];
#pragma unroll
        for (int j = 0; j < ITEMS; ++j) {
            u32 i = threadIdx.x + j * 256;
            if (i < n_here) item[j] = src[start + i];
        }
        if (PAY) {
#pragma unroll
            for (int j = 0; j < ITEMS; ++j) {
                u32 i = threadIdx.x + j * 256;
                if (i < n_here) pay[j] = psrc[start + i];
            }
        }
#pragma unroll
        for (int j = 0; j < ITEMS; ++j) {
            u32 i = threadIdx.x + j * 256;
            if (i < n_here) rk[i] = (u16) atomicAdd(&cnt[item[j].digit(shift, d.bits)], 1u);
        }
        __syncthreads();
        const u32 c = cnt[threadIdx.x];
        u32 total;
        const u32 p = kc_block_exclusive_scan<256>(c, &total, sw);
        loff[threadIdx.x] = p;
        if (c) gbase[threadIdx.x] = atomicAdd((kc_ull *) &cursor[(u64) b * 256 + threadIdx.x], (kc_ull) c);
        cnt[threadIdx.x] = 0;
        __syncthreads();
        // slots inside a digit are handed out in arrival order (the partition is unstable on purpose)
#pragma unroll
        for (int j = 0; j < ITEMS; ++j) {
            u32 i = threadIdx.x + j * 256;
            if (i < n_here) {
                const u32 dg = item[j].digit(shift, d.bits);
                const u32 q = loff[dg] + rk[i];
                stage_k[q] = item[j];
                if (PAY) stage_p[q] = pay[j];
            }
        }
        __syncthreads();
        for (u32 q = threadIdx.x; q < n_here; q += 256) {
            const KWord<L> v = stage_k[q];
            const u32 dg = v.digit(shift, d.bits);
            const u64 idx = gbase[dg] + (q - loff[dg]);
            dst[idx] = v;
            if (PAY) pdst[idx] = stage_p[q];
        }
        __syncthreads();
    }
}

// ---- resolve ---------------------------------------------------------------------------------------------------------
// Bitonic sort of (key, payload) pairs in shared memory by key (whole CTA; any m, see kc_block_bitonic).
template <int L, bool PAY> KC_D void kc_block_bitonic_kv(KWord<L> *sk, u32 *sp, u32 m) {
    u32 P = 2;
    while (P < m) P <<= 1;
    for (u32 k = 2; k <= P; k <<= 1) {
        for (u32 j = k >> 1; j > 0; j >>= 1) {
            for (u32 t = threadIdx.x; t < (P >> 1); t += 256) {
                u32 i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                u32 l = (j == (k >> 1)) ? (i ^ (k - 1)) : (i | j);
                if (l < m && i < m) {
                    KWord<L> a = sk[i], c = sk[l];
                    if (c < a) {
                        sk[i] = c;
                        sk[l] = a;
                        if (PAY) {
                            u32 x = sp[i];
                            sp[i] = sp[l];
                            sp[l] = x;
                        }
                    }
                }
            }
            __syncthreads();
        }
    }
}

static const u32 KC_KS_SUB_SMALL = 32;  // sub-buckets up to this size are sorted by one thread

// One CTA per bucket of at most CAP items (see the file header).  FLAGS: flags != nullptr.  KEYS: unique keys go to
// the front of the bucket's slice of k0, cnt_out receives min(occurrences - 1, 255) (src/parser.h:77,81) and the rest
// of the slice is filled with all-ones words for the compaction that follows (which also applies min_count).
template <int L, bool PAY, bool KEYS>
__global__ void __launch_bounds__(256) kc_ks_resolve_kernel(KWord<L> *k0, const KWord<L> *k1, const u32 *p0, const u32 *p1,
                                                            const SortBucket *small, u32 *flags, u32 min_count, kc_ull *n_unique, u8 *cnt_out) {
    constexpr int CAP = KsCfg<L>::CAP;
    constexpr int SUB_BITS_MAX = 11;
    extern __shared__ __align__(16) unsigned char kc_smem_raw[];
    KWord<L> *sk = reinterpret_cast<KWord<L> *>(kc_smem_raw);
    u32 *sp = reinterpret_cast<u32 *>(sk + CAP);                  // PAY only
    u16 *rnk = reinterpret_cast<u16 *>(sp + (PAY ? CAP : 0));     // rank inside the sub-bucket, later the run heads
    __shared__ u32 sub_cnt[1 << SUB_BITS_MAX];
    __shared__ u32 big_list[64];
    __shared__ u32 n_big;
    __shared__ u32 sw[8];
    const SortBucket d = small[blockIdx.x];
    const KWord<L> *src = (d.parity ? k1 : k0) + d.off;
    const u32 *psrc = (d.parity ? p1 : p0) + d.off;
    KWord<L> *dst = k0 + d.off;
    const u32 size = d.size;
    if (size == 1) {
        if (threadIdx.x == 0) {
            if (min_count <= 1) {
                if (PAY && flags) kc_flag_set(flags, psrc[0]);
                atomicAdd(n_unique, (kc_ull) 1);
            }
            if (KEYS) {
                dst[0] = src[0];
                cnt_out[d.off] = 0;
            }
        }
        return;
    }
    int bits = 1;
    while ((1u << bits) < 2 * size && bits < SUB_BITS_MAX) ++bits;
    if (bits > (int) d.rem) bits = d.rem;
    const u32 n_sub = 1u << bits;
    const int shift = d.rem - bits;
    for (u32 i = threadIdx.x; i < n_sub; i += 256) sub_cnt[i] = 0;
    if (threadIdx.x == 0) n_big = 0;
    __syncthreads();
    // 1. sub-bucket counts and the rank of every item inside its sub-bucket
    for (u32 i = threadIdx.x; i < size; i += 256) rnk[i] = (u16) atomicAdd(&sub_cnt[src[i].digit(shift, bits)], 1u);
    __syncthreads();
    // 2. exclusive scan of the counts (n_sub <= 2048: 8 consecutive entries per thread)
    {
        u32 v[8], c = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            u32 i = threadIdx.x * 8 + j;
            v[j] = i < n_sub ? sub_cnt[i] : 0;
            c += v[j];
        }
        u32 total;
        u32 p = kc_block_exclusive_scan<256>(c, &total, sw);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            u32 i = threadIdx.x * 8 + j;
            if (i < n_sub) {
                sub_cnt[i] = p;
                if (v[j] > KC_KS_SUB_SMALL) {
                    u32 q = atomicAdd(&n_big, 1u);
                    if (q < 64) big_list[q] = i;
                }
            }
            p += v[j];
        }
    }
    __syncthreads();
    // 3. items into shared memory, grouped by sub-bucket (second read of the bucket: it is still in L2)
    for (u32 i = threadIdx.x; i < size; i += 256) {
        const KWord<L> v = src[i];
        const u32 q = sub_cnt[v.digit(shift, bits)] + rnk[i];
        sk[q] = v;
        if (PAY) sp[q] = psrc[i];
    }
    __syncthreads();
    // 4. order inside the sub-buckets (by key only: equal keys need not be ordered among themselves)
    const u32 nbig = n_big;
    if (nbig > 64) {
        kc_block_bitonic_kv<L, PAY>(sk, sp, size);
    } else {
        for (u32 b = threadIdx.x; b < n_sub; b += 256) {
            const u32 lo = sub_cnt[b];
            const u32 hi = (b + 1 < n_sub) ? sub_cnt[b + 1] : size;
            const u32 m = hi - lo;
            if (m < 2 || m > KC_KS_SUB_SMALL) continue;
            for (u32 x = lo + 1; x < hi; ++x) {
                const KWord<L> key = sk[x];
                if (!(key < sk[x - 1])) continue;
                u32 pv = 0;
                if (PAY) pv = sp[x];
                u32 y = x;
                while (y > lo && key < sk[y - 1]) {
                    sk[y] = sk[y - 1];
                    if (PAY) sp[y] = sp[y - 1];
                    --y;
                }
                sk[y] = key;
                if (PAY) sp[y] = pv;
            }
        }
        __syncthreads();
        for (u32 q = 0; q < nbig; ++q) {  // uniform across the CTA
            const u32 b = big_list[q];
            const u32 lo = sub_cnt[b];
            const u32 hi = (b + 1 < n_sub) ? sub_cnt[b + 1] : size;
            kc_block_bitonic_kv<L, PAY>(sk + lo, sp + lo, hi - lo);
        }
    }
    __syncthreads();
    // 5. run heads: thread t owns the items [t * C, (t + 1) * C), so head ranks follow the item order
    u16 *hpos = rnk;
    const u32 C = (size + 255) / 256;
    const u32 i0 = min(size, threadIdx.x * C), i1 = min(size, i0 + C);
    u32 heads = 0;
    for (u32 i = i0; i < i1; ++i) heads += (i == 0 || sk[i] != sk[i - 1]) ? 1u : 0u;
    u32 nu;
    u32 hp = kc_block_exclusive_scan<256>(heads, &nu, sw);
    for (u32 i = i0; i < i1; ++i)
        if (i == 0 || sk[i] != sk[i - 1]) hpos[hp++] = (u16) i;
    __syncthreads();
    // 6. one distinct key per thread: occurrences, smallest position, outputs
    u32 kept = 0;
    for (u32 u = threadIdx.x; u < (KEYS ? size : nu); u += 256) {
        if (u < nu) {
            const u32 h = hpos[u];
            const u32 e = (u + 1 < nu) ? hpos[u + 1] : size;
            const u32 occ = e - h;
            if (occ >= min_count) {
                ++kept;
                if (PAY && flags) {
                    u32 mp = sp[h];
                    for (u32 x = h + 1; x < e; ++x) mp = min(mp, sp[x]);
                    kc_flag_set(flags, mp);
                }
            }
            if (KEYS) {
                dst[u] = sk[h];
                cnt_out[d.off + u] = (u8) min(occ - 1, 255u);
            }
        } else if (KEYS) {
            dst[u] = KWord<L>::ones();
        }
    }
    // 7. kept distinct keys of the bucket -> global count
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) kept += __shfl_down_sync(0xFFFFFFFFu, kept, o);
    if ((threadIdx.x & 31) == 0 && kept) atomicAdd(n_unique, (kc_ull) kept);
}

// FLAGS-only resolve: exact dedup of one bucket through a shared-memory hash table, persistent and software-pipelined.
//   * a CTA walks the bucket list with stride gridDim.x; while it works on bucket b the keys / positions of bucket
//     b + stride are already in flight into registers and the descriptor of b + 2 stride is being fetched, so no
//     global-memory latency sits between the barriers;
//   * the bucket's keys and positions are staged in shared memory; a table slot holds the INDEX of the item that
//     claimed it (one atomicCAS per item), so keys of any width are compared exactly against the staged copy;
//   * only duplicates pay a second atomic: atomicMin of their position into the staged position of the claimer
//     (and an occurrence count when -z needs it);
//   * finally every claimer with enough occurrences flags the smallest position of its key.  Nothing else is written.
// A launch handles the buckets with size in (size_lo, size_hi] and skips the others.
template <int L, int CAPX, bool COUNTED>
__global__ void __launch_bounds__(256) kc_ks_resolve_hash_kernel(const KWord<L> *__restrict__ k0, const KWord<L> *__restrict__ k1,
                                                                 const u32 *__restrict__ p0, const u32 *__restrict__ p1,
                                                                 const SortBucket *__restrict__ small, u32 n_small, u32 size_lo, u32 size_hi,
                                                                 u32 *flags, u32 min_count, kc_ull *n_unique) {
    constexpr int ITEMS = CAPX / 256;
    extern __shared__ __align__(16) unsigned char kc_smem_raw[];
    KWord<L> *sk = reinterpret_cast<KWord<L> *>(kc_smem_raw);
    u32 *tab = reinterpret_cast<u32 *>(sk + CAPX);
    u32 *sp = tab + 3 * CAPX;  // five table rounds: 2 CAPX + CAPX/2 + CAPX/8 + 64 + 64 slots at most
    u32 *occ = sp + CAPX;      // COUNTED only
    const u32 stride = gridDim.x;
    u32 b = blockIdx.x;
    if (b >= n_small) return;
    SortBucket d_cur = small[b], d_next;
    d_next.size = 0;
    u32 bn = b + stride;
    if (bn < n_small) d_next = small[bn];
    KWord<L> cur_k[ITEMS], nxt_k[ITEMS];
    u32 cur_p[ITEMS], nxt_p[ITEMS];
    {
        const bool in_class = d_cur.size > size_lo && d_cur.size <= size_hi;
        const KWord<L> *src = (d_cur.parity ? k1 : k0) + d_cur.off;
        const u32 *psrc = (d_cur.parity ? p1 : p0) + d_cur.off;
#pragma unroll
        for (int j = 0; j < ITEMS; ++j) {
            const u32 i = threadIdx.x + j * 256;
            if (in_class && i < d_cur.size) {
                cur_k[j] = src[i];
                cur_p[j] = psrc[i];
            }
        }
    }
    u32 kept = 0;
    while (true) {
        // prefetch: data of the next bucket, descriptor of the one after it
        const bool next_ok = bn < n_small;
        const bool next_in_class = next_ok && d_next.size > size_lo && d_next.size <= size_hi;
        if (next_in_class) {
            const KWord<L> *src = (d_next.parity ? k1 : k0) + d_next.off;
            const u32 *psrc = (d_next.parity ? p1 : p0) + d_next.off;
#pragma unroll
            for (int j = 0; j < ITEMS; ++j) {
                const u32 i = threadIdx.x + j * 256;
                if (i < d_next.size) {
                    nxt_k[j] = src[i];
                    nxt_p[j] = psrc[i];
                }
            }
        }
        const u32 bnn = bn + stride;
        SortBucket d_next2;
        d_next2.size = 0;
        if (bnn < n_small) d_next2 = small[bnn];
        // resolve the current bucket
        const u32 size = d_cur.size;
        if (size > size_lo && size <= size_hi) {
            int lg = 6;
            while ((1u << lg) < 2 * size) ++lg;
            // stage the bucket and write round 0 of the table
            u64 hs[ITEMS];
            u32 act = 0, rep = 0;  // bit j: item j of this thread is still unsettled / represents its key
#pragma unroll
            for (int j = 0; j < ITEMS; ++j) {
                const u32 i = threadIdx.x + j * 256;
                if (i < size) {
                    sk[i] = cur_k[j];
                    sp[i] = cur_p[j];
                    if (COUNTED) occ[i] = 1;
                    u64 hsh = 0;
#pragma unroll
                    for (int q = 0; q < L; ++q) hsh = (hsh ^ cur_k[j].w[q]) * 0xD6E8FEB86659FD93ULL;
                    hs[j] = hsh;
                    tab[hsh >> (64 - lg)] = i;
                    act |= 1u << j;
                }
            }
            // Rounds of write-then-verify, no atomics for distinct keys: every unsettled item has stored its index in
            // the slot of its key (plain store, some writer wins).  After the barrier the winner of a slot represents
            // its key; an item that finds an equal key there is a duplicate and folds its position into the winner's;
            // an item that finds a different key moves on to the next, smaller table with fresh hash bits.  Items with
            // equal keys take the same path, so they always meet in the same slot of the same round.
            u32 *T = tab;
            int lgr = lg, r = 0;
            __syncthreads();
            while (true) {
                if (r == 5) {
                    // still unsettled after five rounds (~1e-4 of the buckets): classic CAS table with linear probing
                    const u32 n_slots = 1u << lg, mask = n_slots - 1;
                    for (u32 s = threadIdx.x; s < n_slots; s += 256) tab[s] = KC_NONE;
                    __syncthreads();
#pragma unroll
                    for (int j = 0; j < ITEMS; ++j) {
                        if ((act >> j) & 1u) {
                            const u32 i = threadIdx.x + j * 256;
                            u32 s = (u32) (hs[j] >> (64 - lg));
                            while (true) {
                                const u32 old = atomicCAS(&tab[s], KC_NONE, i);
                                if (old == KC_NONE) {
                                    rep |= 1u << j;
                                    break;
                                }
                                if (sk[old] == cur_k[j]) {
                                    atomicMin(&sp[old], cur_p[j]);
                                    if (COUNTED) atomicAdd(&occ[old], 1u);
                                    break;
                                }
                                s = (s + 1) & mask;
                            }
                        }
                    }
                    __syncthreads();
                    break;
                }
                if (act) {
                    u32 *Tn = T + (1u << lgr);
                    const int lgn = lgr - 2 > 6 ? lgr - 2 : 6;
#pragma unroll
                    for (int j = 0; j < ITEMS; ++j) {
                        if ((act >> j) & 1u) {
                            const u32 i = threadIdx.x + j * 256;
                            const u32 o = T[hs[j] >> (64 - lgr)];
                            if (o == i) {
                                rep |= 1u << j;
                                act &= ~(1u << j);
                            } else if (sk[o] == cur_k[j]) {
                                atomicMin(&sp[o], cur_p[j]);
                                if (COUNTED) atomicAdd(&occ[o], 1u);
                                act &= ~(1u << j);
                            } else {
                                hs[j] <<= lgr;
                                if (r < 4) Tn[hs[j] >> (64 - lgn)] = i;
                            }
                        }
                    }
                }
                T += 1u << lgr;
                lgr = lgr - 2 > 6 ? lgr - 2 : 6;
                ++r;
                // barrier (table writes / folded positions become visible) + vote: is any item of the CTA unsettled?
                if (!__syncthreads_or(act != 0)) break;
            }
            // Only the thread's own sp[] / occ[] entries are read from here on, and the next bucket's staging rewrites
            // exactly those, so no barrier is needed before the CTA moves on.
#pragma unroll
            for (int j = 0; j < ITEMS; ++j) {
                const u32 i = threadIdx.x + j * 256;
                if (((rep >> j) & 1u) && (!COUNTED || occ[i] >= min_count)) {
                    kc_flag_set(flags, sp[i]);
                    ++kept;
                }
            }
        }
        if (!next_ok) break;
        d_cur = d_next;
        d_next = d_next2;
        bn = bnn;
#pragma unroll
        for (int j = 0; j < ITEMS; ++j) {
            cur_k[j] = nxt_k[j];
            cur_p[j] = nxt_p[j];
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) kept += __shfl_down_sync(0xFFFFFFFFu, kept, o);
    if ((threadIdx.x & 31) == 0 && kept) atomicAdd(n_unique, (kc_ull) kept);
}

// Buckets that ran out of key bits while still larger than CAP: one distinct key.
template <int L, bool PAY, bool KEYS>
__global__ void __launch_bounds__(256) kc_ks_uniform_kernel(KWord<L> *k0, const KWord<L> *k1, const u32 *p0, const u32 *p1,
                                                            const SortBucket *uniform, u32 *flags, u32 min_count, kc_ull *n_unique, u8 *cnt_out) {
    __shared__ u32 min_pos;
    const SortBucket d = uniform[blockIdx.x];
    const KWord<L> *src = (d.parity ? k1 : k0) + d.off;
    const u32 *psrc = (d.parity ? p1 : p0) + d.off;
    KWord<L> *dst = k0 + d.off;
    const KWord<L> key = src[0];
    if (PAY && flags && d.size >= min_count) {
        if (threadIdx.x == 0) min_pos = 0xFFFFFFFFu;
        __syncthreads();
        u32 m = 0xFFFFFFFFu;
        for (u32 i = threadIdx.x; i < d.size; i += 256) m = min(m, psrc[i]);
        atomicMin(&min_pos, m);
        __syncthreads();
        if (threadIdx.x == 0) kc_flag_set(flags, min_pos);
    }
    if (threadIdx.x == 0 && d.size >= min_count) atomicAdd(n_unique, (kc_ull) 1);
    __syncthreads();
    if (KEYS) {
        for (u32 i = threadIdx.x; i < d.size; i += 256) dst[i] = i == 0 ? key : KWord<L>::ones();
        if (threadIdx.x == 0) cnt_out[d.off] = (u8) min(d.size - 1, 255u);
    }
}

// ---- host driver -----------------------------------------------------------------------------------------------------
// Multi-GPU use (hash-range sharding, kc_grp_exact_flags in group.cuh): the construction is cut at the level-0 boundary.
//   kc_kmerset_hist_only, kc_kmerset_scatter_p2p   level 0 over the window END positions [pos_begin, pos_end) of a sequence
//                 that is resident in full: the scrambled keys and their GLOBAL positions go straight into the owners'
//                 buffers, ordered by level-0 digit (owner rank = digit * n_ranks / 256).
//   kc_kmerset_resolve   the items are given (after the exchange: every occurrence of this rank's hash range, in its
//                 n_pre level-0 buckets) and level 0 is skipped; first-occurrence bits are set at global positions.
struct KsShard {
    u64 pos_begin = 0, pos_end = 0;  // hist / scatter: multiples of EX_TILE (pos_end may also be n_bytes)
    void *keys = nullptr;            // resolve: the items (device, caller-owned)
    u32 *pos = nullptr;
    u64 n_items = 0;
    u32 host_hist[256];              // hist out
    u16 *tile_hist_keep = nullptr;   // caller-owned, (tiles of the slice) * 256 entries: hist out, scatter in
    const u64 *cursor0 = nullptr;    // scatter: host, 256 start cursors (this rank's segment inside each bucket)
    void *const *dst_k = nullptr;    // scatter: device tables of 256 pointers each
    u32 *const *dst_p = nullptr;
    u32 n_pre = 0;                   // resolve: level-0 buckets already in place (>= 1)
    const u64 *pre_off = nullptr, *pre_size = nullptr;  // host arrays
};

template <int L> struct KmerSet {
    u64 n_occ = 0;            // M: k-mer windows seen
    u64 n_kept = 0;           // U: distinct k-mers with >= min_freq occurrences
    KWord<L> *keys = nullptr; // KEYS mode: the n_kept keys in ascending order ...
    u8 *cnt = nullptr;        // ... and min(occurrences - 1, 255) of each
};

// Builds the canonical k-mer set of seq[0, n_bytes).
//   flags != nullptr (bit array over the n_bytes positions, zeroed by the caller): bit p = 1 iff a kept k-mer occurs for the FIRST time in the
//                     window ending at p  (positions travel as the payload);
//   want_keys:        the kept keys (sorted) and their counts are left at the arena position current on entry.
//   shard != nullptr: level 0 is skipped, the construction resolves the level-0 buckets the shard gives (kc_kmerset_resolve).
// Everything else this function allocates is released before it returns.

template <int L, bool PAY, bool KEYS>
KmerSet<L> kc_kmerset_build_impl(CudaExec &ex, const u8 *seq, u64 n_bytes, int k, bool complements, int min_freq, u32 *flags,
                                 u64 *ext_kept_cell, KsShard *shard = nullptr, const u32 *win_mask = nullptr) {
    typedef KsCfg<L> Cfg;
    KmerSet<L> res;
    if (shard && (!PAY || KEYS)) KC_THROW(KC_ERR_INTERNAL, "sharded construction is FLAGS-only");
    if (shard ? shard->n_items == 0 : n_bytes == 0) return res;
    cudaStream_t st = ex.stream;
    const size_t base_mark = ex.arena->mark();
    const u32 cap = Cfg::CAP;
    const u64 n = shard ? shard->n_items : n_bytes;  // upper bound of M
    const u32 big_cap = (u32) (n / cap + 258);
    const u32 small_cap = (u32) (16 * (n / cap) + 4096);
    const u32 uniform_cap = big_cap;

    KWord<L> *out_keys = nullptr;
    u8 *out_cnt = nullptr;

    SortBucket *big_a = ex.alloc<SortBucket>(big_cap);
    SortBucket *big_b = ex.alloc<SortBucket>(big_cap);
    SortBucket *small = ex.alloc<SortBucket>(small_cap);
    SortBucket *uniform = ex.alloc<SortBucket>(uniform_cap);
    u32 *tile_count = ex.alloc<u32>(big_cap + 1);
    u32 *hist = ex.alloc<u32>((u64) big_cap * 256);
    u64 *cursor = ex.alloc<u64>((u64) big_cap * 256);
    u8 *skip = ex.alloc<u8>(big_cap);
    u32 *ctr = ex.alloc<u32>(8);
    u64 *cells = ex.alloc<u64>(2);  // [0] = M, [1] = kept distinct keys
    const u32 ex_blocks = shard ? 0u : (u32) kc_div_up(n_bytes, (u64) Cfg::EX_TILE);
    u16 *tile_hist = ex.alloc<u16>((u64) (ex_blocks ? ex_blocks : 1) * 256);
    ex.fill_bytes(ctr, 0, 32);
    ex.fill_bytes(cells, 0, 16);
    ex.fill_bytes(hist, 0, 256 * 4);

    constexpr bool SCRAMBLE = PAY && !KEYS;  // FLAGS-only: bucket by a bijective hash of the k-mer (see kmer_scramble)
    static KcDevOnce attr_once;  // function attributes are per device
    const int scatter0_smem = Cfg::EX_TILE * ((int) sizeof(KWord<L>) + (PAY ? 2 : 0));
    const int scatter_smem = Cfg::TILE * ((int) sizeof(KWord<L>) + (PAY ? 4 : 0) + 2);
    const int resolve_smem = Cfg::CAP * ((int) sizeof(KWord<L>) + (PAY ? 4 : 0) + 2);
    attr_once.run([&](int) {
        KC_CUDA(cudaFuncSetAttribute(kc_ks_scatter0_kernel<L, PAY, SCRAMBLE>, cudaFuncAttributeMaxDynamicSharedMemorySize, scatter0_smem));
        KC_CUDA(cudaFuncSetAttribute(kc_kv_scatter_kernel<L, PAY>, cudaFuncAttributeMaxDynamicSharedMemorySize, scatter_smem));
        KC_CUDA(cudaFuncSetAttribute(kc_ks_resolve_kernel<L, PAY, KEYS>, cudaFuncAttributeMaxDynamicSharedMemorySize, resolve_smem));
    });

    // ---- level 0 ----
    const int key_bits = SCRAMBLE ? 64 * L : 2 * k;
    const int bits0 = key_bits < Cfg::D0 ? key_bits : Cfg::D0;
    const int shift0 = key_bits - bits0;
    u32 h[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    u64 M = 0;
    KWord<L> *k0 = nullptr, *k1 = nullptr;
    u32 *p0 = nullptr, *p1 = nullptr;
    u8 *cnt_tmp = nullptr;
    if (!shard) {
        {
            CudaExec::Scope sc(ex, KP_KS_HIST0, n_bytes);
            kc_ks_hist0_kernel<L, SCRAMBLE><<<ex_blocks, Cfg::EX_THREADS, 0, st>>>(seq, n_bytes, k, complements ? 1 : 0, shift0, bits0, hist, tile_hist,
                                                                                   0u, win_mask);
        }
        ++ex.launches;
        kc_ks_scan0_kernel<<<1, 256, 0, st>>>(hist, cursor, big_a, big_cap, small, small_cap, uniform, uniform_cap, ctr, cells, cap, Cfg::TILE,
                                             key_bits - bits0);
        ++ex.launches;
        KC_CUDA(cudaGetLastError());
        KC_CUDA(cudaMemcpyAsync(h, ctr, 32, cudaMemcpyDeviceToHost, st));
        KC_CUDA(cudaMemcpyAsync(&M, cells, 8, cudaMemcpyDeviceToHost, st));
        KC_CUDA(cudaStreamSynchronize(st));
        res.n_occ = M;
        if (M == 0) {
            ex.arena->release(base_mark);
            return res;
        }
        if (h[3]) KC_THROW(KC_ERR_INTERNAL, "k-mer set bucket list overflow");
        if (M >= 0xFFFFFFF0ULL) KC_THROW(KC_ERR_TOO_LARGE, "more than 2^32 k-mer occurrences on one GPU");
    } else {
        M = shard->n_items;
        res.n_occ = M;
        if (M >= 0xFFFFFFF0ULL) KC_THROW(KC_ERR_TOO_LARGE, "more than 2^32 k-mer occurrences on one GPU");
        // the owner's level-0 buckets, delivered complete and contiguous by the peers' scatter passes
        std::vector<SortBucket> hs, hb, hu;
        for (u32 i = 0; i < shard->n_pre; ++i) {
            if (shard->pre_size[i] == 0) continue;
            SortBucket b;
            b.off = shard->pre_off[i];
            b.size = (u32) shard->pre_size[i];
            b.rem = (u16) (key_bits - bits0);
            b.parity = 0;
            b.bits = 0;
            if (b.size <= cap) {
                hs.push_back(b);
                if (b.size > 1024u) ++h[5];
            } else if (b.rem == 0) {
                hu.push_back(b);
            } else {
                hb.push_back(b);
                h[4] += (u32) kc_div_up(b.size, (u64) Cfg::TILE);
            }
        }
        h[0] = (u32) hb.size();
        h[1] = (u32) hs.size();
        h[2] = (u32) hu.size();
        if (h[0] > big_cap || h[1] > small_cap || h[2] > uniform_cap) KC_THROW(KC_ERR_INTERNAL, "k-mer set bucket list overflow");
        if (h[0]) KC_CUDA(cudaMemcpyAsync(big_a, hb.data(), hb.size() * sizeof(SortBucket), cudaMemcpyHostToDevice, st));
        if (h[1]) KC_CUDA(cudaMemcpyAsync(small, hs.data(), hs.size() * sizeof(SortBucket), cudaMemcpyHostToDevice, st));
        if (h[2]) KC_CUDA(cudaMemcpyAsync(uniform, hu.data(), hu.size() * sizeof(SortBucket), cudaMemcpyHostToDevice, st));
        u32 init[8] = {h[0], h[1], h[2], 0, h[4], h[5], 0, 0};
        KC_CUDA(cudaMemcpyAsync(ctr, init, 32, cudaMemcpyHostToDevice, st));
        KC_CUDA(cudaStreamSynchronize(st));  // the staging vectors live on this stack frame
    }
    // k1 is allocated last: the KEYS result is compacted into k1 and then copied down to base_mark, and everything
    // allocated before k1 (control arrays, k0, payloads, counts: > U * (8L + 1) bytes) separates the two regions.
    if (!shard) {
        k0 = ex.alloc<KWord<L>>(M);
        if (PAY) {
            p0 = ex.alloc<u32>(M);
            p1 = ex.alloc<u32>(M);
        }
        cnt_tmp = KEYS ? ex.alloc<u8>(M) : nullptr;
        k1 = ex.alloc<KWord<L>>(M);
    } else {
        k0 = reinterpret_cast<KWord<L> *>(shard->keys);
        p0 = shard->pos;
        k1 = ex.alloc<KWord<L>>(M);
        p1 = ex.alloc<u32>(M);
    }
    if (!shard) {
        {
            CudaExec::Scope sc(ex, KP_KS_SCATTER0, n_bytes + M * (sizeof(KWord<L>) + (PAY ? 4 : 0)));
            kc_ks_scatter0_kernel<L, PAY, SCRAMBLE><<<ex_blocks, Cfg::EX_THREADS, scatter0_smem, st>>>(seq, n_bytes, k, complements ? 1 : 0, shift0,
                                                                                                   bits0, cursor, tile_hist, k0, p0, 0u, nullptr,
                                                                                                   nullptr, win_mask);
        }
        ++ex.launches;
        KC_CUDA(cudaGetLastError());
    }

    // ---- levels >= 1 ----
    u32 nb = h[0], n_small = h[1], n_uniform = h[2], n_tiles = h[4], n_small_b = h[5];
    (void) n_small_b;
    SortBucket *cur = big_a, *nxt = big_b;
    const u32 max_ctas = 148 * 8;
    while (nb > 0) {
        kc_sort_prep_kernel<<<(unsigned) kc_div_up(nb, 256), 256, 0, st>>>(cur, nb, cap, Cfg::TILE, tile_count);
        ++ex.launches;
        ex.fill_bytes(tile_count + nb, 0, 4);
        ex.exclusive_scan_nosync(tile_count, tile_count, nb + 1);  // entry nb becomes the total = n_tiles
        ex.fill_bytes(hist, 0, (size_t) nb * 256 * 4);
        const u32 tiles_per_cta = (u32) kc_div_up(n_tiles, max_ctas);
        const u32 ctas = (u32) kc_div_up(n_tiles, tiles_per_cta);
        const u64 level_items = (u64) n_tiles * Cfg::TILE;  // items still in oversized buckets (rounded up to tiles)
        {
            CudaExec::Scope sc(ex, KP_SORT_HIST, level_items * sizeof(KWord<L>));
            kc_kv_hist_kernel<L><<<ctas, 256, 0, st>>>(k0, k1, cur, tile_count, nb, tiles_per_cta, hist);
        }
        ++ex.launches;
        ex.fill_bytes(ctr, 0, 4);       // next-level big counter
        ex.fill_bytes(ctr + 4, 0, 4);   // next-level tile counter
        kc_kv_scan_kernel<<<nb, 256, 0, st>>>(cur, hist, cursor, skip, nxt, big_cap, small, small_cap, uniform, uniform_cap, ctr, cap, Cfg::TILE);
        ++ex.launches;
        {
            CudaExec::Scope sc(ex, KP_SORT_SCATTER, 2 * level_items * (sizeof(KWord<L>) + (PAY ? 4 : 0)));
            kc_kv_scatter_kernel<L, PAY><<<ctas, 256, scatter_smem, st>>>(k0, k1, p0, p1, cur, tile_count, nb, tiles_per_cta, cursor, skip);
        }
        ++ex.launches;
        KC_CUDA(cudaGetLastError());
        KC_CUDA(cudaMemcpyAsync(h, ctr, 32, cudaMemcpyDeviceToHost, st));
        KC_CUDA(cudaStreamSynchronize(st));
        if (h[3]) KC_THROW(KC_ERR_INTERNAL, "k-mer set bucket list overflow");
        nb = h[0];
        n_small = h[1];
        n_uniform = h[2];
        n_tiles = h[4];
        n_small_b = h[5];
        SortBucket *t = cur;
        cur = nxt;
        nxt = t;
    }
    // ---- resolve ----
    // FLAGS-only callers may pass a cell of their own: the count is then left on the device (no read-back here)
    const bool defer_count = !KEYS && ext_kept_cell != nullptr;
    kc_ull *n_unique = reinterpret_cast<kc_ull *>(defer_count ? ext_kept_cell : cells + 1);
    if (n_small) {
        CudaExec::Scope sc(ex, KP_KS_RESOLVE, M * (sizeof(KWord<L>) + (PAY ? 4 : 0)) + (KEYS ? M * (sizeof(KWord<L>) + 1) : 0));
        if constexpr (PAY && !KEYS) {
            // hash resolve in two size classes (class A holds almost every bucket and runs at twice the occupancy)
            constexpr int CA = Cfg::CAP_A < Cfg::CAP ? Cfg::CAP_A : Cfg::CAP;
            const bool counted = min_freq > 1;
            const int per_item = (int) sizeof(KWord<L>) + 12 + 4;  // key + three table slots + position (+ count)
            const int smem_a = CA * (per_item + (counted ? 4 : 0));
            const int smem_b = Cfg::CAP * (per_item + (counted ? 4 : 0));
            // function attributes and occupancy are per device; persistent kernels: exactly as many CTAs as fit on the device
            static KcDevOnce hash_once;
            static int occ_tab[KC_MAX_DEVICES][4];
            const int dev_id = hash_once.run([&](int dv) {
                KC_CUDA(cudaFuncSetAttribute(kc_ks_resolve_hash_kernel<L, CA, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, CA * per_item));
                KC_CUDA(cudaFuncSetAttribute(kc_ks_resolve_hash_kernel<L, CA, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, CA * (per_item + 4)));
                KC_CUDA(cudaFuncSetAttribute(kc_ks_resolve_hash_kernel<L, Cfg::CAP, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::CAP * per_item));
                KC_CUDA(cudaFuncSetAttribute(kc_ks_resolve_hash_kernel<L, Cfg::CAP, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::CAP * (per_item + 4)));
                KC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_tab[dv][0], kc_ks_resolve_hash_kernel<L, CA, false>, 256, CA * per_item));
                KC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_tab[dv][1], kc_ks_resolve_hash_kernel<L, CA, true>, 256, CA * (per_item + 4)));
                KC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_tab[dv][2], kc_ks_resolve_hash_kernel<L, Cfg::CAP, false>, 256, Cfg::CAP * per_item));
                KC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_tab[dv][3], kc_ks_resolve_hash_kernel<L, Cfg::CAP, true>, 256, Cfg::CAP * (per_item + 4)));
            });
            const int n_sm = kc_sm_count(dev_id);
            const int *occ_a = &occ_tab[dev_id][0], *occ_b = &occ_tab[dev_id][2];
            const u32 fit_a = (u32) (n_sm * (occ_a[counted] > 0 ? occ_a[counted] : 1)), fit_b = (u32) (n_sm * (occ_b[counted] > 0 ? occ_b[counted] : 1));
            const u32 grid_a = n_small < fit_a ? n_small : fit_a;
            const u32 grid_b = n_small < fit_b ? n_small : fit_b;
            if (counted) kc_ks_resolve_hash_kernel<L, CA, true><<<grid_a, 256, smem_a, st>>>(k0, k1, p0, p1, small, n_small, 0u, (u32) CA, flags, (u32) min_freq, n_unique);
            else kc_ks_resolve_hash_kernel<L, CA, false><<<grid_a, 256, smem_a, st>>>(k0, k1, p0, p1, small, n_small, 0u, (u32) CA, flags, (u32) min_freq, n_unique);
            ++ex.launches;
            if (CA < Cfg::CAP && n_small_b) {
                if (counted) kc_ks_resolve_hash_kernel<L, Cfg::CAP, true><<<grid_b, 256, smem_b, st>>>(k0, k1, p0, p1, small, n_small, (u32) CA, (u32) Cfg::CAP, flags, (u32) min_freq, n_unique);
                else kc_ks_resolve_hash_kernel<L, Cfg::CAP, false><<<grid_b, 256, smem_b, st>>>(k0, k1, p0, p1, small, n_small, (u32) CA, (u32) Cfg::CAP, flags, (u32) min_freq, n_unique);
                ++ex.launches;
            }
        } else {
            kc_ks_resolve_kernel<L, PAY, KEYS><<<n_small, 256, resolve_smem, st>>>(k0, k1, p0, p1, small, flags, (u32) min_freq, n_unique, cnt_tmp);
            ++ex.launches;
        }
    }
    if (n_uniform) {
        kc_ks_uniform_kernel<L, PAY, KEYS><<<n_uniform, 256, 0, st>>>(k0, k1, p0, p1, uniform, flags, (u32) min_freq, n_unique, cnt_tmp);
        ++ex.launches;
    }
    KC_CUDA(cudaGetLastError());
    const u64 U = defer_count ? ~0ULL : ex.read(cells + 1);
    res.n_kept = U;
    if (KEYS && U) {
        // compact the kept keys into k1 (free by now), then down to the arena position current on entry
        const KWord<L> *srck = k0;
        const u8 *cs = cnt_tmp;
        const u32 need = (u32) (min_freq - 1);
        KWord<L> *ck = k1;
        u8 *cc_dst = PAY ? reinterpret_cast<u8 *>(p1) : ex.alloc<u8>(U);  // the payload buffers are dead by now
        const u64 got = ex.compact_if(
            M, [=] __device__(u64 i) { return srck[i].w[L - 1] != ~0ULL && (u32) cs[i] >= need; },
            [=] __device__(u64 i, u32 r) {
                ck[r] = srck[i];
                cc_dst[r] = cs[i];
            },
            M * (sizeof(KWord<L>) + 1) + U * (sizeof(KWord<L>) + 1));
        if (got != U) KC_THROW(KC_ERR_INTERNAL, "k-mer set compaction disagrees with the resolve count");
        // move to the front of this call's arena region; everything below k1 is dead now
        ex.arena->release(base_mark);
        out_keys = ex.alloc<KWord<L>>(U);
        out_cnt = ex.alloc<u8>(U);
        if ((char *) (out_cnt + U) > (char *) ck || (char *) (out_cnt + U) > (char *) cc_dst)
            KC_THROW(KC_ERR_INTERNAL, "k-mer set result would overlap its source");
        ex.copy_bytes(out_keys, ck, U * sizeof(KWord<L>));
        ex.copy_bytes(out_cnt, cc_dst, U);
        res.keys = out_keys;
        res.cnt = out_cnt;
    } else {
        ex.arena->release(base_mark);
    }
    return res;
}

template <int L>
KmerSet<L> kc_kmerset_build(CudaExec &ex, const u8 *seq, u64 n_bytes, int k, bool complements, int min_freq, u32 *flags, bool want_keys,
                            u64 *ext_kept_cell = nullptr, const u32 *win_mask = nullptr) {
    if (win_mask) {  // maskopt: the set of the k-mers whose window passes the filter, keys only
        if (flags || !want_keys) KC_THROW(KC_ERR_INTERNAL, "window filter is KEYS-only");
        return kc_kmerset_build_impl<L, false, true>(ex, seq, n_bytes, k, complements, min_freq, nullptr, nullptr, nullptr, win_mask);
    }
    if (flags) {
        if (want_keys) return kc_kmerset_build_impl<L, true, true>(ex, seq, n_bytes, k, complements, min_freq, flags, nullptr);
        return kc_kmerset_build_impl<L, true, false>(ex, seq, n_bytes, k, complements, min_freq, flags, ext_kept_cell);
    }
    return kc_kmerset_build_impl<L, false, true>(ex, seq, n_bytes, k, complements, min_freq, nullptr, nullptr);
}

// Fused partition + exchange, phase A: histogram pass over the slice (tile counts are kept in shard->tile_hist_keep).
template <int L> u64 kc_kmerset_hist_only(CudaExec &ex, const u8 *seq, u64 n_bytes, int k, bool complements, KsShard *sh) {
    typedef KsCfg<L> Cfg;
    for (int i = 0; i < 256; ++i) sh->host_hist[i] = 0;
    if (sh->pos_end <= sh->pos_begin) return 0;
    if (sh->pos_begin % Cfg::EX_TILE != 0 || (sh->pos_end % Cfg::EX_TILE != 0 && sh->pos_end != n_bytes) || sh->pos_end > n_bytes)
        KC_THROW(KC_ERR_ARG, "shard boundaries must be multiples of the extraction tile");
    const size_t mark = ex.arena->mark();
    u32 *hist = ex.alloc<u32>(256);
    ex.fill_bytes(hist, 0, 1024);
    const u32 blocks = (u32) kc_div_up(sh->pos_end - sh->pos_begin, (u64) Cfg::EX_TILE);
    {
        CudaExec::Scope sc(ex, KP_KS_HIST0, sh->pos_end - sh->pos_begin);
        kc_ks_hist0_kernel<L, true><<<blocks, Cfg::EX_THREADS, 0, ex.stream>>>(seq, n_bytes, k, complements ? 1 : 0, 64 * L - Cfg::D0, Cfg::D0, hist,
                                                                            sh->tile_hist_keep, (u32) (sh->pos_begin / Cfg::EX_TILE));
    }
    ++ex.launches;
    KC_CUDA(cudaGetLastError());
    ex.read_n(hist, sh->host_hist, 256);
    ex.arena->release(mark);
    u64 m = 0;
    for (int i = 0; i < 256; ++i) m += sh->host_hist[i];
    return m;
}

// Phase B: scatter pass through the peer tables (see kc_ks_scatter0_kernel, P2P = true).  n_items = this rank's items.
template <int L> void kc_kmerset_scatter_p2p(CudaExec &ex, const u8 *seq, u64 n_bytes, int k, bool complements, u64 n_items, KsShard *sh) {
    typedef KsCfg<L> Cfg;
    if (sh->pos_end <= sh->pos_begin) return;
    const size_t mark = ex.arena->mark();
    u64 *cursor = ex.alloc<u64>(256);
    KC_CUDA(cudaMemcpyAsync(cursor, sh->cursor0, 256 * 8, cudaMemcpyHostToDevice, ex.stream));
    const int smem = Cfg::EX_TILE * ((int) sizeof(KWord<L>) + 2);
    static KcDevOnce attr_once;
    attr_once.run([&](int) { KC_CUDA(cudaFuncSetAttribute(kc_ks_scatter0_kernel<L, true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)); });
    const u32 blocks = (u32) kc_div_up(sh->pos_end - sh->pos_begin, (u64) Cfg::EX_TILE);
    {
        CudaExec::Scope sc(ex, KP_KS_SCATTER0, (sh->pos_end - sh->pos_begin) + n_items * (sizeof(KWord<L>) + 4));
        kc_ks_scatter0_kernel<L, true, true, true><<<blocks, Cfg::EX_THREADS, smem, ex.stream>>>(
            seq, n_bytes, k, complements ? 1 : 0, 64 * L - Cfg::D0, Cfg::D0, cursor, sh->tile_hist_keep, nullptr, nullptr,
            (u32) (sh->pos_begin / Cfg::EX_TILE), reinterpret_cast<KWord<L> *const *>(sh->dst_k), sh->dst_p);
    }
    ++ex.launches;
    KC_CUDA(cudaGetLastError());
    KC_CUDA(cudaStreamSynchronize(ex.stream));  // cursor0 is a host stack array of the caller; peers wait on this kernel
    ex.arena->release(mark);
}

// Phase C, on the owner: levels >= 1 and the resolve over the level-0 buckets delivered by phase B (FLAGS-only).
template <int L> u64 kc_kmerset_resolve(CudaExec &ex, int k, int min_freq, u32 *flags, KsShard *shard) {
    return kc_kmerset_build_impl<L, true, false>(ex, nullptr, 0, k, true, min_freq, flags, nullptr, shard).n_kept;
}

#endif  // __CUDACC__
