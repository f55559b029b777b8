// Two neighbours of the compute path that reuse its k-mer set machinery (SURVEY.md §8f rows 3 and 4):
//
//   streaming  `compute -a streaming` (reference src/streaming.h:12-48 Streaming): one pass over the input in file order;
//              a window whose (canonical) k-mer has not been seen before prints its first character in upper case, and a
//              character at most k-1 positions after the latest such window prints in lower case; every other character
//              is dropped.  "Not seen before" is exactly the first-occurrence bit array the from-FASTA compute path builds
//              (kmerset_sig.cuh / kmerset_fast.cuh / kmerset.cuh), so streaming = that construction + one stream compaction.
//
//   maskopt    `maskopt -t max-one | min-one` (reference src/masks.h:40-78 OptimizeOnes, 240-261 Optimize): the set S is the
//              canonical k-mers of the windows that START with an upper-case letter (src/parser.h:41-42 case_sensitive);
//              max-one turns ON every window whose k-mer is in S, min-one only the first such window of each k-mer
//              (the reference erases the k-mer from the hash set once it has been printed ON).  Here: S = the sorted-keys
//              construction over the windows passing a bit filter; "first window of each k-mer" = first-occurrence bits;
//              the hash probe = a binary search in S.
#pragma once
#include "emit.cuh"
#include "kmerset_fast.cuh"
#include "runs.cuh"
#include "set_routes.cuh"

#ifdef __CUDACC__

// 32 START-indexed first-occurrence bits: bit i <=> the window STARTING at 32 * w + i is flagged (flags are END-indexed).
KC_D u32 kc_start_flag_word(const u32 *__restrict__ flags, u64 n_flag_words, i64 w, int k) {
    if (w < 0) return 0u;
    const u64 a = (u64) w + (u64) ((k - 1) >> 5);
    const u32 sh = (u32) (k - 1) & 31u;
    const u32 lo = a < n_flag_words ? flags[a] : 0u;
    const u32 hi = a + 1 < n_flag_words ? flags[a + 1] : 0u;
    return __funnelshift_r(lo, hi, sh);
}

// keep / upper masks of the 32 characters of word w (src/streaming.h:36-42: `lastOne` = latest flagged window).
KC_D void kc_streaming_masks(const u32 *__restrict__ flags, u64 n_flag_words, u64 w, int k, u32 &keep, u32 &upper) {
    upper = kc_start_flag_word(flags, n_flag_words, (i64) w, k);
    // distance from position 32 w - 1 back to the latest flagged start (k or more = out of reach)
    u32 gap = (u32) k;
    const int back = (k - 1 + 31) >> 5;
    for (int b = 1; b <= back; ++b) {
        const u32 pw = kc_start_flag_word(flags, n_flag_words, (i64) w - b, k);
        if (pw) {
            gap = (u32) (32 * (b - 1)) + (u32) __clz(pw);  // highest set bit 31 - clz  ->  distance (31 - bit) + 32 (b - 1)
            break;
        }
    }
    keep = 0;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
        if ((upper >> j) & 1u) gap = 0;
        else if (gap < (u32) k) ++gap;
        if (gap < (u32) k) keep |= 1u << j;  // gap <= k - 1
    }
}

__global__ void __launch_bounds__(256) kc_streaming_count_kernel(const u32 *__restrict__ flags, u64 n_flag_words, u64 n_words, int k,
                                                                 u32 *block_counts) {
    __shared__ u32 sw[8];
    const u64 w = (u64) blockIdx.x * 256 + threadIdx.x;
    u32 c = 0;
    if (w < n_words) {
        u32 keep, upper;
        kc_streaming_masks(flags, n_flag_words, w, k, keep, upper);
        c = __popc(keep);
    }
    u32 total;
    kc_block_exclusive_scan<256>(c, &total, sw);
    if (threadIdx.x == 0) block_counts[blockIdx.x] = total;
}

// Exclusive scan of the per-block counts into 64-bit offsets, out[n] = the total: the kept characters of an input of 2^32 bytes or more
// can number 2^32 and more.  One CTA walks the counts with a running carry, as kc_scan_walk_kernel does (a tile of 1024 counts of at
// most 8192 each sums within 32 bits).
__global__ void __launch_bounds__(256) kc_streaming_offsets_kernel(const u32 *__restrict__ counts, u64 n, u64 *__restrict__ out) {
    __shared__ u32 sw[8];
    u64 carry = 0;
    for (u64 t0 = 0; t0 < n; t0 += 1024) {
        const u64 base = t0 + (u64) threadIdx.x * 4;
        u32 v[4], c = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            v[j] = base + j < n ? counts[base + j] : 0u;
            c += v[j];
        }
        u32 total;
        u64 q = carry + kc_block_exclusive_scan<256>(c, &total, sw);  // ends with a barrier: sw is free for the next tile
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (base + j < n) out[base + j] = q;
            q += v[j];
        }
        carry += total;
    }
    if (threadIdx.x == 0) out[n] = carry;
}

// The kept characters of the block go through shared memory so that the stores to `out` are contiguous.
__global__ void __launch_bounds__(256) kc_streaming_emit_kernel(const u8 *__restrict__ seq, const u32 *__restrict__ flags, u64 n_flag_words,
                                                                u64 n_words, int k, const u64 *__restrict__ block_offsets, u8 *__restrict__ out) {
    __shared__ u32 sw[8];
    __shared__ u8 stage[256 * 32];
    const u64 w = (u64) blockIdx.x * 256 + threadIdx.x;
    u32 keep = 0, upper = 0;
    if (w < n_words) kc_streaming_masks(flags, n_flag_words, w, k, keep, upper);
    u32 total;
    u32 at = kc_block_exclusive_scan<256>(__popc(keep), &total, sw);
    if (keep) {
        const uint4 *src = reinterpret_cast<const uint4 *>(seq + w * 32);  // the sequence buffer is padded to whole words
        const uint4 a = src[0], b = src[1];
        const u32 wd[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
        for (int j = 0; j < 32; ++j) {
            if ((keep >> j) & 1u) {
                const u8 c = (u8) (wd[j >> 2] >> (8 * (j & 3)));
                stage[at++] = ((upper >> j) & 1u) ? (u8) (c & 0xDFu) : (u8) (c | 0x20u);  // src/kmers.h:124-127 Masked
            }
        }
    }
    __syncthreads();
    const u64 base = block_offsets[blockIdx.x];
    for (u32 i = threadIdx.x; i < total; i += 256) out[base + i] = stage[i];
}

struct StreamingResult {
    u8 *ms = nullptr;
    u64 length = 0, n_kept = 0, n_occ = 0;
};

// seq: the framed records, resident in a buffer padded with '\n' up to a multiple of 32 bytes (+ 32).  The constructions each pass
// tries are those of kc_set_ladder (set_routes.cuh).
template <int L>
StreamingResult kc_streaming_run(CudaExec &ex, const u8 *seq, u64 n_bytes, int k, bool complements, int min_freq, SetRoutes &routes) {
    StreamingResult res;
    const size_t fwords = kc_runs_flag_words(n_bytes);
    u32 *flags = ex.arena->alloc_top<u32>(fwords);
    ex.fill_bytes(flags, 0, fwords * 4);
    u64 *cells4 = ex.arena->alloc_top<u64>(4);  // {kept, -, M, overflow status}
    ex.fill_bytes(cells4, 0, 32);
    u64 hc[4] = {0, 0, 0, 0};
    const u32 *win_mask = nullptr;
    auto launch = [&](KcRoute r) {
        return r == KC_ROUTE_SIG ? kc_kmerset_build_sig<L>(ex, seq, n_bytes, k, complements, flags, cells4, routes.sig, nullptr, win_mask)
                                 : kc_kmerset_build_fast<L>(ex, seq, n_bytes, k, complements, 1, flags, cells4, routes.fast);
    };
    auto consume = [&](KcRoute) {
        ex.read_n(cells4, hc, 4);
        if (hc[3] == 0) return true;
        ex.fill_bytes(flags, 0, fwords * 4);
        ex.fill_bytes(cells4, 0, 32);
        return false;
    };
    RoutePolicy pol;
    pol.sig = true;
    pol.fast = min_freq == 1;
    const KcRoute route = kc_set_ladder(routes, pol, n_bytes, *ex.arena, launch, consume);
    if (route != KC_ROUTE_NONE) {
        res.n_kept = hc[2] ? hc[0] : 0;
        res.n_occ = hc[2];
    } else {
        KmerSet<L> set = kc_kmerset_build<L>(ex, seq, n_bytes, k, complements, 1, flags, false, cells4);
        res.n_occ = set.n_occ;
        res.n_kept = set.n_occ ? ex.read(cells4) : 0;
    }
    // -z Z (src/streaming.h:51-107 StreamingFiltered): the window that brings a k-mer's count to Z is ON, i.e. its Z-th
    // occurrence in file order.  Pass t = 2..Z repeats the first-occurrence construction over the windows that were not
    // flagged by the passes before it (window filter of the level-0 kernels): what it flags is every k-mer's t-th occurrence.
    if (min_freq > 1 && res.n_kept) {
        // whole tiles of the signature scan (256 strips); the extraction tiles of the other constructions divide them
        const u64 mwords = kc_div_up(n_bytes, (u64) 256 * KC_EX_STRIP) * 256 + 1;
        u32 *avail = ex.arena->alloc_top<u32>(mwords);
        ex.fill_bytes(avail, 0xFF, mwords * 4);
        win_mask = avail;
        pol.sig = route == KC_ROUTE_SIG;
        pol.fast = false;
        for (int t = 2; t <= min_freq && res.n_kept; ++t) {
            const u32 *f = flags;
            const u64 fw = fwords;
            ex.for_each(mwords, [=] __device__(u64 w) {
                if (w < fw) avail[w] &= ~f[w];
            }, KP_MISC, mwords * 12);
            ex.fill_bytes(flags, 0, fwords * 4);
            ex.fill_bytes(cells4, 0, 32);
            if (kc_set_ladder(routes, pol, n_bytes, *ex.arena, launch, consume) == KC_ROUTE_SIG) {
                res.n_kept = hc[2] ? hc[0] : 0;
                continue;
            }
            KmerSet<L> set = kc_kmerset_build_impl<L, true, false>(ex, seq, n_bytes, k, complements, 1, flags, cells4, nullptr, avail);
            res.n_kept = set.n_occ ? ex.read(cells4) : 0;
        }
    }
    if (res.n_kept == 0) return res;
    const u64 n_words = kc_div_up(n_bytes, 32);
    const u32 blocks = (u32) kc_div_up(n_words, 256);
    u32 *counts = ex.alloc<u32>(blocks);
    {
        CudaExec::Scope sc(ex, KP_RUNS, n_bytes / 8);
        kc_streaming_count_kernel<<<blocks, 256, 0, ex.stream>>>(flags, fwords, n_words, k, counts);
        ++ex.launches;
        KC_CUDA(cudaGetLastError());
    }
    // per-block counts are at most 8192, their running sum is bounded by n_bytes: 64-bit offsets
    u64 *offsets = ex.alloc<u64>((u64) blocks + 1);
    {
        CudaExec::Scope sc(ex, KP_SCAN, (u64) blocks * 12);
        kc_streaming_offsets_kernel<<<1, 256, 0, ex.stream>>>(counts, blocks, offsets);
        ++ex.launches;
        KC_CUDA(cudaGetLastError());
    }
    const u64 total = ex.read(offsets + blocks);
    u8 *out = ex.alloc<u8>(total + 1);
    {
        CudaExec::Scope sc(ex, KP_EMIT, n_bytes + n_bytes / 8 + total);
        kc_streaming_emit_kernel<<<blocks, 256, 0, ex.stream>>>(seq, flags, fwords, n_words, k, offsets, out);
        ++ex.launches;
        KC_CUDA(cudaGetLastError());
    }
    res.ms = out;
    res.length = total;
    return res;
}

struct MaskoptResult {
    u8 *ms = nullptr;
    u64 length = 0, n_kmers = 0;
};

// seq: the superstring (one record) followed by '\n'; len = its length without the '\n'.
template <int L>
MaskoptResult kc_maskopt_run(CudaExec &ex, const u8 *seq, u64 len, int k, bool complements, bool minimize) {
    typedef KsCfg<L> Cfg;
    MaskoptResult res;
    res.length = len;
    u8 *out = ex.arena->alloc_top<u8>(len + 1);
    res.ms = out;
    u32 *err = ex.arena->alloc_top<u32>(2);  // [0] invalid character seen
    ex.fill_bytes(err, 0, 8);
    // src/masks.h:49,74-76: only ACGTacgt may appear (the reference throws after printing; here nothing is printed)
    ex.for_each(len, [=] __device__(u64 p) {
        if (kc_nucleotide_code(seq[p]) > 3) err[0] = 1;
    }, KP_MISC, len);
    if (ex.read(err)) KC_THROW(KC_ERR_BAD_SEQ, "Masked superstring contains invalid characters.");
    if (len < (u64) k) {  // no window at all: everything is part of the trailing k-1 characters
        ex.for_each(len, [=] __device__(u64 p) { out[p] = (u8) (seq[p] | 0x20u); });
        return res;
    }
    const u64 n_bytes = len + 1;
    // window filter over END positions: the window's first character is upper case (src/parser.h:41-42)
    const u64 tiles = kc_div_up(n_bytes, (u64) Cfg::EX_TILE);
    const u64 mwords = tiles * (Cfg::EX_TILE / 32) + 1;
    u32 *win_mask = ex.arena->alloc_top<u32>(mwords);
    ex.for_each(mwords, [=] __device__(u64 w) {
        u32 m = 0;
        for (int i = 0; i < 32; ++i) {
            const u64 p = w * 32 + i;
            if (p + 1 >= (u64) k && p < len && seq[p + 1 - k] <= 'Z') m |= 1u << i;
        }
        win_mask[w] = m;
    }, KP_MISC, len + len / 8);
    u32 *flags = nullptr;
    const size_t fwords = kc_runs_flag_words(n_bytes);
    if (minimize) {
        flags = ex.arena->alloc_top<u32>(fwords);
        ex.fill_bytes(flags, 0, fwords * 4);
    }
    KmerSet<L> set = kc_kmerset_build<L>(ex, seq, n_bytes, k, complements, 1, nullptr, true, nullptr, win_mask);
    res.n_kmers = set.n_kept;
    if (minimize && set.n_kept) {
        u64 *cell = ex.alloc<u64>(1);
        ex.fill_bytes(cell, 0, 8);
        kc_kmerset_build<L>(ex, seq, n_bytes, k, complements, 1, flags, false, cell);
    }
    const KWord<L> *keys = set.keys;
    const u64 n_set = set.n_kept;
    const KmerIndex<L> ix = kc_kmer_index_build<L>(ex, keys, n_set, k);
    // One thread per 32 consecutive window starts: the k-mer rolls from window to window (src/masks.h:50-54), the hash probe of
    // src/masks.h:57-58 is an indexed search in the sorted set, the 32 output letters leave as two 16-byte stores.
    const int top = 2 * (k - 1);
    const int top_limb = top >> 6, top_off = top & 63;
    ex.for_each(kc_div_up(len, 32), [=] __device__(u64 t) {
        const u64 q0 = t * 32;
        const KWord<L> mask = KWord<L>::low_mask(2 * k);
        KWord<L> fwd = KWord<L>::zero(), rc = KWord<L>::zero();
        for (int i = 0; i + 1 < k; ++i) {
            const u64 c = q0 + i < len ? (kc_nucleotide_code(seq[q0 + i]) & 3u) : 0u;
            fwd = fwd.shl(2);
            fwd.w[0] |= c;
            rc = rc.shr(2);
#pragma unroll
            for (int l = 0; l < L; ++l)
                if (l == top_limb) rc.w[l] |= (3 ^ c) << top_off;
        }
        u32 wd[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        for (int j = 0; j < 32; ++j) {
            const u64 q = q0 + j;
            if (q >= len) break;
            const u64 e = q + k - 1;  // END position of the window
            bool on = false;
            if (e < len) {
                const u64 c = kc_nucleotide_code(seq[e]) & 3u;
                fwd = fwd.shl(2);
                fwd.w[0] |= c;
                fwd = fwd & mask;
                rc = rc.shr(2);
#pragma unroll
                for (int l = 0; l < L; ++l)
                    if (l == top_limb) rc.w[l] |= (3 ^ c) << top_off;
                if (n_set && (!minimize || ((flags[e >> 5] >> (e & 31)) & 1u))) {
                    const KWord<L> x = (!complements || fwd < rc) ? fwd : rc;
                    on = kmer_set_contains(keys, n_set, ix, x);
                }
            }
            const u32 ch = seq[q];
            wd[j >> 2] |= (on ? (ch & 0xDFu) : (ch | 0x20u)) << (8 * (j & 3));
        }
        if (q0 + 32 <= len) {
            uint4 *dst = reinterpret_cast<uint4 *>(out + q0);  // `out` is 256-byte aligned (arena), q0 a multiple of 32
            dst[0] = make_uint4(wd[0], wd[1], wd[2], wd[3]);
            dst[1] = make_uint4(wd[4], wd[5], wd[6], wd[7]);
        } else {
            for (u64 q = q0; q < len; ++q) out[q] = (u8) (wd[(q - q0) >> 2] >> (8 * ((q - q0) & 3)));
        }
    }, KP_MAXONE, 2 * len + n_set * sizeof(KWord<L>));
    return res;
}

#endif  // __CUDACC__
