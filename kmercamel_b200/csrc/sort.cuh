// Key-only radix sort of fixed-width words.
//
// This is what stands in for khash's probes on the GPU (reference src/khash.h, src/khash_utils.h): every hash-map probe
// of the reference (src/global.h:73-93) becomes a sort-join over (key, node) tuples packed into one word.
//
// Algorithm: most-significant-digit radix partitioning in global memory until a bucket fits in shared memory,
// then one CTA sorts the bucket in shared memory.
//   * a level = histogram kernel + tiny per-bucket scan kernel + scatter kernel over all buckets still larger
//     than CAP; the digit width of a bucket adapts to its size (1..8 bits) so children land near CAP/4;
//   * scatter is unstable on purpose (keys carry no payload; tuples are made unique by their node id), so
//     output slots are reserved with one global atomicAdd per (tile, digit) and no cross-tile prefix is needed;
//   * a bucket whose items all share the digit is not moved at all, it just descends; a bucket that runs out
//     of key bits holds one distinct key and is emitted as such (this bounds the cost of poly-A style repeats).
// HBM traffic per level is one read (histogram) + one read + one write (scatter) of the participating items.
#pragma once
#include "exec.cuh"
#include "kword.cuh"

struct SortBucket {
    u64 off;
    u32 size;
    u16 rem;    // number of low key bits not partitioned yet
    u8 parity;  // which of the two ping-pong buffers holds the bucket
    u8 bits;    // digit width used when this bucket is partitioned
};

template <int L> struct SortCfg {
    // shared-memory sort capacity (power of two) and scatter tile, sized for 32-64 KB of shared memory
    static constexpr int CAP = L == 1 ? 8192 : (L == 2 ? 4096 : (L <= 4 ? 2048 : 1024));
    static constexpr int TILE = L == 1 ? 4096 : (L == 2 ? 2048 : 1024);
    static constexpr int THREADS = 256;
};

#ifdef __CUDACC__

KC_D u32 kc_upper_bound_u32(const u32 *a, u32 n, u32 v) {  // first index with a[i] > v
    u32 lo = 0, hi = n;
    while (lo < hi) {
        u32 mid = (lo + hi) >> 1;
        if (a[mid] <= v) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

__global__ void kc_sort_root_kernel(SortBucket *dst, SortBucket root) { *dst = root; }

__global__ void kc_sort_prep_kernel(SortBucket *big, u32 nb, u32 cap, u32 tile, u32 *tile_count) {
    u32 b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nb) return;
    SortBucket d = big[b];
    u32 want = (u32) kc_div_up(d.size, cap / 4);
    int bits = 1;
    while ((1u << bits) < want && bits < 8) ++bits;
    if (bits > d.rem) bits = d.rem;
    d.bits = (u8) bits;
    big[b] = d;
    tile_count[b] = (u32) kc_div_up(d.size, tile);
}

template <int L>
__global__ void __launch_bounds__(256) kc_sort_hist_kernel(const KWord<L> *buf0, const KWord<L> *buf1, const SortBucket *big,
                                                           const u32 *tile_prefix, u32 nb, u32 n_tiles, u32 tiles_per_cta,
                                                           u32 *hist) {
    constexpr int TILE = SortCfg<L>::TILE;
    __shared__ u32 sh[256];
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
        SortBucket d = big[b];
        const KWord<L> *src = (d.parity ? buf1 : buf0) + d.off;
        u32 ti = t - tile_prefix[b];
        u32 start = ti * TILE;
        u32 cnt = min((u32) TILE, d.size - start);
        int shift = d.rem - d.bits;
        for (u32 i = threadIdx.x; i < cnt; i += 256) {
            KWord<L> key = src[start + i];
            atomicAdd(&sh[key.digit(shift, d.bits)], 1u);
        }
    }
    __syncthreads();
    if (sh[threadIdx.x]) atomicAdd(&hist[(u64) cur * 256 + threadIdx.x], sh[threadIdx.x]);
}

// One CTA per partitioned bucket: turn its 256 digit counts into child offsets and classify the children.
// ctr[0] = next-level big count, ctr[1] = small count, ctr[2] = uniform count, ctr[3] = overflow flag.
__global__ void __launch_bounds__(256) kc_sort_scan_kernel(const SortBucket *big, const u32 *hist, u64 *cursor, u8 *skip,
                                                           SortBucket *next_big, u32 next_cap, SortBucket *small,
                                                           u32 small_cap, SortBucket *uniform, u32 uniform_cap, u32 *ctr,
                                                           u32 cap) {
    __shared__ u32 sw[8];
    u32 b = blockIdx.x;
    SortBucket d = big[b];
    u32 c = hist[(u64) b * 256 + threadIdx.x];
    u32 total;
    u32 p = kc_block_exclusive_scan_256(c, &total, sw);
    cursor[(u64) b * 256 + threadIdx.x] = d.off + p;
    bool single = (c == d.size);  // every item has this digit: nothing needs to move
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
    } else if (ch.rem == 0) {
        u32 s = atomicAdd(&ctr[2], 1u);
        if (s < uniform_cap) uniform[s] = ch;
        else ctr[3] = 1;
    } else {
        u32 s = atomicAdd(&ctr[0], 1u);
        if (s < next_cap) next_big[s] = ch;
        else ctr[3] = 1;
    }
}

template <int L>
__global__ void __launch_bounds__(256) kc_sort_scatter_kernel(KWord<L> *buf0, KWord<L> *buf1, const SortBucket *big,
                                                              const u32 *tile_prefix, u32 nb, u32 n_tiles, u32 tiles_per_cta,
                                                              u64 *cursor, const u8 *skip) {
    constexpr int TILE = SortCfg<L>::TILE;
    constexpr int ITEMS = TILE / 256;
    extern __shared__ __align__(16) unsigned char kc_smem_raw[];
    KWord<L> *stage = reinterpret_cast<KWord<L> *>(kc_smem_raw);
    __shared__ u32 cnt[256];
    __shared__ u32 loff[256];
    __shared__ u64 gbase[256];
    __shared__ u32 sw[8];
    u32 t0 = blockIdx.x * tiles_per_cta;
    u32 t1 = min(n_tiles, t0 + tiles_per_cta);
    if (t0 >= t1) return;
    u32 b = kc_upper_bound_u32(tile_prefix, nb + 1, t0) - 1;
    cnt[threadIdx.x] = 0;
    __syncthreads();
    for (u32 t = t0; t < t1; ++t) {
        while (t >= tile_prefix[b + 1]) ++b;
        if (skip[b]) continue;
        SortBucket d = big[b];
        const KWord<L> *src = (d.parity ? buf1 : buf0) + d.off;
        KWord<L> *dst = d.parity ? buf0 : buf1;
        u32 ti = t - tile_prefix[b];
        u32 start = ti * TILE;
        u32 n_here = min((u32) TILE, d.size - start);
        int shift = d.rem - d.bits;
        KWord<L> item[ITEMS];
        u32 rank[ITEMS];
#pragma unroll
        for (int j = 0; j < ITEMS; ++j) {
            u32 i = threadIdx.x + j * 256;
            if (i < n_here) {
                item[j] = src[start + i];
                rank[j] = atomicAdd(&cnt[item[j].digit(shift, d.bits)], 1u);
            }
        }
        __syncthreads();
        u32 c = cnt[threadIdx.x];
        u32 total;
        u32 p = kc_block_exclusive_scan_256(c, &total, sw);
        loff[threadIdx.x] = p;
        if (c) gbase[threadIdx.x] = atomicAdd((kc_ull *) &cursor[(u64) b * 256 + threadIdx.x], (kc_ull) c);
        cnt[threadIdx.x] = 0;
        __syncthreads();
#pragma unroll
        for (int j = 0; j < ITEMS; ++j) {
            u32 i = threadIdx.x + j * 256;
            if (i < n_here) stage[loff[item[j].digit(shift, d.bits)] + rank[j]] = item[j];
        }
        __syncthreads();
        for (u32 q = threadIdx.x; q < n_here; q += 256) {
            KWord<L> v = stage[q];
            u32 dg = v.digit(shift, d.bits);
            dst[gbase[dg] + (q - loff[dg])] = v;
        }
        __syncthreads();
    }
}

// Cooperative bitonic sort of the shared-memory segment seg[0..m) by the whole CTA (any m: pairs whose partner
// index is >= m are skipped, which is exact because every compare-exchange moves the larger word up).
template <int L> KC_D void kc_block_bitonic(KWord<L> *seg, u32 m, u32 nthreads = 256) {
    u32 P = 2;
    while (P < m) P <<= 1;
    for (u32 k = 2; k <= P; k <<= 1) {
        for (u32 j = k >> 1; j > 0; j >>= 1) {
            for (u32 t = threadIdx.x; t < (P >> 1); t += nthreads) {
                u32 i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                u32 l = (j == (k >> 1)) ? (i ^ (k - 1)) : (i | j);  // first step of a merge mirrors, the rest are strides
                if (l < m && i < m) {
                    KWord<L> a = seg[i], c = seg[l];
                    if (c < a) {
                        seg[i] = c;
                        seg[l] = a;
                    }
                }
            }
            __syncthreads();
        }
    }
}

// One CTA per bucket of at most CAP items.
//   1. items go global -> registers; each takes a slot in a shared-memory counting sort on its next <= 11 key bits
//      (one shared atomicAdd per item gives digit count and rank at once; order inside a digit is irrelevant);
//   2. after a block scan of the digit counts the items are scattered into shared memory: they are now sorted
//      except inside sub-buckets, which for k-mer data hold ~1 distinct key (plus its duplicates);
//   3. sub-buckets of up to KC_SUB_SMALL items are finished by one thread each (insertion sort in shared memory),
//      the rare larger ones by the whole CTA with a bitonic network.
// ~10 shared-memory touches per item instead of ~110 for a full bitonic sort.
static const u32 KC_SUB_SMALL = 24;
static const int KC_SUB_BITS_MAX = 11;

template <int L>
__global__ void __launch_bounds__(256) kc_sort_local_kernel(KWord<L> *buf0, const KWord<L> *buf1, const SortBucket *small) {
    constexpr int CAP = SortCfg<L>::CAP;
    constexpr int ITEMS = CAP / 256;
    extern __shared__ __align__(16) unsigned char kc_smem_raw[];
    KWord<L> *s = reinterpret_cast<KWord<L> *>(kc_smem_raw);
    __shared__ u32 sub_cnt[1 << KC_SUB_BITS_MAX];              // digit counts, then exclusive starts
    __shared__ u32 big_list[64];
    __shared__ u32 n_big;
    __shared__ u32 sw[8];
    SortBucket d = small[blockIdx.x];
    const KWord<L> *src = (d.parity ? buf1 : buf0) + d.off;
    KWord<L> *dst = buf0 + d.off;
    const u32 size = d.size;
    if (size == 1) {
        if (threadIdx.x == 0) dst[0] = src[0];
        return;
    }
    // digit width: about two sub-buckets per item, bounded by the key bits that are left
    int bits = 1;
    while ((1u << bits) < 2 * size && bits < KC_SUB_BITS_MAX) ++bits;
    if (bits > (int) d.rem) bits = d.rem;
    const u32 n_sub = 1u << bits;
    const int shift = d.rem - bits;
    for (u32 i = threadIdx.x; i < n_sub; i += 256) sub_cnt[i] = 0;
    if (threadIdx.x == 0) n_big = 0;
    __syncthreads();
    KWord<L> item[ITEMS];
    u32 slot[ITEMS];  // digit << 13 | rank inside the digit (rank < CAP <= 8192)
#pragma unroll
    for (int j = 0; j < ITEMS; ++j) {
        u32 i = threadIdx.x + j * 256;
        if (i < size) {
            item[j] = src[i];
            u32 dg = bits ? item[j].digit(shift, bits) : 0;
            slot[j] = (dg << 13) | atomicAdd(&sub_cnt[dg], 1u);
        }
    }
    __syncthreads();
    // exclusive scan of the digit counts (n_sub <= 2048: 8 consecutive entries per thread)
    {
        u32 v[8], c = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            u32 i = threadIdx.x * 8 + j;
            v[j] = i < n_sub ? sub_cnt[i] : 0;
            c += v[j];
        }
        u32 total;
        u32 p = kc_block_exclusive_scan_256(c, &total, sw);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            u32 i = threadIdx.x * 8 + j;
            if (i < n_sub) {
                sub_cnt[i] = p;
                // finish small sub-buckets later from [p, p + v[j]); remember the oversized ones
                if (v[j] > KC_SUB_SMALL) {
                    u32 q = atomicAdd(&n_big, 1u);
                    if (q < 64) big_list[q] = i;
                }
            }
            p += v[j];
        }
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < ITEMS; ++j) {
        u32 i = threadIdx.x + j * 256;
        if (i < size) s[sub_cnt[slot[j] >> 13] + (slot[j] & 8191u)] = item[j];
    }
    __syncthreads();
    const u32 nbig = n_big;
    if (nbig > 64) {
        // pathological bucket (many oversized sub-buckets): sort it whole
        kc_block_bitonic<L>(s, size);
    } else {
        // one thread per small sub-bucket: insertion sort of its segment
        for (u32 b = threadIdx.x; b < n_sub; b += 256) {
            u32 lo = sub_cnt[b];
            u32 hi = (b + 1 < n_sub) ? sub_cnt[b + 1] : size;
            u32 m = hi - lo;
            if (m < 2 || m > KC_SUB_SMALL) continue;
            for (u32 x = lo + 1; x < hi; ++x) {
                KWord<L> key = s[x];
                u32 y = x;
                while (y > lo && key < s[y - 1]) {
                    s[y] = s[y - 1];
                    --y;
                }
                s[y] = key;
            }
        }
        __syncthreads();
        for (u32 q = 0; q < nbig; ++q) {  // uniform across the CTA
            u32 b = big_list[q];
            u32 lo = sub_cnt[b];
            u32 hi = (b + 1 < n_sub) ? sub_cnt[b + 1] : size;
            kc_block_bitonic<L>(s + lo, hi - lo);
        }
    }
    __syncthreads();
    for (u32 i = threadIdx.x; i < size; i += 256) dst[i] = s[i];
}

// Buckets that ran out of key bits: all keys equal, so the bucket is sorted; one left in buf1 is copied back.
template <int L>
__global__ void __launch_bounds__(256) kc_sort_uniform_kernel(KWord<L> *buf0, const KWord<L> *buf1, const SortBucket *uniform) {
    SortBucket d = uniform[blockIdx.x];
    const KWord<L> *src = (d.parity ? buf1 : buf0) + d.off;
    KWord<L> *dst = buf0 + d.off;
    for (u32 i = threadIdx.x; i < d.size; i += 256)
        if (d.parity) dst[i] = src[i];
}

// Bookkeeping of one sort, kept only when the caller passes it (the test hook kc_debug_sort; the product path passes null).
struct KcSortStats {
    u32 levels = 0;                  // radix levels run
    u32 max_big = 0;                 // most buckets partitioned in one level
    u64 n_uniform = 0;               // buckets that ran out of key bits
    std::vector<SortBucket> small;   // every bucket handed to the local kernel
};

// Sort buf0[0..n) ascending on its low key_bits bits (all higher bits must be zero); buf1 is scratch.
//
// Bound of the small-bucket list.  Small buckets collect across levels, and the local kernel sorts them.  A level
// partitioning nb buckets adds at most sum_b 2^bits_b children, and kc_sort_prep_kernel picks 2^bits_b = 2 or
// 2^bits_b < 2 ceil(size_b / (CAP/4)) < 8 size_b / CAP + 2, so with q = n / CAP (rounded down) and nb <= q (each
// partitioned bucket holds more than CAP items) a level adds at most 8 (q + 1) + 2 nb <= 10 q + 8 < small_cap = 16 q + 4096.
// Before a level that could overflow the list, the local kernel sorts the buckets collected so far (they are final and
// disjoint from every bucket still being partitioned) and the list starts empty.
template <int L> void kc_sort(CudaExec &ex, KWord<L> *buf0, KWord<L> *buf1, u64 n, int key_bits, KcSortStats *stats = nullptr) {
    typedef SortCfg<L> Cfg;
    if (n == 0) return;
    if (n >= 0xFFFFFFF0ULL) KC_THROW(KC_ERR_TOO_LARGE, "sort of more than 2^32 items");
    cudaStream_t st = ex.stream;
    size_t mark = ex.arena->mark();
    const u32 cap = Cfg::CAP;
    const u32 big_cap = (u32) (n / cap + 2);
    const u32 small_cap = (u32) (16 * (n / cap) + 4096);
    const u32 uniform_cap = big_cap;
    SortBucket *big_a = ex.alloc<SortBucket>(big_cap);
    SortBucket *big_b = ex.alloc<SortBucket>(big_cap);
    SortBucket *small = ex.alloc<SortBucket>(small_cap);
    SortBucket *uniform = ex.alloc<SortBucket>(uniform_cap);
    u32 *tile_count = ex.alloc<u32>(big_cap + 1);
    u32 *hist = ex.alloc<u32>((u64) big_cap * 256);
    u64 *cursor = ex.alloc<u64>((u64) big_cap * 256);
    u8 *skip = ex.alloc<u8>(big_cap);
    u32 *ctr = ex.alloc<u32>(4);
    ex.fill_bytes(ctr, 0, 16);

    static KcDevOnce attr_once;  // function attributes are per device
    // the CAP * 2 bytes are not used; they keep the local kernel at the occupancy it was tuned at (L = 1: 2 CTAs per SM)
    const int local_smem = Cfg::CAP * (int) sizeof(KWord<L>) + Cfg::CAP * 2;
    const int scatter_smem = Cfg::TILE * (int) sizeof(KWord<L>);
    attr_once.run([&](int) {
        KC_CUDA(cudaFuncSetAttribute(kc_sort_local_kernel<L>, cudaFuncAttributeMaxDynamicSharedMemorySize, local_smem));
        KC_CUDA(cudaFuncSetAttribute(kc_sort_scatter_kernel<L>, cudaFuncAttributeMaxDynamicSharedMemorySize, scatter_smem));
    });

    SortBucket root;
    root.off = 0;
    root.size = (u32) n;
    root.rem = (u16) key_bits;
    root.parity = 0;
    root.bits = 0;
    u32 nb = 0, n_small = 0, n_uniform = 0;
    // the root bucket travels as a kernel argument (a copy from the stack + a stream synchronisation used to put it there)
    if (n <= cap) {
        kc_sort_root_kernel<<<1, 1, 0, st>>>(small, root);
        n_small = 1;
    } else if (root.rem == 0) {
        kc_sort_root_kernel<<<1, 1, 0, st>>>(uniform, root);
        n_uniform = 1;
    } else {
        kc_sort_root_kernel<<<1, 1, 0, st>>>(big_a, root);
        nb = 1;
    }
    ++ex.launches;
    SortBucket *cur = big_a, *nxt = big_b;
    const u32 max_ctas = 148 * 8;
    auto run_local = [&](u64 bytes) {
        if (stats) {
            const size_t at = stats->small.size();
            stats->small.resize(at + n_small);
            KC_CUDA(cudaMemcpyAsync(stats->small.data() + at, small, (size_t) n_small * sizeof(SortBucket), cudaMemcpyDeviceToHost, st));
            KC_CUDA(cudaStreamSynchronize(st));
        }
        CudaExec::Scope sc(ex, KP_SORT_LOCAL, bytes);
        kc_sort_local_kernel<L><<<n_small, 256, local_smem, st>>>(buf0, buf1, small);
        ++ex.launches;
    };
    bool first_level = true;
    while (nb > 0) {
        if (n_small + 8 * (n / cap + 1) + 2 * (u64) nb > small_cap) {  // see the bound above
            run_local(0);
            ex.fill_bytes(ctr + 1, 0, 4);
            n_small = 0;
        }
        if (stats) {
            ++stats->levels;
            if (nb > stats->max_big) stats->max_big = nb;
        }
        kc_sort_prep_kernel<<<(unsigned) kc_div_up(nb, 256), 256, 0, st>>>(cur, nb, cap, Cfg::TILE, tile_count);
        ++ex.launches;
        ex.fill_bytes(tile_count + nb, 0, 4);
        u32 *tile_prefix = tile_count;  // scanned in place; entry nb becomes the total
        u32 n_tiles;
        if (first_level) {  // one bucket: the host knows its tile count (kc_sort_prep_kernel's formula), no read-back
            ex.exclusive_scan_nosync(tile_count, tile_prefix, nb + 1);
            n_tiles = (u32) kc_div_up(n, (u64) Cfg::TILE);
            first_level = false;
        } else {
            n_tiles = ex.exclusive_scan(tile_count, tile_prefix, nb + 1);
        }
        ex.fill_bytes(hist, 0, (size_t) nb * 256 * 4);
        u32 tiles_per_cta = (u32) kc_div_up(n_tiles, max_ctas);
        u32 ctas = (u32) kc_div_up(n_tiles, tiles_per_cta);
        const u64 level_bytes = (u64) n_tiles * Cfg::TILE * sizeof(KWord<L>);  // items still in oversized buckets
        {
            CudaExec::Scope sc(ex, KP_SORT_HIST, level_bytes);
            kc_sort_hist_kernel<L><<<ctas, 256, 0, st>>>(buf0, buf1, cur, tile_prefix, nb, n_tiles, tiles_per_cta, hist);
        }
        ++ex.launches;
        ex.fill_bytes(ctr, 0, 4);  // next-level big counter only
        kc_sort_scan_kernel<<<nb, 256, 0, st>>>(cur, hist, cursor, skip, nxt, big_cap, small, small_cap, uniform,
                                                uniform_cap, ctr, cap);
        ++ex.launches;
        {
            CudaExec::Scope sc(ex, KP_SORT_SCATTER, 2 * level_bytes);
            kc_sort_scatter_kernel<L><<<ctas, 256, scatter_smem, st>>>(buf0, buf1, cur, tile_prefix, nb, n_tiles,
                                                                        tiles_per_cta, cursor, skip);
        }
        ++ex.launches;
        KC_CUDA(cudaGetLastError());
        u32 h[4];
        KC_CUDA(cudaMemcpyAsync(h, ctr, 16, cudaMemcpyDeviceToHost, st));
        KC_CUDA(cudaStreamSynchronize(st));
        if (h[3]) KC_THROW(KC_ERR_INTERNAL, "sort bucket list overflow");
        nb = h[0];
        n_small = h[1];
        n_uniform = h[2];
        SortBucket *t = cur;
        cur = nxt;
        nxt = t;
    }
    if (n_small) run_local(2 * n * sizeof(KWord<L>));
    if (stats) stats->n_uniform = n_uniform;
    if (n_uniform) {
        kc_sort_uniform_kernel<L><<<n_uniform, 256, 0, st>>>(buf0, buf1, uniform);
        ++ex.launches;
    }
    KC_CUDA(cudaGetLastError());
    ex.arena->release(mark);
}

#endif  // __CUDACC__
