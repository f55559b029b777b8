// Key-only radix sort of fixed-width words, with an optional fused dedup + occurrence count.
//
// This is what stands in for khash on the GPU (reference src/khash.h, src/khash_utils.h): the k-mer set of
// src/parser.h:22-85 becomes "sort the occurrences, run-length encode", and every later hash-map probe of the
// reference (src/global.h:73-93) becomes a sort-join over (key, node) tuples packed into one word.
//
// Algorithm: most-significant-digit radix partitioning in global memory until a bucket fits in shared memory,
// then one CTA sorts the bucket in shared memory (bitonic network) and, in dedup mode, run-length encodes it.
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
                                                           u32 *hist, int low_bit) {
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
        int shift = low_bit + d.rem - d.bits;
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
                                                              u64 *cursor, const u8 *skip, int low_bit) {
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
        int shift = low_bit + d.rem - d.bits;
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

// Sort modes: plain sort; dedup where the whole word is the key; dedup where limb 0 is a payload (the position of
// the occurrence) and limbs 1.. are the key — the unique item keeps the smallest payload of its run.
enum { KC_SORT_ONLY = 0, KC_SORT_DEDUP = 1, KC_SORT_DEDUP_PAYLOAD = 2 };

template <int L, int MODE> KC_D bool kc_same_key(const KWord<L> &a, const KWord<L> &b) {
    bool e = true;
#pragma unroll
    for (int i = (MODE == KC_SORT_DEDUP_PAYLOAD ? 1 : 0); i < L; ++i) e = e && (a.w[i] == b.w[i]);
    return e;
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
//      the rare larger ones by the whole CTA with a bitonic network (whole words are compared, so a payload limb
//      orders equal keys by payload).
// In the dedup modes the sorted run is then run-length encoded: unique items go to the front of the bucket's slice
// of buf0, cnt[] receives min(occurrences-1, 255) (the uint8 the reference keeps, src/parser.h:77,81) and the rest
// of the slice is filled with the all-ones word, whose top limb is never that of a k-mer (2k <= 64 L - 2), for
// the compaction pass that follows.  ~10 shared-memory touches per item instead of ~110 for a full bitonic sort.
static const u32 KC_SUB_SMALL = 24;
static const int KC_SUB_BITS_MAX = 11;

template <int L, int MODE>
__global__ void __launch_bounds__(256) kc_sort_local_kernel(KWord<L> *buf0, const KWord<L> *buf1, const SortBucket *small,
                                                            u8 *cnt_out, int low_bit) {
    constexpr int CAP = SortCfg<L>::CAP;
    constexpr int ITEMS = CAP / 256;
    extern __shared__ __align__(16) unsigned char kc_smem_raw[];
    KWord<L> *s = reinterpret_cast<KWord<L> *>(kc_smem_raw);
    u16 *hpos = reinterpret_cast<u16 *>(s + CAP);              // dedup: run heads (CAP entries)
    __shared__ u32 sub_cnt[1 << KC_SUB_BITS_MAX];              // digit counts, then exclusive starts
    __shared__ u32 big_list[64];
    __shared__ u32 n_big;
    __shared__ u32 sw[8];
    __shared__ u32 uniq_total;
    SortBucket d = small[blockIdx.x];
    const KWord<L> *src = (d.parity ? buf1 : buf0) + d.off;
    KWord<L> *dst = buf0 + d.off;
    const u32 size = d.size;
    if (size == 1) {
        if (threadIdx.x == 0) {
            dst[0] = src[0];
            if (MODE != KC_SORT_ONLY) cnt_out[d.off] = 0;
        }
        return;
    }
    // digit width: about two sub-buckets per item, bounded by the key bits that are left
    int bits = 1;
    while ((1u << bits) < 2 * size && bits < KC_SUB_BITS_MAX) ++bits;
    if (bits > (int) d.rem) bits = d.rem;
    const u32 n_sub = 1u << bits;
    const int shift = low_bit + d.rem - bits;
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
    if (MODE == KC_SORT_ONLY) {
        for (u32 i = threadIdx.x; i < size; i += 256) dst[i] = s[i];
        return;
    }
    // run-length encode: hpos[u] = index of the first item of the u-th distinct key (indices < CAP <= 8192 fit u16)
    u32 carry = 0;
    for (u32 base = 0; base < size; base += 256) {  // block-scan the head flags 256 at a time
        u32 i = base + threadIdx.x;
        u32 head = (i < size && (i == 0 || !kc_same_key<L, MODE>(s[i], s[i - 1]))) ? 1u : 0u;
        u32 total;
        u32 p = kc_block_exclusive_scan_256(head, &total, sw);
        if (head) hpos[carry + p] = (u16) i;
        carry += total;
    }
    if (threadIdx.x == 0) uniq_total = carry;
    __syncthreads();
    const u32 nu = uniq_total;
    for (u32 u = threadIdx.x; u < size; u += 256) {
        if (u < nu) {
            u32 h = hpos[u];
            u32 e = (u + 1 < nu) ? hpos[u + 1] : size;
            dst[u] = s[h];  // first of its run: with a payload limb, the smallest payload
            cnt_out[d.off + u] = (u8) min(e - h - 1, 255u);
        } else {
            dst[u] = KWord<L>::ones();
        }
    }
}

// Buckets that ran out of key bits: all keys equal (payloads may differ).
template <int L, int MODE>
__global__ void __launch_bounds__(256) kc_sort_uniform_kernel(KWord<L> *buf0, const KWord<L> *buf1, const SortBucket *uniform,
                                                              u8 *cnt_out) {
    __shared__ kc_ull min_payload;
    SortBucket d = uniform[blockIdx.x];
    const KWord<L> *src = (d.parity ? buf1 : buf0) + d.off;
    KWord<L> *dst = buf0 + d.off;
    KWord<L> key = src[0];
    if (MODE == KC_SORT_DEDUP_PAYLOAD) {
        if (threadIdx.x == 0) min_payload = ~0ULL;
        __syncthreads();
        u64 m = ~0ULL;
        for (u32 i = threadIdx.x; i < d.size; i += 256) m = min(m, src[i].w[0]);
        atomicMin(&min_payload, (kc_ull) m);
        __syncthreads();
        key.w[0] = min_payload;
    }
    __syncthreads();
    for (u32 i = threadIdx.x; i < d.size; i += 256) {
        if (MODE != KC_SORT_ONLY) {
            dst[i] = i == 0 ? key : KWord<L>::ones();
            if (i == 0) cnt_out[d.off] = (u8) min(d.size - 1, 255u);
        } else if (d.parity) {
            dst[i] = src[i];
        }
    }
}

// Bookkeeping of one sort, kept only when the caller passes it (the test hook kc_debug_sort; the product path passes null).
struct KcSortStats {
    u32 levels = 0;                  // radix levels run
    u32 max_big = 0;                 // most buckets partitioned in one level
    u64 n_uniform = 0;               // buckets that ran out of key bits
    std::vector<SortBucket> small;   // every bucket handed to the local kernel
};

// Radix levels consume the bits [low_bit, key_bits) from the top; bits below low_bit only matter to the final
// shared-memory sort (which compares whole words).
//
// Bound of the small-bucket list.  Small buckets collect across levels, and the local kernel sorts them.  A level
// partitioning nb buckets adds at most sum_b 2^bits_b children, and kc_sort_prep_kernel picks 2^bits_b = 2 or
// 2^bits_b < 2 ceil(size_b / (CAP/4)) < 8 size_b / CAP + 2, so with q = n / CAP (rounded down) and nb <= q (each
// partitioned bucket holds more than CAP items) a level adds at most 8 (q + 1) + 2 nb <= 10 q + 8 < small_cap = 16 q + 4096.
// Before a level that could overflow the list, the local kernel sorts the buckets collected so far (they are final and
// disjoint from every bucket still being partitioned) and the list starts empty.
template <int L, int MODE>
void kc_sort_impl(CudaExec &ex, KWord<L> *buf0, KWord<L> *buf1, u64 n, int key_bits, int low_bit, u8 *cnt_tmp,
                  KcSortStats *stats = nullptr) {
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
    const int local_smem = Cfg::CAP * (int) sizeof(KWord<L>) + Cfg::CAP * 2;
    const int scatter_smem = Cfg::TILE * (int) sizeof(KWord<L>);
    attr_once.run([&](int) {
        KC_CUDA(cudaFuncSetAttribute(kc_sort_local_kernel<L, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, local_smem));
        KC_CUDA(cudaFuncSetAttribute(kc_sort_scatter_kernel<L>, cudaFuncAttributeMaxDynamicSharedMemorySize, scatter_smem));
    });

    SortBucket root;
    root.off = 0;
    root.size = (u32) n;
    root.rem = (u16) (key_bits - low_bit);
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
        kc_sort_local_kernel<L, MODE><<<n_small, 256, local_smem, st>>>(buf0, buf1, small, cnt_tmp, low_bit);
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
            kc_sort_hist_kernel<L><<<ctas, 256, 0, st>>>(buf0, buf1, cur, tile_prefix, nb, n_tiles, tiles_per_cta, hist, low_bit);
        }
        ++ex.launches;
        ex.fill_bytes(ctr, 0, 4);  // next-level big counter only
        kc_sort_scan_kernel<<<nb, 256, 0, st>>>(cur, hist, cursor, skip, nxt, big_cap, small, small_cap, uniform,
                                                uniform_cap, ctr, cap);
        ++ex.launches;
        {
            CudaExec::Scope sc(ex, KP_SORT_SCATTER, 2 * level_bytes);
            kc_sort_scatter_kernel<L><<<ctas, 256, scatter_smem, st>>>(buf0, buf1, cur, tile_prefix, nb, n_tiles,
                                                                        tiles_per_cta, cursor, skip, low_bit);
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
        kc_sort_uniform_kernel<L, MODE><<<n_uniform, 256, 0, st>>>(buf0, buf1, uniform, cnt_tmp);
        ++ex.launches;
    }
    KC_CUDA(cudaGetLastError());
    ex.arena->release(mark);
}

// Sort buf0[0..n) ascending on its low key_bits bits (all higher bits must be zero); buf1 is scratch.
template <int L> void kc_sort(CudaExec &ex, KWord<L> *buf0, KWord<L> *buf1, u64 n, int key_bits) {
    kc_sort_impl<L, KC_SORT_ONLY>(ex, buf0, buf1, n, key_bits, 0, nullptr);
}

// Sort + dedup + count.  On return out_keys[0..U) holds the distinct keys with at least min_freq occurrences in
// ascending order and out_cnt[0..U) their min(occurrences-1, 255); buf0 is destroyed.  out_keys may be buf1.
// PAYLOAD = true: limb 0 of every word is a payload (not part of the key); the surviving word of a key carries the
// smallest payload of its occurrences.  key_bits counts from bit 0 of the whole word in both cases.
template <int L, bool PAYLOAD>
u64 kc_sort_dedup(CudaExec &ex, KWord<L> *buf0, KWord<L> *buf1, u8 *cnt_tmp, KWord<L> *out_keys, u8 *out_cnt, u64 n,
                  int key_bits, int min_freq) {
    if (n == 0) return 0;
    kc_sort_impl<L, PAYLOAD ? KC_SORT_DEDUP_PAYLOAD : KC_SORT_DEDUP>(ex, buf0, buf1, n, key_bits, PAYLOAD ? 64 : 0, cnt_tmp);
    const KWord<L> *src = buf0;
    const u8 *cs = cnt_tmp;
    const u32 need = (u32) (min_freq - 1);
    return ex.compact_if(
        n, [=] __device__(u64 i) { return src[i].w[L - 1] != ~0ULL && (u32) cs[i] >= need; },
        [=] __device__(u64 i, u32 r) {
            out_keys[r] = src[i];
            out_cnt[r] = cs[i];
        },
        n * (sizeof(KWord<L>) + 1));
}

#endif  // __CUDACC__
