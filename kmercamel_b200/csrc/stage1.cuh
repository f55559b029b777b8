// Stage 1: k-mer set construction (reference src/parser.h:22-141 AddKMers / AddKMersWithFrequencies /
// ReadKMers[Filtered], src/khash_utils.h:143-159) as  extract -> radix sort -> run-length encode.
//
// Input is the framed sequence stream: the record sequences concatenated, separated by one non-ACGT byte.  A
// k-mer window is valid iff its k bytes are all ACGT/acgt, which reproduces both the reference's restart on
// N-like bytes (src/parser.h:32-37) and "windows never span records" (one AddKMers call per record,
// src/parser.h:112-114).
//
// kc_extract_kernel: one thread per strip of 32 consecutive window END positions.
//   * the CTA loads its 8 KiB of bytes once (two 16-byte loads per thread, fully coalesced), converts them
//     4 bytes at a time with SIMD-in-register arithmetic to 2-bit codes + 1 validity bit, and parks one packed
//     64-bit code word + one 32-bit validity word per strip in shared memory (plus 4 halo words to the left);
//   * k < 32: every window is a funnel shift of (previous word : own word) — no rolling dependency; the reverse
//     complement rolls in registers (src/parser.h:39-40); k >= 32 rolls both strands over KWord<L>;
//   * canonical = min(forward, reverse complement) (src/parser.h:44), or forward with -u;
//   * output slots are reserved with ONE atomicAdd per CTA (order is irrelevant: the sort follows); 8-byte
//     words are staged per warp in shared memory so the global stores are full-line coalesced.
// Algorithmic HBM bytes: n_bytes read + M * 8L written.
#pragma once
#include "exec.cuh"
#include "kword.cuh"
#include "sort.cuh"

#ifdef __CUDACC__

static const int KC_EX_THREADS = 256;
static const int KC_EX_STRIP = 32;
static const int KC_EX_HALO = 4;  // halo words: 4 * 32 >= 127 - 1 preceding bases

// 4 ASCII bytes (byte 0 = first base) -> 8 bits of codes (first base in the top 2 bits) and 4 validity bits.
KC_D void kc_pack4(u32 w, u32 &codes, u32 &valid) {
    u32 c = ((w >> 1) ^ (w >> 2)) & 0x03030303u;  // A,a->0 C,c->1 G,g->2 T,t->3
    codes = (c * 0x40100401u) >> 24;
    // valid = the case-folded byte IS the letter its code stands for: A = 0x41, C = A + 2, G = A + 6, T = A + 19, rebuilt for the four bytes
    // at once (three multiply-adds; four emulated __vcmpeq4 cost twice the instructions), then the zero bytes of the difference
    const u32 c0 = c & 0x01010101u, c1 = (c >> 1) & 0x01010101u;
    const u32 expect = 0x41414141u + c0 * 2u + c1 * 6u + (c0 & c1) * 11u;
    const u32 d = (w & 0xDFDFDFDFu) ^ expect;
    const u32 z = ~(((d & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | d) & 0x80808080u;  // bit 7 of every byte that is zero
    valid = (((z >> 7) * 0x08040201u) >> 24) & 0xFu;
}

// WITH_POS = false: out[] receives the canonical k-mers (KWord<L>).
// WITH_POS = true : out[] receives KWord<L+1> items {limb 0 = END position of the window in seq, limbs 1.. = k-mer},
//                   the input of the first-occurrence dedup (kc_sort_dedup<L+1, true>).
template <int L, bool WITH_POS>
__global__ void __launch_bounds__(KC_EX_THREADS) kc_extract_kernel(const u8 *__restrict__ seq, u64 n_bytes, int k, int complements,
                                                                    KWord<L + (WITH_POS ? 1 : 0)> *__restrict__ out, kc_ull *counter) {
    __shared__ u64 pk[KC_EX_HALO + KC_EX_THREADS];
    __shared__ u32 vm[KC_EX_HALO + KC_EX_THREADS];
    __shared__ u32 sw[8];
    __shared__ kc_ull block_base;
    extern __shared__ __align__(16) unsigned char kc_smem_raw[];  // L == 1: 8 warps * 1024 staged words

    const i64 block_pos0 = (i64) blockIdx.x * (KC_EX_THREADS * KC_EX_STRIP);
    for (int wi = threadIdx.x; wi < KC_EX_HALO + KC_EX_THREADS; wi += KC_EX_THREADS) {
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
    __syncthreads();

    const int widx = KC_EX_HALO + threadIdx.x;
    const u64 mine = pk[widx];
    const u32 myv = vm[widx];
    // windows ending in this strip that are valid: run length of valid codes, seeded from the halo
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
    const u32 cnt = __popc(em);
    u32 block_total;
    const u32 my_off = kc_block_exclusive_scan_256(cnt, &block_total, sw);
    if (threadIdx.x == 0 && block_total) block_base = atomicAdd(counter, (kc_ull) block_total);
    __syncthreads();
    if (block_total == 0) return;

    if (L == 1) {
        // ---- 64-bit fast path (k < 32): funnel shifts ---------------------------------------------------
        u64 *stage = reinterpret_cast<u64 *>(kc_smem_raw) + (threadIdx.x >> 5) * (32 * KC_EX_STRIP);
        const u32 lane = threadIdx.x & 31;
        u32 warp_off = cnt;  // inclusive warp scan of cnt
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            u32 t = __shfl_up_sync(0xFFFFFFFFu, warp_off, o);
            if (lane >= (u32) o) warp_off += t;
        }
        const u32 warp_total = __shfl_sync(0xFFFFFFFFu, warp_off, 31);
        u32 pos = warp_off - cnt;
        kc_ull gpos = block_base + my_off;                     // WITH_POS: direct 16-byte stores
        const u64 strip_pos0 = (u64) block_pos0 + (u64) threadIdx.x * KC_EX_STRIP;
        if (em) {
            const u64 prev = pk[widx - 1];
            const u64 mask = (k == 32) ? ~0ULL : ((1ULL << (2 * k)) - 1);
            const int top = 2 * (k - 1);
            // rc of the k-1 bases preceding the strip, already shifted right by one base (see DESIGN.md)
            KWord<1> pw;
            pw.w[0] = prev & ((1ULL << top) - 1);
            u64 rcs = k > 1 ? kmer_reverse_complement(pw, k - 1).w[0] : 0;
#pragma unroll
            for (int j = 0; j < KC_EX_STRIP; ++j) {
                const int sh = 2 * (31 - j);
                u64 fwd = (mine >> sh);
                if (j < 31) fwd |= prev << (2 * (j + 1));
                fwd &= mask;
                u64 c = (mine >> sh) & 3;
                u64 rcf = rcs | ((3 ^ c) << top);
                rcs = rcf >> 2;
                if ((em >> (31 - j)) & 1) {
                    const u64 canon = (!complements || fwd < rcf) ? fwd : rcf;
                    if (WITH_POS) {
                        *reinterpret_cast<ulonglong2 *>(&out[gpos++]) = make_ulonglong2(strip_pos0 + j, canon);
                    } else {
                        stage[pos++] = canon;
                    }
                }
            }
        }
        if (!WITH_POS) {
            __syncwarp();
            // the warp's first global slot: block base + slots of the preceding warps = my_off of lane 0
            const kc_ull warp_base = block_base + __shfl_sync(0xFFFFFFFFu, my_off, 0);
            u64 *o64 = reinterpret_cast<u64 *>(out);
            for (u32 q = lane; q < warp_total; q += 32) o64[warp_base + q] = stage[q];
        }
    } else {
        // ---- generic path: roll both strands over KWord<L> ---------------------------------------------
        if (!em) return;
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
        kc_ull pos = block_base + my_off;
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
                KWord<L + (WITH_POS ? 1 : 0)> item;
                if (WITH_POS) item.w[0] = (u64) block_pos0 + (u64) threadIdx.x * KC_EX_STRIP + j;
#pragma unroll
                for (int i = 0; i < L; ++i) item.w[i + (WITH_POS ? 1 : 0)] = canon.w[i];
                out[pos++] = item;
            }
        }
    }
}

// Extract every canonical k-mer occurrence of seq[0..n_bytes) into out (capacity n_bytes); returns M.
template <int L, bool WITH_POS>
u64 kc_extract_kmers(CudaExec &ex, const u8 *seq, u64 n_bytes, int k, bool complements, KWord<L + (WITH_POS ? 1 : 0)> *out) {
    if (n_bytes == 0) return 0;
    size_t mark = ex.arena->mark();
    kc_ull *counter = reinterpret_cast<kc_ull *>(ex.alloc<u64>(1));
    ex.fill_bytes(counter, 0, 8);
    u64 blocks = kc_div_up(n_bytes, (u64) KC_EX_THREADS * KC_EX_STRIP);
    const int smem = (L == 1 && !WITH_POS) ? 8 * 32 * KC_EX_STRIP * 8 : 0;
    static KcDevOnce attr_once;  // function attributes are per device
    if (smem) attr_once.run([&](int) { KC_CUDA(cudaFuncSetAttribute(kc_extract_kernel<L, WITH_POS>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)); });
    {
        // algorithmic bytes: the input once; the M item bytes written are added below once M is known
        CudaExec::Scope sc(ex, KP_EXTRACT, n_bytes);
        kc_extract_kernel<L, WITH_POS><<<(unsigned) blocks, KC_EX_THREADS, smem, ex.stream>>>(seq, n_bytes, k, complements ? 1 : 0,
                                                                                               out, counter);
    }
    ++ex.launches;
    KC_CUDA(cudaGetLastError());
    u64 m = ex.read(reinterpret_cast<u64 *>(counter));
    if (ex.prof && ex.prof->enabled) ex.prof->bytes[KP_EXTRACT] += m * sizeof(KWord<L + (WITH_POS ? 1 : 0)>);
    ex.arena->release(mark);
    return m;
}

// First and last k-mer of the node seq[off .. off + len), len >= k.
template <int L> KC_D void kc_node_end_kmers(const u8 *seq, u64 off, u64 len, int k, KWord<L> &first, KWord<L> &last) {
    KWord<L> f = KWord<L>::zero(), l = KWord<L>::zero();
    for (int i = 0; i < k; ++i) {
        f = f.shl(2);
        f.w[0] |= kc_nucleotide_code(seq[off + i]) & 3;
        l = l.shl(2);
        l.w[0] |= kc_nucleotide_code(seq[off + len - k + i]) & 3;
    }
    first = f;
    last = l;
}

// `-S`: first and last k-mer of every record (reference src/simplitigs.h:68-76) and input validation
// (src/simplitigs.h:82 asserts ACGT only; records shorter than k have no k-mer and are rejected here).
template <int L>
void kc_extract_node_ends(CudaExec &ex, const u8 *seq, u64 n_bytes, const u64 *rec_off, const u64 *rec_len, u64 n_recs, int k,
                          KWord<L> *first, KWord<L> *last, u32 *error_flag, bool validate_bytes) {
    ex.for_each(n_recs, [=] __device__(u64 r) {
        u64 off = rec_off[r], len = rec_len[r];
        if (len < (u64) k) {
            *error_flag = 1;
            return;
        }
        kc_node_end_kmers<L>(seq, off, len, k, first[r], last[r]);
    });
    if (!validate_bytes) return;
    // every byte that is not a record separator must be a nucleotide
    ex.for_each(n_bytes, [=] __device__(u64 p) {
        u8 c = seq[p];
        if (c != '\n' && kc_nucleotide_code(c) > 3) *error_flag = 1;
    });
}

#endif  // __CUDACC__
