// kc_kmer_digest over first-occurrence bits: the digest of a k-mer set is (n, sum h, xor h) over its k-mers, and a set built as
// first-occurrence flags (kmerset_sig.cuh) holds each k-mer exactly once, at its first window.  So the digest is one pass over the
// sequence that hashes the flagged windows: no sorted key array, which is what lets the digest take inputs of 2^32 bytes and more.
#pragma once
#include "kmerset.cuh"

// h of one k-mer: the splitmix64 finaliser folded over the limbs (include/kcgpu.h, kc_kmer_digest)
KC_HD u64 kc_mix64(u64 x) {
    x ^= x >> 30;
    x *= 0xbf58476d1ce4e5b9ULL;
    x ^= x >> 27;
    x *= 0x94d049bb133111ebULL;
    x ^= x >> 31;
    return x;
}

template <int L> KC_HD u64 kc_kmer_hash(const KWord<L> &x) {
    u64 h = kc_mix64(x.w[0] + 0x9e3779b97f4a7c15ULL);
#pragma unroll
    for (int l = 1; l < L; ++l) h = kc_mix64(h ^ (x.w[l] + 0x9e3779b97f4a7c15ULL * (u64) (l + 1)));
    return h;
}

#ifdef __CUDACC__

static const int KC_DIGEST_THREADS = 256;
static const u64 KC_DIGEST_TILE = KC_DIGEST_THREADS * KC_EX_STRIP;  // window END positions per tile

// acc[0] += flagged windows, acc[1] += sum of their h, acc[2] ^= xor of their h.  One 32-window strip per thread (flag word w = strip
// w), persistent CTAs over the tiles; a tile without a flag is skipped before its sequence is read.  One set of atomics per CTA.
template <int L>
__global__ void __launch_bounds__(KC_DIGEST_THREADS) kc_flag_digest_kernel(const u8 *__restrict__ seq, u64 n_bytes, const u32 *__restrict__ flags,
                                                                            u64 n_flag_words, int k, int complements, u64 n_tiles, kc_ull *acc) {
    constexpr int T = KC_DIGEST_THREADS;
    __shared__ u64 pk[KC_EX_HALO + T];
    __shared__ u32 vm[KC_EX_HALO + T];
    __shared__ u64 red[3][T / 32];
    u64 n = 0, s = 0, x = 0;
    for (u64 tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const u64 w = tile * T + threadIdx.x;
        const u32 f = w < n_flag_words ? flags[w] : 0u;
        if (!__syncthreads_or(f != 0u)) continue;
        kc_tile_load<T>(seq, n_bytes, (i64) (tile * KC_DIGEST_TILE), pk, vm);
        __syncthreads();
        kc_strip_windows<L>(pk, KC_EX_HALO + threadIdx.x, __brev(f), k, complements, [&](int, const KWord<L> &c) {
            const u64 h = kc_kmer_hash<L>(c);
            ++n;
            s += h;
            x ^= h;
        });
        __syncthreads();  // pk is loaded again by the next tile
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        n += __shfl_xor_sync(0xFFFFFFFFu, n, o);
        s += __shfl_xor_sync(0xFFFFFFFFu, s, o);
        x ^= __shfl_xor_sync(0xFFFFFFFFu, x, o);
    }
    if ((threadIdx.x & 31) == 0) {
        red[0][threadIdx.x >> 5] = n;
        red[1][threadIdx.x >> 5] = s;
        red[2][threadIdx.x >> 5] = x;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int i = 1; i < T / 32; ++i) {
            n += red[0][i];
            s += red[1][i];
            x ^= red[2][i];
        }
        if (n) {
            atomicAdd(&acc[0], (kc_ull) n);
            atomicAdd(&acc[1], (kc_ull) s);
            atomicXor(&acc[2], (kc_ull) x);
        }
    }
}

// Launches the digest of the flagged windows of seq (n_bytes, the buffer padded to whole 32-byte words) into acc[0..2] (zeroed by the
// caller) on ex.stream.
template <int L> void kc_flag_digest(CudaExec &ex, const u8 *seq, u64 n_bytes, const u32 *flags, u64 n_flag_words, int k, bool complements, kc_ull *acc) {
    const u64 tiles = kc_div_up(n_bytes, KC_DIGEST_TILE);
    if (tiles == 0) return;
    int dev = 0;
    KC_CUDA(cudaGetDevice(&dev));
    const u64 fit = (u64) kc_sm_count(dev) * 8;
    CudaExec::Scope sc(ex, KP_MISC, n_bytes + n_bytes / 8);
    kc_flag_digest_kernel<L><<<(unsigned) (tiles < fit ? tiles : fit), KC_DIGEST_THREADS, 0, ex.stream>>>(seq, n_bytes, flags, n_flag_words, k, complements ? 1 : 0,
                                                                                                           tiles, acc);
    ++ex.launches;
    KC_CUDA(cudaGetLastError());
}

#endif  // __CUDACC__
