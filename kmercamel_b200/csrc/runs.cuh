// First-occurrence runs: the nodes of the overlap stage in the from-FASTA regime (see kcgpu.cu run_stage1_runs and run_tail).
//
// Bit p of the flag array marks a window END position p whose k-mer is a kept k-mer occurring there for the first time.  A
// maximal run of consecutive flagged positions e_s..e_t is the node seq[e_s - k + 1 .. e_t].  Every run has one
// start and one end and both appear in the same order, so one count pass + one scan + one emit pass number them:
// the run of an end at position q is (number of starts at positions <= q) - 1.
#pragma once
#include "exec.cuh"
#include "kmerset.cuh"
#include "sort.cuh"

#ifdef __CUDACC__

static const int KC_RUN_WORDS = 4;                          // consecutive words of the bit array per thread
static const int KC_RUN_PER_THREAD = 32 * KC_RUN_WORDS;
static const int KC_RUN_TILE = 256 * KC_RUN_PER_THREAD;

// The thread's KC_RUN_WORDS x 32 flags (bit i of f[j] = position 32 (word + j) + i) and the flags just before and after them.  The
// bit array has one zero word of padding at the end.
KC_D void kc_runs_load(const u32 *flags, u64 word, u64 n_words, u32 (&f)[KC_RUN_WORDS], u32 &prev, u32 &next) {
#pragma unroll
    for (int j = 0; j < KC_RUN_WORDS; ++j) f[j] = word + j < n_words ? flags[word + j] : 0u;
    prev = word && word <= n_words ? flags[word - 1] >> 31 : 0u;
    next = word + KC_RUN_WORDS <= n_words ? flags[word + KC_RUN_WORDS] & 1u : 0u;
}

// starts / ends of runs inside word j, given the last flag before it and the first one after it
KC_D u32 kc_runs_starts(u32 f, u32 prev) { return f & ~((f << 1) | prev); }
KC_D u32 kc_runs_ends(u32 f, u32 next) { return f & ~((f >> 1) | (next << 31)); }

__global__ void __launch_bounds__(256) kc_runs_count_kernel(const u32 *flags, u64 n_words, u32 *block_counts, kc_ull *total_runs) {
    kc_pdl_wait();
    __shared__ u32 sw[8];
    const u64 word = ((u64) blockIdx.x * 256 + threadIdx.x) * KC_RUN_WORDS;
    u32 f[KC_RUN_WORDS], prev, next;
    kc_runs_load(flags, word, n_words, f, prev, next);
    u32 c = 0;
#pragma unroll
    for (int j = 0; j < KC_RUN_WORDS; ++j) c += __popc(kc_runs_starts(f[j], j ? f[j - 1] >> 31 : prev));
    u32 total;
    kc_block_exclusive_scan<256>(c, &total, sw);
    if (threadIdx.x == 0) {
        block_counts[blockIdx.x] = total;
        if (total) atomicAdd(total_runs, (kc_ull) total);
    }
}

// rec_off[r] = END position of the first window of run r, rec_len[r] = END position of its last window.
// spec_total == nullptr: block_offsets = exclusive prefix of the per-block run counts.  Otherwise (speculative tail, kcgpu.cu) it holds
// the counts themselves and *spec_total their sum: the kernel writes nothing when that exceeds spec_cap, and a block that holds a run
// start or end sums the counts before it (one block in ~10^4 on a genome), instead of a scan launch in between.
__global__ void __launch_bounds__(256) kc_runs_emit_kernel(const u32 *flags, u64 n_words, const u32 *block_offsets, u64 *rec_off, u64 *rec_len,
                                                           const kc_ull *spec_total = nullptr, u64 spec_cap = 0) {
    kc_pdl_wait();
    __shared__ u32 sw[8];
    if (spec_total && *spec_total > spec_cap) return;
    const u64 word = ((u64) blockIdx.x * 256 + threadIdx.x) * KC_RUN_WORDS;
    u32 f[KC_RUN_WORDS], prev, next;
    kc_runs_load(flags, word, n_words, f, prev, next);
    u32 c = 0, any = 0;
#pragma unroll
    for (int j = 0; j < KC_RUN_WORDS; ++j) {
        c += __popc(kc_runs_starts(f[j], j ? f[j - 1] >> 31 : prev));
        any |= kc_runs_ends(f[j], j + 1 < KC_RUN_WORDS ? f[j + 1] & 1u : next);
    }
    if (!__syncthreads_or(c | any)) return;  // no run starts or ends here: nothing to write
    u32 total;
    u32 before = kc_block_exclusive_scan<256>(c, &total, sw);
    if (spec_total) {
        u32 sum = 0;
        for (u32 b = threadIdx.x; b < blockIdx.x; b += 256) sum += block_offsets[b];
        u32 all;
        kc_block_exclusive_scan<256>(sum, &all, sw);
        before += all;
    } else {
        before += block_offsets[blockIdx.x];
    }
#pragma unroll
    for (int j = 0; j < KC_RUN_WORDS; ++j) {
        const u64 base = (word + j) * 32;
        const u32 starts = kc_runs_starts(f[j], j ? f[j - 1] >> 31 : prev);
        const u32 ends = kc_runs_ends(f[j], j + 1 < KC_RUN_WORDS ? f[j + 1] & 1u : next);
        u32 s = starts;
        u32 r = before;
        while (s) {
            const int i = __ffs(s) - 1;
            s &= s - 1;
            rec_off[r++] = base + i;
        }
        u32 e = ends;
        while (e) {  // the run of an end at bit i: (starts at positions <= its position) - 1
            const int i = __ffs(e) - 1;
            e &= e - 1;
            rec_len[before + __popc(starts & (0xFFFFFFFFu >> (31 - i))) - 1] = base + i;
        }
        before += __popc(starts);
    }
}

struct RunNodes {
    const u64 *rec_off = nullptr, *rec_len = nullptr;  // arena top end (or the -S records)
    u64 n_runs = 0;
};

// flags: bit array of kc_runs_flag_words(n_pos) words, bits >= n_pos zero.
inline size_t kc_runs_flag_words(u64 n_pos) { return (size_t) kc_div_up(n_pos, 32) + 1; }

// cells: device words {kept distinct k-mers (already accumulated), number of runs (zero on entry) [, M, status]}; all
// n_cells of them come back to the host with ONE synchronising read (host_cells).  With n_cells == 4 a non-zero status
// word (kmerset_fast.cuh: a slot overflowed, the flags are incomplete) makes the function return before it allocates
// anything: *aborted = true and the caller rebuilds the flags with the exact construction.
inline RunNodes kc_runs_from_flags(CudaExec &ex, const u32 *flags, u64 n_pos, int k, u64 *cells, u64 *host_cells, int n_cells = 2,
                                   bool *aborted = nullptr) {
    RunNodes runs;
    for (int i = 0; i < n_cells; ++i) host_cells[i] = 0;
    if (aborted) *aborted = false;
    if (n_pos == 0) return runs;
    const size_t mark = ex.arena->mark();
    const u64 n_words = kc_div_up(n_pos, 32);
    const u32 blocks = (u32) kc_div_up(n_pos, (u64) KC_RUN_TILE);
    u32 *counts = ex.alloc<u32>(blocks);
    {
        CudaExec::Scope sc(ex, KP_RUNS, n_pos / 8);
        kc_runs_count_kernel<<<blocks, 256, 0, ex.stream>>>(flags, n_words, counts, reinterpret_cast<kc_ull *>(cells + 1));
    }
    ++ex.launches;
    KC_CUDA(cudaGetLastError());
    ex.exclusive_scan_nosync(counts, counts, blocks);
    ex.read_n(cells, host_cells, (size_t) n_cells);
    if (n_cells >= 4 && host_cells[3] != 0) {
        if (aborted) *aborted = true;
        ex.arena->release(mark);
        return runs;
    }
    const u64 n_runs = host_cells[1];
    // run numbers are 32-bit in the emit kernel (and node ids in the overlap stage); an input of 2^32 bytes or more can have more runs
    if (n_runs >= 0xFFFFFFF0ULL) KC_THROW(KC_ERR_TOO_LARGE, "too many first-occurrence runs for one GPU");
    if (n_runs == 0) {
        ex.arena->release(mark);
        return runs;
    }
    u64 *rec_off = ex.arena->alloc_top<u64>(n_runs), *rec_len = ex.arena->alloc_top<u64>(n_runs);
    {
        CudaExec::Scope sc(ex, KP_RUNS, n_pos / 8 + 16 * n_runs);
        kc_runs_emit_kernel<<<blocks, 256, 0, ex.stream>>>(flags, n_words, counts, rec_off, rec_len);
    }
    ++ex.launches;
    KC_CUDA(cudaGetLastError());
    // window END positions e_s..e_t  ->  bytes [e_s - k + 1, e_t]
    ex.for_each(n_runs, [=] __device__(u64 r) {
        const u64 e_s = rec_off[r], e_t = rec_len[r];
        rec_len[r] = e_t - e_s + k;
        rec_off[r] = e_s - (k - 1);
    }, KP_RUNS, 32 * n_runs);
    ex.arena->release(mark);
    runs.rec_off = rec_off;
    runs.rec_len = rec_len;
    runs.n_runs = n_runs;
    return runs;
}

// ---- sparse switch (reference src/main.cpp:94,175-181) ---------------------------------------------------------------------
// PartialPreSort (src/global_sparse.h:14-35): a STABLE counting sort on the top min(2k, 8) bits of the k-mer.  Stable = sorted by
// (digit, original index), a unique 40-bit key, so any sort of those keys is the stable order: key[i] = digit(i) << 32 | i goes
// through the radix sort of sort.cuh and the low 32 bits come back as the permutation (new position -> old index).
template <class DigitOf> u64 *kc_partial_presort_perm(CudaExec &ex, u64 n, DigitOf digit_of) {
    KWord<1> *keys = ex.alloc<KWord<1>>(n), *tmp = ex.alloc<KWord<1>>(n);
    ex.for_each(n, [=] __device__(u64 i) { keys[i].w[0] = ((u64) digit_of(i) << 32) | i; }, KP_MISC, n * 16);
    kc_sort<1>(ex, keys, tmp, n, 40);
    return reinterpret_cast<u64 *>(keys);
}

// When the simplitigs are barely longer than k-mers (5 n >= U) the reference drops them and runs the greedy on the individual
// k-mers: simplitigs_to_kmer_vec (src/simplitigs.h:53-65: every k-mer of every simplitig, in simplitig order, in the
// orientation it has there) followed by PartialPreSort.  Here a simplitig is a first-occurrence run, so its k-mers are the
// windows of the run in input order and orientation: node i = k bytes at off[i], digit = its first min(k, 4) bases.
inline RunNodes kc_kmer_nodes_from_runs(CudaExec &ex, const u8 *seq, const RunNodes &runs, int k) {
    RunNodes out;
    const u64 n_runs = runs.n_runs;
    if (n_runs == 0) return out;
    const size_t mark = ex.arena->mark();
    u32 *pre = ex.alloc<u32>(n_runs + 1);
    const u64 *r_off = runs.rec_off, *r_len = runs.rec_len;
    ex.for_each(n_runs + 1, [=] __device__(u64 r) { pre[r] = r < n_runs ? (u32) (r_len[r] - (u64) k + 1) : 0u; }, KP_RUNS, n_runs * 12);
    const u64 U = ex.exclusive_scan(pre, pre, n_runs + 1);
    if (U >= 0xFFFFFFF0ULL) KC_THROW(KC_ERR_TOO_LARGE, "too many k-mer nodes for one GPU");
    u64 *n_off = ex.arena->alloc_top<u64>(U), *n_len = ex.arena->alloc_top<u64>(U);
    u64 *tmp_off = ex.alloc<u64>(U);
    ex.for_each(U, [=] __device__(u64 i) {
        const u32 r = kc_upper_bound_u32(pre, (u32) n_runs + 1, (u32) i) - 1;
        tmp_off[i] = r_off[r] + (i - pre[r]);
    }, KP_RUNS, U * 12);
    const int nb = k < 4 ? k : 4;  // SORT_FIRST_BITS = min(2k, 8) bits = the first nb bases
    const u64 *perm = kc_partial_presort_perm(ex, U, [=] __device__(u64 i) {
        u32 d = 0;
        for (int j = 0; j < nb; ++j) d = (d << 2) | (kc_nucleotide_code(seq[tmp_off[i] + j]) & 3u);
        return d;
    });
    ex.for_each(U, [=] __device__(u64 j) {
        n_off[j] = tmp_off[perm[j] & 0xFFFFFFFFULL];
        n_len[j] = (u64) k;
    }, KP_RUNS, U * 32);
    ex.arena->release(mark);
    out.rec_off = n_off;
    out.rec_len = n_len;
    out.n_runs = U;
    return out;
}

#endif  // __CUDACC__
