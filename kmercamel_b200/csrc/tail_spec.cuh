// Speculative tail of the from-FASTA single-GPU path (kcgpu.cu run_tail_spec).
//
// A genome leaves a few dozen first-occurrence runs, far below what the one-CTA kernels of the tail take.  So instead of reading the run
// count back after the signature construction and sizing the tail from it, the host queues the whole tail sized for KC_SPEC_RUNS runs
// and every kernel reads the real count from the device.  When the guess does not hold (too many runs, the sparse switch, an empty set, a
// signature bucket that overflowed), kc_spec_nodes_kernel says why and the kernels after it do nothing; the host learns it from the one
// read-back at the end and runs the ordinary tail.
#pragma once
#include "engine.cuh"
#include "runs.cuh"
#include "stage1.cuh"

// Runs the speculative tail is sized for: N <= 1024 virtual nodes with reverse complements, what kc_rank_small_kernel and the staged
// state of kc_small_engine_kernel (SmallCfg::NS) take.
static const u32 KC_SPEC_RUNS = 512;

// The status block of one call, read back to the host with ONE copy after the last kernel of the tail is queued (u64 words):
//   [0, 4)   cells of the signature construction: {kept, runs, M, signature status}
//   [4, 6)   spec: u32 {status, n, N} (kc_spec_nodes_kernel)
//   [6, 12)  the emission's cell (EmitSpec)
//   [12, 84) the small engine's status words (KC_SMALL_STATUS_WORDS u32)
static const u32 KC_SPEC_SPEC = 4, KC_SPEC_EMIT = 6, KC_SPEC_SMALL = 12;
static const u32 KC_SPEC_BLOCK_WORDS = KC_SPEC_SMALL + KC_SMALL_STATUS_WORDS / 2;

enum KcSpecStatus : u32 { KC_SPEC_OK = 0, KC_SPEC_SIG_OVERFLOW = 1, KC_SPEC_EMPTY = 2, KC_SPEC_TOO_MANY = 3, KC_SPEC_SPARSE = 4 };

#ifdef __CUDACC__

// One CTA.  cells = {kept distinct k-mers, runs, M, signature status}; rec_off / rec_len hold the window END positions of the runs
// (kc_runs_emit_kernel).  Writes spec = {status, n, N} (n = N = 0 unless the status is KC_SPEC_OK) and, when it is: the runs as byte
// ranges, their first / last k-mers (kc_extract_node_ends), the initial path state (Engine::init_state), the identity live lists and the
// zeroed level masks of the small engine (mask_words of them).
template <int L>
__global__ void __launch_bounds__(1024) kc_spec_nodes_kernel(const u64 *cells, u32 *spec, bool sparse_switch, bool complements, const u8 *seq, int k,
                                                            u64 *rec_off, u64 *rec_len, KWord<L> *first, KWord<L> *last, PathState st, u8 *ban_flag,
                                                            u32 *ban_ctr, u32 *live_s, u32 *live_p, u32 *masks, u32 mask_words) {
    const u64 kept = cells[0], runs = cells[1], M = cells[2];
    const u64 U = M ? kept : 0;
    const u32 status = cells[3] ? KC_SPEC_SIG_OVERFLOW
                       : U == 0 ? KC_SPEC_EMPTY
                       : runs > KC_SPEC_RUNS ? KC_SPEC_TOO_MANY
                       : sparse_switch && runs * 5 >= U ? KC_SPEC_SPARSE  // src/main.cpp:175-181, as in run_pipeline
                                                        : KC_SPEC_OK;
    const u32 n = status == KC_SPEC_OK ? (u32) runs : 0u, N = complements ? 2 * n : n;
    if (threadIdx.x == 0) {
        spec[0] = status;
        spec[1] = n;
        spec[2] = N;
    }
    if (status != KC_SPEC_OK) return;
    for (u32 r = threadIdx.x; r < n; r += blockDim.x) {  // window END positions e_s..e_t  ->  bytes [e_s - k + 1, e_t]
        const u64 e_s = rec_off[r], e_t = rec_len[r];
        const u64 off = e_s - (k - 1), len = e_t - e_s + k;
        rec_off[r] = off;
        rec_len[r] = len;
        kc_node_end_kmers<L>(seq, off, len, k, first[r], last[r]);
    }
    for (u32 v = threadIdx.x; v < N; v += blockDim.x) {
        st.edge_from[v] = KC_NONE;
        st.edge_to[v] = KC_NONE;
        st.ovl[v] = 255;
        ban_flag[v] = 0;
        st.chain_head[v] = v;
        st.chain_tail[v] = v;
        live_s[v] = v;
        live_p[v] = v;
    }
    for (u32 i = threadIdx.x; i < mask_words; i += blockDim.x) masks[i] = 0;
    if (threadIdx.x < 4) ban_ctr[threadIdx.x] = 0;
}

#endif  // __CUDACC__
