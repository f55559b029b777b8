// Greedy overlap Hamiltonian path on the GPU (reference src/global.h:43-133 and its k-mer-node twin
// src/global_sparse.h:42-132), one overlap length d at a time.
//
// What the reference does sequentially — for d = k-1..0, for 16 batches of prefix nodes, for every suffix-free
// node i in ascending order: take the largest still prefix-free node j of the batch with pre_d(j) == suf_d(i),
// j != rc(i), j != first(i) — is restated as a priority-ordered matching and evaluated level by level:
//
//   1. build one tuple per free suffix end (key = suf_d(last k-mer), order = i) and per free prefix end
//      (key = pre_d(first k-mer), order = (batch(j), descending j)), each packed into ONE word
//      [key | role | batch | id] so that a key-only radix sort yields, per key, the suffix nodes in ascending
//      id followed by the prefix nodes in exactly the order the reference's linked lists are walked
//      (src/global.h:73-85 pushes at the head, hence descending j inside a batch);
//   2. a key whose run holds both roles is an active group.  With reverse complements the groups of key and
//      rc(key) mirror each other (accepting i->j also accepts rc(j)->rc(i), src/global.h:110-112), so one
//      thread replays the reference's loop over the PAIR of groups, events merged in the reference's global
//      order (batch, i).  Everything a pair touches (edge slots of its own nodes) is private to it;
//   3. the only coupling between pairs is the cycle test j == first(i) (src/global.h:97).  Each pair tracks
//      chain merges it makes itself and uses the level-start snapshot for the rest.  A stale snapshot can
//      only produce a false accept, and a false accept closes a cycle in (old edges + this level's edges).
//      Cycles are found by pointer doubling over this level's edges with chains contracted; in each cycle the
//      edge with the largest order stamp is the one the sequential loop would have refused: it is banned and
//      the level is replayed.  `strict` bans only the globally earliest such edge per round (provably the first
//      divergence from the sequential run — used when the reference's tie order must be reproduced, i.e.
//      `-S`); otherwise all cycle closers are banned at once;
//   4. chain ends (first/last of src/global.h:53-60,116-121) are updated from the doubling result.
//
// The same code runs the d = k-1 level over k-mer nodes when the input is a FASTA (the reference builds
// simplitigs there, src/simplitigs.h:105-205; its merge order is khash-iteration order and unspecified, see
// DESIGN.md) and every level of `-S` inputs, where the output is byte-identical to the reference.
#pragma once
#include "exec.cuh"
#include "kword.cuh"
#include "sort.cuh"
#ifdef KC_HOST_EMUL
#include <algorithm>
#endif

// ---- nodes ------------------------------------------------------------------------------------------
// Virtual node ids 0..N-1; with complements N = 2n and id >= n is the reverse complement of id - n
// (src/global.h:16-25).
template <int L> struct NodeView {
    const KWord<L> *first;  // first k-mer of node v < n
    const KWord<L> *last;   // last k-mer of node v < n (== first for k-mer nodes)
    u32 n, N;
    int k;
    bool complements;
    KC_HD u32 mirror(u32 v) const { return v < n ? v + n : v - n; }
    KC_HD KWord<L> first_kmer(u32 v) const { return v < n ? first[v] : kmer_reverse_complement(last[v - n], k); }
    KC_HD KWord<L> last_kmer(u32 v) const { return v < n ? last[v] : kmer_reverse_complement(first[v - n], k); }
};

struct PathState {
    u32 *edge_from;   // src/global.h:49 edgeFrom, KC_NONE = none
    u32 *edge_to;     // inverse; edge_to[j] != NONE  <=>  prefixForbidden[j] (src/global.h:52)
    u8 *ovl;          // src/global.h:50 overlaps, 255 = none
    u32 *chain_head;  // for a chain tail t: the chain's head (src/global.h:53 first[])
    u32 *chain_tail;  // for a chain head h: the chain's tail (src/global.h:54 last[])
};

// ---- tuples -----------------------------------------------------------------------------------------
// limb 0 = meta << 27, limbs 1..L = key.  meta (37 bits) = role(1) | batch(4) | id-or-~id (32).
static const int KC_META_SHIFT = 27;
static const u64 KC_ROLE_P = 1ULL << 36;

template <int L> KC_HD KWord<L + 1> tuple_make(const KWord<L> &key, u64 meta) {
    KWord<L + 1> t;
    t.w[0] = meta << KC_META_SHIFT;
#pragma unroll
    for (int i = 0; i < L; ++i) t.w[i + 1] = key.w[i];
    return t;
}
template <int LT> KC_HD KWord<LT - 1> tuple_key(const KWord<LT> &t) {
    KWord<LT - 1> k;
#pragma unroll
    for (int i = 0; i < LT - 1; ++i) k.w[i] = t.w[i + 1];
    return k;
}
template <int LT> KC_HD bool tuple_is_prefix(const KWord<LT> &t) { return (t.w[0] >> (36 + KC_META_SHIFT)) & 1; }
template <int LT> KC_HD u32 tuple_part(const KWord<LT> &t) { return (u32) (t.w[0] >> (32 + KC_META_SHIFT)) & 15u; }
template <int LT> KC_HD u32 tuple_node(const KWord<LT> &t) {
    u32 id = (u32) (t.w[0] >> KC_META_SHIFT);
    return tuple_is_prefix(t) ? ~id : id;
}

// first index in [lo, hi) whose tuple is >= probe
template <int LT> KC_HD u64 tuple_lower_bound(const KWord<LT> *T, u64 lo, u64 hi, const KWord<LT> &probe) {
    while (lo < hi) {
        u64 mid = (lo + hi) >> 1;
        if (T[mid] < probe) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// ---- sort dispatch ------------------------------------------------------------------------------------
#ifdef __CUDACC__
template <int LL> void exec_sort(CudaExec &ex, KWord<LL> *a, KWord<LL> *b, u64 n, int key_bits) { kc_sort<LL>(ex, a, b, n, key_bits); }
#endif
#ifdef KC_HOST_EMUL
template <int LL> void exec_sort(HostExec &, KWord<LL> *a, KWord<LL> *, u64 n, int) {
    std::sort(a, a + n, [](const KWord<LL> &x, const KWord<LL> &y) { return x < y; });
}
#endif

// ---- per-level device state -----------------------------------------------------------------------------
template <int L> struct LevelCtx {
    NodeView<L> nv;
    PathState st;
    const KWord<L + 1> *T;  // sorted tuples
    u64 nt;
    int d;
    u32 batch;      // src/global.h:48 batchSize = N / 16 + 1
    u32 *head_w;    // working copy of chain_head for this level (owned by the pair holding the node's suffix slot)
    u32 *tail_w;    // working copy of chain_tail (owned by the pair holding the node's prefix slot)
    u64 *stamp;     // order stamp of the edge leaving a node: (batch(j) << 32) | i of the PRIMARY event
    u8 *prim;       // 1 = edge accepted as primary, 0 = as the mirror of a primary
    const u8 *ban_flag;
    const u32 *ban_i, *ban_j;
    u32 n_bans;
    bool check_cycles;  // false in lower-bound mode (src/global.h:95-97 skips the rc and cycle tests)
};

// One thread replays the reference loop for one (key, rc(key)) pair of groups.
template <int L> struct SimulatePairFn {
    LevelCtx<L> c;
    const u32 *group_pstart;  // index of the first prefix tuple of every active group

    KC_HD bool banned(u32 i, u32 j) const {
        if (!c.ban_flag[i]) return false;
        for (u32 b = 0; b < c.n_bans; ++b)
            if (c.ban_i[b] == i && c.ban_j[b] == j) return true;
        return false;
    }
    KC_HD bool owns_suffix(u32 v, const KWord<L> &ka, const KWord<L> &kb) const {
        if (c.d == 0) return true;  // one group holds every end
        KWord<L> s = kmer_suffix(c.nv.last_kmer(v), c.d);
        return s == ka || s == kb;
    }
    KC_HD bool owns_prefix(u32 v, const KWord<L> &ka, const KWord<L> &kb) const {
        if (c.d == 0) return true;
        KWord<L> p = kmer_prefix(c.nv.first_kmer(v), c.nv.k, c.d);
        return p == ka || p == kb;
    }
    KC_HD void link(u32 x, u32 y, u64 stampv, u8 primary, const KWord<L> &ka, const KWord<L> &kb) const {
        c.st.edge_from[x] = y;  // src/global.h:114-115,121
        c.st.edge_to[y] = x;
        c.st.ovl[x] = (u8) c.d;
        c.stamp[x] = stampv;
        c.prim[x] = primary;
        u32 h = c.head_w[x], t = c.tail_w[y];  // src/global.h:116-120, restricted to entries this pair owns
        if (owns_suffix(t, ka, kb)) c.head_w[t] = h;
        if (owns_prefix(h, ka, kb)) c.tail_w[h] = t;
    }

    KC_HD void operator()(u64 g) const {
        const KWord<L + 1> *T = c.T;
        const u64 p_beg = group_pstart[g];
        const KWord<L> ka = tuple_key(T[p_beg]);
        KWord<L> kb = ka;
        bool two = false;
        if (c.nv.complements) {
            kb = kmer_reverse_complement(ka, c.d);
            if (kb < ka) return;  // the thread of rc(key) replays this pair
            two = kb != ka;
        }
        // group A = key ka.  The probe with the maximal meta (prefix role, batch 15, ~id = 0xFFFFFFFF i.e. node 0) is
        // never a real tuple because node 0 lies in batch 0, so the lower bound is the end of the group.
        const u64 meta_max = (1ULL << 37) - 1;
        const u64 s_beg = tuple_lower_bound(T, (u64) 0, p_beg, tuple_make(ka, 0));
        const u64 s_end = p_beg;
        const u64 pa_end = tuple_lower_bound(T, p_beg, c.nt, tuple_make(ka, meta_max));
        // group B = key kb (mirror)
        u64 s2_beg = 0, s2_end = 0, p2_beg = 0, p2_end = 0;
        if (two) {
            s2_beg = tuple_lower_bound(T, (u64) 0, c.nt, tuple_make(kb, 0));
            s2_end = tuple_lower_bound(T, s2_beg, c.nt, tuple_make(kb, KC_ROLE_P));
            p2_beg = s2_end;
            p2_end = tuple_lower_bound(T, p2_beg, c.nt, tuple_make(kb, meta_max));
        }
        u64 ca = p_beg, cb = p2_beg;  // per-batch run cursors
        for (u32 part = 0; part < 16; ++part) {  // src/global.h:66
            u64 ra0 = ca;
            while (ca < pa_end && tuple_part(T[ca]) == part) ++ca;
            u64 ra1 = ca;
            u64 rb0 = cb;
            while (cb < p2_end && tuple_part(T[cb]) == part) ++cb;
            u64 rb1 = cb;
            if (ra0 == ra1 && rb0 == rb1) continue;
            u64 fa = ra0, fb = rb0;  // first possibly-free candidate of each run
            u64 ia = s_beg, ib = s2_beg;
            while (true) {  // src/global.h:86: suffix nodes in ascending id, merged over both groups
                u32 va = (ia < s_end && fa < ra1) ? tuple_node(T[ia]) : KC_NONE;
                u32 vb = (ib < s2_end && fb < rb1) ? tuple_node(T[ib]) : KC_NONE;
                if (va == KC_NONE && vb == KC_NONE) break;
                u32 i;
                u64 *front;
                u64 rend;
                if (va < vb) {
                    i = va;
                    ++ia;
                    front = &fa;
                    rend = ra1;
                } else {
                    i = vb;
                    ++ib;
                    front = &fb;
                    rend = rb1;
                }
                if (c.st.edge_from[i] != KC_NONE) continue;  // suffixForbidden
                while (*front < rend && c.st.edge_to[tuple_node(T[*front])] != KC_NONE) ++*front;
                for (u64 q = *front; q < rend; ++q) {  // src/global.h:93-106
                    u32 j = tuple_node(T[q]);
                    if (c.st.edge_to[j] != KC_NONE) continue;
                    if (c.check_cycles) {
                        if (c.nv.complements && j == c.nv.mirror(i)) continue;
                        if (j == c.head_w[i]) continue;
                        if (banned(i, j)) continue;
                    }
                    u64 stampv = ((u64) part << 32) | i;
                    link(i, j, stampv, 1, ka, kb);
                    if (c.nv.complements) link(c.nv.mirror(j), c.nv.mirror(i), stampv, 0, ka, kb);  // src/global.h:110-112
                    break;
                }
            }
        }
    }
};

// ---- pointer doubling in ONE cooperative kernel ---------------------------------------------------------------------------
// The validation of a level contracts this level's edges by pointer doubling: ceil(log2(ne)) + 1 rounds, each a pass over the ne
// slots that must see the previous round complete.  As separate launches that was 444 of the 1263 launches of a 126 k-node input
// (profiles/r02e_path_stage_310M.json), each ~7 us for microseconds of work.  Here the rounds are iterations of one persistent
// grid separated by grid-wide barriers, and the loop ends as soon as a round found nothing left to jump over (chains made of this
// level's edges are short: a handful of rounds instead of 17); slots on a cycle never resolve and keep the loop going for the full
// count, exactly as before.  Results always end in the `a` arrays.
#ifdef __CUDACC__
#include <cooperative_groups.h>
__global__ void __launch_bounds__(256) kc_doubling_kernel(u32 *jump_a, u32 *jump_b, u32 *fin_a, u32 *fin_b, u64 *max_a, u64 *max_b, u32 ne, int rounds,
                                                          u32 *active /*[3], zeroed*/, const u32 *ne_dev /* non-null: the slot count lives on the device, ne is its upper bound */) {
    cooperative_groups::grid_group grid = cooperative_groups::this_grid();
    if (ne_dev) ne = *ne_dev;
    u32 *ja = jump_a, *jb = jump_b, *fa = fin_a, *fb = fin_b;
    u64 *ma = max_a, *mb = max_b;
    const u32 stride = gridDim.x * blockDim.x;
    int it = 0;
    for (; it < rounds; ++it) {
        bool any = false;
        for (u32 r = blockIdx.x * blockDim.x + threadIdx.x; r < ne; r += stride) {
            const u32 j = ja[r];
            if (j == KC_NONE) {
                jb[r] = KC_NONE;
                fb[r] = fa[r];
                mb[r] = ma[r];
            } else {
                any = true;
                jb[r] = ja[j];
                fb[r] = fa[j];
                const u64 m1 = ma[r], m2 = ma[j];
                mb[r] = m1 > m2 ? m1 : m2;
            }
        }
        if (__syncthreads_or(any) && threadIdx.x == 0) atomicOr(&active[it % 3], 1u);
        // the flag of the NEXT round: last read after the barrier of round it - 2, which every thread has left (all passed the barrier of
        // round it - 1); with only two flags a slow thread could still be reading the one being cleared
        if (blockIdx.x == 0 && threadIdx.x == 0) active[(it + 1) % 3] = 0;
        grid.sync();
        u32 *t = ja; ja = jb; jb = t;
        t = fa; fa = fb; fb = t;
        u64 *m = ma; ma = mb; mb = m;
        const u32 more = *reinterpret_cast<volatile u32 *>(&active[it % 3]);
        if (!more) {  // every slot was resolved BEFORE this round: it only copied a -> b
            ++it;
            break;
        }
    }
    if (ja != jump_a) {  // an odd number of rounds: bring the results home
        grid.sync();
        for (u32 r = blockIdx.x * blockDim.x + threadIdx.x; r < ne; r += stride) {
            jump_a[r] = ja[r];
            fin_a[r] = fa[r];
            max_a[r] = ma[r];
        }
    }
}
#endif

#include "small_engine.cuh"

// ---- engine -------------------------------------------------------------------------------------------
struct EngineStats {
    u64 levels_run = 0, tuples_sorted = 0, groups = 0, edges = 0, ban_rounds = 0, bans = 0;
};

template <class Exec, int L> struct Engine {
    Exec &ex;
    NodeView<L> nv;
    PathState st;
    bool strict;
    bool lower_bound;
    bool use_small = true;      // hand the tail of the level loop to the single-CTA kernel (small_engine.cuh)
    bool fast_levels = true;    // queue a whole level without host round trips and read its counts back once (run_level)
    int small_threads_opt = 0;  // 0 = by size; 256 / 512 (option "small_threads")
    EngineStats stats;

    // live end lists (ascending node id); nullptr = identity 0..N-1
    u32 *live_s = nullptr, *live_p = nullptr;
    u32 *list_buf[4] = {nullptr, nullptr, nullptr, nullptr};  // live_s generations 0 / 1, live_p generations 0 / 1
    int list_gen = 0;
    u64 n_s = 0, n_p = 0;
    u32 *head_w, *tail_w, *slot_of;
    u64 *stamp;
    u8 *prim, *ban_flag;
    u32 *ban_i, *ban_j, *ban_ctr;
    static const u32 BAN_CAP = 1u << 20;

    Engine(Exec &e, const NodeView<L> &v, bool strict_, bool lower_bound_) : ex(e), nv(v), strict(strict_), lower_bound(lower_bound_) {}

    // Speculative tail (kcgpu.cu): the real node count is on the device ({n, N} at n_dev) and nv holds its cap; the caller's kernel
    // initialised the state, the identity live lists and the small engine's level masks (small_masks), and the status words of the
    // single-CTA engine go to small_status, which the caller reads back with its own results (apply_small_status).
    const u32 *n_dev = nullptr;
    u32 *small_status = nullptr, *small_masks = nullptr;

    void alloc_state() {
        const u64 N = nv.N;
        st.edge_from = ex.template alloc<u32>(N);
        st.edge_to = ex.template alloc<u32>(N);
        st.ovl = ex.template alloc<u8>(N);
        st.chain_head = ex.template alloc<u32>(N);
        st.chain_tail = ex.template alloc<u32>(N);
        head_w = ex.template alloc<u32>(N);
        tail_w = ex.template alloc<u32>(N);
        slot_of = ex.template alloc<u32>(N);
        stamp = ex.template alloc<u64>(N);
        prim = ex.template alloc<u8>(N);
        ban_flag = ex.template alloc<u8>(N);
        ban_i = ex.template alloc<u32>(BAN_CAP);
        ban_j = ex.template alloc<u32>(BAN_CAP);
        ban_ctr = ex.template alloc<u32>(4);
    }

    void init_state() {
        alloc_state();
        const u64 N = nv.N;
        // one kernel instead of five fills and a kernel: on a genome the stage is a dozen tiny operations, each ~2 us of stream time
        PathState s = st;
        u8 *bf = ban_flag;
        u32 *bc = ban_ctr;
        ex.for_each(N, [=] KC_HD_LAMBDA(u64 v) {
            s.edge_from[v] = KC_NONE;
            s.edge_to[v] = KC_NONE;
            s.ovl[v] = 255;
            bf[v] = 0;
            s.chain_head[v] = (u32) v;
            s.chain_tail[v] = (u32) v;
            if (v < 4) bc[v] = 0;
        });
        if (N < 4) ex.fill_bytes(ban_ctr, 0, 16);
        n_s = n_p = N;
    }

    // Runs levels d = k-1 .. 0 (src/global.h:63).
    void run() {
        for (int d = nv.k - 1; d >= 0; --d) {
            const u64 done = lower_bound ? 0 : (nv.complements ? 2 : 1);
            if (n_s <= done) break;  // one path (two mirror paths) left: nothing can merge any more
            if (run_small(d)) break;
            run_level(d);
        }
    }

    u32 *small_out = nullptr;  // device status words of a launched kc_small_engine_kernel that have not been checked yet
    int small_d = 0;

    // Deferred error check + statistics of run_small (synchronises the stream).
    void check_small() {
#ifdef __CUDACC__
        if constexpr (Exec::is_device) {
            if (!small_out) return;
            u32 h[KC_SMALL_STATUS_WORDS];
            ex.read_n(small_out, h, KC_SMALL_STATUS_WORDS);
            small_out = nullptr;
            apply_small_status(h);
        }
#endif
    }

    // Statistics and error of a single-CTA engine run from its status words (read back by check_small or by the caller).
    void apply_small_status(const u32 *h) {
        if (std::getenv("KC_TRACE")) {
            std::fprintf(stderr, "[kc_trace] small engine: n_s=%llu n_p=%llu levels=%u groups=%u edges=%u ban_rounds=%u bans=%u; clocks per level (* = run):",
                         (unsigned long long) n_s, (unsigned long long) n_p, h[1], h[2], h[3], h[4], h[5]);
            for (int dd = small_d; dd >= 0; --dd) std::fprintf(stderr, " d%d=%u%s", dd, h[8 + dd] & 0x7FFFFFFFu, (h[8 + dd] >> 31) ? "*" : "");
            std::fprintf(stderr, "; phases: stage+mask=%u tuples=%u sort=%u groups=%u replay=%u validate+commit=%u lists=%u writeback=%u\n", h[136], h[137],
                         h[138], h[139], h[140], h[141], h[142], h[143]);
        }
        if (h[0]) KC_THROW(KC_ERR_INTERNAL, "ban list overflow");
        stats.levels_run += h[1];
        stats.groups += h[2];
        stats.edges += h[3];
        stats.ban_rounds += h[4];
        stats.bans += h[5];
    }

    // Runs levels d..0 in one kernel when the free ends fit in shared memory.  Device policy only.
    bool run_small(int d) {
#ifdef __CUDACC__
        if constexpr (Exec::is_device) {
            if (!use_small || lower_bound || n_s + n_p > SmallCfg<L>::T) return false;
            if (!live_s) {  // identity lists were implicit
                u32 *a = ex.template alloc<u32>(n_s), *b = ex.template alloc<u32>(n_p);
                ex.for_each(nv.N, [=] KC_HD_LAMBDA(u64 i) {
                    a[i] = (u32) i;
                    b[i] = (u32) i;
                });
                live_s = a;
                live_p = b;
            }
            SmallEngineArgs<L> a;
            a.nv = nv;
            a.st = st;
            a.live_s_a = live_s;
            a.live_p_a = live_p;
            a.live_s_b = ex.template alloc<u32>(n_s);
            a.live_p_b = ex.template alloc<u32>(n_p);
            a.n_s = (u32) n_s;
            a.n_p = (u32) n_p;
            a.head_w = head_w;
            a.tail_w = tail_w;
            a.slot_of = slot_of;
            a.stamp = stamp;
            a.prim = prim;
            a.ban_flag = ban_flag;
            a.ban_i = ban_i;
            a.ban_j = ban_j;
            a.ban_cap = BAN_CAP;
            a.d_start = d;
            a.strict = strict;
            // status words, then the level masks: [4] for the whole problem, then four words per end (two copies each: they travel with
            // the live lists); one allocation, one fill
            u32 *lvl_mask;
            if (n_dev) {
                a.out = small_status;
                lvl_mask = small_masks;
            } else {
                a.out = ex.template alloc<u32>(KC_SMALL_STATUS_WORDS + kc_small_mask_words(n_s, n_p) + 4 * (n_s + n_p));
                lvl_mask = a.out + KC_SMALL_STATUS_WORDS;
                ex.fill_bytes(a.out, 0, (KC_SMALL_STATUS_WORDS + kc_small_mask_words(n_s, n_p)) * 4);
            }
            a.n_dev = n_dev;
            a.lvl_mask_in = lvl_mask;
            a.end_mask_s_a = lvl_mask + 4;
            a.end_mask_p_a = a.end_mask_s_a + 4 * n_s;
            a.end_mask_s_b = a.end_mask_p_a + 4 * n_p;
            a.end_mask_p_b = a.end_mask_s_b + 4 * n_s;
            const int mask_smem = (int) (SmallCfg<L>::T * sizeof(KWord<L + 1>));
            static KcDevOnce once;  // function attributes are per device
            once.run([&](int) {
                KC_CUDA(cudaFuncSetAttribute(kc_small_engine_kernel<L>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int) SmallCfg<L>::SMEM));
                KC_CUDA(cudaFuncSetAttribute(kc_small_level_mask_kernel<L>, cudaFuncAttributeMaxDynamicSharedMemorySize, mask_smem));
            });
            {   // which levels can accept an edge at all: one CTA per two levels (the engine kernel used to do this alone)
                typename Exec::Scope sc(ex, KP_SMALL_ENGINE, 0);
                const u32 per_cta = kc_small_mask_levels_per_cta<L>((u32) n_s, (u32) n_p);
                ex.launch(kc_small_level_mask_kernel<L>, (unsigned) kc_div_up((u64) d + 1, per_cta), 256, mask_smem, nv, (const u32 *) live_s,
                          (const u32 *) live_p, (u32) n_s, (u32) n_p, d, lvl_mask, a.end_mask_s_a, a.end_mask_p_a, n_dev);
            }
            {
                typename Exec::Scope sc(ex, KP_SMALL_ENGINE, 0);
                // (measured: one warp instead of 256 threads makes the kernel 1.7x slower on configs[1] — the levels are
                // bound by the work per phase, not by the block barriers)
                // 512 threads once the sort has work for them: two threads per tuple in the rank sort (129..256 tuples), more than two
                // items per thread in the bitonic network (> 512 tuples)
                const u64 nt0 = n_s + n_p;
                // (speculative tail: the count is not known here; 256 vs 512 threads is within 1.5 % at 50 records, r02z_small_engine_trace.txt)
                const unsigned small_threads = small_threads_opt ? (unsigned) small_threads_opt
                                               : n_dev || (nt0 > 128 && nt0 <= 256) || nt0 > 512 ? 512u : 256u;
                ex.launch(kc_small_engine_kernel<L>, 1, small_threads, SmallCfg<L>::SMEM, a);
            }
            // The status words are read back by check_small() after the caller's next synchronisation point: the kernels of the
            // emission stage are queued behind this one without a host round trip.
            small_out = n_dev ? nullptr : a.out;
            small_d = d;
            return true;
        }
#endif
        (void) d;
        return false;
    }

    void run_level(int d) {
        typedef KWord<L + 1> TW;
        const u64 nt = n_s + n_p;
        if (n_s == 0 || n_p == 0) return;
        ++stats.levels_run;
        stats.tuples_sorted += nt;
        if (!list_buf[0]) {  // two generations of each live list, allocated once (the lists only shrink): the next generation goes where the one before last was
            for (int i = 0; i < 4; ++i) list_buf[i] = ex.template alloc<u32>(i < 2 ? n_s : n_p);
        }
        size_t mark = ex.arena->mark();
        TW *T = ex.template alloc<TW>(nt);
        TW *T2 = ex.template alloc<TW>(nt);
        const NodeView<L> v = nv;
        // The 16 prefix batches of src/global.h:48,66-72 only fix the reference's tie order.  It is reproduced for -S
        // input (strict); from FASTA the reference's own node order is khash order, i.e. unspecified, so every prefix
        // goes into batch 0 and a group is replayed with one pass over its suffixes instead of 16.
        const u32 batch = strict ? nv.N / 16 + 1 : nv.N + 1;
        const u32 *ls = live_s, *lp = live_p;
        const u64 ns = n_s, np = n_p;
        u32 *hw = head_w, *tw = tail_w;
        const PathState s = st;
        // 1. tuples (+ working copies of the chain ends of the live nodes)
        ex.for_each(nt, [=] KC_HD_LAMBDA(u64 i) {
            if (i < ns) {
                u32 x = ls ? ls[i] : (u32) i;
                T[i] = tuple_make(kmer_suffix(v.last_kmer(x), d), (u64) x);
                hw[x] = s.chain_head[x];
            } else {
                u32 x = lp ? lp[i - ns] : (u32) (i - ns);
                u64 meta = KC_ROLE_P | ((u64) (x / batch) << 32) | (u64) (u32) ~x;
                T[i] = tuple_make(kmer_prefix(v.first_kmer(x), v.k, d), meta);
                tw[x] = s.chain_tail[x];
            }
        }, KP_TUPLES, nt * (sizeof(KWord<L>) + sizeof(TW)));
        // 2. sort by (key, role, batch, id order)
        exec_sort<L + 1>(ex, T, T2, nt, 64 + 2 * d);
        // 3. active groups = positions where a prefix run starts right after a suffix run of the same key
        u32 *group_pstart = ex.template alloc<u32>(np);
        const TW *Tc = T;
        auto is_group = [=] KC_HD_LAMBDA(u64 i) {
            if (i == 0) return false;
            TW a = Tc[i - 1], b = Tc[i];
            return tuple_is_prefix(b) && !tuple_is_prefix(a) && tuple_key(a) == tuple_key(b);
        };
        auto put_group = [=] KC_HD_LAMBDA(u64 i, u32 r) { group_pstart[r] = (u32) i; };
        LevelCtx<L> c;
        c.nv = nv;
        c.st = st;
        c.T = T;
        c.nt = nt;
        c.d = d;
        c.batch = batch;
        c.head_w = head_w;
        c.tail_w = tail_w;
        c.stamp = stamp;
        c.prim = prim;
        c.ban_flag = ban_flag;
        c.ban_i = ban_i;
        c.ban_j = ban_j;
        c.n_bans = 0;
        c.check_cycles = !lower_bound;
        u32 *new_tail = ex.template alloc<u32>(ns);
        u32 *so = slot_of;
        auto has_edge = [=] KC_HD_LAMBDA(u64 i) { return s.edge_from[ls ? ls[i] : (u32) i] != KC_NONE; };
        auto put_edge = [=] KC_HD_LAMBDA(u64 i, u32 r) {
            u32 x = ls ? ls[i] : (u32) i;
            new_tail[r] = x;
            so[x] = r;
        };
        u64 n_groups = 0, n_edges = 0;
        u32 n_bans = 0;
        bool settled = false, lists_done = false, cycles_pending = false;
#ifdef __CUDACC__
        if constexpr (Exec::is_device) if (fast_levels && (lower_bound || doubling_blocks() > 0)) {
            // The whole level queued WITHOUT a host round trip, as if it had no cycle (nearly every level): groups, replay, this level's
            // edges, pointer doubling, commit (skipped on the device if a cycle turns up), the next live lists — every count stays on
            // the device, kernels are launched for its upper bound and check it — then ONE read-back of {groups, edges, cycle slots, new
            // list sizes}.  Five synchronising read-backs per level used to separate these steps: on a 126 k-node genome the stage was
            // bound by them, not by work (profiles/r02k_path_stage_310M.json).  A cycle (rare) falls into the step-by-step loop below.
            u64 *cells = ex.template alloc<u64>(6);  // groups, edges, new n_s, new n_p, cycle slots, min over the cycles of the max stamp
            ex.fill_bytes(cells, 0, 40);
            ex.fill_bytes(cells + 5, 0xFF, 8);
            u32 *c_groups = reinterpret_cast<u32 *>(cells), *c_edges = reinterpret_cast<u32 *>(cells + 1);
            u32 *c_ns = reinterpret_cast<u32 *>(cells + 2), *c_np = reinterpret_cast<u32 *>(cells + 3);
            ex.compact_if_nosync(nt, is_group, put_group, c_groups);
            {
                SimulatePairFn<L> sim{c, group_pstart};
                ex.for_each(ns < np ? ns : np, [=] __device__(u64 g) {
                    if (g < *c_groups) sim(g);
                }, KP_SIMULATE);
            }
            ex.compact_if_nosync(ns, has_edge, put_edge, c_edges);
            bool queued = true;
            u32 *jump_a = nullptr, *fin_a = nullptr;
            u64 *max_a = nullptr;
            if (!lower_bound) {
                const u32 ub = (u32) ns;
                jump_a = ex.template alloc<u32>(ub);
                u32 *jump_b = ex.template alloc<u32>(ub);
                fin_a = ex.template alloc<u32>(ub);
                u32 *fin_b = ex.template alloc<u32>(ub);
                max_a = ex.template alloc<u64>(ub);
                u64 *max_b = ex.template alloc<u64>(ub);
                const u64 *stp = stamp;
                u32 *ja = jump_a, *fa = fin_a;
                u64 *ma = max_a;
                ex.for_each(ub, [=] __device__(u64 r) {
                    if (r >= *c_edges) return;
                    u32 x = new_tail[r];
                    u32 t = s.chain_tail[s.edge_from[x]];
                    bool cont = s.edge_from[t] != KC_NONE;
                    ja[r] = cont ? so[t] : KC_NONE;
                    fa[r] = t;
                    ma[r] = stp[x];
                }, KP_DOUBLING, (u64) ub * 36);
                queued = doubling_fused(jump_a, jump_b, fin_a, fin_b, max_a, max_b, ub, kc_ceil_log2(ub) + 1, c_edges);
                if (queued) {
                    ex.for_each(ub, [=] __device__(u64 r) {
                        if (r < *c_edges && ja[r] != KC_NONE) {
                            atomicAdd((kc_ull *) &cells[4], (kc_ull) 1);
                            atomicMin((kc_ull *) &cells[5], (kc_ull) ma[r]);
                        }
                    });
                    ex.for_each(ub, [=] __device__(u64 r) {  // 7. commit the chain ends, unless a cycle was found
                        if (r >= *c_edges || cells[4] != 0) return;
                        u32 x = new_tail[r];
                        u32 h = s.chain_head[x];
                        if (s.edge_to[h] == KC_NONE) {
                            u32 t = fa[r];
                            s.chain_tail[h] = t;
                            s.chain_head[t] = h;
                        }
                    }, KP_COMMIT, (u64) ub * 16);
                }
            }
            if (queued) {
                const u32 *src_s = live_s, *src_p = live_p;
                u32 *dst_s = list_buf[list_gen], *dst_p = list_buf[2 + list_gen];
                ex.compact_if_nosync(ns, [=] __device__(u64 i) { return s.edge_from[src_s ? src_s[i] : (u32) i] == KC_NONE; },
                                     [=] __device__(u64 i, u32 r) { dst_s[r] = src_s ? src_s[i] : (u32) i; }, c_ns);
                ex.compact_if_nosync(np, [=] __device__(u64 i) { return s.edge_to[src_p ? src_p[i] : (u32) i] == KC_NONE; },
                                     [=] __device__(u64 i, u32 r) { dst_p[r] = src_p ? src_p[i] : (u32) i; }, c_np);
                u64 h[5];
                ex.read_n(cells, h, 5);
                n_groups = h[0];
                n_edges = h[1];
                stats.groups += n_groups;
                if (h[4] == 0) {  // no cycle: the level stands
                    settled = true;
                    if (n_edges) {
                        live_s = dst_s;
                        live_p = dst_p;
                        list_gen ^= 1;
                        n_s = h[2];
                        n_p = h[3];
                    }
                    lists_done = true;
                } else {  // ban the cycle closers (validate_and_commit's last step) and replay step by step
                    const u64 *stp = stamp;
                    const u32 *ja = jump_a;
                    const u64 *ma = max_a;
                    const bool only_first = strict;
                    const NodeView<L> v = nv;
                    const u8 *pr = prim;
                    u32 *bi = ban_i, *bj = ban_j, *bc = ban_ctr;
                    u8 *bf = ban_flag;
                    const u32 cap = BAN_CAP;
                    ex.for_each(n_edges, [=] __device__(u64 r) {
                        if (ja[r] == KC_NONE) return;
                        u32 x = new_tail[r];
                        if (stp[x] != ma[r]) return;
                        if (only_first && ma[r] != cells[5]) return;
                        u32 y = s.edge_from[x];
                        u32 pi = x, pj = y;
                        if (!pr[x]) {
                            pi = v.mirror(y);
                            pj = v.mirror(x);
                        }
                        u32 slot = atomicAdd(bc, v.complements ? 2u : 1u);
                        if (slot + 2 <= cap) {
                            bi[slot] = pi;
                            bj[slot] = pj;
                            bf[pi] = 1;
                            if (v.complements) {
                                bi[slot + 1] = v.mirror(pj);
                                bj[slot + 1] = v.mirror(pi);
                                bf[v.mirror(pj)] = 1;
                            }
                        }
                    });
                    cycles_pending = true;
                }
            }
        }
#endif
        if (!settled && !cycles_pending) {
            n_groups = ex.compact_if(nt, is_group, put_group);
            stats.groups += n_groups;
        }
        if (n_groups == 0) {
            ex.arena->release(mark);
            return;
        }
        while (!settled) {
            if (!cycles_pending) {
                // 4. replay every pair of groups
                c.n_bans = n_bans;
                SimulatePairFn<L> sim{c, group_pstart};
                ex.for_each(n_groups, sim, KP_SIMULATE);
                // 5. edges of this level, one slot per edge
                n_edges = ex.compact_if(ns, has_edge, put_edge);
                if (n_edges == 0 || lower_bound) break;
                if (validate_and_commit(c, new_tail, n_edges, n_bans)) break;
            }
            cycles_pending = false;
            // 6. cycles found: bans were appended; undo this level's edges and replay
            ++stats.ban_rounds;
            n_bans = ex.read(ban_ctr);
            if (n_bans > BAN_CAP) KC_THROW(KC_ERR_INTERNAL, "ban list overflow");
            ex.for_each(nt, [=] KC_HD_LAMBDA(u64 i) {
                if (i < ns) {
                    u32 x = ls ? ls[i] : (u32) i;
                    u32 y = s.edge_from[x];
                    if (y != KC_NONE) {
                        s.edge_to[y] = KC_NONE;
                        s.edge_from[x] = KC_NONE;
                        s.ovl[x] = 255;
                    }
                    hw[x] = s.chain_head[x];
                } else {
                    u32 x = lp ? lp[i - ns] : (u32) (i - ns);
                    tw[x] = s.chain_tail[x];
                }
            });
        }
        if (lower_bound && n_edges) commit_lower_bound();
        stats.edges += n_edges;
        stats.bans += n_bans;
        if (std::getenv("KC_TRACE"))
            std::fprintf(stderr, "[kc_trace] level d=%d: free ends %llu + %llu, groups %llu, edges %llu, bans %u\n", d, (unsigned long long) ns, (unsigned long long) np,
                         (unsigned long long) n_groups, (unsigned long long) n_edges, n_bans);
        // clear ban flags for the next level
        if (n_bans) {
            u8 *bf = ban_flag;
            const u32 *bi = ban_i;
            ex.for_each(n_bans, [=] KC_HD_LAMBDA(u64 b) { bf[bi[b]] = 0; });
            ex.fill_bytes(ban_ctr, 0, 16);
        }
        ex.arena->release(mark);
        // 8. shrink the live lists.  Only a level that accepted edges changes them; the lists only ever shrink, so the new ones are
        //    compacted straight into buffers of the old size (one compaction per list instead of count + allocate + compact)
        if (n_edges && !lists_done) {
            const u32 *src_s = live_s, *src_p = live_p;
            u32 *dst_s = list_buf[list_gen], *dst_p = list_buf[2 + list_gen];
            list_gen ^= 1;
            n_s = ex.compact_if(
                ns, [=] KC_HD_LAMBDA(u64 i) { return s.edge_from[src_s ? src_s[i] : (u32) i] == KC_NONE; },
                [=] KC_HD_LAMBDA(u64 i, u32 r) { dst_s[r] = src_s ? src_s[i] : (u32) i; });
            n_p = ex.compact_if(
                np, [=] KC_HD_LAMBDA(u64 i) { return s.edge_to[src_p ? src_p[i] : (u32) i] == KC_NONE; },
                [=] KC_HD_LAMBDA(u64 i, u32 r) { dst_p[r] = src_p ? src_p[i] : (u32) i; });
            live_s = dst_s;
            live_p = dst_p;
        }
    }

#ifdef __CUDACC__
    // All rounds of the doubling in one cooperative launch (kc_doubling_kernel); false = not available, the caller loops over launches.
    // co-resident blocks of kc_doubling_kernel on this device; 0 = no cooperative launch
    static int doubling_blocks() {
        static KcDevOnce once;
        static int max_blocks[KC_MAX_DEVICES];
        const int dev = once.run([&](int dv) {
            int coop = 0, per_sm = 0;
            KC_CUDA(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dv));
            KC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kc_doubling_kernel, 256, 0));
            max_blocks[dv] = coop ? per_sm * kc_sm_count(dv) : 0;
        });
        return max_blocks[dev];
    }
    bool doubling_fused(u32 *jump_a, u32 *jump_b, u32 *fin_a, u32 *fin_b, u64 *max_a, u64 *max_b, u32 ne, int rounds, const u32 *ne_dev = nullptr) {
        const int max_blocks_dev = doubling_blocks();
        if (max_blocks_dev <= 0) return false;
        u32 *active = ex.template alloc<u32>(4);
        ex.fill_bytes(active, 0, 16);
        u32 blocks = (u32) kc_div_up((u64) ne, 256);
        if (blocks > (u32) max_blocks_dev) blocks = (u32) max_blocks_dev;
        void *args[] = {&jump_a, &jump_b, &fin_a, &fin_b, &max_a, &max_b, &ne, &rounds, &active, &ne_dev};
        typename Exec::Scope sc(ex, KP_DOUBLING, (u64) ne * 32 * 4);
        KC_CUDA(cudaLaunchCooperativeKernel(reinterpret_cast<void *>(kc_doubling_kernel), dim3(blocks), dim3(256), args, 0, ex.stream));
        ++ex.launches;
        return true;
    }
#endif

    // Pointer doubling over this level's edges with chains contracted.  Returns true when the edge set is
    // acyclic (and the chain ends have been updated); false after appending bans for the cycle closers.
    bool validate_and_commit(const LevelCtx<L> &c, const u32 *new_tail, u64 n_edges, u32 n_bans_before) {
        size_t mark = ex.arena->mark();
        const u32 ne = (u32) n_edges;
        u32 *jump_a = ex.template alloc<u32>(ne), *jump_b = ex.template alloc<u32>(ne);
        u32 *fin_a = ex.template alloc<u32>(ne), *fin_b = ex.template alloc<u32>(ne);
        u64 *max_a = ex.template alloc<u64>(ne), *max_b = ex.template alloc<u64>(ne);
        const PathState s = st;
        const u32 *so = slot_of;
        const u64 *stp = stamp;
        ex.for_each(ne, [=] KC_HD_LAMBDA(u64 r) {
            u32 x = new_tail[r];
            u32 t = s.chain_tail[s.edge_from[x]];  // tail of the chain x now leads into (level-start snapshot)
            bool cont = s.edge_from[t] != KC_NONE;
            jump_a[r] = cont ? so[t] : KC_NONE;
            fin_a[r] = t;
            max_a[r] = stp[x];
        }, KP_DOUBLING, (u64) ne * 36);
        int rounds = kc_ceil_log2(ne) + 1;
        bool fused = false;
#ifdef __CUDACC__
        if constexpr (Exec::is_device) fused = doubling_fused(jump_a, jump_b, fin_a, fin_b, max_a, max_b, ne, rounds);
#endif
        for (int it = 0; it < rounds && !fused; ++it) {
            const u32 *ja = jump_a, *fa = fin_a;
            const u64 *ma = max_a;
            u32 *jb = jump_b, *fb = fin_b;
            u64 *mb = max_b;
            ex.for_each(ne, [=] KC_HD_LAMBDA(u64 r) {
                u32 j = ja[r];
                if (j == KC_NONE) {
                    jb[r] = KC_NONE;
                    fb[r] = fa[r];
                    mb[r] = ma[r];
                } else {
                    jb[r] = ja[j];
                    fb[r] = fa[j];
                    u64 m1 = ma[r], m2 = ma[j];
                    mb[r] = m1 > m2 ? m1 : m2;
                }
            }, KP_DOUBLING, (u64) ne * 32);
            u32 *t = jump_a; jump_a = jump_b; jump_b = t;
            t = fin_a; fin_a = fin_b; fin_b = t;
            u64 *m = max_a; max_a = max_b; max_b = m;
        }
        // unresolved slots lie on cycles
        u64 *cell = ex.template alloc<u64>(2);  // [0] = number of cycle slots, [1] = min over cycles of the max stamp
        ex.fill_bytes(cell, 0, 8);
        ex.fill_bytes(cell + 1, 0xFF, 8);
        {
            const u32 *ja = jump_a;
            const u64 *ma = max_a;
            ex.for_each(ne, [=] KC_HD_LAMBDA(u64 r) {
                if (ja[r] != KC_NONE) {
                    KC_ATOMIC_ADD((kc_ull *) &cell[0], (kc_ull) 1);
                    KC_ATOMIC_MIN((kc_ull *) &cell[1], (kc_ull) ma[r]);
                }
            });
        }
        u64 n_cyc = ex.read(cell);
        if (n_cyc == 0) {
            // 7. commit chain ends (src/global.h:116-120 for the whole level at once)
            const u32 *fa = fin_a;
            ex.for_each(ne, [=] KC_HD_LAMBDA(u64 r) {
                u32 x = new_tail[r];
                u32 h = s.chain_head[x];
                if (s.edge_to[h] == KC_NONE) {  // x's chain is the first of its merged run
                    u32 t = fa[r];
                    s.chain_tail[h] = t;
                    s.chain_head[t] = h;
                }
            }, KP_COMMIT, (u64) ne * 16);
            ex.arena->release(mark);
            return true;
        }
        {
            const u32 *ja = jump_a;
            const u64 *ma = max_a;
            const bool only_first = strict;
            const NodeView<L> v = nv;
            const u8 *pr = prim;
            u32 *bi = ban_i, *bj = ban_j, *bc = ban_ctr;
            u8 *bf = ban_flag;
            const u32 cap = BAN_CAP;
            ex.for_each(ne, [=] KC_HD_LAMBDA(u64 r) {
                if (ja[r] == KC_NONE) return;
                u32 x = new_tail[r];
                if (stp[x] != ma[r]) return;                 // not the closer of its cycle
                if (only_first && ma[r] != cell[1]) return;  // strict: only the earliest divergence is certain
                u32 y = s.edge_from[x];
                u32 pi = x, pj = y;
                if (!pr[x]) {  // mirror edge: its primary is rc(y) -> rc(x)
                    pi = v.mirror(y);
                    pj = v.mirror(x);
                }
                u32 slot = KC_ATOMIC_ADD(bc, v.complements ? 2u : 1u);
                if (slot + 2 <= cap) {
                    bi[slot] = pi;
                    bj[slot] = pj;
                    bf[pi] = 1;
                    if (v.complements) {  // the same pair seen from the other strand stays refused as well
                        bi[slot + 1] = v.mirror(pj);
                        bj[slot + 1] = v.mirror(pi);
                        bf[v.mirror(pj)] = 1;
                    }
                }
            });
        }
        (void) n_bans_before;
        ex.arena->release(mark);
        return false;
    }

    // Lower-bound mode keeps cycles (src/lower_bound.h:9-22); chain ends are not needed afterwards because the
    // rc / cycle tests are off, but first/last are still spliced by the reference — irrelevant to its result.
    void commit_lower_bound() {}
};
