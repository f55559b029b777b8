// Small-problem tail of the overlap stage: once the free suffix + prefix ends fit in shared memory, every remaining
// level d runs inside ONE single-CTA kernel — tuples are built and sorted in shared memory, group pairs are
// replayed by the same SimulatePairFn the multi-kernel path uses, and the cycle validation / ban / replay loop of
// engine.cuh is done with __syncthreads() instead of kernel boundaries.  Results are identical to the host-driven
// levels (same code for the pair replay, same ban rule); what disappears is ~10 launches and 2-3 host
// synchronisations per level, which is what a genome-like input (few runs left after the first levels) pays for.
#pragma once
// (included from the middle of engine.cuh, after LevelCtx / SimulatePairFn)

// Status words of one kc_small_engine_kernel run (SmallEngineArgs::out), and the zeroed words of its level masks that follow them:
// [4] for the whole problem, then four words per end (the second copies of the ping-pong pairs need no zeroing).
static const u32 KC_SMALL_STATUS_WORDS = 8 + 128 + 8;
KC_HD u64 kc_small_mask_words(u64 n_s, u64 n_p) { return 4 + 4 * (n_s + n_p); }

#ifdef __CUDACC__

template <int L> struct SmallCfg {
    static constexpr u32 T = L <= 2 ? 4096 : 2048;  // tuple capacity (free suffix ends + free prefix ends)
    static constexpr u32 H = T / 2;
    static constexpr u32 NS = 1024;  // up to this many virtual nodes the whole path state lives in shared memory
    static constexpr u32 RANK_SORT = 384;      // up to this many tuples: rank sort (no barriers) instead of the bitonic network
    // Staging the first / last k-mers of the nodes in shared memory next to the path state was tried and made the kernel slower:
    static constexpr bool STAGE_KMERS = false;  // measured on B200: 0.159 -> 0.179 ms at 100 free ends, 0.22 -> 0.25 at 200 (the k-mers were L1 hits already)
    static constexpr size_t SMEM = (size_t) T * sizeof(KWord<L + 1>) + (size_t) H * (4 * 6 + 8 * 2) + (size_t) NS * (8 + 4 * 7 + 3) +
                                   (STAGE_KMERS ? (size_t) NS * 2 * sizeof(KWord<L>) + 16 : 0);
};

template <int L> struct SmallEngineArgs {
    NodeView<L> nv;
    PathState st;
    u32 *live_s_a, *live_p_a, *live_s_b, *live_p_b;  // ping-pong live lists
    u32 n_s, n_p;
    u32 *head_w, *tail_w, *slot_of;
    u64 *stamp;
    u8 *prim, *ban_flag;
    u32 *ban_i, *ban_j;
    u32 ban_cap;
    int d_start;
    bool strict;
    u32 *out;  // [0] error, [1] levels run, [2] groups, [3] edges, [4] ban rounds, [5] bans, [8 + d] clocks spent in level d (KC_TRACE)
    const u32 *lvl_mask_in;  // [4] bit d: some (suffix, prefix) pair of the initial free ends agrees on d bases (kc_small_level_mask_kernel)
    // [4 * n_s], [4 * n_p]: the same per END (bit d of the four words of initial list position i: end i has a partner at level d);
    // ping-pong copies travel with the live lists
    u32 *end_mask_s_a, *end_mask_p_a, *end_mask_s_b, *end_mask_p_b;
    const u32 *n_dev;  // != nullptr: {n, N} on the device (speculative tail, kcgpu.cu); nv, n_s and n_p then hold their caps
};

// Levels of one CTA of kc_small_level_mask_kernel (host and device must agree): as many hash tables as fit next to the parked k-mers,
// at most KC_SMALL_MASK_LEVELS.  Few levels per CTA = many CTAs: the join of one level is independent of every other level.
static const u32 KC_SMALL_MASK_LEVELS = 2;
template <int L> KC_HD u32 kc_small_mask_table_slots(u32 n_p) {
    u32 H2 = 64;
    while (H2 < 2 * n_p) H2 <<= 1;
    return H2;
}
template <int L> KC_HD u32 kc_small_mask_levels_per_cta(u32 n_s, u32 n_p) {
    const u32 avail = (u32) ((SmallCfg<L>::T * sizeof(KWord<L + 1>) - (size_t) (n_s + n_p) * sizeof(KWord<L>)) / 4);
    u32 G = avail / kc_small_mask_table_slots<L>(n_p);
    if (G > KC_SMALL_MASK_LEVELS) G = KC_SMALL_MASK_LEVELS;
    return G < 1 ? 1 : G;
}

// Find out ONCE at which levels any free suffix can meet any free prefix.  The live sets only shrink, so a level whose bit is clear
// can never accept an edge and the engine skips it.  An EXACT hash join per level: the prefix keys of level d go into an
// open-addressing table of end indices (keys are compared through the parked k-mers, so there are no false positives — a bit filter
// lit up at every level once ~800 x 800 ends were alive, and all 31 levels of a 400-record genome ran at ~40 us each although only 11
// could accept an edge); the suffix keys probe it.  This used to be the first phase of the single-CTA engine kernel: 17 % of its
// clocks at 100 ends, 32 % at 800 (all (level, end) pairs through one CTA).  The levels are independent, so they now spread over
// (d_start + 1) / levels-per-CTA CTAs that run at the same time.
// The join also says WHICH ends have a partner at a level (end_mask_s / end_mask_p, bit d of the end's four words): an end without one
// can never be in an active group of that level, and the engine leaves it out of the level's tuples — at the high levels of a genome
// a handful of the ~200 free ends take part, and the tuple sort was 30 % of the engine's clocks.
template <int L>
__global__ void __launch_bounds__(256) kc_small_level_mask_kernel(NodeView<L> v, const u32 *__restrict__ ls, const u32 *__restrict__ lp, u32 n_s, u32 n_p,
                                                                  int d_start, u32 *mask_out /* [4], zeroed */, u32 *end_mask_s /* [4 n_s], zeroed */,
                                                                  u32 *end_mask_p /* [4 n_p], zeroed */, const u32 *n_dev /* see SmallEngineArgs */) {
    extern __shared__ __align__(16) unsigned char kc_smem_raw[];
    __shared__ u32 s_hits;
    const u32 tid = threadIdx.x, NT = blockDim.x;
    const u32 G = kc_small_mask_levels_per_cta<L>(n_s, n_p);  // from the sizes the grid was launched for
    if (n_dev) {  // the real counts are at most the caps: fewer k-mers to park, smaller tables
        v.n = n_dev[0];
        v.N = n_dev[1];
        n_s = n_p = v.N;
    }
    KWord<L> *pk = reinterpret_cast<KWord<L> *>(kc_smem_raw), *sk = pk + n_p;
    u32 *tab = reinterpret_cast<u32 *>(sk + n_s);
    const u32 H2 = kc_small_mask_table_slots<L>(n_p);
    const int d_hi = d_start - (int) (blockIdx.x * G);
    if (d_hi < 0) return;
    const u32 g = (u32) (d_hi + 1) < G ? (u32) (d_hi + 1) : G;  // levels d_hi, d_hi - 1, ..., d_hi - g + 1
    for (u32 i = tid; i < n_p; i += NT) pk[i] = v.first_kmer(lp[i]);
    for (u32 i = tid; i < n_s; i += NT) sk[i] = v.last_kmer(ls[i]);
    for (u32 i = tid; i < g * H2; i += NT) tab[i] = KC_NONE;
    if (tid == 0) s_hits = 0;
    __syncthreads();
    for (u32 item = tid; item < g * n_p; item += NT) {  // (level, prefix end) pairs spread over the whole block
        const u32 lev = item / n_p, i = item - lev * n_p;
        const int d = d_hi - (int) lev;
        u32 *tb = tab + lev * H2;
        const KWord<L> key = kmer_prefix(pk[i], v.k, d);
        u64 h = 0;
#pragma unroll
        for (int q = 0; q < L; ++q) h = (h ^ key.w[q]) * 0x9E3779B97F4A7C15ULL;
        u32 sl = (u32) (h >> 40) & (H2 - 1);
        while (true) {
            const u32 old = atomicCAS(&tb[sl], KC_NONE, i);
            if (old == KC_NONE || kmer_prefix(pk[old], v.k, d) == key) break;
            sl = (sl + 1) & (H2 - 1);
        }
    }
    __syncthreads();
    constexpr u32 PROBED = 0x80000000u;  // table entry: a suffix key has met this prefix key
    u32 hits = 0;
    for (u32 item = tid; item < g * n_s; item += NT) {
        const u32 lev = item / n_s, i = item - lev * n_s;
        const int d = d_hi - (int) lev;
        u32 *tb = tab + lev * H2;
        const KWord<L> key = kmer_suffix(sk[i], d);
        u64 h = 0;
#pragma unroll
        for (int q = 0; q < L; ++q) h = (h ^ key.w[q]) * 0x9E3779B97F4A7C15ULL;
        u32 sl = (u32) (h >> 40) & (H2 - 1);
        while (true) {
            const u32 o = tb[sl];
            if (o == KC_NONE) break;
            if (kmer_prefix(pk[o & ~PROBED], v.k, d) == key) {
                hits |= 1u << lev;
                if (!(o & PROBED)) tb[sl] = o | PROBED;  // (several writers, one value)
                atomicOr(&end_mask_s[4 * i + ((u32) d >> 5)], 1u << (d & 31));
                break;
            }
            sl = (sl + 1) & (H2 - 1);
        }
    }
    if (hits) atomicOr(&s_hits, hits);
    __syncthreads();
    if (tid == 0) {
        const u32 hm = s_hits;
        for (u32 lev = 0; lev < g; ++lev)
            if ((hm >> lev) & 1u) atomicOr(&mask_out[(d_hi - (int) lev) >> 5], 1u << ((d_hi - (int) lev) & 31));
    }
    const u32 hm = s_hits;
    for (u32 item = tid; item < g * n_p; item += NT) {  // the prefix ends whose key was met
        const u32 lev = item / n_p, i = item - lev * n_p;
        if (!((hm >> lev) & 1u)) continue;
        const int d = d_hi - (int) lev;
        const u32 *tb = tab + lev * H2;
        const KWord<L> key = kmer_prefix(pk[i], v.k, d);
        u64 h = 0;
#pragma unroll
        for (int q = 0; q < L; ++q) h = (h ^ key.w[q]) * 0x9E3779B97F4A7C15ULL;
        u32 sl = (u32) (h >> 40) & (H2 - 1);
        while (true) {  // the key is in the table
            const u32 o = tb[sl];
            if (kmer_prefix(pk[o & ~PROBED], v.k, d) == key) {
                if (o & PROBED) atomicOr(&end_mask_p[4 * i + ((u32) d >> 5)], 1u << (d & 31));
                break;
            }
            sl = (sl + 1) & (H2 - 1);
        }
    }
}

template <int L> __global__ void __launch_bounds__(512) kc_small_engine_kernel(SmallEngineArgs<L> a) {
    typedef KWord<L + 1> TW;
    constexpr u32 TCAP = SmallCfg<L>::T, HCAP = SmallCfg<L>::H;
    extern __shared__ __align__(16) unsigned char kc_smem_raw[];
    TW *const T0 = reinterpret_cast<TW *>(kc_smem_raw);
    TW *T = T0;
    u64 *max0 = reinterpret_cast<u64 *>(T0 + TCAP);
    u64 *max1 = max0 + HCAP;
    u32 *group_pstart = reinterpret_cast<u32 *>(max1 + HCAP);
    u32 *new_tail = group_pstart + HCAP;
    u32 *jump0 = new_tail + HCAP, *jump1 = jump0 + HCAP, *fin0 = jump1 + HCAP, *fin1 = fin0 + HCAP;
    __shared__ u32 s_groups, s_edges, s_cyc, s_bans, s_live_s, s_live_p;
    __shared__ u32 lvl_mask[4];  // bit d: some (suffix, prefix) pair of the initial free ends agrees on d bases
    __shared__ kc_ull s_min;
    const u32 tid = threadIdx.x;
    const u32 NT = blockDim.x;  // 256, or one warp for tiny problems (block barriers then cost next to nothing)
    NodeView<L> v = a.nv;
    if (a.n_dev) {
        v.n = a.n_dev[0];
        v.N = a.n_dev[1];
    }
    PathState s = a.st;
    u32 *head_w = a.head_w, *tail_w = a.tail_w, *slot_of = a.slot_of;
    u64 *stamp = a.stamp;
    u8 *prim = a.prim, *ban_flag = a.ban_flag;
    // Small inputs (a genome: a few dozen first-occurrence runs): the replay of a big group is ONE thread chasing
    // edge / chain-end entries it has just written, i.e. an L2 round trip per access when the state is in global
    // memory.  With N <= NS the state is staged in shared memory for the whole kernel and written back at the end.
    const bool local_state = v.N <= SmallCfg<L>::NS;
    if (local_state) {
        constexpr u32 NS = SmallCfg<L>::NS;
        u64 *l_stamp = reinterpret_cast<u64 *>(fin1 + HCAP);
        u32 *l32 = reinterpret_cast<u32 *>(l_stamp + NS);
        u8 *l8 = reinterpret_cast<u8 *>(l32 + 7 * NS);
        for (u32 i = tid; i < v.N; i += NT) {
            l32[i] = s.edge_from[i];
            l32[NS + i] = s.edge_to[i];
            l32[2 * NS + i] = s.chain_head[i];
            l32[3 * NS + i] = s.chain_tail[i];
            l8[i] = s.ovl[i];
            l8[2 * NS + i] = 0;
        }
        s.edge_from = l32;
        s.edge_to = l32 + NS;
        s.chain_head = l32 + 2 * NS;
        s.chain_tail = l32 + 3 * NS;
        head_w = l32 + 4 * NS;
        tail_w = l32 + 5 * NS;
        slot_of = l32 + 6 * NS;
        stamp = l_stamp;
        s.ovl = l8;
        prim = l8 + NS;
        ban_flag = l8 + 2 * NS;
        if constexpr (SmallCfg<L>::STAGE_KMERS) {
            KWord<L> *lk = reinterpret_cast<KWord<L> *>((reinterpret_cast<uintptr_t>(l8 + 3 * NS) + 15) & ~(uintptr_t) 15);
            for (u32 i = tid; i < v.n; i += NT) {
                lk[i] = a.nv.first[i];
                lk[NS + i] = a.nv.last[i];
            }
            v.first = lk;
            v.last = lk + NS;
        }
        __syncthreads();
    }
    u32 n_s = a.n_dev ? v.N : a.n_s, n_p = a.n_dev ? v.N : a.n_p;
    u32 *ls = a.live_s_a, *lp = a.live_p_a, *ls2 = a.live_s_b, *lp2 = a.live_p_b;
    u32 *ms = a.end_mask_s_a, *mp = a.end_mask_p_a, *ms2 = a.end_mask_s_b, *mp2 = a.end_mask_p_b;
    __shared__ u32 s_nt;
    const u32 batch = a.strict ? v.N / 16 + 1 : v.N + 1;  // see Engine::run_level
    const u32 done = v.complements ? 2u : 1u;
    u32 st_levels = 0, st_groups = 0, st_edges = 0, st_rounds = 0, st_bans = 0;
    long long ph[8] = {0, 0, 0, 0, 0, 0, 0, 0};  // KC_TRACE: clocks per phase, summed over the levels (thread 0)
    long long ph_t = clock64();
#define KC_PH(i) do { const long long kc_now = clock64(); ph[i] += kc_now - ph_t; ph_t = kc_now; } while (0)

    // the levels at which any free suffix can meet any free prefix (kc_small_level_mask_kernel)
    if (tid < 4) lvl_mask[tid] = a.lvl_mask_in[tid];
    __syncthreads();

    KC_PH(0);  // state staging
    for (int d = a.d_start; d >= 0; --d) {
        if (n_s <= done || n_p == 0) break;
        const long long lvl_t0 = clock64();
        // A level whose bit is clear cannot accept an edge (the live sets only shrink): skipped without touching memory.
        if (!((lvl_mask[d >> 5] >> (d & 31)) & 1u)) continue;  // uniform: no barrier needed
        ++st_levels;
        const u32 n_live = n_s + n_p;
        T = T0;
        if (tid == 0) {
            s_nt = 0;
            s_groups = 0;
            s_bans = 0;
        }
        __syncthreads();
        // 1. working copies of the chain ends; tuples of the ends that had a partner at this level when the kernel started (the others
        //    cannot be in an active group; the order of the tuples is irrelevant, the sort follows)
        for (u32 i = tid; i < n_live; i += NT) {
            if (i < n_s) {
                u32 x = ls[i];
                head_w[x] = s.chain_head[x];
                if ((ms[4 * i + ((u32) d >> 5)] >> (d & 31)) & 1u) T[atomicAdd(&s_nt, 1u)] = tuple_make(kmer_suffix(v.last_kmer(x), d), (u64) x);
            } else {
                u32 x = lp[i - n_s];
                tail_w[x] = s.chain_tail[x];
                if ((mp[4 * (i - n_s) + ((u32) d >> 5)] >> (d & 31)) & 1u) {
                    u64 meta = KC_ROLE_P | ((u64) (x / batch) << 32) | (u64) (u32) ~x;
                    T[atomicAdd(&s_nt, 1u)] = tuple_make(kmer_prefix(v.first_kmer(x), v.k, d), meta);
                }
            }
        }
        for (u32 i = tid; i < n_live && i <= SmallCfg<L>::RANK_SORT; i += NT) group_pstart[i] = 0;  // partial ranks of the rank sort
        __syncthreads();
        const u32 nt = s_nt;
        KC_PH(1);  // tuples
        // 2. sort.  Tiny levels: every thread ranks its tuple against all others (tuples are distinct: they carry role
        // and node id) and drops it at its rank in the upper half of the tuple buffer — two barriers instead of the
        // 36+ of a bitonic network over 256 slots.
        if (nt <= SmallCfg<L>::RANK_SORT) {
            TW *dst = T0 + HCAP;
            const u32 P = nt ? (NT / nt < 8u ? NT / nt : 8u) : 0u;  // threads per tuple
            if (P >= 2) {
                // each of a tuple's P threads counts the smaller tuples in its share of the buffer (consecutive threads hold consecutive
                // tuples and walk the same share: the loads broadcast); the partial ranks meet in rk[] (zeroed in the tuple phase)
                u32 *rk = group_pstart;
                if (tid < nt * P) {
                    const u32 part = tid / nt, i = tid - part * nt;
                    const u32 j0 = part * nt / P, j1 = (part + 1) * nt / P;
                    const TW mine = T0[i];
                    u32 r = 0;
#pragma unroll 8
                    for (u32 j = j0; j < j1; ++j) r += T0[j] < mine ? 1u : 0u;
                    atomicAdd(&rk[i], r);
                }
                __syncthreads();
                for (u32 i = tid; i < nt; i += NT) dst[rk[i]] = T0[i];
            } else {
                for (u32 i = tid; i < nt; i += NT) {
                    const TW mine = T0[i];
                    u32 r = 0;
#pragma unroll 8
                    for (u32 j = 0; j < nt; ++j) r += T0[j] < mine ? 1u : 0u;
                    dst[r] = mine;
                }
            }
            T = dst;
            __syncthreads();
        } else {
            kc_block_bitonic<L + 1>(T, nt, NT);
        }
        KC_PH(2);  // sort
        // 3. active groups
        for (u32 i = tid + 1; i < nt; i += NT) {
            TW p = T[i - 1], q = T[i];
            if (tuple_is_prefix(q) && !tuple_is_prefix(p) && tuple_key(p) == tuple_key(q)) group_pstart[atomicAdd(&s_groups, 1u)] = i;
        }
        __syncthreads();
        const u32 n_groups = s_groups;
        st_groups += n_groups;
        KC_PH(3);  // group detection
        if (n_groups) {
            LevelCtx<L> c;
            c.nv = v;
            c.st = s;
            c.T = T;
            c.nt = nt;
            c.d = d;
            c.batch = batch;
            c.head_w = head_w;
            c.tail_w = tail_w;
            c.stamp = stamp;
            c.prim = prim;
            c.ban_flag = ban_flag;
            c.ban_i = a.ban_i;
            c.ban_j = a.ban_j;
            c.check_cycles = true;
            u32 n_bans = 0;
            while (true) {
                // 4. replay every pair of groups
                c.n_bans = n_bans;
                SimulatePairFn<L> sim{c, group_pstart};
                for (u32 g = tid; g < n_groups; g += NT) sim((u64) g);
                if (tid == 0) {
                    s_edges = 0;
                    s_cyc = 0;
                    s_min = ~0ULL;
                }
                __syncthreads();
                KC_PH(4);  // replay
                // 5. this level's edges
                for (u32 i = tid; i < n_s; i += NT) {
                    u32 x = ls[i];
                    if (s.edge_from[x] != KC_NONE) {
                        u32 r = atomicAdd(&s_edges, 1u);
                        new_tail[r] = x;
                        slot_of[x] = r;
                    }
                }
                __syncthreads();
                const u32 ne = s_edges;
                if (ne == 0) break;
                for (u32 r = tid; r < ne; r += NT) {
                    u32 x = new_tail[r];
                    u32 t = s.chain_tail[s.edge_from[x]];
                    bool cont = s.edge_from[t] != KC_NONE;
                    jump0[r] = cont ? slot_of[t] : KC_NONE;
                    fin0[r] = t;
                    max0[r] = stamp[x];
                }
                __syncthreads();
                u32 *ja = jump0, *jb = jump1, *fa = fin0, *fb = fin1;
                u64 *ma = max0, *mb = max1;
                int rounds = 1;
                while ((1u << (rounds - 1)) < ne) ++rounds;
                for (int it = 0; it < rounds; ++it) {
                    for (u32 r = tid; r < ne; r += NT) {
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
                    }
                    __syncthreads();
                    u32 *t32 = ja; ja = jb; jb = t32;
                    t32 = fa; fa = fb; fb = t32;
                    u64 *t64 = ma; ma = mb; mb = t64;
                }
                for (u32 r = tid; r < ne; r += NT)
                    if (ja[r] != KC_NONE) {
                        atomicAdd(&s_cyc, 1u);
                        atomicMin(&s_min, (kc_ull) ma[r]);
                    }
                __syncthreads();
                if (s_cyc == 0) {
                    // 7. commit the chain ends
                    for (u32 r = tid; r < ne; r += NT) {
                        u32 x = new_tail[r];
                        u32 h = s.chain_head[x];
                        if (s.edge_to[h] == KC_NONE) {
                            u32 t = fa[r];
                            s.chain_tail[h] = t;
                            s.chain_head[t] = h;
                        }
                    }
                    st_edges += ne;
                    __syncthreads();
                    break;
                }
                // 6. ban the cycle closers, undo the level, replay
                const kc_ull first_stamp = s_min;
                for (u32 r = tid; r < ne; r += NT) {
                    if (ja[r] == KC_NONE) continue;
                    u32 x = new_tail[r];
                    if (stamp[x] != ma[r]) continue;
                    if (a.strict && ma[r] != first_stamp) continue;
                    u32 y = s.edge_from[x];
                    u32 pi = x, pj = y;
                    if (!prim[x]) {
                        pi = v.mirror(y);
                        pj = v.mirror(x);
                    }
                    u32 slot = atomicAdd(&s_bans, v.complements ? 2u : 1u);
                    if (slot + 2 <= a.ban_cap) {
                        a.ban_i[slot] = pi;
                        a.ban_j[slot] = pj;
                        ban_flag[pi] = 1;
                        if (v.complements) {
                            a.ban_i[slot + 1] = v.mirror(pj);
                            a.ban_j[slot + 1] = v.mirror(pi);
                            ban_flag[v.mirror(pj)] = 1;
                        }
                    }
                }
                __syncthreads();
                n_bans = s_bans;
                ++st_rounds;
                if (n_bans + 2 > a.ban_cap) {
                    if (tid == 0) a.out[0] = 1;
                    return;
                }
                for (u32 i = tid; i < n_live; i += NT) {
                    if (i < n_s) {
                        u32 x = ls[i];
                        u32 y = s.edge_from[x];
                        if (y != KC_NONE) {
                            s.edge_to[y] = KC_NONE;
                            s.edge_from[x] = KC_NONE;
                            s.ovl[x] = 255;
                        }
                        head_w[x] = s.chain_head[x];
                    } else {
                        u32 x = lp[i - n_s];
                        tail_w[x] = s.chain_tail[x];
                    }
                }
                __syncthreads();
            }
            for (u32 b = tid; b < n_bans; b += NT) ban_flag[a.ban_i[b]] = 0;
            st_bans += n_bans;
            KC_PH(5);  // edges, cycle validation, commit
        }
        // 8. shrink the live lists (their order is irrelevant: the tuple sort orders by id)
        if (tid == 0) {
            s_live_s = 0;
            s_live_p = 0;
        }
        __syncthreads();
        for (u32 i = tid; i < n_s; i += NT) {
            u32 x = ls[i];
            if (s.edge_from[x] == KC_NONE) {
                const u32 to = atomicAdd(&s_live_s, 1u);
                ls2[to] = x;
                *reinterpret_cast<uint4 *>(ms2 + 4 * to) = *reinterpret_cast<const uint4 *>(ms + 4 * i);
            }
        }
        for (u32 i = tid; i < n_p; i += NT) {
            u32 x = lp[i];
            if (s.edge_to[x] == KC_NONE) {
                const u32 to = atomicAdd(&s_live_p, 1u);
                lp2[to] = x;
                *reinterpret_cast<uint4 *>(mp2 + 4 * to) = *reinterpret_cast<const uint4 *>(mp + 4 * i);
            }
        }
        __syncthreads();
        n_s = s_live_s;
        n_p = s_live_p;
        u32 *t32 = ls; ls = ls2; ls2 = t32;
        t32 = lp; lp = lp2; lp2 = t32;
        t32 = ms; ms = ms2; ms2 = t32;
        t32 = mp; mp = mp2; mp2 = t32;
        __syncthreads();
        KC_PH(6);  // live lists
        if (tid == 0) a.out[8 + d] = (u32) (clock64() - lvl_t0) | 0x80000000u;  // top bit: the level was run, not skipped
    }
    if (local_state) {  // write the path back for the emission stage
        __syncthreads();
        for (u32 i = tid; i < v.N; i += NT) {
            a.st.edge_from[i] = s.edge_from[i];
            a.st.edge_to[i] = s.edge_to[i];
            a.st.chain_head[i] = s.chain_head[i];
            a.st.chain_tail[i] = s.chain_tail[i];
            a.st.ovl[i] = s.ovl[i];
        }
    }
    KC_PH(7);  // write-back
    if (tid == 0) {
        for (int i = 0; i < 8; ++i) a.out[8 + 128 + i] = (u32) ph[i];
        a.out[1] = st_levels;
        a.out[2] = st_groups;
        a.out[3] = st_edges;
        a.out[4] = st_rounds;
        a.out[5] = st_bans;
    }
}

#undef KC_PH

#endif  // __CUDACC__
