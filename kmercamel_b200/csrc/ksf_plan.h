// Plan of the histogram-free (fixed-slot) k-mer set construction of kmerset_fast.cuh: how many MSD partition levels, how many
// key bits each consumes, and the slot size of every level, all from the input size alone.  Pure host C++ (no CUDA), so that
// tests/host_emul can check the invariants the kernels rely on:
//   * a level's digit is at most 8 bits wide (the kernels keep 256 counters per tile);
//   * every slot size is a multiple of 32 items, so slots stay 128-byte aligned for 4-byte positions and 256-byte aligned for
//     8-byte keys — the 16-byte bulk and cp.async copies of tiles and leaves (kc_ksf_scatter_pf_kernel, kc_ksf_resolve*_kernel)
//     need that;
//   * all partition digits together stay inside the top limb of the scrambled word (KWord::digit_top);
//   * a leaf slot holds KSF_LEAF_CAP items, the capacity of the shared-memory resolve.
#pragma once
#include <cmath>
#include <cstdint>

static const uint32_t KSF_LEAF_CAP = 1024;  // capacity of the shared-memory leaf resolve (kc_ksf_resolve*_kernel)
static const int KSF_MAX_LEVELS = 4;

struct KsfTuning {
    bool enabled = true;
    uint32_t leaf_target = 768;   // mean leaf size aimed at (the leaf slot holds KSF_LEAF_CAP)
    double sigmas = 8.0;     // slot = mean + sigmas * sqrt(mean) (+ 2 %) items; 0 forces overflows (tests)
    uint64_t min_items = 1u << 16;  // smaller inputs take the exact path (nothing to gain)
    int max_ctas = 148 * 16; // level >= 1 scatter grid: at most this many CTAs, each walking a run of consecutive tiles
};

struct KsfPlan {
    bool ok = false;
    int n_levels = 0;
    int bits[KSF_MAX_LEVELS];   // digit width of level i
    int cum[KSF_MAX_LEVELS];    // key bits consumed after level i
    uint64_t cap[KSF_MAX_LEVELS];    // slot size (items) of one bucket produced by level i
    uint64_t slots[2] = {0, 0};      // items the ping (even levels) / pong (odd levels) buffers must hold
    uint64_t n_leaf = 0;
};

inline KsfPlan kc_ksf_plan(uint64_t m_upper, const KsfTuning &t) {
    KsfPlan p;
    if (!t.enabled || m_upper < t.min_items) return p;
    int total_bits = 1;
    while (total_bits < 40 && (m_upper >> total_bits) > t.leaf_target) ++total_bits;
    const int levels = (total_bits + 7) / 8;
    if (levels > KSF_MAX_LEVELS) return p;
    p.n_levels = levels;
    int cum = 0;
    for (int i = 0; i < levels; ++i) {
        p.bits[i] = total_bits / levels + (i < total_bits % levels ? 1 : 0);
        cum += p.bits[i];
        p.cum[i] = cum;
        const double mean = (double) m_upper / (double) (1ULL << cum);
        uint64_t cap = (uint64_t) std::ceil(mean + t.sigmas * std::sqrt(mean) + (t.sigmas > 0 ? 0.02 * mean + 64.0 : 0.0));
        cap = (cap + 31) / 32 * 32;
        if (i == levels - 1) cap = KSF_LEAF_CAP;
        if (cap >= 0xFFFFFFFFULL) return p;
        p.cap[i] = cap;
        const uint64_t need = (1ULL << cum) * cap;
        if (need > p.slots[i & 1]) p.slots[i & 1] = need;
    }
    p.n_leaf = 1ULL << cum;
    p.ok = true;
    return p;
}

// ---- multi-GPU (group.cuh): hash-range sharding of the same construction ---------------------------------------------------
// Level 0 runs on every rank over its slice of the level-0 tiles; level-0 digit d belongs to rank owner(d) = d * n_ranks /
// n_digits (contiguous digit ranges), and the items a sender produces for d go into the sub-slot (d, sender) of the owner's
// receive buffer: cap_sub items, planned like every other slot from the slice size alone.  From level 1 on the owner works
// alone, with the plan of the WHOLE input (its buckets hold the items of all senders).
static const int KSF_MAX_RANKS = 16;
inline uint64_t ksf_div_up(uint64_t a, uint64_t b) { return (a + b - 1) / b; }

// Geometry of one job, the same on every rank (computed from n_bytes, the tuning and the group size alone).
struct KsfGroupPlan {
    bool ok = false;
    KsfPlan pl;
    int n_ranks = 1;
    uint32_t n_digits = 0;      // level-0 buckets = 1 << pl.bits[0]
    uint32_t tiles = 0;         // level-0 tiles of the whole input
    uint64_t cap_sub = 0;       // items per (digit, sender) sub-slot
    uint32_t dig_max = 0;       // most digits any rank owns
    uint32_t tile_begin(int r) const { return (uint32_t) ((uint64_t) tiles * (uint64_t) r / (uint64_t) n_ranks); }
    uint32_t dig_begin(int r) const { return (uint32_t) (((uint64_t) r * n_digits + (uint64_t) n_ranks - 1) / (uint64_t) n_ranks); }  // owner(d) = d * n_ranks / n_digits
    uint32_t owner(uint32_t d) const { return (uint32_t) ((uint64_t) d * (uint64_t) n_ranks / n_digits); }
    uint64_t recv_items() const { return (uint64_t) dig_max * (uint64_t) n_ranks * cap_sub; }  // receive slots every rank must provide
};

inline KsfGroupPlan kc_ksf_group_plan(uint64_t n_bytes, int n_ranks, uint64_t ex_tile, const KsfTuning &tune) {
    KsfGroupPlan g;
    g.pl = kc_ksf_plan(n_bytes, tune);
    g.n_ranks = n_ranks;
    if (!g.pl.ok || g.pl.n_levels < 2 || n_ranks < 1 || n_ranks > KSF_MAX_RANKS) return g;  // one level: the leaves would be split by sender
    g.n_digits = 1u << g.pl.bits[0];
    if (g.n_digits < (uint32_t) n_ranks) return g;
    g.tiles = (uint32_t) ksf_div_up(n_bytes, ex_tile);
    const uint64_t slice_tiles = ksf_div_up((uint64_t) g.tiles, (uint64_t) n_ranks);
    const double mean = (double) (slice_tiles * ex_tile) / (double) g.n_digits;
    uint64_t cap = (uint64_t) std::ceil(mean + tune.sigmas * std::sqrt(mean) + (tune.sigmas > 0 ? 0.02 * mean + 64.0 : 0.0));
    cap = (cap + 31) / 32 * 32;
    if (cap >= 0xFFFFFFFFULL) return g;
    g.cap_sub = cap;
    for (int r = 0; r < n_ranks; ++r) {
        const uint32_t n = g.dig_begin(r + 1) - g.dig_begin(r);
        g.dig_max = n > g.dig_max ? n : g.dig_max;
    }
    g.ok = true;
    return g;
}

