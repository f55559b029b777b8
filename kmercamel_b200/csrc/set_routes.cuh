// Which construction builds the first-occurrence bits of a from-FASTA input, and what a context remembers when one fails.
//
// Three constructions can build the bits.  The signature buckets (kmerset_sig.cuh, k >= 26) and the fixed slots (kmerset_fast.cuh)
// are fast but can overflow: a status word reports it after the fact, and the bits are then incomplete.  The exact construction
// (kmerset.cuh, or kc_grp_exact_flags on a group) always stands.  kc_set_ladder runs the two that can overflow, in that order, and
// returns the one whose bits stood; the caller then runs its own last route.  The policy of each entry point:
//
//   compute, lowerbound, group ranks (SetRoutes::compute_policy)
//       signature buckets without -M and -z, fixed slots without -M.  With option fast_heuristics a rung is skipped when it
//       overflowed on an input of similar size (SizeMemo::near) earlier in this context, and the fixed slots are skipped under -z
//       too: -z announces a read set with coverage, whose leaf slots overflow (configs[3] at full size lost 70 ms to the wasted
//       attempt).  An overflow is remembered whether or not fast_heuristics is on.  A group tries the fixed slots only when its
//       group plan applies and fits the heap.  Last route: the exact construction (sorted keys with -M).  Inside the signature
//       rung compute may try the speculative tail (tail_spec.cuh); its own memory is `tail`.
//   kmer_digest without -z
//       the signature buckets only, then the sorted-keys digest.
//   streaming
//       pass 1: the signature buckets, then the fixed slots without -z, then the exact construction.  Passes 2..Z of -z: the
//       signature buckets only if they stood in pass 1 (an overflow falls back to the filtered exact pass for that pass only).
//   Digest and streaming count runs and fallbacks but neither consult nor write the memories: a read set digested or streamed does
//   not change which construction a later compute tries.
//
// Inputs of KC_POS32_BYTES or more need 64-bit window positions, which only the signature buckets carry: they never reach the fixed
// slots, and a signature rung that does not apply or overflows fails the call.
#pragma once
#include "kmerset_sig.cuh"

#define KC_LARGE_ONLY "inputs of 2^32 bytes or more are built by the signature construction only (k >= 26, no -z, no -M, no -S)"

// The input size of the last call on which a construction failed (0 = none).
struct SizeMemo {
    u64 bytes = 0;
    bool near(u64 nb) const { return bytes && nb >= bytes / 2 && nb <= bytes * 2; }
    void remember(u64 nb) { bytes = nb; }
};

enum KcRoute { KC_ROUTE_SIG, KC_ROUTE_FAST, KC_ROUTE_NONE };

struct RoutePolicy {
    bool sig = false, fast = false;  // the rungs that may run
    bool remember = false;           // write an overflow into the rung's memory
};

struct RungState {
    u64 runs = 0, fallbacks = 0;  // stats "<rung>_runs" and "<rung>_fallbacks": bits that stood / overflowed
    SizeMemo overflow;
};

struct SetRoutes {
    SigTuning sig;          // options sig_*
    KsfTuning fast;         // options fast_*
    bool heuristics = true; // option fast_heuristics: consult the memories
    RungState sig_rung, fast_rung;
    SizeMemo tail;          // the speculative tail did not hold

    RoutePolicy compute_policy(const kc_params &p, u64 nb) const {
        RoutePolicy q;
        q.sig = !p.want_maxone && p.min_frequency == 1 && (nb >= KC_POS32_BYTES || !(heuristics && sig_rung.overflow.near(nb)));
        q.fast = !p.want_maxone && !(heuristics && (p.min_frequency > 1 || fast_rung.overflow.near(nb)));
        q.remember = true;
        return q;
    }
};

// launch(route) queues the construction into flags and cells the caller owns (zeroed) and returns false when its plan does not
// apply (nothing queued).  consume(route) queues what reads the bits, does the call's one read-back and returns whether the status
// word was clear; when it was not, consume leaves what the next route needs cleared, and the arena is restored to where it was
// before the rung.
template <class Launch, class Consume>
KcRoute kc_set_ladder(SetRoutes &r, const RoutePolicy &pol, u64 nb, Arena &arena, Launch launch, Consume consume) {
    const bool large = nb >= KC_POS32_BYTES;
    auto attempt = [&](KcRoute route, RungState &st) {
        const ArenaMark mark = arena.checkpoint();
        if (!launch(route)) {
            if (large) KC_THROW(KC_ERR_TOO_LARGE, KC_LARGE_ONLY "; its bucket plan does not fit this input");
            return false;
        }
        if (consume(route)) {
            ++st.runs;
            return true;
        }
        ++st.fallbacks;
        if (pol.remember) st.overflow.remember(nb);
        if (large) KC_THROW(KC_ERR_TOO_LARGE, KC_LARGE_ONLY "; it overflowed on this input (too repetitive)");
        arena.restore(mark);
        return false;
    };
    if (pol.sig && attempt(KC_ROUTE_SIG, r.sig_rung)) return KC_ROUTE_SIG;
    if (large) KC_THROW(KC_ERR_INTERNAL, "an input of 2^32 bytes or more reached the 32-bit set constructions");
    if (pol.fast && attempt(KC_ROUTE_FAST, r.fast_rung)) return KC_ROUTE_FAST;
    return KC_ROUTE_NONE;
}
