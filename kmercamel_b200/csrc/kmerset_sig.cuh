// K-mer set construction by SIGNATURE buckets (super-k-mers) for the FLAGS regime: the same result as kmerset_fast.cuh /
// kmerset.cuh — bit p of the flag array set iff the k-mer of the window ending at p occurs there for the first time
// (reference src/parser.h:22-141 AddKMers / ReadKMers + khash) — with ~10 x less HBM traffic and two kernels instead of three.
//
// The partition passes of kmerset_fast.cuh move every k-mer occurrence as a 12-byte (key, position) item: 1 + 12 (level 0)
// + 12 + 12 (level 1) + 12 (leaf resolve) = 49 bytes per k-mer, and their cost is the shared-memory ranking of those items.
// Here the unit that travels is a RECORD: up to 8 consecutive windows of one 32-position strip whose k-mers share a
// signature, 8 bytes for ~5 windows.  The k-mers themselves are re-created from the 2-bit packed sequence (0.25 bytes per
// base, written by the scan) inside the CTA that resolves the bucket.
//
//   signature of a k-mer  = the smallest hash among the canonical M-mers at its W = 16 CENTRAL M-mer positions
//                           (M = 16 / 15 for k >= 30, 12 / 11 for 26 <= k < 30; chosen so that k - M - (W - 1) is even:
//                           the central range is then mirror-symmetric, a k-mer and its reverse complement see the same
//                           set of canonical M-mers, and every occurrence of a canonical k-mer gets the same signature);
//   bucket                = floor(n_buckets * (1 - (1 - s)^13)), s = signature / 2^32.  The minimum of W uniform hashes has
//                           distribution 1 - (1 - s)^W; exponent W would spread the WINDOWS evenly over the buckets, but a large
//                           signature changes hands after ~2 windows where a small one lasts for 16, so the last buckets would
//                           hold twice the RECORDS of the first ones — and the capacity of a bucket is counted in records.
//                           Exponent 13 evens the records out (simulation over 16 M windows: octile means within 6 %);
//   kc_sig_scan_kernel    sequence -> 2-bit codes (as level 0 of the other constructions; the code words also go to HBM) -> 47
//                           M-mer hashes per strip by static funnel shifts of the strip's 128-bit code window and of its reverse
//                           complement -> sliding minimum by doubling (2, 4, 8, 16) in registers -> runs of equal signature, cut
//                           into records of <= 8 windows: one atomicAdd on the bucket's counter reserves the record slot, one
//                           8-byte store writes {position, length}.  Also writes the valid-window bits ("clear the losers"
//                           flags, kmerset_fast.cuh).
//   kc_sig_resolve_kernel persistent CTAs, one bucket (<= 256 records) at a time, ONE THREAD PER RECORD: two 8-byte loads fetch
//                           the record's code words (one bucket ahead, into registers), the first k-mer is a funnel shift, the
//                           next ones roll (forward and reverse complement, src/parser.h:39-40); item t of record r lives in
//                           slot t * 256 + r of the shared-memory arrays (conflict-free, no prefix sums), and the tables of
//                           kc_ksf_resolve2_kernel resolve them: plain-store table T1, one barrier, CAS fallback T2; every folded
//                           duplicate clears the bit of the larger position.  (Handing the windows of a warp's records out one
//                           per lane — dense lanes, direct funnel extraction — was measured: more instructions per window.)
//
// HBM bytes per k-mer (L = 1): 1 (sequence) + 0.25 (code words written) + 1.6 (record written) + 1.6 (record read) + ~3 (code
// words re-read, 16 bytes per record) = ~7.5 instead of 49.
//
// A bucket that exceeds its capacity (heavily repeated sequence, read sets with coverage) sets the status word; the caller
// discards the flags and uses the other constructions, exactly like an overflow in kmerset_fast.cuh.  Inputs of 2^32 bytes or more
// have no other construction (theirs carry 32-bit positions): there the call fails.
#pragma once
#include "kmerset_fast.cuh"

struct SigTuning {
    bool enabled = true;
    uint32_t load_pct = 0;             // mean records per bucket in percent of the bucket capacity; 0 = planned from the input size (kc_sig_plan)
    uint64_t min_items = 1u << 16;     // smaller inputs: nothing to gain
};

static const int KC_SIG_W = 16;
static const int KC_SIG_PIECE = 8;          // windows per record at most
static const u32 KC_SIG_REC_CAP = 256;      // records per bucket = threads of the resolving CTA
static const u32 KC_SIG_SLOTS = KC_SIG_PIECE * KC_SIG_REC_CAP;  // item t of record r lives in slot t * REC_CAP + r
static const double KC_SIG_WINDOWS_PER_RECORD = 5.16;          // random sequence, runs cut by the 32-window strips and into pieces of 8

struct SigPlan {
    bool ok = false;
    int m = 0;          // M-mer length
    int a = 0;          // the central range of a window ending at e: M-mers ending at e - a - (W - 1) .. e - a
    u32 n_buckets = 0;
    double mean_records = 0;  // per bucket
    double clump = 1.5;       // sigma of a bucket's record count = clump * sqrt(mean)
};

inline SigPlan kc_sig_plan(u64 n_bytes, int k, const SigTuning &t) {
    SigPlan p;
    if (!t.enabled || n_bytes < t.min_items) return p;
    static const int ms[4] = {16, 15, 12, 11};
    for (int i = 0; i < 4 && !p.m; ++i) {
        const int d = k - ms[i] - (KC_SIG_W - 1);
        if (d >= 0 && d % 2 == 0) {
            p.m = ms[i];
            p.a = d / 2;
        }
    }
    if (!p.m) return p;
    // How full may a bucket be on average?  Its record count spreads like a clumped Poisson variable: runs of windows are cut into
    // several records (factor ~1.5 on sigma, measured), and every further occurrence of a signature M-mer in the input drops its
    // records into the same bucket — chance repeats alone are 2 n / 4^M per M-mer (1.4 at 3.1 Gbp with M = 16: the first north-star run
    // overflowed with the fixed 55 % load that fits 50-500 Mbp).  The fullest of nb buckets sits ~sqrt(2 ln nb) sigma above the mean, the
    // first buckets get ~6 % more than the mean: solve 1.06 m + z * clump * sqrt(m) = 256 for m.
    const double mu = 2.0 * (double) n_bytes / std::pow(4.0, (double) p.m);
    p.clump = 1.5 * std::sqrt(1.0 + mu);
    const double z = std::sqrt(2.0 * std::log((double) n_bytes / 500.0 + 16.0)) + 2.0;  // + 2: repeats of real sequence on top of the chance ones
    const double zc = z * p.clump;
    const double x = (-zc + std::sqrt(zc * zc + 4.0 * 1.06 * KC_SIG_REC_CAP)) / (2.0 * 1.06);
    p.mean_records = t.load_pct ? KC_SIG_REC_CAP * (t.load_pct / 100.0) : x * x;
    if (p.mean_records < 32.0) {  // far too clumpy for buckets of 256 records (short M-mers on a large input)
        p.m = 0;
        return p;
    }
    const double mean_windows = p.mean_records * KC_SIG_WINDOWS_PER_RECORD;
    const u64 nb = (u64) ((double) n_bytes / (mean_windows > 1.0 ? mean_windows : 1.0)) + 1;
    if (nb >= (1u << 27)) return p;
    p.n_buckets = (u32) (nb < 64 ? 64 : nb);
    p.ok = true;
    return p;
}

// Arena bytes of kc_kmerset_build_sig besides the sequence and the flags: record rows, code words, bucket counters.
inline u64 kc_sig_arena_bytes(const SigPlan &p, u64 n_bytes) {
    const u64 tiles = (n_bytes + 256 * 32 - 1) / (256 * 32);
    return (u64) p.n_buckets * KC_SIG_REC_CAP * 8 + tiles * 256 * 8 + (u64) p.n_buckets * 4 + (3u << 10);
}

#ifdef __CUDACC__

// Reverse complement of 16 bases held in one 32-bit word.
KC_D u32 kc_revcomp16(u32 w) {
    u32 b = __brev(w);  // symbols reversed, the two bits of every symbol swapped
    b = ((b >> 1) & 0x55555555u) | ((b & 0x55555555u) << 1);
    return ~b;
}

// Bits [SH, SH + 31] of the 128-bit value x[0] : x[1] : x[2] : x[3] (x[0] most significant), SH static.
template <int SH> KC_D u32 kc_bits128(const u32 (&x)[4]) {
    constexpr int wr = SH >> 5, off = SH & 31;  // word index from the right
    const u32 lo = x[3 - wr];
    if constexpr (off == 0) {
        return lo;
    } else {
        const u32 hi = wr + 1 <= 3 ? x[3 - (wr + 1 <= 3 ? wr + 1 : 3)] : 0u;
        return __funnelshift_r(lo, hi, off);
    }
}

template <int M, int I> struct SigHashLoop {
    KC_D static void run(const u32 (&x)[4], const u32 (&y)[4], u32 *H) {
        constexpr u32 mask = M == 16 ? 0xFFFFFFFFu : ((1u << (2 * M)) - 1u);
        const u32 f = kc_bits128<128 - 2 * (I + M)>(x) & mask;  // bases I .. I + M - 1 of the code window
        const u32 r = kc_bits128<2 * I>(y) & mask;               // their reverse complement
        u32 h = (f < r ? f : r) * 0x9E3779B1u;
        h ^= h >> 15;
        h *= 0x85EBCA6Bu;
        H[I] = h;
        SigHashLoop<M, I + 1>::run(x, y, H);
    }
};
template <int M> struct SigHashLoop<M, 32 + KC_SIG_W - 1> {
    KC_D static void run(const u32 (&)[4], const u32 (&)[4], u32 *) {}
};

// signature -> bucket (see the header): floor(n_buckets * (1 - (1 - s)^13))
KC_D u32 kc_sig_bucket(u32 sig, u32 n_buckets) {
    const u32 u1 = ~sig;
    const u32 u2 = __umulhi(u1, u1), u4 = __umulhi(u2, u2), u8 = __umulhi(u4, u4);
    const u32 u13 = __umulhi(__umulhi(u8, u4), u1);
    return __umulhi(~u13, n_buckets);
}

// A record: END position of its first window in bits 0..31 (low half) and 35..63 (bits 32..60 of the position), windows - 1 in
// bits 32..34.  Below 2^32 the word is the plain {position, length} of a 32-bit layout.
KC_HD u64 kc_sig_record(u64 pos, u32 len) { return (pos & 0xFFFFFFFFULL) | ((u64) (len - 1) << 32) | ((pos >> 32) << 35); }
KC_HD u64 kc_sig_record_pos(u64 rec) { return (rec & 0xFFFFFFFFULL) | ((rec >> 35) << 32); }
KC_HD u32 kc_sig_record_len(u64 rec) { return ((u32) (rec >> 32) & 7u) + 1u; }

// Multi-GPU (group.cuh): bucket b belongs to rank b % n; rank r's records for it go into the sub-slot (b / n, r) of the owner's
// receive array (sub_cap records, reserved with a LOCAL counter: no remote atomics), the code words and the valid-window words of
// the rank's slice go to every rank.
struct SigPeers {
    u64 *recs[KC_MAX_PEERS];     // receive array of rank o: [bucket / n][sender][sub_cap]
    u64 *packed[KC_MAX_PEERS];   // code words of the whole sequence, one copy per rank
    u32 *flags[KC_MAX_PEERS];    // first-occurrence bits, one copy per rank
    u32 *cnt[KC_MAX_PEERS];      // fill counts of the sub-slots of rank o: [bucket / n][sender]
    int n, rank;
    u32 magic;                   // floor(2^32 / n) + 1: b / n = umulhi(b, magic) for b < 2^28 (n >= 2; one rank owns everything)
    u32 sub_cap;
};

// packed[s] = the 2-bit codes of bases 32 s .. 32 s + 31 (first base in the top bits); every strip of every tile is written.
template <int M, bool P2P>
__global__ void __launch_bounds__(256) kc_sig_scan_kernel(const u8 *__restrict__ seq, u64 n_bytes, int k, int a, u32 n_buckets, u32 *cursor,
                                                          u64 *__restrict__ recs, u64 *__restrict__ packed, u32 *__restrict__ flags, u64 n_flag_words,
                                                          u32 tile0, kc_ull *m_cell, u32 *status, const u32 *__restrict__ win_mask, const SigPeers sp) {
    kc_pdl_wait();
    constexpr int T = 256;
    constexpr int NH = 32 + KC_SIG_W - 1;  // M-mer hashes a strip needs
    __shared__ u64 pk[KC_EX_HALO + T];
    __shared__ u32 vm[KC_EX_HALO + T];
    __shared__ u32 ssig[KC_EX_STRIP * T];  // signature of the window ending at strip base j of thread t at [j * T + t]
    const i64 block_pos0 = (i64) (tile0 + blockIdx.x) * (T * KC_EX_STRIP);
    kc_tile_load<T>(seq, n_bytes, block_pos0, pk, vm);
    __syncthreads();
    const int widx = KC_EX_HALO + threadIdx.x;
    if (P2P) {
        for (int r = 0; r < sp.n; ++r) sp.packed[r][(u64) (block_pos0 >> 5) + threadIdx.x] = pk[widx];
    } else {
        packed[(u64) (block_pos0 >> 5) + threadIdx.x] = pk[widx];
    }
    u32 em;
    {   // genomes: every base of the strip and of the k - 1 before it is a nucleotide (warp-uniform most of the time)
        const int need = (k - 1 + 31) >> 5;  // words to the left that a window of the strip can reach into
        bool all = vm[widx] == 0xFFFFFFFFu;
#pragma unroll
        for (int w = 1; w <= KC_EX_HALO; ++w) all = all && (w > need || vm[widx - w] == 0xFFFFFFFFu);
        em = all ? 0xFFFFFFFFu : kc_strip_emit_mask(vm, widx, k);
    }
    em &= kc_strip_window_filter(win_mask, block_pos0);
    {   // clear-the-losers flags: every window starts as "first occurrence" (bit p & 31 of word p >> 5 = window END p).  The flags do
        // not arrive zeroed: every word is written, the ones past the last tile (the padding word) by the last thread of that tile
        const u64 w = (u64) (block_pos0 >> 5) + threadIdx.x;
        if (P2P) {
            if (w < n_flag_words)
                for (int r = 0; r < sp.n; ++r) sp.flags[r][w] = __brev(em);
        } else if (w < n_flag_words) {
            flags[w] = __brev(em);
            if (threadIdx.x == T - 1 && (u64) block_pos0 + T * KC_EX_STRIP >= n_bytes)
                for (u64 x = w + 1; x < n_flag_words; ++x) flags[x] = 0;
        }
    }
    {
        u32 c = __popc(em);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) c += __shfl_down_sync(0xFFFFFFFFu, c, o);
        if ((threadIdx.x & 31) == 0 && c) atomicAdd(m_cell, (kc_ull) c);
    }
    if (!em) return;
    // the 64 bases that end with the strip's last M-mer: base t of the code window = strip base t - back
    const int back = a + (KC_SIG_W - 2) + M;
    const int g0 = widx * 32 - back;
    const int wi0 = g0 >> 5, sb = 2 * (g0 & 31);
    const u64 p0 = pk[wi0], p1 = pk[wi0 + 1], p2 = wi0 + 2 <= widx ? pk[wi0 + 2] : 0ULL;
    const u64 X0 = sb ? (p0 << sb) | (p1 >> (64 - sb)) : p0;
    const u64 X1 = sb ? (p1 << sb) | (p2 >> (64 - sb)) : p1;
    const u32 x[4] = {(u32) (X0 >> 32), (u32) X0, (u32) (X1 >> 32), (u32) X1};
    const u32 y[4] = {kc_revcomp16(x[3]), kc_revcomp16(x[2]), kc_revcomp16(x[1]), kc_revcomp16(x[0])};
    u32 H[NH];
    SigHashLoop<M, 0>::run(x, y, H);
    // sliding minimum over W = 16 hashes by doubling; H[j] = signature of the window ending at strip base j
#pragma unroll
    for (int i = 0; i < NH - 1; ++i) H[i] = min(H[i], H[i + 1]);
#pragma unroll
    for (int i = 0; i < NH - 3; ++i) H[i] = min(H[i], H[i + 2]);
#pragma unroll
    for (int i = 0; i < NH - 7; ++i) H[i] = min(H[i], H[i + 4]);
#pragma unroll
    for (int i = 0; i < NH - 15; ++i) H[i] = min(H[i], H[i + 8]);
    u32 neq = 1u;  // bit j: the signature changes at window j
#pragma unroll
    for (int j = 0; j < KC_EX_STRIP; ++j) {
        ssig[j * T + threadIdx.x] = H[j];
        if (j) neq |= (H[j] != H[j - 1] ? 1u : 0u) << j;
    }
    const u32 emr = __brev(em);                          // bit j = window ending at strip base j
    const u32 run_starts = emr & (neq | ~(emr << 1));    // a run: valid windows of one signature
    // The pieces (<= 8 windows) of the runs, bit-parallel: a run is cut every 8 windows from its start, i.e. window p starts a piece
    // iff it starts a run, or window p - 8 starts a piece and windows p - 7 .. p all continue its run.  (A loop over the runs that
    // listed the pieces in shared memory first was 19 % of the kernel's instructions.)
    const u32 cont = emr & ~run_starts;
    u32 c8 = cont & (cont << 1);
    c8 &= c8 << 2;
    c8 &= c8 << 4;                                       // bit p: windows p - 7 .. p continue the run of window p - 8
    u32 ps = run_starts;
    {
        u32 q = (run_starts << 8) & c8;
        ps |= q;
        q = (q << 8) & c8;
        ps |= q;
        q = (q << 8) & c8;
        ps |= q;
    }
    const u32 bound = ps | ~emr;                         // a piece ends before the next piece or the next window that is not valid
    // eight pieces per round, so that their atomics are in flight together (one at a time, the thread waited ~0.7 us for each
    // slot: 51 % of the kernel's stall samples)
    const u64 pos0 = (u64) block_pos0 + threadIdx.x * KC_EX_STRIP;
    const u64 rec_hi = kc_sig_record(pos0, 1u) & ~0xFFFFFFFFULL;  // bits 35..63, the same for the whole strip (32 | 2^32)
    bool over = false;
    while (ps) {
        u32 bk[8], slot[8], e[8];
        bool on[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            on[u] = ps != 0;
            const u32 j = ((u32) __ffs(ps) - 1u) & 31u;
            ps &= ps - 1u;
            const u32 rest = bound & (0xFFFFFFFEu << j);
            const u32 len = (rest ? (u32) __ffs(rest) - 1u : 32u) - j;
            e[u] = (j << 3) | (len - 1u);
            bk[u] = kc_sig_bucket(ssig[j * T + threadIdx.x], n_buckets);
        }
#pragma unroll
        for (int u = 0; u < 8; ++u)
            if (on[u]) slot[u] = atomicAdd(&cursor[bk[u]], 1u);
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            if (on[u]) {
                const u64 rec = kc_sig_record((u32) pos0 + (e[u] >> 3), (e[u] & 7u) + 1u) | rec_hi;
                if (P2P) {  // into the rank's own staging array; kc_sig_ship_kernel sends whole sub-slots
                    if (slot[u] < sp.sub_cap) recs[(u64) bk[u] * sp.sub_cap + slot[u]] = rec;
                    else over = true;
                } else {
                    if (slot[u] < KC_SIG_REC_CAP) recs[(u64) bk[u] * KC_SIG_REC_CAP + slot[u]] = rec;
                    else over = true;
                }
            }
        }
    }
    if (over) status[0] = 1;
}

// After the scan of a group rank, its records (staged per bucket in its own HBM) travel to the owners as DENSE STREAMS: one
// stream per owner, the owner's buckets in ascending order, plus the offsets of the buckets inside the stream.
//   kc_sig_om_counts_kernel   fill count of bucket lb * n + o at index o * nbr + lb ("owner-major"; nbr = buckets a rank owns at most)
//   exclusive scan             -> offsets into one dense array (all owners back to back)
//   kc_sig_compact_kernel     a warp per bucket: staged records -> their place in the dense array (local)
//   kc_sig_ship_kernel        owner o's part of the dense array -> region `rank` of o's receive array, and the nbr + 1 offsets
//                             relative to its start -> o's offset table, both as long coalesced runs
// Measured before: every record as an 8-byte store of its own across NVLink, 0.57 ms for 39 MB at two GPUs; one run per
// (bucket, sender) sub-slot, 0.65 ms at eight GPUs (1.6 M small packets per rank).  NVLink wants few, large writes.
__global__ void __launch_bounds__(256) kc_sig_om_counts_kernel(const u32 *__restrict__ cursor, u32 n_buckets, u32 nbr, u32 n_ranks, u32 sub_cap, u32 *cnt_om) {
    const u32 i = blockIdx.x * 256 + threadIdx.x;
    if (i > n_ranks * nbr) return;
    u32 c = 0;
    if (i < n_ranks * nbr) {
        const u32 o = i / nbr, lb = i - o * nbr;
        const u64 b = (u64) lb * n_ranks + o;
        if (b < n_buckets) {
            c = cursor[b];
            c = c < sub_cap ? c : sub_cap;
        }
    }
    cnt_om[i] = c;  // entry n_ranks * nbr = 0: the scan leaves the total there
}

__global__ void __launch_bounds__(256) kc_sig_compact_kernel(const u32 *__restrict__ cursor, const u64 *__restrict__ staged, const u32 *__restrict__ off_om,
                                                             u32 n_buckets, u32 nbr, u32 n_ranks, u32 sub_cap, u64 *__restrict__ dense, u64 dense_cap, u32 *status) {
    const u32 i = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31u;
    if (i >= n_ranks * nbr) return;
    const u32 o = i / nbr, lb = i - o * nbr;
    const u64 b = (u64) lb * n_ranks + o;
    if (b >= n_buckets) return;
    u32 c = cursor[b];
    c = c < sub_cap ? c : sub_cap;
    const u64 *src = staged + b * sub_cap;
    const u32 at = off_om[i];
    if ((u64) at + c > dense_cap) {  // far more records than windows / 5 (the caller falls back)
        if (lane == 0) status[0] = 1;
        return;
    }
    u64 *dst = dense + at;
    for (u32 j = lane; j < c; j += 32) dst[j] = src[j];
}

// grid = (chunks, n_ranks): block (c, o) copies every gridDim.x-th 256-record piece of owner o's stream
__global__ void __launch_bounds__(256) kc_sig_ship_kernel(const u64 *__restrict__ dense, const u32 *__restrict__ off_om, u32 nbr, u32 region_cap, u32 *status,
                                                          const SigPeers sp) {
    const u32 o = blockIdx.y;
    const u32 base = off_om[o * nbr], len = off_om[(o + 1) * nbr] - base;
    u32 *od = sp.cnt[o] + (u64) (u32) sp.rank * (nbr + 1);
    if (len > region_cap || status[0]) {  // the owner must still find a valid table: all buckets empty (the status word makes every rank fall back)
        if (threadIdx.x == 0 && blockIdx.x == 0) status[0] = 1;
        for (u32 j = blockIdx.x * 256 + threadIdx.x; j <= nbr; j += gridDim.x * 256) od[j] = 0;
        return;
    }
    u64 *dst = sp.recs[o] + (u64) (u32) sp.rank * region_cap;
    for (u32 j = blockIdx.x * 256 + threadIdx.x; j < len; j += gridDim.x * 256) dst[j] = dense[base + j];
    for (u32 j = blockIdx.x * 256 + threadIdx.x; j <= nbr; j += gridDim.x * 256) od[j] = off_om[o * nbr + j] - base;
}

// Owner side, before the resolve: the pieces of a bucket in the senders' streams -> one row of 256 records per bucket (a warp per
// bucket), its record count next to it.  Letting every thread of the resolve look its record up in the n offset tables was measured:
// 0.38 -> 0.60 ms at eight GPUs (16 loads per thread and bucket); this pass costs 0.06 ms.
__global__ void __launch_bounds__(256) kc_sig_gather_kernel(const u32 *__restrict__ offsets, u32 off_stride, const u64 *__restrict__ streams, u32 region_cap,
                                                            u32 n_senders, u32 n_owned, u32 *__restrict__ cnt_bm, u64 *__restrict__ recs_bm) {
    const u32 lb = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31u;
    if (lb >= n_owned) return;
    u32 o0 = 0, cs = 0;
    if (lane < n_senders) {
        const u32 *of = offsets + (u64) lane * off_stride + lb;
        o0 = of[0];
        cs = of[1] - o0;
    }
    u32 incl = cs;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const u32 v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (lane >= (u32) o) incl += v;
    }
    const u32 pre = incl - cs, total = __shfl_sync(0xFFFFFFFFu, incl, 31);
    if (lane == 0) cnt_bm[lb] = total;  // > 256: the resolve raises the status word
    const u32 n_copy = total < KC_SIG_REC_CAP ? total : KC_SIG_REC_CAP;
    for (u32 tb = 0; tb < n_copy; tb += 32) {
        const u32 t = tb + lane;
        u64 src = ~0ULL;
        for (u32 sd = 0; sd < n_senders; ++sd) {
            const u32 ps = __shfl_sync(0xFFFFFFFFu, pre, sd), cc = __shfl_sync(0xFFFFFFFFu, cs, sd), oo = __shfl_sync(0xFFFFFFFFu, o0, sd);
            if (t >= ps && t < ps + cc) src = (u64) sd * region_cap + oo + (t - ps);
        }
        if (t < n_copy && src != ~0ULL) recs_bm[(u64) lb * KC_SIG_REC_CAP + t] = streams[src];
    }
}

template <int L> struct SigCfg {
    static constexpr int THREADS = (int) KC_SIG_REC_CAP;
    static constexpr int NW = L + 1;                                     // 32-base code words a window can reach into
    static constexpr u32 T1N = 4 * KC_SIG_SLOTS, T2N = KC_SIG_SLOTS / 4;  // T2 takes the items that lose their T1 slot to another key (~4 %)
    static constexpr int T1_BITS = 13;
    static constexpr int MIN_CTAS = L == 1 ? 5 : (L == 2 ? 3 : 2);      // resident CTAs per SM the shared memory allows
    static int smem(bool pos64 = false) { return (int) (KC_SIG_SLOTS * (sizeof(KWord<L>) + 4) + (pos64 ? KC_SIG_REC_CAP * 8 : 0) + T1N * 2 + T2N * 4); }
};

// Reverse the 32 two-bit symbols of a limb through the bit-reversal instruction (kc_reverse_symbols64 of kword.cuh walks a
// five-step swap network: ~4 x the instructions).
KC_D u64 kc_reverse_symbols64_brev(u64 w) {
    const u64 b = __brevll(w);  // symbols reversed, the two bits of every symbol swapped
    return ((b >> 1) & 0x5555555555555555ULL) | ((b & 0x5555555555555555ULL) << 1);
}

// Hash of a canonical k-mer for the tables of the resolve: a sum of 32-bit products (one multiply-add per half limb instead of a
// 64-bit product per limb); T1 takes the top bits, T2 a second mix of all of them.
template <int L> KC_D u32 kc_sig_hash(const KWord<L> &c) {
    constexpr u32 C[8] = {0x9E3779B1u, 0x85EBCA6Bu, 0xC2B2AE35u, 0x27D4EB2Fu, 0x165667B1u, 0xD3A2646Du, 0xFD7046C5u, 0xB55A4F09u};
    u32 h = 0;
#pragma unroll
    for (int q = 0; q < L; ++q) h += (u32) c.w[q] * C[2 * q] + (u32) (c.w[q] >> 32) * C[2 * q + 1];
    return h;
}
KC_D u32 kc_sig_hash2(u32 h) {
    h ^= h >> 15;
    return (h * 0x2C1B3C6Du) >> 16;
}

// The code words a record's windows can reach into: word NW - 1 = the strip of the record, the others to its left.
template <int NW, bool POS64> KC_D void kc_sig_load_words(const u64 *__restrict__ packed, u64 rec, bool have, u64 (&w)[NW]) {
    if constexpr (POS64) {
        const u64 strip = kc_sig_record_pos(rec) >> 5;
#pragma unroll
        for (int wi = 0; wi < NW; ++wi) w[wi] = have && strip >= (u64) (NW - 1 - wi) ? __ldg(&packed[strip - (u64) (NW - 1 - wi)]) : 0ULL;
    } else {
        const u32 strip = (u32) rec >> 5;
#pragma unroll
        for (int wi = 0; wi < NW; ++wi) w[wi] = have && strip >= (u32) (NW - 1 - wi) ? __ldg(&packed[strip - (u32) (NW - 1 - wi)]) : 0ULL;
    }
}

// One bucket at a time, ONE THREAD PER RECORD: item t of record r lives in slot t * 256 + r of the shared-memory arrays
// (conflict-free, no prefix sums).  The first k-mer of a record is a funnel shift of its code words, the next ones roll: forward
// word left by one base, reverse complement right by one base (src/parser.h:39-40; L = 1 keeps the reverse complement
// left-aligned, so that every shift of the roll is static).  The record of bucket n + 2 and the code words of bucket n + 1 are
// in flight (registers) while bucket n is resolved: no thread waits for HBM between the barriers.
//
// All eight windows of a record are computed whatever its length and only the stores are predicated: in a warp of 32 records
// some record has 8 windows practically always, so branches around every window saved nothing and cost the reconvergence
// points (16 BSSY / BSYNC pairs per bucket) and the overlap of the eight independent hash / store chains (0.315 -> 0.289 ms on
// configs[1]).  Fewer threads per CTA (160 / 192 with a second round for the records beyond, 6 CTAs per SM) were measured and change
// nothing: 0.287 - 0.293 ms.
//
// POS64 (inputs of more than 2^32 bytes): window positions need 64 bits, and a shared array of them would cost the L = 1 instance one
// of its five resident CTAs, so an item stands for its position by its slot (position = rp[slot % RC] + slot / RC, rp = the 256
// record positions) and a duplicate folds by a CAS loop on slots.  A separate instance because this decode, in one code path for all
// sizes, made the resolve 3 % slower on configs[1] (0.2442 -> 0.2515 ms, two back-to-back pairs on one B200 at 1000 W).
template <int L, bool MULTI, bool UNI, bool POS64 = false>
__global__ void __launch_bounds__(SigCfg<L>::THREADS, SigCfg<L>::MIN_CTAS) kc_sig_resolve_kernel(const u64 *__restrict__ packed, int k,
                                                                                                const u32 *__restrict__ cursor, const u64 *__restrict__ recs,
                                                                                                u32 n_buckets, KsfFlagPeers fl, kc_ull *n_unique, u32 *status,
                                                                                                u32 n_senders, u32 sub_cap, u32 off_stride) {
    // MULTI: the buckets are this rank's (kc_sig_gather_kernel has lined their records up), a duplicate clears its bit on every rank
    kc_pdl_wait();
    // the CTAs finish unevenly: the next kernel (the run count) may place its CTAs on the SMs this one leaves
    kc_pdl_trigger();
    typedef SigCfg<L> Cfg;
    constexpr u32 RC = KC_SIG_REC_CAP, T2N = Cfg::T2N;
    constexpr int NW = Cfg::NW, P = KC_SIG_PIECE;
    static_assert((1u << Cfg::T1_BITS) == Cfg::T1N, "T1 size");
    extern __shared__ __align__(16) unsigned char kc_smem_raw[];
    KWord<L> *sk = reinterpret_cast<KWord<L> *>(kc_smem_raw);  // [SLOTS] canonical k-mer of the item in slot t * RC + r
    u64 *rp = reinterpret_cast<u64 *>(sk + KC_SIG_SLOTS);       // POS64: [RC] END position of the first window of record r
    // [SLOTS] its window END position (the smallest one of its key, once folded); POS64: the slot of that position
    u32 *sp = reinterpret_cast<u32 *>(rp + (POS64 ? RC : 0));
    u32 *T2 = sp + KC_SIG_SLOTS;                                // [T2N]
    u16 *T1 = reinterpret_cast<u16 *>(T2 + T2N);                // [T1N]
    const KWord<L> kmask = KWord<L>::low_mask(2 * k);
    u32 kept = 0;
    const u32 stride = gridDim.x;
    u32 b = blockIdx.x;
    auto fetch = [&](u32 bb, u32 &nr, u64 &rec) {
        nr = 0;
        rec = 0;
        if (bb >= n_buckets) return;
        nr = cursor[bb];
        rec = recs[(u64) bb * RC + threadIdx.x];
    };
    // record r (its code words in w) -> the canonical k-mers of its windows into slots t * RC + r, their T1 slots into h1
    auto spread = [&](const u64 rec, const u64 (&w)[NW], const u32 r, u32 (&h1)[P]) -> u32 {
        const u32 pos = (u32) rec, len = kc_sig_record_len(rec);
        if (POS64) rp[r] = kc_sig_record_pos(rec);
        const int sh = 2 * (31 - (int) (pos & 31u));
        const u64 mine = w[NW - 1];
        const u64 ms = sh ? mine << (64 - sh) : 0ULL;  // the bases behind the first window, left-aligned
        if constexpr (L == 1) {
            // The record's k + 7 bases (first window + the 7 bases behind it) as one 96-bit value F2 : F1 : F0, right-aligned, and
            // their reverse complement R2 : R1 : R0: window t is bits [14 - 2 t, 14 - 2 t + 2 k) of F and its reverse complement bits
            // [2 t, 2 t + 2 k) of R — two funnel shifts by constants and one mask per strand and window, where rolling both strands
            // (extract the next base, shift, or, mask; shift back into place to compare) cost twice that.  k >= 26 here (kc_sig_plan):
            // the low word of a k-mer needs no mask.
            const u64 f0 = (sh ? (mine >> sh) | (w[0] << (64 - sh)) : mine) & kmask.w[0];
            const u64 lo64 = (f0 << 14) | (ms >> 50);
            const u32 F0 = (u32) lo64, F1 = (u32) (lo64 >> 32), F2 = (u32) (f0 >> 50);
            const u32 mh = (u32) (kmask.w[0] >> 32);
            u32 R0 = 0, R1 = 0, R2 = 0;
            if (!UNI) {
                const u32 V0 = kc_revcomp16(F2), V1 = kc_revcomp16(F1), V2 = kc_revcomp16(F0);  // the 48 symbols reversed and complemented
                const int q = 96 - 2 * (k + 7);                                               // ... and right-aligned again
                R0 = __funnelshift_r(V0, V1, q);
                R1 = __funnelshift_r(V1, V2, q);
                R2 = V2 >> q;
            }
#pragma unroll
            for (int t = 0; t < P; ++t) {
                const int sf = 14 - 2 * t, sr = 2 * t;
                u32 cl = sf ? __funnelshift_r(F0, F1, sf) : F0;
                u32 ch = (sf ? __funnelshift_r(F1, F2, sf) : F1) & mh;
                if (!UNI) {
                    const u32 rl = sr ? __funnelshift_r(R0, R1, sr) : R0;
                    const u32 rh = (sr ? __funnelshift_r(R1, R2, sr) : R1) & mh;
                    const bool take_r = (((u64) rh << 32) | rl) < (((u64) ch << 32) | cl);
                    cl = take_r ? rl : cl;
                    ch = take_r ? rh : ch;
                }
                KWord<1> canon;
                canon.w[0] = ((u64) ch << 32) | cl;
                const u32 slot = (u32) t * RC + r;
                h1[t] = kc_sig_hash<1>(canon) >> (32 - Cfg::T1_BITS);
                if ((u32) t < len) {
                    sk[slot] = canon;
                    sp[slot] = POS64 ? slot : pos + (u32) t;
                    T1[h1[t]] = (u16) slot;
                }
            }
        } else {
            // the same with L + 1 limbs: F = the k + 7 bases right-aligned, R = their reverse complement
            KWord<L> f;
#pragma unroll
            for (int l = 0; l < L; ++l) f.w[l] = sh ? (w[NW - 1 - l] >> sh) | (w[NW - 2 - l] << (64 - sh)) : w[NW - 1 - l];
            f = f & kmask;
            KWord<L + 1> F, R;
            F.w[0] = (f.w[0] << 14) | (ms >> 50);
#pragma unroll
            for (int i = 1; i < L; ++i) F.w[i] = (f.w[i] << 14) | (f.w[i - 1] >> 50);
            F.w[L] = f.w[L - 1] >> 50;
            if (!UNI) {
#pragma unroll
                for (int i = 0; i <= L; ++i) R.w[i] = ~kc_reverse_symbols64_brev(F.w[L - i]);
                R = R.shr(64 * (L + 1) - 2 * (k + 7));
            }
#pragma unroll
            for (int t = 0; t < P; ++t) {
                const int sf = 14 - 2 * t, sr = 2 * t;
                KWord<L> canon;
#pragma unroll
                for (int j = 0; j < L; ++j) canon.w[j] = sf ? (F.w[j] >> sf) | (F.w[j + 1] << (64 - sf)) : F.w[j];
                canon = canon & kmask;
                if (!UNI) {
                    KWord<L> rt;
#pragma unroll
                    for (int j = 0; j < L; ++j) rt.w[j] = sr ? (R.w[j] >> sr) | (R.w[j + 1] << (64 - sr)) : R.w[j];
                    rt = rt & kmask;
                    if (rt < canon) canon = rt;
                }
                const u32 slot = (u32) t * RC + r;
                h1[t] = kc_sig_hash<L>(canon) >> (32 - Cfg::T1_BITS);
                if ((u32) t < len) {
                    sk[slot] = canon;
                    sp[slot] = POS64 ? slot : pos + (u32) t;
                    T1[h1[t]] = (u16) slot;
                }
            }
        }
        return len;
    };
    auto pos_of = [&](const u32 slot) -> u64 { return rp[slot % RC] + slot / RC; };
    // a duplicate of the key that slot o represents: the smaller position stays in sp[o], the bit of the larger one is cleared
    // (POS64: an atomicMin by position as a CAS loop on slots)
    auto fold = [&](const u32 o, const u32 slot) {
        if constexpr (!POS64) {
            const u32 mine_p = sp[slot];
            const u32 was = atomicMin(&sp[o], mine_p);
            kc_flag_clear_all<MULTI>(fl, was > mine_p ? was : mine_p);
            return;
        }
        const u64 mine_p = pos_of(slot);
        u32 cur = sp[o];
        for (;;) {
            const u64 cur_p = pos_of(cur);
            if (cur_p < mine_p) {
                kc_flag_clear_all<MULTI>(fl, mine_p);
                return;
            }
            const u32 was = atomicCAS(&sp[o], cur, slot);
            if (was == cur) {
                kc_flag_clear_all<MULTI>(fl, cur_p);
                return;
            }
            cur = was;
        }
    };
    // an item that did not win its T1 slot: equal key = duplicate (fold); different key -> T2 with CAS + linear probing
    auto settle = [&](const u32 slot) {
        const KWord<L> key = sk[slot];
        const u32 h = kc_sig_hash<L>(key);
        const u32 o = T1[h >> (32 - Cfg::T1_BITS)];
        if (sk[o] == key) {
            fold(o, slot);
        } else {
            u32 s2 = kc_sig_hash2(h) & (T2N - 1);
#pragma unroll 1
            for (u32 probes = 0;; ++probes) {
                if (probes == T2N) {  // T2 is full (never seen: it would take > 512 T1 collisions in one bucket)
                    status[0] = 1;
                    break;
                }
                const u32 old = atomicCAS(&T2[s2], KC_NONE, slot);
                if (old == KC_NONE) {
                    ++kept;
                    break;
                }
                if (sk[old] == key) {
                    fold(old, slot);
                    break;
                }
                s2 = (s2 + 1) & (T2N - 1);
            }
        }
    };
    u32 nr0, nr1;
    u64 rec0, rec1;
    fetch(b, nr0, rec0);
    fetch(b + stride, nr1, rec1);
    u64 w0[NW], w1[NW];
    kc_sig_load_words<NW, POS64>(packed, rec0, threadIdx.x < nr0 && nr0 <= RC, w0);
    for (; b < n_buckets; b += stride) {
        u32 nr2;
        u64 rec2;
        fetch(b + 2 * stride, nr2, rec2);
        kc_sig_load_words<NW, POS64>(packed, rec1, threadIdx.x < nr1 && nr1 <= RC, w1);
        const u32 n_rec = nr0;
        const bool skip = n_rec == 0 || n_rec > RC;  // uniform over the CTA
        if (n_rec > RC && threadIdx.x == 0) status[0] = 1;  // the scan has set the status word already
        if (!skip) {
            static_assert(T2N / 4 <= (u32) Cfg::THREADS, "one uint4 of T2 per thread");
            if (threadIdx.x < T2N / 4) reinterpret_cast<uint4 *>(T2)[threadIdx.x] = make_uint4(KC_NONE, KC_NONE, KC_NONE, KC_NONE);
            // P1: the thread's record -> its k-mers, canonical, into the tables
            const bool have = threadIdx.x < n_rec;
            u32 len = 0;
            u32 h1[P];
            if (have) len = spread(rec0, w0, threadIdx.x, h1);
            __syncthreads();
            // P2: the winner of a T1 slot represents its key (~92 % of the items: done).  The others are listed in a bit mask and
            //     handled in a loop of their own (a thread has ~0.4 of them; inside the unrolled pass over t every warp paid the
            //     slow path eight times).  Dealing a warp's losers out one per lane through a list in shared memory — one dense
            //     round instead of the 2-3 rounds of the unluckiest lane — was measured: 0.289 -> 0.298 ms.
            if (have) {
                u32 win = 0;
#pragma unroll
                for (int t = 0; t < P; ++t) win |= (T1[h1[t]] == (u32) t * RC + threadIdx.x ? 1u : 0u) << t;
                const u32 all = (1u << len) - 1u;
                kept += __popc(win & all);
                u32 slow = all & ~win;
                while (slow) {
                    const u32 t = (u32) __ffs(slow) - 1u;
                    slow &= slow - 1u;
                    settle(t * RC + threadIdx.x);
                }
            }
            __syncthreads();  // the next bucket's P1 overwrites sk / sp / T1 / T2
        }
        nr0 = nr1;
        nr1 = nr2;
        rec0 = rec1;
        rec1 = rec2;
#pragma unroll
        for (int wi = 0; wi < NW; ++wi) w0[wi] = w1[wi];
    }
#pragma unroll
    for (int o2 = 16; o2 > 0; o2 >>= 1) kept += __shfl_down_sync(0xFFFFFFFFu, kept, o2);
    if ((threadIdx.x & 31) == 0 && kept) atomicAdd(n_unique, (kc_ull) kept);
}

template <int L> struct SigKernels {
    typedef SigCfg<L> Cfg;
    struct Dev {
        int n_sm = 0, occ = 0;
        int occ_multi64 = 0;  // the group's instance for inputs of 2^32 bytes or more
    };
    static const Dev &prepare() {
        static KcDevOnce once;
        static Dev dev[KC_MAX_DEVICES];
        const int d = once.run([&](int dv) {
            KC_CUDA(cudaFuncSetAttribute(kc_sig_resolve_kernel<L, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::smem()));
            KC_CUDA(cudaFuncSetAttribute(kc_sig_resolve_kernel<L, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::smem()));
            KC_CUDA(cudaFuncSetAttribute(kc_sig_resolve_kernel<L, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::smem()));
            KC_CUDA(cudaFuncSetAttribute(kc_sig_resolve_kernel<L, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::smem()));
            KC_CUDA(cudaFuncSetAttribute(kc_sig_resolve_kernel<L, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::smem(true)));
            KC_CUDA(cudaFuncSetAttribute(kc_sig_resolve_kernel<L, false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::smem(true)));
            KC_CUDA(cudaFuncSetAttribute(kc_sig_resolve_kernel<L, true, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::smem(true)));
            KC_CUDA(cudaFuncSetAttribute(kc_sig_resolve_kernel<L, true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::smem(true)));
            dev[dv].n_sm = kc_sm_count(dv);
            KC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&dev[dv].occ, kc_sig_resolve_kernel<L, false, false>, Cfg::THREADS, Cfg::smem()));
            KC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&dev[dv].occ_multi64, kc_sig_resolve_kernel<L, true, false, true>, Cfg::THREADS, Cfg::smem(true)));
        });
        return dev[d];
    }
};

template <bool P2P>
inline void kc_sig_scan_launch(CudaExec &ex, int m, u32 blocks, const u8 *seq, u64 n_bytes, int k, int a, u32 n_buckets, u32 *cursor, u64 *recs, u64 *packed,
                               u32 *flags, u64 n_flag_words, u32 tile0, kc_ull *m_cell, u32 *status, const u32 *win_mask, const SigPeers &sp) {
    auto *kern = m == 16 ? kc_sig_scan_kernel<16, P2P> : m == 15 ? kc_sig_scan_kernel<15, P2P> : m == 12 ? kc_sig_scan_kernel<12, P2P> : kc_sig_scan_kernel<11, P2P>;
    ex.launch(kern, blocks, 256, 0, seq, n_bytes, k, a, n_buckets, cursor, recs, packed, flags, n_flag_words, tile0, m_cell, status, win_mask, sp);
}

// Launches the construction on ex.stream and returns without synchronising; same contract as kc_kmerset_build_fast:
//   cells[0] += distinct k-mers, cells[2] = M (k-mer windows), low word of cells[3] = overflow status.  The flags (kc_runs_flag_words
// of n_bytes) need not arrive zeroed; the cells must, unless zero_cells > 0: then the construction zeroes cells[0, zero_cells) first
// (with its bucket counters in the same memset when `cells` is the arena's top block).
// Returns false (nothing launched) when the plan does not apply.
template <int L>
bool kc_kmerset_build_sig(CudaExec &ex, const u8 *seq, u64 n_bytes, int k, bool complements, u32 *flags, u64 *cells, const SigTuning &tune,
                          InputChunks *chunks = nullptr, const u32 *win_mask = nullptr, SigPlan *plan_out = nullptr, u32 zero_cells = 0) {
    typedef SigCfg<L> Cfg;
    typedef SigKernels<L> KK;
    const SigPlan pl = kc_sig_plan(n_bytes, k, tune);
    if (plan_out) *plan_out = pl;
    if (!pl.ok) return false;
    const typename KK::Dev &dv = KK::prepare();
    cudaStream_t st = ex.stream;
    const size_t base_mark = ex.arena->mark();
    constexpr u64 TILE = 256 * KC_EX_STRIP;
    const u32 blocks = (u32) kc_div_up(n_bytes, TILE);
    u64 *recs = ex.alloc<u64>((u64) pl.n_buckets * KC_SIG_REC_CAP);
    u64 *packed = ex.alloc<u64>((u64) blocks * 256);
    // the bucket counters go to the arena top, right below `cells` when the caller has just allocated them there: one memset for both
    const ArenaMark top_mark = ex.arena->checkpoint();
    u32 *cursor = ex.arena->alloc_top<u32>(pl.n_buckets);
    const size_t cursor_bytes = kc_align_up((u64) pl.n_buckets * 4, 256);
    if (zero_cells && reinterpret_cast<char *>(cursor) + cursor_bytes == reinterpret_cast<char *>(cells)) {
        ex.fill_bytes(cursor, 0, cursor_bytes + (size_t) zero_cells * 8);
    } else {
        ex.fill_bytes(cursor, 0, cursor_bytes);
        ex.fill_bytes(cells, 0, (size_t) zero_cells * 8);
    }
    const u64 n_flag_words = kc_div_up(n_bytes, (u64) 32) + 1;
    u32 *status = reinterpret_cast<u32 *>(cells + 3);
    kc_ull *m_cell = reinterpret_cast<kc_ull *>(cells + 2);
    {
        const int n_parts = chunks && chunks->n > 1 && !chunks->waited ? chunks->n : 1;
        if (chunks && n_parts == 1) chunks->wait_all(st);
        for (int c = 0; c < n_parts; ++c) {
            u32 t0 = 0, t1 = blocks;
            if (n_parts > 1) {
                KC_CUDA(cudaStreamWaitEvent(st, chunks->ev[c], 0));
                t0 = (u32) std::min<u64>(blocks, (u64) c * (chunks->chunk_bytes / TILE));
                t1 = c == n_parts - 1 ? blocks : (u32) std::min<u64>(blocks, (u64) (c + 1) * (chunks->chunk_bytes / TILE));
            }
            if (t1 <= t0) continue;
            const u64 part_bytes = std::min<u64>(n_bytes, (u64) t1 * TILE) - (u64) t0 * TILE;
            // sequence read, code words + flag words + records written
            CudaExec::Scope sc(ex, KP_KS_SCATTER0, part_bytes + part_bytes / 4 + part_bytes / 8 + (u64) (part_bytes * 8 / KC_SIG_WINDOWS_PER_RECORD));
            kc_sig_scan_launch<false>(ex, pl.m, t1 - t0, seq, n_bytes, k, pl.a, pl.n_buckets, cursor, recs, packed, flags, n_flag_words, t0, m_cell,
                                      status, win_mask, SigPeers());
        }
        if (chunks) chunks->waited = true;
    }
    {
        const u32 fit = (u32) (dv.n_sm * (dv.occ > 0 ? dv.occ : 1));
        const u32 grid = pl.n_buckets < fit ? pl.n_buckets : fit;
        // records read, two code words per record
        CudaExec::Scope sc(ex, KP_KS_RESOLVE, (u64) (n_bytes * (8 + 8 * Cfg::NW) / KC_SIG_WINDOWS_PER_RECORD));
        const bool pos64 = n_bytes > 0xFFFFFFFFULL;  // a window END position may need more than 32 bits
        auto *kern = complements ? (pos64 ? kc_sig_resolve_kernel<L, false, false, true> : kc_sig_resolve_kernel<L, false, false, false>)
                                 : (pos64 ? kc_sig_resolve_kernel<L, false, true, true> : kc_sig_resolve_kernel<L, false, true, false>);
        ex.launch(kern, grid, Cfg::THREADS, Cfg::smem(pos64), packed, k, cursor, recs, pl.n_buckets, kc_ksf_own_flags(flags), reinterpret_cast<kc_ull *>(cells),
                  status, 1u, KC_SIG_REC_CAP, 0u);
    }
    ex.arena->restore({base_mark, top_mark.top});
    return true;
}

// ---- multi-GPU (group.cuh) -----------------------------------------------------------------------------------------------------
// Records a (bucket, sender) sub-slot must hold: the bucket's mean share + 6 sigma (records arrive in clumps: sigma ~ 1.5 sqrt(mean)).
inline u32 kc_sig_sub_cap(const SigPlan &pl, int n_ranks) {
    const double mean = pl.mean_records / n_ranks;
    u32 cap = (u32) (mean * 1.06 + 7.0 * pl.clump * std::sqrt(mean) + 8.0);
    cap = (cap + 31) / 32 * 32;
    return cap < KC_SIG_REC_CAP ? cap : KC_SIG_REC_CAP;
}
inline u32 kc_sig_owned_buckets(u32 n_buckets, int n_ranks, int rank) { return (n_buckets + (u32) n_ranks - 1u - (u32) rank) / (u32) n_ranks; }

// Records one (sender, owner) stream must hold: the pair's share of the slice's records + 15 % + slack.  The kernels take it as a
// u32: kc_grp_large_bound (group.cuh) refuses the inputs where it reaches 2^32.
inline u64 kc_sig_region_cap(u64 n_bytes, int n_ranks) {
    const double per_pair = (double) n_bytes / n_ranks / KC_SIG_WINDOWS_PER_RECORD / n_ranks;
    return ((u64) (per_pair * 1.15) + 8192 + 31) / 32 * 32;
}
// Records the dense stream of a slice of slice_bytes may hold (kc_sig_compact_kernel reports more through the status word).
inline u64 kc_sig_dense_cap(u64 slice_bytes, int n_ranks) { return (u64) (slice_bytes / KC_SIG_WINDOWS_PER_RECORD * 1.3) + (u64) n_ranks * 8192 + 65536; }
// The most buckets any plan gives an input of up to n_bytes: kc_sig_plan keeps at least 32 records per bucket and fewer than 2^27 buckets.
inline u64 kc_sig_max_buckets(u64 n_bytes) {
    const u64 nb = (u64) ((double) n_bytes / (32.0 * KC_SIG_WINDOWS_PER_RECORD)) + 1;
    return nb < 64 ? 64 : (nb < (1u << 27) ? nb : (1u << 27));
}
// Bytes of the largest slice of the tiles a rank of n_ranks scans (kc_sig_group_scan).
inline u64 kc_sig_max_slice(u64 n_bytes, int n_ranks) {
    constexpr u64 TILE = 256 * KC_EX_STRIP;
    const u64 tiles = (n_bytes + TILE - 1) / TILE;
    return std::min<u64>(n_bytes, (tiles + (u64) n_ranks - 1) / (u64) n_ranks * TILE);
}

// Arena bytes of kc_grp_sig_flags on one rank: bucket counters, records staged per bucket, owner-major offsets and the dense stream
// of its slice (kc_sig_group_scan), then the gathered rows of the buckets it owns (kc_sig_group_resolve), + scan scratch.
inline u64 kc_sig_group_arena_bytes(const SigPlan &p, u64 n_bytes, int n_ranks) {
    const u64 nb = p.n_buckets, nbr = (nb + (u64) n_ranks - 1) / (u64) n_ranks;
    const u64 scan = nb * 4 + nb * kc_sig_sub_cap(p, n_ranks) * 8 + ((u64) n_ranks * nbr + 1) * 8 + kc_sig_dense_cap(kc_sig_max_slice(n_bytes, n_ranks), n_ranks) * 8;
    return scan + nbr * (4 + 8 * (u64) KC_SIG_REC_CAP) + (64u << 20);
}

// The scan of this rank's slice of the tiles (records staged per bucket, code words and valid-window words to every rank), then the
// staged records as dense streams to the owners.  cells: {-, -, M of the slice (+=), status (low word)}.
inline void kc_sig_group_scan(CudaExec &ex, const u8 *seq, u64 n_bytes, int k, const SigPlan &pl, const SigPeers &sp, u32 region_cap, u64 *cells) {
    constexpr u64 TILE = 256 * KC_EX_STRIP;
    const u32 tiles = (u32) kc_div_up(n_bytes, TILE);
    const u32 t0 = (u32) ((u64) tiles * (u32) sp.rank / (u32) sp.n), t1 = (u32) ((u64) tiles * ((u32) sp.rank + 1) / (u32) sp.n);
    const u32 nbr = kc_sig_owned_buckets(pl.n_buckets, sp.n, 0), n_om = (u32) sp.n * nbr;
    u32 *cursor = ex.alloc<u32>(pl.n_buckets);
    u64 *staged = ex.alloc<u64>((u64) pl.n_buckets * sp.sub_cap);
    u32 *off_om = ex.alloc<u32>((u64) n_om + 1);
    u32 *status = reinterpret_cast<u32 *>(cells + 3);
    ex.fill_bytes(cursor, 0, (size_t) pl.n_buckets * 4);
    u64 slice_bytes = 0;
    if (t1 > t0) {
        slice_bytes = std::min<u64>(n_bytes, (u64) t1 * TILE) - (u64) t0 * TILE;
        CudaExec::Scope sc(ex, KP_KS_SCATTER0, slice_bytes + (slice_bytes / 4 + slice_bytes / 8) * (u64) sp.n + (u64) (slice_bytes * 8 / KC_SIG_WINDOWS_PER_RECORD));
        kc_sig_scan_launch<true>(ex, pl.m, t1 - t0, seq, n_bytes, k, pl.a, pl.n_buckets, cursor, staged, nullptr, nullptr, kc_div_up(n_bytes, (u64) 32), t0,
                                 reinterpret_cast<kc_ull *>(cells + 2), status, nullptr, sp);
    }
    kc_sig_om_counts_kernel<<<(unsigned) kc_div_up((u64) n_om + 1, 256), 256, 0, ex.stream>>>(cursor, pl.n_buckets, nbr, (u32) sp.n, sp.sub_cap, off_om);
    ++ex.launches;
    KC_CUDA(cudaGetLastError());
    ex.exclusive_scan_nosync(off_om, off_om, (u64) n_om + 1);
    const u64 dense_cap = kc_sig_dense_cap(slice_bytes, sp.n);
    u64 *dense = ex.alloc<u64>(dense_cap);
    {
        const u64 rec_bytes = (u64) (slice_bytes * 8 / KC_SIG_WINDOWS_PER_RECORD);
        CudaExec::Scope sc(ex, KP_SORT_MISC, 4 * rec_bytes);  // compact: read + write; ship: read + write
        kc_sig_compact_kernel<<<(unsigned) kc_div_up((u64) n_om, 8), 256, 0, ex.stream>>>(cursor, staged, off_om, pl.n_buckets, nbr, (u32) sp.n, sp.sub_cap, dense, dense_cap,
                                                                                             status);
        kc_sig_ship_kernel<<<dim3(128, (unsigned) sp.n), 256, 0, ex.stream>>>(dense, off_om, nbr, region_cap, status, sp);
        ex.launches += 2;
        KC_CUDA(cudaGetLastError());
    }
}

// Owner side: the buckets of this rank (the senders' streams + offset tables in its own heap, code words of the whole sequence) ->
// losers cleared in every rank's flags.  cells: {kept (+=), -, -, status (low word)}.
template <int L>
void kc_sig_group_resolve(CudaExec &ex, const u64 *packed, int k, bool complements, u32 n_owned, const u32 *offsets, u32 off_stride, const u64 *recv, int n_ranks,
                          u32 region_cap, const KsfFlagPeers &all_flags, u64 *cells, u64 n_bytes) {
    typedef SigCfg<L> Cfg;
    typedef SigKernels<L> KK;
    if (n_owned == 0) return;
    const typename KK::Dev &dv = KK::prepare();
    const u32 fit = (u32) (dv.n_sm * (dv.occ > 0 ? dv.occ : 1));
    const u32 grid = n_owned < fit ? n_owned : fit;
    u32 *cnt_bm = ex.alloc<u32>(n_owned);
    u64 *recs_bm = ex.alloc<u64>((u64) n_owned * KC_SIG_REC_CAP);
    {
        CudaExec::Scope sc(ex, KP_SORT_MISC, (u64) (n_bytes / n_ranks * 16 / KC_SIG_WINDOWS_PER_RECORD));
        kc_sig_gather_kernel<<<(unsigned) kc_div_up((u64) n_owned, 8), 256, 0, ex.stream>>>(offsets, off_stride, recv, region_cap, (u32) n_ranks, n_owned, cnt_bm, recs_bm);
        ++ex.launches;
        KC_CUDA(cudaGetLastError());
    }
    CudaExec::Scope sc(ex, KP_KS_RESOLVE, (u64) (n_bytes / n_ranks * (8 + 8 * Cfg::NW) / KC_SIG_WINDOWS_PER_RECORD));
    if (n_bytes > 0xFFFFFFFFULL) {  // a window END position may need more than 32 bits (as in kc_kmerset_build_sig)
        const u32 fit64 = (u32) (dv.n_sm * (dv.occ_multi64 > 0 ? dv.occ_multi64 : 1));
        auto *kern = complements ? kc_sig_resolve_kernel<L, true, false, true> : kc_sig_resolve_kernel<L, true, true, true>;
        kern<<<n_owned < fit64 ? n_owned : fit64, Cfg::THREADS, Cfg::smem(true), ex.stream>>>(packed, k, cnt_bm, recs_bm, n_owned, all_flags, reinterpret_cast<kc_ull *>(cells),
                                                                                         reinterpret_cast<u32 *>(cells + 3), (u32) n_ranks, KC_SIG_REC_CAP, 0u);
    } else if (complements)
        kc_sig_resolve_kernel<L, true, false><<<grid, Cfg::THREADS, Cfg::smem(), ex.stream>>>(packed, k, cnt_bm, recs_bm, n_owned, all_flags, reinterpret_cast<kc_ull *>(cells),
                                                                                            reinterpret_cast<u32 *>(cells + 3), (u32) n_ranks, KC_SIG_REC_CAP, 0u);
    else
        kc_sig_resolve_kernel<L, true, true><<<grid, Cfg::THREADS, Cfg::smem(), ex.stream>>>(packed, k, cnt_bm, recs_bm, n_owned, all_flags, reinterpret_cast<kc_ull *>(cells),
                                                                                           reinterpret_cast<u32 *>(cells + 3), (u32) n_ranks, KC_SIG_REC_CAP, 0u);
    ++ex.launches;
    KC_CUDA(cudaGetLastError());
}

#endif  // __CUDACC__
