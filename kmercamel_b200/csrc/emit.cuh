// Masked-superstring emission (reference src/global.h:149-210 SuperstringFromPath and its k-mer-node twin
// src/global_sparse.h:137-202).
//
// The reference walks edgeFrom[] from the lowest-numbered node without a predecessor and streams characters.
// Here the walk becomes a weighted list ranking (pointer doubling over edge_from with the number of characters
// each node contributes as weight), after which every node of the printed strand knows its output offset and
// all characters are written in parallel:
//     node v contributes its first len(v) - overlap(v) bases: the first len(v)-k+1 of them upper case (a
//     represented k-mer starts there), the rest lower case; the last node of the path contributes all len(v).
// `-M` (max-one mask, src/global.h:185-195): a lower-case position outside the final k-1 becomes upper case
// iff the k-mer that starts there in the superstring (or its reverse complement) is in the k-mer set; the
// hash-set probe becomes a binary search in the sorted set.
#pragma once
#include "engine.cuh"

template <int L> struct NodeSeq {
    const KWord<L> *kmers;  // != nullptr: node v < n is the single k-mer kmers[v]
    const u8 *seq;          // otherwise node v < n is the record seq[rec_off[v] .. +rec_len[v])
    const u64 *rec_off, *rec_len;
    u32 n;
    int k;
    KC_HD u64 length(u32 v) const { return kmers ? (u64) k : rec_len[v < n ? v : v - n]; }
    // 2-bit symbol at position pos of virtual node v (v >= n: reverse complement, src/global.h:24-25)
    KC_HD u32 symbol(u32 v, u64 pos) const {
        if (kmers) {
            if (v < n) return kmer_symbol(kmers[v], k, (int) pos);
            return 3u - kmer_symbol(kmers[v - n], k, k - 1 - (int) pos);
        }
        if (v < n) return kc_nucleotide_code(seq[rec_off[v] + pos]);
        u32 u = v - n;
        return 3u - kc_nucleotide_code(seq[rec_off[u] + rec_len[u] - 1 - pos]);
    }
};

KC_HD u8 kc_letter(u32 sym, bool upper) {
    const u32 packed = 'A' | ('C' << 8) | ('G' << 16) | ('T' << 24);  // src/kmers.h:97 letters
    u8 c = (u8) (packed >> (8 * sym));
    return upper ? c : (u8) (c + ('a' - 'A'));  // src/kmers.h:124-127 Masked
}

// Bucket index over the top `bits` bits of the 2k-bit k-mers of a SORTED set: start[b] = first position whose k-mer has a
// top-bits value >= b (start[2^bits] = n).  Cuts the ~log2(n) dependent DRAM probes of a binary search down to the index
// read plus a search inside one bucket (about two keys when 2^bits ~ n / 2).
template <int L> struct KmerIndex {
    const u32 *start = nullptr;
    int bits = 0, shift = 0;
};

template <int L> KC_HD bool kmer_set_contains(const KWord<L> *keys, u64 n, const KmerIndex<L> &ix, const KWord<L> &x) {
    u64 lo = 0, hi = n;
    if (ix.start) {
        const u32 b = x.digit(ix.shift, ix.bits);
        lo = ix.start[b];
        hi = ix.start[b + 1];
    }
    while (lo < hi) {
        const u64 mid = (lo + hi) >> 1;
        if (keys[mid] < x) lo = mid + 1;
        else hi = mid;
    }
    return lo < n && keys[lo] == x;  // src/khash_utils.h:98-103 containsKMer on the canonical k-mer
}

static const u32 KC_EMIT_SHORT = 128;   // contributions up to this many characters: one thread
static const u32 KC_EMIT_CHUNK = 16384;  // longer ones: chunks of this many characters, 256 work items each (KC_EMIT_SUB x 16 bytes per item:
static const u32 KC_EMIT_SUB = 4;        // the search for the chunk's node and its metadata loads are paid once for 64 bytes of output)

#ifdef __CUDACC__
template <int L> KmerIndex<L> kc_kmer_index_build(CudaExec &ex, const KWord<L> *keys, u64 n, int k) {
    KmerIndex<L> ix;
    if (n < 1024 || n >= 0xFFFFFFFFULL) return ix;  // small sets: a plain binary search stays in cache
    int bits = kc_ceil_log2(n) - 1;
    if (bits > 24) bits = 24;
    if (bits > 2 * k) bits = 2 * k;
    const u64 nb = 1ULL << bits;
    u32 *start = ex.alloc<u32>(nb + 1);
    const int shift = 2 * k - bits;
    ex.for_each(n + 1, [=] __device__(u64 i) {
        const u64 b_prev = i == 0 ? 0 : (u64) keys[i - 1].digit(shift, bits) + 1;  // first bucket not yet started
        const u64 b_cur = i == n ? nb : (u64) keys[i].digit(shift, bits);
        for (u64 b = b_prev; b <= b_cur; ++b) start[b] = (u32) i;
    }, KP_MISC, n * sizeof(KWord<L>) + nb * 4);
    ix.start = start;
    ix.bits = bits;
    ix.shift = shift;
    return ix;
}

static const u32 KC_RANK_SMALL = 1024;

// Chunks of KC_EMIT_CHUNK output characters that node v writes, given its rank (the record-node emission of kc_emit_superstring).
KC_HD u32 kc_emit_node_chunks(u64 cnt, u64 off, u64 s_begin, u64 s_end) {
    if (cnt <= KC_EMIT_SHORT) return 0;
    // the node's chunks start at its 16-byte aligned first byte; only those that meet the slice [s_begin, s_end) of this
    // rank are enumerated (a rank of an 8-GPU job used to walk all chunks of the whole superstring: 0.26 ms instead of 0.06)
    const u64 a0 = off & ~(u64) 15, a1 = off + cnt;
    const u64 lo = a0 > s_begin ? a0 : s_begin, hi = a1 < s_end ? a1 : s_end;
    return lo < hi ? (u32) ((hi - a0 + KC_EMIT_CHUNK - 1) / KC_EMIT_CHUNK - (lo - a0) / KC_EMIT_CHUNK) : 0u;
}

// List ranking of up to KC_RANK_SMALL nodes by one CTA in shared memory (same recurrences as the multi-kernel path).
// chunks != nullptr (the deferred emission of a whole superstring): the same CTA also writes the exclusive prefix of the chunk counts
// (chunks[0..N], N + 1 entries) and the characters of the short contributions into ms, which would otherwise take three more launches.
// n_dev != nullptr: {n, N} on the device, and N is their cap (the entries past the real N get no chunks).
template <int L>
__global__ void __launch_bounds__(256) kc_rank_small_kernel(PathState s, NodeSeq<L> q, u32 N, u32 *fin_out, u64 *dist_out, u64 *cell,
                                                            const u32 *n_dev, u32 *chunks, u8 *ms) {
    __shared__ u32 jump[2][KC_RANK_SMALL], fin[2][KC_RANK_SMALL];
    __shared__ u64 dist[2][KC_RANK_SMALL];
    __shared__ u32 s_start, s_cyc;
    __shared__ u32 sw[8];
    kc_pdl_wait();
    kc_pdl_trigger();  // one CTA: the next kernel's launch overlaps this one
    const u32 n_cells = N;  // chunks[] has n_cells + 1 entries
    if (n_dev) {
        q.n = n_dev[0];
        N = n_dev[1];
    }
    if (threadIdx.x == 0) {
        s_start = KC_NONE;
        s_cyc = 0;
    }
    __syncthreads();
    for (u32 v = threadIdx.x; v < N; v += 256) {
        const u32 nx = s.edge_from[v];
        jump[0][v] = nx;
        fin[0][v] = v;
        dist[0][v] = q.length(v) - (nx != KC_NONE ? (u64) s.ovl[v] : 0);
        if (s.edge_to[v] == KC_NONE) atomicMin(&s_start, v);  // src/global.h:156-161 start
    }
    __syncthreads();
    int rounds = 1;
    while ((1u << (rounds - 1)) < N) ++rounds;
    int cur = 0;
    for (int it = 0; it < rounds; ++it) {
        for (u32 v = threadIdx.x; v < N; v += 256) {
            const u32 j = jump[cur][v];
            if (j == KC_NONE) {
                jump[cur ^ 1][v] = KC_NONE;
                fin[cur ^ 1][v] = fin[cur][v];
                dist[cur ^ 1][v] = dist[cur][v];
            } else {
                jump[cur ^ 1][v] = jump[cur][j];
                fin[cur ^ 1][v] = fin[cur][j];
                dist[cur ^ 1][v] = dist[cur][v] + dist[cur][j];
            }
        }
        __syncthreads();
        cur ^= 1;
    }
    for (u32 v = threadIdx.x; v < N; v += 256) {
        fin_out[v] = fin[cur][v];
        dist_out[v] = dist[cur][v];
        if (jump[cur][v] != KC_NONE) s_cyc = 1;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const u32 st0 = s_start;
        cell[0] = st0 == KC_NONE ? ~0ULL : (u64) st0;
        cell[1] = s_cyc ? 0 : 1;
        cell[2] = st0 < N ? dist[cur][st0] : 0;
        cell[3] = st0 < N ? fin[cur][st0] : 0;
    }
    if (!chunks) return;
    const u32 st0 = s_start;
    const u64 total = st0 < N ? dist[cur][st0] : 0;
    const u32 fin_start = st0 < N ? fin[cur][st0] : 0;
    u32 carry = 0;
    for (u32 t0 = 0; t0 <= n_cells; t0 += 1024) {  // exclusive scan over n_cells + 1 entries, four per thread
        const u32 base = t0 + threadIdx.x * 4;
        u32 c4[4], c = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const u32 v = base + j;
            c4[j] = 0;
            if (v < N && fin[cur][v] == fin_start) {
                const u64 cnt = q.length(v) - (s.edge_from[v] != KC_NONE ? (u64) s.ovl[v] : 0);
                c4[j] = kc_emit_node_chunks(cnt, total - dist[cur][v], 0, total);
            }
            c += c4[j];
        }
        u32 tile;
        u32 p = kc_block_exclusive_scan_256(c, &tile, sw) + carry;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (base + j <= n_cells) chunks[base + j] = p;
            p += c4[j];
        }
        carry += tile;
        __syncthreads();  // sw is reused by the next tile
    }
    for (u32 v = threadIdx.x; v < N; v += 256) {  // the short contributions, one thread each
        if (fin[cur][v] != fin_start) continue;
        const u64 len = q.length(v);
        const u64 cnt = len - (s.edge_from[v] != KC_NONE ? (u64) s.ovl[v] : 0);
        if (cnt > KC_EMIT_SHORT) continue;
        const u64 off = total - dist[cur][v];
        const u64 n_upper = len - q.k + 1;
        for (u64 j = 0; j < cnt && off + j < total; ++j) ms[off + j] = kc_letter(q.symbol(v, j), j < n_upper);
    }
}
#endif

struct EmitResult {
    u8 *ms = nullptr;      // device, `length` bytes
    u8 *maxone = nullptr;  // device, `length` bytes, or nullptr
    u64 length = 0;        // of the WHOLE superstring
    u64 n_printed = 0;     // nodes on the printed strand
    u64 slice_begin = 0, slice_len = 0;  // the part of it that `ms` holds (the whole superstring unless a slice was asked for)
};

// The speculative tail of kcgpu.cu: the node count is on the device ({n, N} at n_dev; nv and ns hold its cap) and the emission's
// cell goes to `cell`, which the caller reads back with the rest of its status (kc_emit_check on words 0..3 of it).
struct EmitSpec {
    const u32 *n_dev;
    u64 *cell;  // 6 words
};

// The host's checks of the emission's cell {start node, 0 if a cycle survived, length, ...}.
inline void kc_emit_check(const u64 *info, u64 N, u64 total_ub) {
    if (info[0] >= N) KC_THROW(KC_ERR_INTERNAL, "no start node: the path cover contains only cycles");
    if (info[1] == 0) KC_THROW(KC_ERR_INTERNAL, "cycle in the final path cover");
    if (total_ub && info[2] > total_ub) KC_THROW(KC_ERR_INTERNAL, "superstring longer than its bound");
}

// set_keys: sorted distinct (canonical when complements) k-mers, needed only for want_maxone.
template <class Exec, int L>
EmitResult kc_emit_superstring(Exec &ex, const NodeSeq<L> &ns, const NodeView<L> &nv, const PathState &st,
                               const KWord<L> *set_keys, u64 n_set, bool want_maxone, u32 slice_index = 0, u32 n_slices = 1, u64 total_ub = 0,
                               const EmitSpec *spec = nullptr) {
    // total_ub: an upper bound of the superstring length known to the caller (0 = none).  With it, a small problem (one-CTA list
    // ranking, record nodes, whole superstring) is emitted WITHOUT reading the length back first: the kernels take the length and the
    // printed strand from the device cell, the buffer and the launches are sized by the bound, and the one read-back comes after the
    // last kernel is queued — the GPU does not idle through a host round trip in the middle of a 0.7 ms job.
    EmitResult res;
    const u64 N = nv.N;
    const int k = nv.k;
    size_t mark = ex.arena->mark();
    u32 *jump_a = ex.template alloc<u32>(N), *jump_b = ex.template alloc<u32>(N);
    u32 *fin_a = ex.template alloc<u32>(N), *fin_b = ex.template alloc<u32>(N);
    u64 *dist_a = ex.template alloc<u64>(N), *dist_b = ex.template alloc<u64>(N);
    u64 *cell = spec ? spec->cell : ex.template alloc<u64>(6);  // [0] start node, [1] 0 if a cycle survived, [2..4] info for the host
    const u32 *n_dev = spec ? spec->n_dev : nullptr;
    const PathState s = st;
    const NodeSeq<L> q = ns, q0 = ns;
    bool ranked = false;
    bool deferred = false;
    u8 *ms_pre = nullptr;
    u32 *chunks_pre = nullptr;
#ifdef __CUDACC__
    if constexpr (Exec::is_device) {
        if (N <= KC_RANK_SMALL) {  // the whole list ranking in one CTA (a genome leaves a few dozen nodes)
            deferred = total_ub && !ns.kmers && !want_maxone && n_slices == 1;
            if (deferred) {
                ms_pre = ex.template alloc<u8>(total_ub + 1);
                chunks_pre = ex.template alloc<u32>(N + 1);
            }
            typename Exec::Scope sc(ex, KP_RANK, N * 25);
            ex.launch(kc_rank_small_kernel<L>, 1, 256, 0, s, q, (u32) N, fin_a, dist_a, cell, n_dev, chunks_pre, ms_pre);
            ranked = true;
        }
    }
#endif
    if (spec && !deferred) KC_THROW(KC_ERR_INTERNAL, "the speculative tail needs the deferred one-CTA emission");
    if (!ranked) {
        ex.fill_bytes(cell, 0xFF, 16);
        ex.for_each(N, [=] KC_HD_LAMBDA(u64 vv) {
            u32 v = (u32) vv;
            u32 nx = s.edge_from[v];
            jump_a[v] = nx;
            fin_a[v] = v;
            dist_a[v] = q.length(v) - (nx != KC_NONE ? (u64) s.ovl[v] : 0);  // characters contributed by v
            if (s.edge_to[v] == KC_NONE) KC_ATOMIC_MIN((kc_ull *) &cell[0], (kc_ull) v);  // src/global.h:156-161 start
        }, KP_RANK, N * 25);
        int rounds = kc_ceil_log2(N) + 1;
        for (int it = 0; it < rounds; ++it) {
            const u32 *ja = jump_a, *fa = fin_a;
            const u64 *da = dist_a;
            u32 *jb = jump_b, *fb = fin_b;
            u64 *db = dist_b;
            ex.for_each(N, [=] KC_HD_LAMBDA(u64 v) {
                u32 j = ja[v];
                if (j == KC_NONE) {
                    jb[v] = KC_NONE;
                    fb[v] = fa[v];
                    db[v] = da[v];
                } else {
                    jb[v] = ja[j];
                    fb[v] = fa[j];
                    db[v] = da[v] + da[j];
                }
            }, KP_RANK, N * 32);
            u32 *t = jump_a; jump_a = jump_b; jump_b = t;
            t = fin_a; fin_a = fin_b; fin_b = t;
            u64 *m = dist_a; dist_a = dist_b; dist_b = m;
        }
        {
            const u32 *ja = jump_a;
            ex.for_each(N, [=] KC_HD_LAMBDA(u64 v) {
                if (ja[v] != KC_NONE) cell[1] = 0;  // a cycle survived: engine bug
            });
            const u32 *fa = fin_a;
            const u64 *da = dist_a;
            const u64 NN = N;
            ex.for_each(1, [=] KC_HD_LAMBDA(u64) {  // everything the host needs, in one place
                const u64 st0 = cell[0];
                cell[2] = st0 < NN ? da[st0] : 0;
                cell[3] = st0 < NN ? fa[st0] : 0;
            });
        }
    }
    const u64 *cellp = deferred ? cell : nullptr;  // deferred: the kernels below read the length and the printed strand from here
    u64 info[4] = {0, 1, total_ub, 0};
    if (!deferred) {
        ex.read_n(cell, info, 4);
        kc_emit_check(info, N, 0);
    }
    const u64 total_h = info[2];  // deferred: the bound (sizes the buffer and the launches)
    const u32 fin_start_h = (u32) info[3];
    const u64 total = total_h;
    // results live below the scratch: release the scratch first, then allocate outputs, then re-reserve scratch
    // is not possible with a bump arena, so outputs are allocated after the scratch and the scratch is leaked
    // until the caller releases its own mark.
    // Multi-GPU: every rank walks the same path and writes only its slice [s_begin, s_end) of the superstring (boundaries are
    // multiples of 16, so the 16-byte stores below stay aligned); `ms` is biased so that ms[a] is superstring position a.
    if (n_slices > 1 && (ns.kmers || want_maxone)) KC_THROW(KC_ERR_ARG, "sliced emission is for record nodes without -M");
    const u64 s_begin = n_slices > 1 ? ((total / n_slices) * slice_index) & ~(u64) 15 : 0;
    const u64 s_end_h = n_slices > 1 && slice_index + 1 < n_slices ? ((total / n_slices) * (slice_index + 1)) & ~(u64) 15 : total;
    const u64 s_end = s_end_h;
    const u32 fin_start = fin_start_h;
    u8 *ms_base = deferred ? ms_pre : ex.template alloc<u8>(s_end - s_begin + 1);
    u8 *ms = ms_base - s_begin;
    res.ms = ms_base;
    res.length = total;
    res.slice_begin = s_begin;
    res.slice_len = s_end - s_begin;
    const u32 *fa = fin_a;
    const u64 *da = dist_a;
    if (ns.kmers) {
        ex.for_each(N, [=] KC_HD_LAMBDA(u64 vv) {
            u32 v = (u32) vv;
            if (fa[v] != fin_start) return;
            u64 off = total - da[v];
            u32 cnt = (u32) (k - (s.edge_from[v] != KC_NONE ? (int) s.ovl[v] : 0));
            KWord<L> x = q.kmers[v < q.n ? v : v - q.n];
            if (v >= q.n) x = kmer_reverse_complement(x, k);
            for (u32 j = 0; j < cnt; ++j) ms[off + j] = kc_letter(kmer_symbol(x, k, (int) j), j == 0);
        }, KP_EMIT, N * 12 + (u64) q.n * sizeof(KWord<L>) + total);
    } else {
        // Record nodes.  Short contributions: one thread per node.  Long ones (simplitigs, first-occurrence runs of
        // a genome can span megabases) are cut into chunks of KC_EMIT_CHUNK characters; one group of 256 work items
        // writes one chunk with coalesced stores.
        // Chunks are laid out on the OUTPUT: a chunk is 256 work items x 16 bytes, 16-byte aligned in `ms`, so a full
        // item is one st.global.v4 and a warp writes 512 contiguous bytes (the per-character version spent 0.16 ms
        // on 50 MB; byte stores, not DRAM, were the bound).
        // Deferred: kc_rank_small_kernel has written the chunk prefix and the short contributions already.
        u32 *chunks = deferred ? chunks_pre : ex.template alloc<u32>(N + 1);
        if (!deferred) {
            ex.for_each(N + 1, [=] KC_HD_LAMBDA(u64 vv) {
                u32 c = 0;
                if (vv < N && fa[vv] == fin_start_h) {
                    u32 v = (u32) vv;
                    u64 cnt = q.length(v) - (s.edge_from[v] != KC_NONE ? (u64) s.ovl[v] : 0);
                    c = kc_emit_node_chunks(cnt, total_h - da[v], s_begin, s_end_h);
                }
                chunks[vv] = c;
            }, KP_EMIT, N * 12);
        }
        // Few nodes: launch for an upper bound of the chunk count (a node's chunks span at most its characters + 15 bytes of
        // alignment) and let the surplus work items exit, instead of reading the exact count back.
        u32 n_chunks = 0;
        bool bounded = false;
#ifdef __CUDACC__
        if constexpr (Exec::is_device) {
            if (N <= 65536) {
                bounded = true;
                if (!deferred) ex.exclusive_scan_nosync(chunks, chunks, N + 1);
                n_chunks = (u32) ((s_end - s_begin) / KC_EMIT_CHUNK + 2 * N + 1);
            }
        }
#endif
        if (!bounded) n_chunks = ex.exclusive_scan(chunks, chunks, N + 1);
        if (!deferred) ex.for_each(N, [=] KC_HD_LAMBDA(u64 vv) {
            const u64 total = total_h;
            const u32 fin_start = fin_start_h;
            const u64 s_end = s_end_h;
            u32 v = (u32) vv;
            if (fa[v] != fin_start) return;
            u64 len = q.length(v);
            u64 cnt = len - (s.edge_from[v] != KC_NONE ? (u64) s.ovl[v] : 0);
            if (cnt > KC_EMIT_SHORT) return;
            u64 off = total - da[v];
            if (off >= s_end || off + cnt <= s_begin) return;
            u64 n_upper = len - k + 1;
            for (u64 j = 0; j < cnt; ++j)
                if (off + j >= s_begin && off + j < s_end) ms[off + j] = kc_letter(q.symbol(v, j), j < n_upper);
        }, KP_EMIT, N * 12);
        ex.for_each((u64) n_chunks * 256, [=] KC_HD_LAMBDA(u64 w) {
            const u64 total = cellp ? cellp[2] : total_h;
            const u64 s_end = cellp ? total : s_end_h;
            NodeSeq<L> q = q0;
            if (n_dev) q.n = n_dev[0];
            u32 chunk = (u32) (w >> 8), lane = (u32) (w & 255);
            if (chunk >= chunks[N]) return;  // chunks[N] = the exact number of chunks
            // node owning this chunk: last v with chunks[v] <= chunk (chunks[] is the exclusive prefix, N+1 entries)
            u32 lo = 0, hi = (u32) N;
            while (lo < hi) {
                u32 mid = (lo + hi + 1) >> 1;
                if (chunks[mid] <= chunk) lo = mid;
                else hi = mid - 1;
            }
            u32 v = lo;
            u64 len = q.length(v);
            u64 cnt = len - (s.edge_from[v] != KC_NONE ? (u64) s.ovl[v] : 0);
            u64 n_upper = len - k + 1;
            u64 off = total - da[v];
            // output bytes [a0, a0 + 16) of this item, clipped to the node's [off, off + cnt)
            const u64 n0 = off & ~(u64) 15;                                             // first chunk of the node that meets the slice
            const u64 skip = n0 < s_begin ? (s_begin - n0) / KC_EMIT_CHUNK : 0;
            const u64 c0 = n0 + ((u64) (chunk - chunks[v]) + skip) * KC_EMIT_CHUNK + (u64) lane * 16;
            static_assert(KC_EMIT_CHUNK == KC_EMIT_SUB * 256 * 16, "a chunk is 256 work items x KC_EMIT_SUB x 16 bytes");
            for (u32 sub = 0; sub < KC_EMIT_SUB; ++sub) {
            u64 a0 = c0 + (u64) sub * (256 * 16);
            u64 b0 = a0 < off ? off : a0;
            u64 b1 = a0 + 16 < off + cnt ? a0 + 16 : off + cnt;
            if (b0 < s_begin) b0 = s_begin;  // slice boundaries are multiples of 16: an item is inside or outside as a whole
            if (b1 > s_end) b1 = s_end;
            if (b0 >= b1) continue;
            const u64 j0 = b0 - off;
#ifdef __CUDA_ARCH__
            const bool one_case = j0 + 16 <= n_upper || j0 >= n_upper;
#else
            const bool one_case = false;  // host emulation (tests): the per-character path below
#endif
            if (b1 - b0 == 16 && one_case) {
#ifdef __CUDA_ARCH__
                // Whole item with one case: 16 source bytes in five aligned words, case (and, on the mirror strand, order and
                // complement) changed four characters at a time.  Node characters are ACGT in either case by construction
                // (first-occurrence runs span valid windows only, -S records were validated).
                const u32 u = v < q.n ? v : v - q.n;
                const u64 src0 = v < q.n ? q.rec_off[u] + j0 : q.rec_off[u] + q.rec_len[u] - 16 - j0;
                const u32 *wp = reinterpret_cast<const u32 *>(q.seq + (src0 & ~(u64) 3));
                const u32 sh = (u32) (src0 & 3) * 8;
                u32 in[5];
#pragma unroll
                for (int x = 0; x < 4; ++x) in[x] = wp[x];
                in[4] = sh ? wp[4] : 0u;
                u32 wd[4];
#pragma unroll
                for (int x = 0; x < 4; ++x) wd[x] = __funnelshift_r(in[x], in[x + 1], sh) & 0xDFDFDFDFu;  // upper case
                if (v >= q.n) {
                    u32 r[4];
#pragma unroll
                    for (int x = 0; x < 4; ++x) {
                        const u32 t = __byte_perm(wd[3 - x], 0u, 0x0123);
                        const u32 cg = ((t >> 1) & 0x01010101u) * 0xFFu;              // bytes holding C or G
                        r[x] = t ^ ((cg & 0x04040404u) | (~cg & 0x15151515u));        // C <-> G, A <-> T
                    }
#pragma unroll
                    for (int x = 0; x < 4; ++x) wd[x] = r[x];
                }
                if (j0 >= n_upper) {
#pragma unroll
                    for (int x = 0; x < 4; ++x) wd[x] |= 0x20202020u;
                }
                *reinterpret_cast<uint4 *>(ms + b0) = make_uint4(wd[0], wd[1], wd[2], wd[3]);
#endif
            } else if (b1 - b0 == 16) {
                u32 wd[4];
                u64 j = b0 - off;
                for (int x = 0; x < 4; ++x) {
                    u32 t = 0;
                    for (int y = 0; y < 4; ++y) t |= (u32) kc_letter(q.symbol(v, j + 4 * x + y), j + 4 * x + y < n_upper) << (8 * y);
                    wd[x] = t;
                }
                *reinterpret_cast<uint4 *>(ms + b0) = make_uint4(wd[0], wd[1], wd[2], wd[3]);
            } else {
                for (u64 a = b0; a < b1; ++a) ms[a] = kc_letter(q.symbol(v, a - off), a - off < n_upper);
            }
            }
        }, KP_EMIT, 2 * total);
    }
    if (want_maxone) {
        u8 *mo = ex.template alloc<u8>(total + 1);
        res.maxone = mo;
        const bool complements = nv.complements;
        KmerIndex<L> ix;
#ifdef __CUDACC__
        if constexpr (Exec::is_device) ix = kc_kmer_index_build<L>(ex, set_keys, n_set, k);
#endif
        ex.for_each(total, [=] KC_HD_LAMBDA(u64 p) {
            u8 c = ms[p];
            if (c <= 'Z' || p + k > total) {  // already ON, or inside the trailing k-1 (src/global.h:200-208)
                mo[p] = c;
                return;
            }
            KWord<L> x = KWord<L>::zero();
            for (int i = 0; i < k; ++i) x = x.shl(2) | KWord<L>::from_u64(kc_nucleotide_code(ms[p + i]));
            if (complements) {
                KWord<L> r = kmer_reverse_complement(x, k);
                if (r < x) x = r;
            }
            const bool present = kmer_set_contains(set_keys, n_set, ix, x);
            mo[p] = present ? (u8) (c - ('a' - 'A')) : c;
        }, KP_MAXONE, 2 * total);
    }
    if (deferred && !spec) {  // the one read-back of the stage, after its last kernel was queued
        ex.read_n(cell, info, 4);
        kc_emit_check(info, N, total_ub);
        res.length = info[2];
        res.slice_len = info[2];
    }
    res.n_printed = nv.n;  // one strand: every node or its mirror
    (void) mark;
    return res;
}
