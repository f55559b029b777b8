// TEST INFRASTRUCTURE ONLY — see oracle.h.  Plain single-threaded C++ restatement of the reference's
// `compute` hot path; each function cites the reference file:line it follows.  Nothing here is ever
// linked into the product.
#include "oracle.h"

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <unordered_map>
#include <vector>

namespace {

// src/kmers.h:15-32 nucleotideToInt — A/a C/c G/g T/t -> 0..3, everything else 4.
inline int nucleotide_to_int(uint8_t c) {
    switch (c) {
        case 'A': case 'a': return 0;
        case 'C': case 'c': return 1;
        case 'G': case 'g': return 2;
        case 'T': case 't': return 3;
        default: return 4;
    }
}

const char kLetters[4] = {'A', 'C', 'G', 'T'};  // src/kmers.h:97

// Fixed-width unsigned integer of L 64-bit limbs, limb 0 least significant (the layout of uint64_t,
// __uint128_t and src/uint256_t/uint256_t.include:49-55).
template <int L> struct Word {
    uint64_t w[L];
    Word() { std::memset(w, 0, sizeof(w)); }
    explicit Word(uint64_t v) {
        std::memset(w, 0, sizeof(w));
        w[0] = v;
    }
    bool operator==(const Word &o) const { return std::memcmp(w, o.w, sizeof(w)) == 0; }
    bool operator!=(const Word &o) const { return !(*this == o); }
    bool operator<(const Word &o) const {
        for (int i = L - 1; i >= 0; --i)
            if (w[i] != o.w[i]) return w[i] < o.w[i];
        return false;
    }
    Word shl(int bits) const {
        Word r;
        int limb = bits / 64, off = bits % 64;
        for (int i = L - 1; i >= 0; --i) {
            uint64_t v = 0;
            if (i - limb >= 0) {
                v = w[i - limb] << off;
                if (off && i - limb - 1 >= 0) v |= w[i - limb - 1] >> (64 - off);
            }
            r.w[i] = v;
        }
        return r;
    }
    Word shr(int bits) const {
        Word r;
        int limb = bits / 64, off = bits % 64;
        for (int i = 0; i < L; ++i) {
            uint64_t v = 0;
            if (i + limb < L) {
                v = w[i + limb] >> off;
                if (off && i + limb + 1 < L) v |= w[i + limb + 1] << (64 - off);
            }
            r.w[i] = v;
        }
        return r;
    }
    Word operator|(const Word &o) const {
        Word r;
        for (int i = 0; i < L; ++i) r.w[i] = w[i] | o.w[i];
        return r;
    }
    Word operator&(const Word &o) const {
        Word r;
        for (int i = 0; i < L; ++i) r.w[i] = w[i] & o.w[i];
        return r;
    }
    static Word low_mask(int bits) {  // (1 << bits) - 1, bits < 64*L
        Word r;
        for (int i = 0; i < L; ++i) {
            int lo = i * 64;
            if (bits >= lo + 64) r.w[i] = ~0ULL;
            else if (bits > lo) r.w[i] = (1ULL << (bits - lo)) - 1;
        }
        return r;
    }
};

template <int L> struct WordHash {
    size_t operator()(const Word<L> &x) const {
        uint64_t h = 0x9e3779b97f4a7c15ULL;
        for (int i = 0; i < L; ++i) {
            h ^= x.w[i] + 0x9e3779b97f4a7c15ULL + (h << 6) + (h >> 2);
            h *= 0xff51afd7ed558ccdULL;
            h ^= h >> 33;
        }
        return (size_t) h;
    }
};

// src/kmers.h:35-44
template <int L> Word<L> bit_prefix(const Word<L> &x, int k, int d) { return x.shr((k - d) * 2); }
template <int L> Word<L> bit_suffix(const Word<L> &x, int d) { return x & Word<L>::low_mask(2 * d); }

// src/kmers.h:92-95: reverse the order of the k 2-bit symbols and complement each (3 - symbol).
// Restated symbol by symbol instead of with the word-parallel swap network; the result is the same number.
template <int L> Word<L> reverse_complement(const Word<L> &x, int k) {
    Word<L> r;
    for (int i = 0; i < k; ++i) {
        uint64_t sym = (x.w[(2 * i) / 64] >> ((2 * i) % 64)) & 3;  // symbol i counted from the right
        int dst = 2 * (k - 1 - i);
        r.w[dst / 64] |= (3 - sym) << (dst % 64);
    }
    return r;
}

template <int L> int symbol_at(const Word<L> &x, int k, int index) {  // src/kmers.h:99-102 AtIndex
    int bit = 2 * (k - index - 1);
    return (int) ((x.w[bit / 64] >> (bit % 64)) & 3);
}

template <int L> void store(const Word<L> &x, uint64_t *out) { std::memcpy(out, x.w, sizeof(x.w)); }
template <int L> Word<L> load(const uint64_t *in) {
    Word<L> r;
    std::memcpy(r.w, in, sizeof(r.w));
    return r;
}

// ---------------------------------------------------------------------------------------------------
// Stage 1: src/parser.h:53-85.  Instead of a khash map the occurrences are collected and sorted; the
// observable result (key -> min(occurrences-1,255)) is identical.
template <int L>
int count_kmers(const uint8_t *seq, const uint64_t *rec_off, const uint64_t *rec_len, uint64_t n_rec, int k,
                bool complements, uint64_t **keys_out, uint8_t **vals_out, uint64_t *n_out) {
    std::vector<Word<L>> occ;
    const Word<L> mask = Word<L>::low_mask(2 * k);
    const int shift = 2 * (k - 1);
    for (uint64_t r = 0; r < n_rec; ++r) {
        const uint8_t *s = seq + rec_off[r];
        int64_t current_length = 0;
        Word<L> cur, rc;
        for (uint64_t i = 0; i < rec_len[r]; ++i) {
            int data = nucleotide_to_int(s[i]);
            if (data >= 4) {  // parser.h:63-68 restart on a non-ACGT byte
                cur = Word<L>();
                rc = Word<L>();
                current_length = 0;
                continue;
            }
            cur = (cur.shl(2) | Word<L>((uint64_t) data)) & mask;               // parser.h:69
            rc = rc.shr(2) | Word<L>((uint64_t) (3 ^ data)).shl(shift);         // parser.h:70
            if (++current_length >= k)                                            // parser.h:71
                occ.push_back((!complements || cur < rc) ? cur : rc);             // parser.h:73
        }
    }
    std::sort(occ.begin(), occ.end());
    std::vector<Word<L>> keys;
    std::vector<uint8_t> vals;
    for (size_t i = 0; i < occ.size();) {
        size_t j = i;
        while (j < occ.size() && occ[j] == occ[i]) ++j;
        keys.push_back(occ[i]);
        vals.push_back((uint8_t) std::min<size_t>(255, j - i - 1));  // parser.h:77,81
        i = j;
    }
    *n_out = keys.size();
    *keys_out = (uint64_t *) std::malloc(std::max<size_t>(1, keys.size() * L * 8));
    *vals_out = (uint8_t *) std::malloc(std::max<size_t>(1, keys.size()));
    for (size_t i = 0; i < keys.size(); ++i) store(keys[i], *keys_out + i * L);
    if (!vals.empty()) std::memcpy(*vals_out, vals.data(), vals.size());
    return 0;
}

// ---------------------------------------------------------------------------------------------------
// Stage 3: src/global.h:43-133 line by line, with std::unordered_map standing in for the khash map.
// `parts` is the number of prefix batches: 16 is the reference (MEMORY_REDUCTION_FACTOR, global.h:48,66); 1 puts every prefix into
// one batch, the tie order of the product's from-FASTA engine (engine.cuh, strict = false).
template <int L>
int overlap_path(const uint64_t *first_in, const uint64_t *last_in, uint64_t n, int k, bool complements,
                 bool lower_bound, int64_t *edge_from, uint8_t *overlaps, int parts = 16) {
    const size_t NONE = (size_t) -1;
    const size_t count = n * (1 + (complements ? 1 : 0));                         // global.h:47
    const size_t batch = count / parts + 1;                                       // global.h:48
    std::vector<Word<L>> node_first(count), node_last(count);                     // accessPrefix/accessSuffix, global.h:16-21
    for (size_t i = 0; i < n; ++i) {
        node_first[i] = load<L>(first_in + i * L);
        node_last[i] = load<L>(last_in + i * L);
    }
    if (complements)
        for (size_t i = 0; i < n; ++i) {
            node_first[n + i] = reverse_complement(node_last[i], k);
            node_last[n + i] = reverse_complement(node_first[i], k);
        }
    std::vector<size_t> ef(count, NONE);
    std::vector<uint8_t> ov(count, 255);
    std::vector<char> suffix_forbidden(count, 0), prefix_forbidden(count, 0);
    std::vector<size_t> first(n), last(n), next(batch);
    for (size_t i = 0; i < n; ++i) first[i] = last[i] = i;
    // accessFirstLast, global.h:28-29
    auto access_fl = [&](const std::vector<size_t> &a, const std::vector<size_t> &b, size_t index) -> size_t {
        return n > index ? a[index] : (b[index - n] + n) % (2 * n);
    };
    std::unordered_map<Word<L>, size_t, WordHash<L>> prefixes;
    for (int d = k - 1; d >= 0; --d) {                                            // global.h:63
        for (int part = 0; part < parts; ++part) {                                // global.h:66
            prefixes.clear();
            std::fill(next.begin(), next.end(), NONE);
            size_t to = std::min(count, (size_t) (part + 1) * batch);
            size_t from = (size_t) part * batch;
            for (size_t i = from; i < to; ++i)                                    // global.h:73-85
                if (!prefix_forbidden[i]) {
                    next[i - from] = NONE;
                    Word<L> prefix = bit_prefix(node_first[i], k, d);
                    auto it = prefixes.find(prefix);
                    if (it != prefixes.end()) {
                        next[i - from] = it->second;
                        it->second = i;
                    } else {
                        prefixes.emplace(prefix, i);
                    }
                }
            for (size_t i = 0; i < count; ++i)                                    // global.h:86-125
                if (!suffix_forbidden[i]) {
                    Word<L> suffix = bit_suffix(node_last[i], d);
                    auto it = prefixes.find(suffix);
                    if (it == prefixes.end()) continue;
                    size_t previous, j;
                    previous = j = it->second;
                    while (j != NONE &&
                           ((!lower_bound && (i + n) % (2 * n) == j) ||
                            (!lower_bound && access_fl(first, last, i) == j) || prefix_forbidden[j])) {
                        size_t new_j = next[j - from];
                        if (prefix_forbidden[j]) next[previous - from] = new_j;
                        else previous = j;
                        j = new_j;
                    }
                    if (j == NONE) continue;
                    size_t xs[2] = {i, 0}, ys[2] = {j, 0};
                    int n_edges = 1;
                    if (complements) {                                            // global.h:110-112
                        xs[1] = (j + n) % count;
                        ys[1] = (i + n) % count;
                        n_edges = 2;
                    }
                    for (int e = 0; e < n_edges; ++e) {                           // global.h:113-122
                        size_t x = xs[e], y = ys[e];
                        ef[x] = y;
                        ov[x] = (uint8_t) d;
                        prefix_forbidden[y] = 1;
                        size_t last_y = access_fl(last, first, y);
                        size_t first_x = access_fl(first, last, x);
                        if (last_y < n) first[last_y] = first_x;
                        if (first_x < n) last[first_x] = last_y;
                        suffix_forbidden[x] = 1;
                    }
                    next[previous - from] = next[j - from];                       // global.h:123
                }
        }
    }
    for (size_t i = 0; i < count; ++i) {
        edge_from[i] = ef[i] == NONE ? -1 : (int64_t) ef[i];
        overlaps[i] = ov[i];
    }
    return 0;
}

// ---------------------------------------------------------------------------------------------------
// The nodes of the product's from-FASTA regime (kmercamel_b200/csrc/runs.cuh): the window END position of the first occurrence, in
// input order, of every kept canonical k-mer (occurring at least min_frequency times, counted as in count_kmers) is marked; a maximal
// run of consecutive marked ends e_s..e_t is the node seq[e_s - k + 1 .. e_t].  Positions are seq offsets, so records must be
// separated by a non-ACGT byte for runs not to cross them (the framing of records_to_arrays).
template <int L>
int first_occurrence_runs(const uint8_t *seq, const uint64_t *rec_off, const uint64_t *rec_len, uint64_t n_rec, int k,
                          bool complements, int min_frequency, uint64_t **off_out, uint64_t **len_out, uint64_t *n_out,
                          uint64_t *n_kept_out) {
    std::vector<std::pair<Word<L>, uint64_t>> occ;  // (canonical k-mer, window end)
    const Word<L> mask = Word<L>::low_mask(2 * k);
    const int shift = 2 * (k - 1);
    for (uint64_t r = 0; r < n_rec; ++r) {
        const uint8_t *s = seq + rec_off[r];
        int64_t current_length = 0;
        Word<L> cur, rc;
        for (uint64_t i = 0; i < rec_len[r]; ++i) {
            int data = nucleotide_to_int(s[i]);
            if (data >= 4) {
                cur = Word<L>();
                rc = Word<L>();
                current_length = 0;
                continue;
            }
            cur = (cur.shl(2) | Word<L>((uint64_t) data)) & mask;
            rc = rc.shr(2) | Word<L>((uint64_t) (3 ^ data)).shl(shift);
            if (++current_length >= k) occ.emplace_back((!complements || cur < rc) ? cur : rc, rec_off[r] + i);
        }
    }
    std::sort(occ.begin(), occ.end(), [](const std::pair<Word<L>, uint64_t> &a, const std::pair<Word<L>, uint64_t> &b) {
        return a.first < b.first || (a.first == b.first && a.second < b.second);
    });
    std::vector<uint64_t> ends;
    for (size_t i = 0; i < occ.size();) {
        size_t j = i;
        while (j < occ.size() && occ[j].first == occ[i].first) ++j;
        if (j - i >= (size_t) min_frequency) ends.push_back(occ[i].second);
        i = j;
    }
    *n_kept_out = ends.size();
    std::sort(ends.begin(), ends.end());
    std::vector<uint64_t> offs, lens;
    for (size_t i = 0; i < ends.size();) {
        size_t j = i + 1;
        while (j < ends.size() && ends[j] == ends[j - 1] + 1) ++j;
        offs.push_back(ends[i] - (uint64_t) (k - 1));
        lens.push_back(ends[j - 1] - ends[i] + (uint64_t) k);
        i = j;
    }
    *n_out = offs.size();
    *off_out = (uint64_t *) std::malloc(std::max<size_t>(1, offs.size() * 8));
    *len_out = (uint64_t *) std::malloc(std::max<size_t>(1, lens.size() * 8));
    if (!offs.empty()) {
        std::memcpy(*off_out, offs.data(), offs.size() * 8);
        std::memcpy(*len_out, lens.data(), lens.size() * 8);
    }
    return 0;
}

// ---------------------------------------------------------------------------------------------------
// Nodes as sequences (src/simplitigs.h:11-37,78-87); index >= n is the reverse complement (global.h:24-25).
struct Nodes {
    const uint8_t *seq;
    const uint64_t *off, *len;
    uint64_t n;
    uint64_t length(size_t v) const { return len[v < n ? v : v - n]; }
    int symbol(size_t v, uint64_t pos) const {  // 2-bit symbol at position pos of virtual node v
        if (v < n) return nucleotide_to_int(seq[off[v] + pos]);
        size_t u = v - n;
        return 3 - nucleotide_to_int(seq[off[u] + len[u] - 1 - pos]);
    }
};

template <int L> Word<L> kmer_at(const Nodes &nodes, size_t v, uint64_t index, int k) {  // simplitigs.h:30-38
    Word<L> r;
    for (int i = 0; i < k; ++i) r = r.shl(2) | Word<L>((uint64_t) nodes.symbol(v, index + i));
    return r;
}

template <int L> bool contains(const std::vector<Word<L>> &set, const Word<L> &x, int k, bool complements) {
    // khash_utils.h:98-103 containsKMer over a sorted vector
    bool ret = std::binary_search(set.begin(), set.end(), x);
    if (complements) ret |= std::binary_search(set.begin(), set.end(), reverse_complement(x, k));
    return ret;
}

inline char masked(char upper, bool mask) { return mask ? upper : (char) (upper + ('a' - 'A')); }  // kmers.h:124-127

// src/global.h:149-210
template <int L>
int superstring(const Nodes &nodes, int k, bool complements, const int64_t *edge_from, const uint8_t *overlaps,
                const std::vector<Word<L>> *set, std::vector<uint8_t> &ms, std::vector<uint8_t> *maxone) {
    const size_t count = nodes.n * (1 + (complements ? 1 : 0));
    std::vector<char> is_start(count, 1);                                         // global.h:156-161
    for (size_t i = 0; i < count; ++i)
        if (edge_from[i] >= 0) is_start[edge_from[i]] = 0;
    size_t start = 0;
    for (; start < count && !is_start[start]; ++start) {}
    if (start == count) return 1;
    auto print_start = [&](size_t v) {                                            // global.h:136-143
        uint64_t cnt = nodes.length(v) - k + 1;
        for (uint64_t i = 0; i < cnt; ++i) {
            char c = kLetters[nodes.symbol(v, i)];
            ms.push_back((uint8_t) c);
            if (maxone) maxone->push_back((uint8_t) c);
        }
    };
    Word<L> last = kmer_at<L>(nodes, start, nodes.length(start) - k, k);
    print_start(start);
    const Word<L> kmask = Word<L>::low_mask(2 * k);
    while (edge_from[start] >= 0) {                                               // global.h:176
        int ov = overlaps[start];
        size_t nxt = (size_t) edge_from[start];
        for (int j = 1; j < k - ov; ++j)                                          // global.h:180-182: last[1 .. k-ov)
            ms.push_back((uint8_t) masked(kLetters[symbol_at(last, k, j)], false));
        if (maxone) {
            Word<L> current = kmer_at<L>(nodes, nxt, 0, k);
            for (int j = 0; j < k - ov - 1; ++j) {                                // global.h:184-195
                last = (last.shl(2) | Word<L>((uint64_t) symbol_at(current, k, ov + j))) & kmask;
                maxone->push_back((uint8_t) masked(kLetters[symbol_at(last, k, 0)], contains(*set, last, k, complements)));
            }
        }
        last = kmer_at<L>(nodes, nxt, nodes.length(nxt) - k, k);
        print_start(nxt);
        start = nxt;
    }
    for (int j = 1; j < k; ++j) {                                                 // global.h:200-205 trailing k-1
        char c = masked(kLetters[symbol_at(last, k, j)], false);
        ms.push_back((uint8_t) c);
        if (maxone) maxone->push_back((uint8_t) c);
    }
    return 0;
}

uint8_t *to_malloc(const std::vector<uint8_t> &v) {
    uint8_t *p = (uint8_t *) std::malloc(std::max<size_t>(1, v.size()));
    if (!v.empty()) std::memcpy(p, v.data(), v.size());
    return p;
}

template <int L>
int superstring_entry(const uint8_t *seq, const uint64_t *rec_off, const uint64_t *rec_len, uint64_t n, int k,
                      bool complements, const int64_t *edge_from, const uint8_t *overlaps, const uint64_t *set_keys,
                      uint64_t n_set, uint8_t **ms_out, uint8_t **maxone_out, uint64_t *len_out) {
    Nodes nodes{seq, rec_off, rec_len, n};
    std::vector<Word<L>> set;
    if (maxone_out) {
        set.resize(n_set);
        for (uint64_t i = 0; i < n_set; ++i) set[i] = load<L>(set_keys + i * L);
        std::sort(set.begin(), set.end());
    }
    std::vector<uint8_t> ms, mo;
    int rc = superstring<L>(nodes, k, complements, edge_from, overlaps, maxone_out ? &set : nullptr, ms,
                            maxone_out ? &mo : nullptr);
    if (rc) return rc;
    *ms_out = to_malloc(ms);
    if (maxone_out) *maxone_out = to_malloc(mo);
    *len_out = ms.size();
    return 0;
}

// src/main.cpp:171-187 with -S, then src/global.h:217-226
template <int L>
int compute_from_simplitigs(const uint8_t *seq, const uint64_t *rec_off, const uint64_t *rec_len, uint64_t n, int k,
                            bool complements, bool want_maxone, uint8_t **ms_out, uint8_t **maxone_out,
                            uint64_t *len_out) {
    if (n == 0) return 1;  // global.h:219-221 "input cannot be empty"
    Nodes nodes{seq, rec_off, rec_len, n};
    for (uint64_t r = 0; r < n; ++r) {
        if (rec_len[r] < (uint64_t) k) return 2;
        for (uint64_t i = 0; i < rec_len[r]; ++i)
            if (nucleotide_to_int(seq[rec_off[r] + i]) > 3) return 3;  // simplitigs.h:82 assert
    }
    std::vector<uint64_t> first(n * L), last(n * L);
    for (uint64_t r = 0; r < n; ++r) {
        store(kmer_at<L>(nodes, r, 0, k), &first[r * L]);
        store(kmer_at<L>(nodes, r, rec_len[r] - k, k), &last[r * L]);
    }
    const size_t count = n * (1 + (complements ? 1 : 0));
    std::vector<int64_t> ef(count);
    std::vector<uint8_t> ov(count);
    overlap_path<L>(first.data(), last.data(), n, k, complements, false, ef.data(), ov.data());
    std::vector<Word<L>> set;
    if (want_maxone) {  // fill_kmers, simplitigs.h:41-51: the k-mers as they occur, not canonicalised
        for (uint64_t r = 0; r < n; ++r)
            for (uint64_t i = 0; i + k <= rec_len[r]; ++i) set.push_back(kmer_at<L>(nodes, r, i, k));
        std::sort(set.begin(), set.end());
        set.erase(std::unique(set.begin(), set.end()), set.end());
    }
    std::vector<uint8_t> ms, mo;
    int rc = superstring<L>(nodes, k, complements, ef.data(), ov.data(), want_maxone ? &set : nullptr, ms,
                            want_maxone ? &mo : nullptr);
    if (rc) return rc;
    *ms_out = to_malloc(ms);
    if (want_maxone) *maxone_out = to_malloc(mo);
    *len_out = ms.size();
    return 0;
}

// verify.py:41-57 through conversions.h:45-72: every upper-case position p starts a represented k-mer
// (ms2spss copies the run of upper-case letters plus the k-1 letters that follow, truncated at the end).
template <int L>
int ms_kmers(const uint8_t *ms, uint64_t len, int k, bool complements, uint64_t **keys_out, uint64_t *n_out,
             uint64_t *n_on_out) {
    std::vector<Word<L>> on;
    for (uint64_t p = 0; p + k <= len; ++p) {
        if (ms[p] > 'Z') continue;  // conversions.h:6-8 is_upper
        Word<L> x;
        bool ok = true;
        for (int i = 0; i < k; ++i) {
            int s = nucleotide_to_int(ms[p + i]);
            if (s > 3) { ok = false; break; }
            x = x.shl(2) | Word<L>((uint64_t) s);
        }
        if (!ok) continue;
        if (complements) {
            Word<L> rc = reverse_complement(x, k);
            if (rc < x) x = rc;
        }
        on.push_back(x);
    }
    *n_on_out = on.size();
    std::sort(on.begin(), on.end());
    on.erase(std::unique(on.begin(), on.end()), on.end());
    *n_out = on.size();
    *keys_out = (uint64_t *) std::malloc(std::max<size_t>(1, on.size() * L * 8));
    for (size_t i = 0; i < on.size(); ++i) store(on[i], *keys_out + i * L);
    return 0;
}


// ---------------------------------------------------------------------------------------------------
// `compute -a streaming [-z]`: src/streaming.h:12-48 (Streaming) and :51-107 (StreamingFiltered), restated with one
// occurrence counter per canonical k-mer.  Streaming stores the k-mer as read and probes both orientations
// (src/khash_utils.h:98-103 containsKMer), which is the same as one entry per canonical k-mer; StreamingFiltered keeps
// min(255, occurrences - 1) and turns a window ON when `count + 1 == min_frequency` (:96), i.e. at the z-th occurrence.
inline uint8_t masked_char(uint8_t c, bool mask) {  // src/kmers.h:124-127
    const int d = (int) (c <= 'Z') - (int) mask;
    return (uint8_t) (c + d * ('a' - 'A'));
}

template <int L>
int streaming(const uint8_t *seq, const uint64_t *rec_off, const uint64_t *rec_len, uint64_t n_rec, int k, bool complements,
              int min_frequency, uint8_t **out, uint64_t *len_out) {
    std::unordered_map<Word<L>, uint32_t, WordHash<L>> seen;  // canonical k-mer -> stored uint8 value (occurrences - 1, saturating)
    std::vector<uint8_t> of;
    const Word<L> mask = Word<L>::low_mask(2 * k);
    for (uint64_t r = 0; r < n_rec; ++r) {
        const uint8_t *s = seq + rec_off[r];
        const uint64_t l = rec_len[r];
        Word<L> kmer;
        uint64_t first_index = (uint64_t) k - 1;
        int64_t last_one = -(int64_t) k;
        for (uint64_t i = 0; i < l + (uint64_t) k - 1; ++i) {
            int c = 4;
            if (i < l) c = nucleotide_to_int(s[i]);
            if (c >= 4) {
                kmer = Word<L>();
                first_index = i + (uint64_t) k;
            }
            kmer = (kmer.shl(2) | Word<L>((uint64_t) c)) & mask;  // c = 4 spills into the next symbol exactly as in the reference
            bool on = false;
            if (i >= first_index) {
                Word<L> canon = kmer;
                if (complements) {
                    const Word<L> rc = reverse_complement(kmer, k);
                    if (rc < canon) canon = rc;
                }
                auto it = seen.find(canon);
                uint32_t count = 0;
                if (it != seen.end()) {
                    count = it->second + 1;
                    it->second = std::min<uint32_t>(255, count);
                } else {
                    seen.emplace(canon, 0u);
                }
                on = count + 1 == (uint32_t) min_frequency;
            }
            if (on) {
                of.push_back(masked_char(s[i - k + 1], true));
                last_one = (int64_t) i;
            } else if ((int64_t) i <= last_one + k - 1) {
                of.push_back(masked_char(s[i - k + 1], false));
            }
        }
    }
    *len_out = of.size();
    *out = (uint8_t *) std::malloc(of.size() + 1);
    if (!*out) return -1;
    if (!of.empty()) std::memcpy(*out, of.data(), of.size());
    return 0;
}

// `maskopt -t max-one | min-one`: Optimize (src/masks.h:240-261) = AddKMers(case_sensitive = true) (src/parser.h:22-49)
// followed by OptimizeOnes (src/masks.h:40-78).  Returns 1 when the superstring holds a non-ACGT letter (the reference
// throws std::invalid_argument after printing).  out: n letters.
template <int L>
int maskopt(const uint8_t *ms, uint64_t n, int k, bool complements, bool minimize, uint8_t *out) {
    std::unordered_map<Word<L>, uint32_t, WordHash<L>> set;
    const Word<L> mask = Word<L>::low_mask(2 * k);
    const int shift = 2 * (k - 1);
    {   // AddKMers, case sensitive: the window must start with an upper-case letter
        Word<L> cur, rc;
        int64_t cur_len = 0;
        std::vector<uint8_t> upper(n, 0);
        for (uint64_t i = 0; i < n; ++i) {
            const int d = nucleotide_to_int(ms[i]);
            if (d >= 4) {
                cur = rc = Word<L>();
                cur_len = 0;
                continue;
            }
            cur = (cur.shl(2) | Word<L>((uint64_t) d)) & mask;
            rc = rc.shr(2) | Word<L>((uint64_t) (3 ^ d)).shl(shift);
            upper[i] = ms[i] <= 'Z';
            if (++cur_len >= k && upper[i - k + 1]) set.emplace((!complements || cur < rc) ? cur : rc, 1u);
        }
    }
    int bad = 0;
    Word<L> cur, rc;
    for (uint64_t i = 0; i < n; ++i) {
        const int d = nucleotide_to_int(ms[i]);
        if (d >= 4) bad = 1;
        cur = (cur.shl(2) | Word<L>((uint64_t) d)) & mask;
        rc = rc.shr(2) | Word<L>((uint64_t) (3 ^ d)).shl(shift);
        if (i + 1 >= (uint64_t) k) {
            const Word<L> canon = (!complements || cur < rc) ? cur : rc;
            auto it = set.find(canon);
            const bool contained = it != set.end();
            out[i - k + 1] = masked_char(ms[i - k + 1], contained);
            if (minimize && contained) set.erase(it);
        }
    }
    for (uint64_t i = n >= (uint64_t) k ? n - k + 1 : n; i < n; ++i) out[i] = masked_char(ms[i], false);
    return bad;
}

}  // namespace

#define DISPATCH(k, fn, ...)                                  \
    do {                                                      \
        if ((k) < 1 || (k) > 127) return -1;                  \
        if ((k) < 32) return fn<1>(__VA_ARGS__);              \
        if ((k) < 64) return fn<2>(__VA_ARGS__);              \
        return fn<4>(__VA_ARGS__);                            \
    } while (0)

extern "C" {

int orc_limbs_for_k(int k) { return k < 32 ? 1 : (k < 64 ? 2 : 4); }  // src/main.cpp:309-315

int orc_count_kmers(const uint8_t *seq, const uint64_t *rec_off, const uint64_t *rec_len, uint64_t n_rec, int k,
                    int complements, uint64_t **keys_out, uint8_t **vals_out, uint64_t *n_out) {
    DISPATCH(k, count_kmers, seq, rec_off, rec_len, n_rec, k, complements != 0, keys_out, vals_out, n_out);
}

void orc_reverse_complement(const uint64_t *in, int k, uint64_t *out) {
    if (k < 32) store(reverse_complement(load<1>(in), k), out);
    else if (k < 64) store(reverse_complement(load<2>(in), k), out);
    else store(reverse_complement(load<4>(in), k), out);
}

void orc_bit_prefix(const uint64_t *in, int k, int d, uint64_t *out) {
    if (k < 32) store(bit_prefix(load<1>(in), k, d), out);
    else if (k < 64) store(bit_prefix(load<2>(in), k, d), out);
    else store(bit_prefix(load<4>(in), k, d), out);
}

void orc_bit_suffix(const uint64_t *in, int k, int d, uint64_t *out) {
    if (k < 32) store(bit_suffix(load<1>(in), d), out);
    else if (k < 64) store(bit_suffix(load<2>(in), d), out);
    else store(bit_suffix(load<4>(in), d), out);
}

int orc_overlap_path(const uint64_t *first, const uint64_t *last, uint64_t n, int k, int complements,
                     int lower_bound, int64_t *edge_from, uint8_t *overlaps) {
    DISPATCH(k, overlap_path, first, last, n, k, complements != 0, lower_bound != 0, edge_from, overlaps, 16);
}

int orc_overlap_path_parts(const uint64_t *first, const uint64_t *last, uint64_t n, int k, int complements,
                           int lower_bound, int parts, int64_t *edge_from, uint8_t *overlaps) {
    if (parts < 1 || parts > 16) return -1;
    DISPATCH(k, overlap_path, first, last, n, k, complements != 0, lower_bound != 0, edge_from, overlaps, parts);
}

int orc_first_occurrence_runs(const uint8_t *seq, const uint64_t *rec_off, const uint64_t *rec_len, uint64_t n_rec, int k,
                              int complements, int min_frequency, uint64_t **off_out, uint64_t **len_out, uint64_t *n_out,
                              uint64_t *n_kept_out) {
    if (min_frequency < 1) return -1;
    DISPATCH(k, first_occurrence_runs, seq, rec_off, rec_len, n_rec, k, complements != 0, min_frequency, off_out, len_out, n_out,
             n_kept_out);
}

int orc_superstring(const uint8_t *seq, const uint64_t *rec_off, const uint64_t *rec_len, uint64_t n, int k,
                    int complements, const int64_t *edge_from, const uint8_t *overlaps, const uint64_t *set_keys,
                    uint64_t n_set, uint8_t **ms_out, uint8_t **maxone_out, uint64_t *len_out) {
    DISPATCH(k, superstring_entry, seq, rec_off, rec_len, n, k, complements != 0, edge_from, overlaps, set_keys,
             n_set, ms_out, maxone_out, len_out);
}

int orc_compute_from_simplitigs(const uint8_t *seq, const uint64_t *rec_off, const uint64_t *rec_len, uint64_t n,
                                int k, int complements, int want_maxone, uint8_t **ms_out, uint8_t **maxone_out,
                                uint64_t *len_out) {
    DISPATCH(k, compute_from_simplitigs, seq, rec_off, rec_len, n, k, complements != 0, want_maxone != 0, ms_out,
             maxone_out, len_out);
}

int orc_ms_kmers(const uint8_t *ms, uint64_t len, int k, int complements, uint64_t **keys_out, uint64_t *n_out,
                 uint64_t *n_on_out) {
    DISPATCH(k, ms_kmers, ms, len, k, complements != 0, keys_out, n_out, n_on_out);
}

int orc_streaming(const uint8_t *seq, const uint64_t *rec_off, const uint64_t *rec_len, uint64_t n_rec, int k, int complements,
                  int min_frequency, uint8_t **out, uint64_t *len_out) {
    DISPATCH(k, streaming, seq, rec_off, rec_len, n_rec, k, complements != 0, min_frequency, out, len_out);
}

int orc_maskopt(const uint8_t *ms, uint64_t n, int k, int complements, int minimize, uint8_t *out) {
    DISPATCH(k, maskopt, ms, n, k, complements != 0, minimize != 0, out);
}

void orc_free(void *p) { std::free(p); }

}  // extern "C"
