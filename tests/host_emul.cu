// TESTS ONLY — serial host emulation of the engine / emission control flow (KC_HOST_EMUL).
//
// The build container has no GPU, so this binary instantiates kmercamel_b200/csrc/engine.cuh and emit.cuh with
// HostExec (a for-loop per "kernel", std::sort for the radix sort) to debug the level logic against the oracle.
// It is not part of libkcgpu.so and the product never runs it; the GPU tests exercise the real kernels.
//
//   host_emul path <k> <complements> <strict> <lower_bound>   records on stdin, one per line
//       -> "edge_from overlap" per virtual node
//   host_emul ms <k> <complements> <strict> <maxone>          records on stdin (nodes = records, like -S)
//       -> superstring, then (maxone) the max-one string
//   host_emul kmers <k> <complements> <strict> <maxone>       records on stdin; nodes = sorted distinct canonical
//       k-mers of the records (the from-FASTA regime) -> superstring [, max-one]
//   host_emul plan <m_upper> <leaf_target> <sigmas> 0         the fixed-slot plan of csrc/ksf_plan.h for an input of m_upper
//       windows -> "ok levels n_leaf slots0 slots1", then "bits cum cap" per level
//
// KC_ARENA_POISON=<0..255> in the environment fills every arena block with that byte before it is handed out (the option
// "arena_poison" of the library): the output must not change.
#include "../kmercamel_b200/csrc/emit.cuh"
#include "../kmercamel_b200/csrc/engine.cuh"
#include "../kmercamel_b200/csrc/ksf_plan.h"

#include <iostream>
#include <string>
#include <vector>

template <int L> KWord<L> kmer_of(const std::string &s, size_t pos, int k) {
    KWord<L> x = KWord<L>::zero();
    for (int i = 0; i < k; ++i) {
        x = x.shl(2);
        x.w[0] |= kc_nucleotide_code((u8) s[pos + i]) & 3;
    }
    return x;
}

static int arena_poison = -1;

template <int L> int run(const std::string &mode, int k, bool complements, bool strict, bool flag, const std::vector<std::string> &recs) {
    Arena arena;
    arena.cap = (size_t) 1 << 30;
    arena.base = (char *) std::malloc(arena.cap);
    arena.poison = arena_poison;
    arena.reset();
    HostExec ex{&arena};
    std::vector<KWord<L>> set;
    for (auto &r : recs)
        for (size_t i = 0; i + k <= r.size(); ++i) {
            KWord<L> x = kmer_of<L>(r, i, k);
            if (complements) {
                KWord<L> rc = kmer_reverse_complement(x, k);
                if (rc < x) x = rc;
            }
            set.push_back(x);
        }
    std::sort(set.begin(), set.end(), [](const KWord<L> &a, const KWord<L> &b) { return a < b; });
    set.erase(std::unique(set.begin(), set.end(), [](const KWord<L> &a, const KWord<L> &b) { return a == b; }), set.end());

    NodeView<L> nv;
    NodeSeq<L> ns;
    nv.k = ns.k = k;
    nv.complements = complements;
    std::vector<KWord<L>> first, last;
    std::string seq;
    std::vector<u64> off, len;
    if (mode == "kmers") {
        nv.first = nv.last = set.data();
        nv.n = (u32) set.size();
        ns.kmers = set.data();
        ns.seq = nullptr;
        ns.rec_off = ns.rec_len = nullptr;
    } else {
        for (auto &r : recs) {
            first.push_back(kmer_of<L>(r, 0, k));
            last.push_back(kmer_of<L>(r, r.size() - k, k));
            off.push_back(seq.size());
            len.push_back(r.size());
            seq += r;
            seq += '\n';
        }
        nv.first = first.data();
        nv.last = last.data();
        nv.n = (u32) recs.size();
        ns.kmers = nullptr;
        ns.seq = (const u8 *) seq.data();
        ns.rec_off = off.data();
        ns.rec_len = len.data();
    }
    nv.N = nv.n * (complements ? 2u : 1u);
    ns.n = nv.n;
    const bool lower_bound = mode == "path" && flag;
    Engine<HostExec, L> eng(ex, nv, strict, lower_bound);
    eng.init_state();
    eng.run();
    if (mode == "path") {
        for (u32 v = 0; v < nv.N; ++v)
            std::cout << (eng.st.edge_from[v] == KC_NONE ? -1LL : (long long) eng.st.edge_from[v]) << " " << (int) eng.st.ovl[v] << "\n";
    } else {
        EmitResult er = kc_emit_superstring<HostExec, L>(ex, ns, nv, eng.st, set.data(), set.size(), flag);
        std::cout << std::string((const char *) er.ms, er.length) << "\n";
        if (flag) std::cout << std::string((const char *) er.maxone, er.length) << "\n";
    }
    std::cerr << "levels=" << eng.stats.levels_run << " groups=" << eng.stats.groups << " edges=" << eng.stats.edges
              << " ban_rounds=" << eng.stats.ban_rounds << " bans=" << eng.stats.bans << "\n";
    std::free(arena.base);
    return 0;
}

int main(int argc, char **argv) {
    if (argc < 6) return 64;
    std::string mode = argv[1];
    if (const char *e = std::getenv("KC_ARENA_POISON")) arena_poison = std::atoi(e);
    if (mode == "plan") {
        KsfTuning t;
        t.leaf_target = (uint32_t) std::atoi(argv[3]);
        t.sigmas = std::atof(argv[4]);
        const KsfPlan pl = kc_ksf_plan(std::strtoull(argv[2], nullptr, 10), t);
        std::cout << (pl.ok ? 1 : 0) << " " << pl.n_levels << " " << pl.n_leaf << " " << pl.slots[0] << " " << pl.slots[1] << "\n";
        for (int i = 0; pl.ok && i < pl.n_levels; ++i) std::cout << pl.bits[i] << " " << pl.cum[i] << " " << pl.cap[i] << "\n";
        return 0;
    }
    int k = std::atoi(argv[2]);
    bool complements = std::atoi(argv[3]) != 0, strict = std::atoi(argv[4]) != 0, flag = std::atoi(argv[5]) != 0;
    std::vector<std::string> recs;
    std::string line;
    while (std::getline(std::cin, line))
        if (!line.empty()) recs.push_back(line);
    try {
        if (k < 32) return run<1>(mode, k, complements, strict, flag, recs);
        if (k < 64) return run<2>(mode, k, complements, strict, flag, recs);
        return run<4>(mode, k, complements, strict, flag, recs);
    } catch (const KcError &e) {
        std::cerr << "error " << e.code << ": " << e.what << " (" << e.file << ":" << e.line << ")\n";
        return 1;
    }
}
