// kmercamel (B200) — host side of `kmercamel compute`: flags, file reading, FASTA framing, output writing.
// Everything between "bytes in memory" and "masked superstring in memory" happens on the GPU behind the C ABI of
// include/kcgpu.h; this file mirrors the user-visible behaviour of the reference CLI for the compute sub-command:
// flags and validation (reference src/main.cpp:214-316), the header line (src/parser.h:167-179), the stderr stage
// log (src/parser.h:159-164, src/main.cpp:133,160,174, src/global.h:223,225) and the two-line .msfa output.
// The neighbouring sub-commands are mirrored as well: lowerbound (src/main.cpp:378-443), `compute -a streaming`
// (src/main.cpp:139-144), maskopt -t max-one|min-one (src/main.cpp:318-376) and the four text conversions ms2mssep,
// mssep2ms, ms2spss, spss2ms (src/main.cpp:444-667, src/conversions.h).  `verify` (not in the reference CLI) is the -V check on
// an input file and a written superstring.
#include <kcgpu.h>
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>
#include <zlib.h>

#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <fstream>
#include <iomanip>
#include <iostream>
#include <string>
#include <thread>
#include <vector>

static const char *VERSION = "kmercamel-b200 0.1 (compute path of KmerCamel v2.3.0)";
static const int MAX_K = 127;  // reference src/main.cpp:93

// Successful end of a GPU sub-command: everything has been written and flushed by the caller.  Tearing the CUDA context
// down in user mode costs about as much as creating it (~1 s on a B200 box, more than all the work on a 50 Mbp input), so
// the process leaves it to the operating system.
[[noreturn]] static void finish_ok() {
    std::cout.flush();
    std::cerr.flush();
    std::fflush(nullptr);
    _exit(0);
}

static double now_ms() {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

static void write_log(const std::string &message) {  // src/parser.h:159-164
    auto snapshot = std::chrono::system_clock::now();
    std::time_t time = std::chrono::system_clock::to_time_t(snapshot);
    std::tm *time_tm = std::localtime(&time);
    std::cerr << "[" << std::put_time(time_tm, "%H:%M:%S") << "] " << message << std::endl;
}

static void write_name(const std::string &dataset, int k, bool maxone, bool unidirectional, std::ostream &of,
                       const char *algorithm = "greedy") {  // src/parser.h:167-179
    of << ">maskedsuperstring dataset='" << dataset << "' k=" << k << " alg=" << algorithm << " mask=" << (maxone ? "max-one " : "min-one ")
       << "mode=" << (unidirectional ? "unidirectional" : "bidirectional") << std::endl;
}

static int usage() {
    std::cerr << std::endl;
    std::cerr << "Program: kmercamel (B200-native masked superstring computation)" << std::endl;
    std::cerr << "Version: " << VERSION << std::endl;
    std::cerr << std::endl;
    std::cerr << "Usage:   kmercamel compute [options] <fasta>" << std::endl;
    std::cerr << "         kmercamel lowerbound [-k INT] [-u] [-S] [-z INT] [-g INT] <fasta>" << std::endl;
    std::cerr << "         kmercamel maskopt -k INT [-t max-one|min-one] [-u] [-o FILE] [-g INT] <ms>" << std::endl;
    std::cerr << "         kmercamel verify -k INT [-u] [-z INT] [-g INT] <fasta> <msfa>" << std::endl;
    std::cerr << "         kmercamel ms2mssep -m FILE [-s FILE] <ms>     |  mssep2ms [-m FILE] [-s FILE] [-o FILE]" << std::endl;
    std::cerr << "         kmercamel ms2spss -k INT [-o FILE] <ms>       |  spss2ms -k INT [-o FILE] <fasta>" << std::endl << std::endl;
    std::cerr << "Options:" << std::endl;
    std::cerr << "  -k INT   - k-mer size (required; up to " << MAX_K << ")" << std::endl;
    std::cerr << "  -a STR   - the algorithm [greedy (default), streaming]" << std::endl;
    std::cerr << "  -o FILE  - output file [default: stdout]" << std::endl;
    std::cerr << "  -u       - treat k-mer and its reverse complement as distinct" << std::endl;
    std::cerr << "  -S       - assume the input are simplitigs / matchtigs / unitigs" << std::endl;
    std::cerr << "  -M FILE  - also output the masked superstring with the mask maximizing the number of ones" << std::endl;
    std::cerr << "  -z INT   - keep only k-mers with at least this many occurrences [default: 1]" << std::endl;
    std::cerr << "  -g LIST  - CUDA device ordinal(s), e.g. 0 or 0,1,2,3 or 0-7 [default: 0]; several devices shard the k-mer set" << std::endl;
    std::cerr << "             construction of `compute` (from FASTA, without -S / -M) by hash range over NVLink" << std::endl;
    std::cerr << "  -V       - verify: the k-mer set the output represents must equal the k-mer set of the input (digest on the GPU)" << std::endl;
    std::cerr << "  -h       - print help" << std::endl;
    std::cerr << std::endl;
    return 1;
}

// "-g 0", "-g 0,1,2", "-g 0-7", "-g 0-3,6" -> device ordinals (an ordinal may repeat: the ranks then share that GPU)
static bool parse_devices(const std::string &arg, std::vector<int> &out) {
    out.clear();
    size_t at = 0;
    while (at <= arg.size()) {
        const size_t comma = std::min(arg.find(',', at), arg.size());
        const std::string part = arg.substr(at, comma - at);
        if (part.empty() || part.find_first_not_of("0123456789-") != std::string::npos) return false;
        const size_t dash = part.find('-');
        try {
            if (dash == std::string::npos) {
                out.push_back(std::stoi(part));
            } else {
                const int a = std::stoi(part.substr(0, dash)), b = std::stoi(part.substr(dash + 1));
                if (b < a) return false;
                for (int d = a; d <= b; ++d) out.push_back(d);
            }
        } catch (std::exception &) {
            return false;
        }
        at = comma + 1;
    }
    for (int d : out)
        if (d < 0) return false;
    return !out.empty() && out.size() <= 16;
}

// CUDA initialisation enumerates every GPU of the box (5 s on an 8-GPU node for a job that uses one of them).  Unless the caller
// already restricts the visible devices, expose only the ones named by -g and renumber them 0, 1, ...; must run before the first
// CUDA call of the process.
static void restrict_visible_devices(std::vector<int> &devices) {
    if (std::getenv("CUDA_VISIBLE_DEVICES")) return;
    std::vector<int> uniq;
    for (int d : devices) {
        bool seen = false;
        for (int u : uniq) seen = seen || u == d;
        if (!seen) uniq.push_back(d);
    }
    std::string list;
    for (size_t i = 0; i < uniq.size(); ++i) list += (i ? "," : "") + std::to_string(uniq[i]);
    if (setenv("CUDA_VISIBLE_DEVICES", list.c_str(), 0) != 0) return;
    for (int &d : devices)
        for (size_t i = 0; i < uniq.size(); ++i)
            if (uniq[i] == d) {
                d = (int) i;
                break;
            }
}

// Whole file (plain or gzip, "-" = stdin) into memory; zlib detects the format as in src/parser.h:88-101.  A regular file that
// does not start with the gzip magic is read with plain read() calls into a buffer of its size (gzread passes such a file
// through at ~0.8 GB/s and the doubling vector touches every page twice: 4 s for the 3.1 GB of the human-scale input).
static bool read_all(const std::string &path, std::vector<unsigned char> &data) {
    if (path != "-") {
        int fd = ::open(path.c_str(), O_RDONLY);
        if (fd < 0) return false;
        struct stat st;
        unsigned char magic[2] = {0, 0};
        if (::fstat(fd, &st) == 0 && S_ISREG(st.st_mode) && ::pread(fd, magic, 2, 0) >= 0 && !(magic[0] == 0x1f && magic[1] == 0x8b)) {
            const size_t size = (size_t) st.st_size;
            data.resize(size);
            // several readers: page-cache copies are memcpy-bound per thread
            const int n_thr = size > (64u << 20) ? 8 : 1;
            std::vector<std::thread> th;
            bool ok = true;
            for (int t = 0; t < n_thr; ++t)
                th.emplace_back([&, t] {
                    size_t at = size * (size_t) t / (size_t) n_thr;
                    const size_t end = size * (size_t) (t + 1) / (size_t) n_thr;
                    while (at < end) {
                        const ssize_t got = ::pread(fd, data.data() + at, std::min<size_t>(end - at, 1u << 30), (off_t) at);
                        if (got <= 0) {
                            ok = false;
                            return;
                        }
                        at += (size_t) got;
                    }
                });
            for (auto &x : th) x.join();
            ::close(fd);
            return ok;
        }
        ::close(fd);
    }
    FILE *in = path == "-" ? stdin : std::fopen(path.c_str(), "r");
    if (!in) return false;
    gzFile fp = gzdopen(fileno(in), "r");
    if (!fp) return false;
    gzbuffer(fp, 1 << 20);
    size_t cap = 1 << 24;
    data.resize(cap);
    size_t len = 0;
    while (true) {
        if (len == cap) {
            cap *= 2;
            data.resize(cap);
        }
        int got = gzread(fp, data.data() + len, (unsigned) std::min<size_t>(cap - len, 1u << 30));
        if (got <= 0) break;
        len += (size_t) got;
    }
    data.resize(len);
    gzclose(fp);
    return true;
}

// `compute` (src/main.cpp:214-316) and `lowerbound` (src/main.cpp:378-443) share everything up to the overlap stage.
static int camel_compute(int argc, char **argv, bool lower_bound) {
    std::string path;
    if (argc > 1 && std::string(argv[argc - 1]) != "-h") {  // src/main.cpp:217-220: the input is the LAST argument
        path = argv[argc - 1];
        argc--;
    }
    int k = 0, device = 0;
    std::vector<int> devices{0};
    long min_frequency = 1;
    std::string out_path, mask_path, algorithm = "greedy";
    bool complements = true, assume_simplitigs = false, d_set = false, verify = false;
    int opt;
    try {
        while ((opt = getopt(argc, argv, lower_bound ? "k:huxSz:g:" : "k:d:a:o:huxM:Sz:g:V")) != -1) {  // src/main.cpp:234,391
            switch (opt) {
                case 'o': out_path = optarg; break;
                case 'k': k = std::stoi(optarg); break;
                case 'd': d_set = true; (void) std::stoi(optarg); break;
                case 'a': algorithm = optarg; break;
                case 'u': complements = false; break;
                case 'x':
                    std::cerr << "Warning: The parameter -x currently has no effect due to the improvement in the underlying algorithm." << std::endl;
                    break;
                case 'M': mask_path = optarg; break;
                case 'S': assume_simplitigs = true; break;
                case 'z': min_frequency = std::stol(optarg); break;
                case 'g':
                    if (!parse_devices(optarg, devices)) {
                        std::cerr << "-g takes CUDA device ordinals, e.g. 0 or 0,1,2,3 or 0-7." << std::endl;
                        return usage();
                    }
                    device = devices[0];
                    break;
                case 'V': verify = true; break;
                case 'h': usage(); return 0;
                default: return usage();
            }
        }
    } catch (std::exception &) {
        return usage();
    }
    if (algorithm == "global") algorithm = "greedy";  // src/main.cpp:97-106
    if (path.empty()) {
        std::cerr << "Required positional parameter path to the file not set." << std::endl;
        return usage();
    }
    if (k == 0) {
        std::cerr << "Required parameter k not set." << std::endl;
        return usage();
    } else if (k < 0) {
        std::cerr << "k must be positive." << std::endl;
        return usage();
    } else if (algorithm != "greedy" && (algorithm != "streaming" || lower_bound)) {
        std::cerr << "Algorithm '" << algorithm << "' is not part of the GPU compute path; use the reference build for it." << std::endl;
        return usage();
    } else if (k > MAX_K) {
        std::cerr << "k > " << MAX_K << " not supported for the algorithm 'greedy'." << std::endl;
        return usage();
    } else if (d_set) {
        std::cerr << "Unsupported argument d for algorithm '" << algorithm << "'." << std::endl;
        return usage();
    } else if (!mask_path.empty() && algorithm != "greedy") {  // src/main.cpp:296-298
        std::cerr << "Outputting mask with maximum number of ones is only supported for the global greedy algorithm." << std::endl;
        return usage();
    } else if (assume_simplitigs && algorithm != "greedy") {  // src/main.cpp:299-301
        std::cerr << "Assuming simplitigs is only supported for the global greedy algorithm." << std::endl;
        return usage();
    } else if (min_frequency >= 256 || min_frequency < 1) {
        std::cerr << "Minimum frequency '-z' must be between 1 and 255." << std::endl;
        return usage();
    } else if (min_frequency != 1 && assume_simplitigs) {
        std::cerr << "Inputting simplitigs is not compatible with frequency filterring." << std::endl;
        return usage();
    }

    if (!lower_bound) write_log("Started computation of a masked superstring from '" + path + "'.");
    else write_log("Started computation of a masked superstring length lower bound from '" + path + "'.");  // src/main.cpp:134
    const double t_start = now_ms();
    const int device_asked = device;
    restrict_visible_devices(devices);
    device = devices[0];
    // several devices: the k-mer set construction of the from-FASTA greedy is sharded over them; every other mode runs on the first
    bool multi = devices.size() > 1 && !lower_bound && algorithm == "greedy" && !assume_simplitigs && mask_path.empty();
    if (devices.size() > 1 && !multi) write_log("Note: -S, -M, streaming and lowerbound run on one GPU; using device " + std::to_string(device_asked) + ".");
    // the CUDA context(s) (~1 s) are created while the file is read and framed
    kc_ctx *ctx = nullptr;
    kc_group *group = nullptr;
    int rc_init = KC_OK;
    double t_init_done = 0;
    std::thread init_thread([&] {
        if (multi) {
            rc_init = kc_init_multi((int) devices.size(), devices.data(), &group);
            if (rc_init == KC_OK) ctx = kc_group_ctx(group, 0);
        } else {
            rc_init = kc_init(device, nullptr, &ctx);
        }
        t_init_done = now_ms();
    });
    struct Joiner {
        std::thread &t;
        ~Joiner() {
            if (t.joinable()) t.join();
        }
    } joiner{init_thread};
    std::vector<unsigned char> data;
    if (!read_all(path, data)) {
        std::cerr << "couldn't open file " << path << std::endl;  // src/parser.h:95-97 throws invalid_argument
        return 1;
    }
    const double t_read = now_ms();
    uint8_t *seq = nullptr;
    uint64_t n_bytes = 0, n_recs = 0, *rec_off = nullptr, *rec_len = nullptr;
    int rc = kc_frame_fasta(data.data(), data.size(), &seq, &n_bytes, &rec_off, &rec_len, &n_recs);
    if (rc != KC_OK) {
        std::cerr << "framing failed: " << kc_strerror(rc) << std::endl;
        return 1;
    }
    std::vector<unsigned char>().swap(data);
    const double t_frame = now_ms();
    // 64-bit window positions (include/kcgpu.h KC_POS32_BYTES): one GPU; -V would hold input and output at once, `verify` checks the file
    const bool large = n_bytes >= KC_POS32_BYTES;
    if (large && verify) {
        std::cerr << "kmercamel compute: verification not available for inputs of 2^32 bytes or more (" << n_bytes << " sequence bytes)" << std::endl;
        return 1;
    }

    init_thread.join();
    rc = rc_init;
    if (rc == KC_OK && multi && large) {
        kc_group_destroy(group);
        group = nullptr;
        ctx = nullptr;
        multi = false;
        write_log("Note: inputs of 2^32 bytes or more run on one GPU; using device " + std::to_string(device_asked) + ".");
        rc = kc_init(device, nullptr, &ctx);
    }
    const double t_init = now_ms();
    if (rc != KC_OK) {
        std::cerr << "cannot initialise CUDA device " << device_asked << (multi ? " (and the other devices of -g; all need peer access to each other)" : "") << ": "
                  << kc_strerror(rc) << " (this build has no CPU path)" << std::endl;
        return 1;
    }
    kc_params p{k, complements ? 1 : 0, (int) min_frequency, assume_simplitigs ? 1 : 0, mask_path.empty() ? 0 : 1};
    kc_input in{seq, n_bytes, rec_off, rec_len, n_recs};
    kc_output out;
    std::memset(&out, 0, sizeof(out));
    uint64_t bound = 0;
    if (algorithm == "streaming") {  // src/main.cpp:139-144: header, then Streaming / StreamingFiltered
        rc = kc_streaming(ctx, &p, &in, &out);
        (void) verify;
        if (rc != KC_OK) {
            std::cerr << "kmercamel compute -a streaming failed: " << kc_strerror(rc) << ": " << kc_last_error(ctx) << std::endl;
            kc_destroy(ctx);
            return 1;
        }
        std::ofstream output;
        std::ostream *of = &std::cout;
        if (!out_path.empty()) {
            output.open(out_path);
            of = &output;
        }
        write_name(path, k, false, !complements, *of, "streaming");
        of->write(reinterpret_cast<const char *>(out.ms), (std::streamsize) out.length);
        *of << std::endl;
        write_log("Finished masked superstring computation.");
        if (output.is_open()) output.close();
        finish_ok();
    }
    rc = lower_bound ? kc_lower_bound(ctx, &p, &in, &bound, &out) : (multi ? kc_group_compute(group, &p, &in, &out) : kc_compute(ctx, &p, &in, &out));
    const double t_compute = now_ms();
    if (rc == KC_ERR_EMPTY && !assume_simplitigs) {  // src/main.cpp:155-158
        std::cerr << "Path '" << path << "' contains no k-mers. Make sure that your file is a FASTA or gzipped FASTA." << std::endl;
        if (!multi) kc_destroy(ctx);
        return usage();
    }
    if (rc != KC_OK) {
        std::cerr << "kmercamel " << (lower_bound ? "lowerbound" : "compute") << " failed: " << kc_strerror(rc) << ": "
                  << (multi ? kc_group_last_error(group) : kc_last_error(ctx)) << std::endl;
        if (!multi) kc_destroy(ctx);
        return 1;
    }
    if (!assume_simplitigs)
        write_log("Finished collecting k-mers: " + std::to_string(out.n_kmers) + " " + std::to_string(k) + "-mers.");
    write_log("Finished 1. part: simplitigs (" + std::to_string(out.n_simplitigs) + " simplitigs).");  // src/main.cpp:174
    if (!assume_simplitigs && out.n_simplitigs * 5 >= out.n_kmers)                                       // src/main.cpp:175-176
        write_log("2. part: Number of simplitigs over threshold, computing directly from k-mers.");
    write_log("Finished 2. part: Hamiltonian path.");
    if (lower_bound) {  // src/lower_bound.h:21, src/main.cpp:182,210
        write_log("Finished 3. part: lower bound = " + std::to_string(bound) + ".");
        std::cout << bound << std::endl;
        finish_ok();
    }
    write_log("Finished 3. part: masked superstring (l=" + std::to_string(out.length) + ").");
    char times[256];
    std::snprintf(times, sizeof(times), "GPU stages [ms]: extract %.3f, count %.3f, path %.3f, emit %.3f, total %.3f; %llu kernels",
                  out.t.extract_ms, out.t.count_ms, out.t.path_ms, out.t.emit_ms, out.t.total_ms, (unsigned long long) out.n_launches);
    write_log(times);
    {   // which k-mer set construction ran (kmerset_sig.cuh: signature buckets; kmerset_fast.cuh / kmerset.cuh otherwise)
        uint64_t sig_runs = 0, sig_fb = 0;
        kc_ctx *c0 = multi ? kc_group_ctx(group, 0) : ctx;
        if (c0 && kc_get_stat(c0, "sig_runs", &sig_runs) == KC_OK && kc_get_stat(c0, "sig_fallbacks", &sig_fb) == KC_OK && !assume_simplitigs)
            write_log(std::string("k-mer set construction: ") + (sig_runs ? "signature buckets (super-k-mer records)" : (sig_fb ? "signature buckets overflowed, fixed slots / exact" : "fixed slots / exact")) + ".");
    }
    if (multi) write_log("k-mer set construction sharded by hash range over " + std::to_string(devices.size()) + " GPUs.");
    bool verified_ok = true;
    if (verify) {  // what the reference's verify.py checks: the superstring represents exactly the k-mer set of the input
        uint64_t d_in[4], d_out[4];
        kc_input ms_in{out.ms, out.length, nullptr, nullptr, 0};
        kc_params pv = p;
        pv.min_frequency = 1;
        int rv = kc_kmer_digest(ctx, &p, &in, 0, d_in);
        if (rv == KC_OK) rv = kc_kmer_digest(ctx, &pv, &ms_in, 1, d_out);
        if (rv != KC_OK) {
            std::cerr << "verification could not run: " << kc_strerror(rv) << ": " << kc_last_error(ctx) << std::endl;
            return 1;
        }
        verified_ok = d_in[0] == d_out[0] && d_in[1] == d_out[1] && d_in[2] == d_out[2] && d_in[0] == out.n_kmers;
        char vb[256];
        std::snprintf(vb, sizeof(vb), "Verification %s: input %llu k-mers (digest %016llx %016llx), output represents %llu (digest %016llx %016llx).",
                      verified_ok ? "passed" : "FAILED", (unsigned long long) d_in[0], (unsigned long long) d_in[1], (unsigned long long) d_in[2],
                      (unsigned long long) d_out[0], (unsigned long long) d_out[1], (unsigned long long) d_out[2]);
        write_log(vb);
    }
    const double t_verify = now_ms();

    std::ofstream output, mask_output;
    std::ostream *of = &std::cout;
    if (!out_path.empty()) {
        output.open(out_path);
        of = &output;
    }
    write_name(path, k, false, !complements, *of);
    of->write(reinterpret_cast<const char *>(out.ms), (std::streamsize) out.length);
    *of << std::endl;  // src/main.cpp:210
    if (!mask_path.empty()) {
        mask_output.open(mask_path);
        write_name(path, k, true, !complements, mask_output);
        mask_output.write(reinterpret_cast<const char *>(out.ms_maxone), (std::streamsize) out.length);
        mask_output << std::endl;  // src/global.h:206-208
    }
    if (of == &output) output.flush();
    std::snprintf(times, sizeof(times), "Host stages [ms]: read %.1f, frame %.1f, CUDA context %.1f (in the background; waited %.1f), compute incl. H2D/D2H and arena %.1f, verify %.1f, write %.1f, total %.1f",
                  t_read - t_start, t_frame - t_read, t_init_done - t_start, t_init - t_frame, t_compute - t_init, t_verify - t_compute, now_ms() - t_verify, now_ms() - t_start);
    write_log(times);
    if (!verified_ok) {
        std::cout.flush();
        std::fflush(nullptr);
        _exit(2);
    }
    if (output.is_open()) output.close();
    if (mask_output.is_open()) mask_output.close();
    finish_ok();
}

// Reads the file and frames it; returns false after printing the reason.
static bool load_framed(const std::string &path, std::vector<unsigned char> &data, uint8_t **seq, uint64_t *n_bytes, uint64_t **rec_off,
                        uint64_t **rec_len, uint64_t *n_recs) {
    if (!read_all(path, data)) {
        std::cerr << "couldn't open file " << path << std::endl;
        return false;
    }
    int rc = kc_frame_fasta(data.data(), data.size(), seq, n_bytes, rec_off, rec_len, n_recs);
    if (rc != KC_OK) {
        std::cerr << "framing failed: " << kc_strerror(rc) << std::endl;
        return false;
    }
    return true;
}

// The -V check on two files: the k-mer set of input.fa against the set the masked superstring in superstring.msfa represents (its only
// record).  Both sets are digested on the GPU (kc_kmer_digest), which takes inputs of 2^32 bytes and more as well, where `compute -V`
// cannot keep the input and the output together.  Exit code 0 = the sets are equal, 2 = they differ, 1 = error.
static int camel_verify(int argc, char **argv) {
    int k = 0, device = 0;
    long min_frequency = 1;
    bool complements = true;
    int opt;
    try {
        while ((opt = getopt(argc, argv, "k:uz:g:h")) != -1) {
            switch (opt) {
                case 'k': k = std::stoi(optarg); break;
                case 'u': complements = false; break;
                case 'z': min_frequency = std::stol(optarg); break;
                case 'g': device = std::stoi(optarg); break;
                case 'h': usage(); return 0;
                default: return usage();
            }
        }
    } catch (std::exception &) {
        return usage();
    }
    if (argc - optind != 2) {
        std::cerr << "verify takes two files: the input FASTA and the masked superstring (.msfa)." << std::endl;
        return usage();
    }
    const std::string in_path = argv[optind], ms_path = argv[optind + 1];
    if (k == 0) {
        std::cerr << "Required parameter k not set." << std::endl;
        return usage();
    } else if (k < 0 || k > MAX_K) {
        std::cerr << "k must be in 1.." << MAX_K << "." << std::endl;
        return usage();
    } else if (min_frequency >= 256 || min_frequency < 1) {
        std::cerr << "Minimum frequency '-z' must be between 1 and 255." << std::endl;
        return usage();
    }
    write_log("Started verification of '" + ms_path + "' against '" + in_path + "'.");
    kc_ctx *ctx = nullptr;
    {
        std::vector<int> dv{device};
        restrict_visible_devices(dv);
        device = dv[0];
    }
    int rc = kc_init(device, nullptr, &ctx);
    if (rc != KC_OK) {
        std::cerr << "cannot initialise CUDA device " << device << ": " << kc_strerror(rc) << " (this build has no CPU path)" << std::endl;
        return 1;
    }
    kc_params p{k, complements ? 1 : 0, (int) min_frequency, 0, 0};
    kc_params pv = p;
    pv.min_frequency = 1;
    uint64_t d_in[4], d_out[4];
    {
        std::vector<unsigned char> data;
        uint8_t *seq = nullptr;
        uint64_t n_bytes = 0, n_recs = 0, *rec_off = nullptr, *rec_len = nullptr;
        if (!load_framed(in_path, data, &seq, &n_bytes, &rec_off, &rec_len, &n_recs)) return 1;
        std::vector<unsigned char>().swap(data);
        kc_input in{seq, n_bytes, rec_off, rec_len, n_recs};
        rc = kc_kmer_digest(ctx, &p, &in, 0, d_in);
        kc_free(seq);
        kc_free(rec_off);
        kc_free(rec_len);
    }
    if (rc == KC_OK) {
        std::vector<unsigned char> data;
        uint8_t *seq = nullptr;
        uint64_t n_bytes = 0, n_recs = 0, *rec_off = nullptr, *rec_len = nullptr;
        if (!load_framed(ms_path, data, &seq, &n_bytes, &rec_off, &rec_len, &n_recs)) return 1;
        std::vector<unsigned char>().swap(data);
        if (n_recs > 1) {  // as maskopt: the superstring is ONE record (src/masks.h:258)
            std::cerr << "Expecting only a single FASTA record -- the masked superstring." << std::endl;
            return 1;
        }
        kc_input ms_in{seq + (n_recs ? rec_off[0] : 0), n_recs ? rec_len[0] : 0, nullptr, nullptr, 0};
        rc = kc_kmer_digest(ctx, &pv, &ms_in, 1, d_out);
        kc_free(seq);
        kc_free(rec_off);
        kc_free(rec_len);
    }
    if (rc != KC_OK) {
        std::cerr << "verification could not run: " << kc_strerror(rc) << ": " << kc_last_error(ctx) << std::endl;
        return 1;
    }
    const bool ok = d_in[0] == d_out[0] && d_in[1] == d_out[1] && d_in[2] == d_out[2];
    char vb[256];
    std::snprintf(vb, sizeof(vb), "Verification %s: input %llu k-mers (digest %016llx %016llx), output represents %llu (digest %016llx %016llx).",
                  ok ? "passed" : "FAILED", (unsigned long long) d_in[0], (unsigned long long) d_in[1], (unsigned long long) d_in[2],
                  (unsigned long long) d_out[0], (unsigned long long) d_out[1], (unsigned long long) d_out[2]);
    write_log(vb);
    std::cerr.flush();
    std::fflush(nullptr);
    _exit(ok ? 0 : 2);
}

// `maskopt` (src/main.cpp:318-376, src/masks.h:240-261): max-one and min-one on the GPU; min-run needs an ILP solver.
static int camel_optimize(int argc, char **argv) {
    std::string path;
    if (argc > 1 && std::string(argv[argc - 1]) != "-h") {
        path = argv[argc - 1];
        argc--;
    }
    int k = 0, device = 0;
    std::string out_path, algorithm = "max-one";
    bool complements = true;
    int opt;
    try {
        while ((opt = getopt(argc, argv, "k:t:o:hug:")) != -1) {
            switch (opt) {
                case 'o': out_path = optarg; break;
                case 'k': k = std::stoi(optarg); break;
                case 't': algorithm = optarg; break;
                case 'u': complements = false; break;
                case 'g': device = std::stoi(optarg); break;
                case 'h': usage(); return 0;
                default: return usage();
            }
        }
    } catch (std::exception &) {
        return usage();
    }
    if (algorithm == "maxone") algorithm = "max-one";  // src/main.cpp:109-115
    if (algorithm == "minone") algorithm = "min-one";
    if (path.empty()) {
        std::cerr << "Required positional parameter path to the file not set." << std::endl;
        return usage();
    }
    if (k == 0) {
        std::cerr << "Required parameter k not set." << std::endl;
        return usage();
    } else if (k < 0) {
        std::cerr << "k must be positive." << std::endl;
        return usage();
    } else if (k > MAX_K) {
        std::cerr << "k > " << MAX_K << " not supported." << std::endl;
        return usage();
    }
    if (algorithm != "max-one" && algorithm != "min-one") {
        std::cerr << "Algorithm '" + algorithm + "' not recognized by the GPU build (max-one, min-one)." << std::endl;
        return usage();
    }
    write_log("Started optimization of a masked superstring from '" + path + "'.");
    std::vector<unsigned char> data;
    uint8_t *seq = nullptr;
    uint64_t n_bytes = 0, n_recs = 0, *rec_off = nullptr, *rec_len = nullptr;
    if (!load_framed(path, data, &seq, &n_bytes, &rec_off, &rec_len, &n_recs)) return 1;
    uint64_t span[5] = {0, 0, 0, 0, 0};
    kc_fasta_first_header(data.data(), data.size(), span);
    kc_ctx *ctx = nullptr;
    {
        std::vector<int> dv{device};
        restrict_visible_devices(dv);
        device = dv[0];
    }
    int rc = kc_init(device, nullptr, &ctx);
    if (rc != KC_OK) {
        std::cerr << "cannot initialise CUDA device " << device << ": " << kc_strerror(rc) << " (this build has no CPU path)" << std::endl;
        return 1;
    }
    const uint64_t len = n_recs ? rec_len[0] : 0;  // ReadMaskedSuperstring: the first record (src/parser.h:145-150)
    kc_output out;
    std::memset(&out, 0, sizeof(out));
    rc = kc_maskopt(ctx, seq + (n_recs ? rec_off[0] : 0), len, k, complements ? 1 : 0, algorithm == "min-one" ? 1 : 0, &out);
    if (rc != KC_OK) {
        std::cerr << "kmercamel maskopt failed: " << kc_strerror(rc) << ": " << kc_last_error(ctx) << std::endl;
        kc_destroy(ctx);
        return 1;
    }
    std::ofstream output;
    std::ostream *of = &std::cout;
    if (!out_path.empty()) {
        output.open(out_path);
        of = &output;
    }
    *of << ">";  // ReprintSequenceHeader, src/masks.h:27-37
    of->write(reinterpret_cast<const char *>(data.data() + span[0]), (std::streamsize) span[1]);
    *of << " reoptimized=" << algorithm;
    if (span[2]) {
        *of << " ";
        of->write(reinterpret_cast<const char *>(data.data() + span[3]), (std::streamsize) span[4]);
    }
    *of << std::endl;
    of->write(reinterpret_cast<const char *>(out.ms), (std::streamsize) out.length);
    *of << std::endl;
    if (len >= (uint64_t) k && out.ms[len - k] > 'Z')  // src/masks.h:63-66 mask convention
        std::cerr << "Warning: the mask after optimization violates the mask convention as there are more than k-1 trailing zeros "
                     "(more than k-1 trailing lowercase characters)." << std::endl;
    if (n_recs > 1) {  // AssertEOF, src/masks.h:258 (the reference throws after having written the output)
        std::cerr << "Expecting only a single FASTA record -- the masked superstring." << std::endl;
        return 1;
    }
    write_log("Finished optimization.");
    if (output.is_open()) output.close();
    finish_ok();
}

// The four text conversions (src/main.cpp:444-667): host only.
static int camel_convert(const std::string &sub, int argc, char **argv) {
    const bool has_path = sub != "mssep2ms";
    std::string path;
    if (has_path && argc > 1 && std::string(argv[argc - 1]) != "-h") {
        path = argv[argc - 1];
        argc--;
    }
    std::string out_path, mask_path, sup_path;
    int k = 0, opt;
    const bool needs_k = sub == "ms2spss" || sub == "spss2ms";
    try {
        while ((opt = getopt(argc, argv, needs_k ? "o:k:h" : (sub == "ms2mssep" ? "m:s:h" : "m:s:o:h"))) != -1) {
            switch (opt) {
                case 'o': out_path = optarg; break;
                case 'k': k = std::stoi(optarg); break;
                case 'm':
                    if (!mask_path.empty()) {
                        std::cerr << "Error: -m parameter provided multiple times" << std::endl;
                        return usage();
                    }
                    mask_path = optarg;
                    break;
                case 's':
                    if (!sup_path.empty()) {
                        std::cerr << "Error: -s parameter provided multiple times" << std::endl;
                        return usage();
                    }
                    sup_path = optarg;
                    break;
                case 'h': usage(); return 0;
                default: return usage();
            }
        }
    } catch (std::exception &) {
        return usage();
    }
    if (has_path && path.empty()) {
        std::cerr << "Required positional parameter path to the file not set." << std::endl;
        return usage();
    }
    if (needs_k && k == 0) {
        std::cerr << "Required parameter k not set." << std::endl;
        return usage();
    } else if (needs_k && k < 0) {
        std::cerr << "k must be positive." << std::endl;
        return usage();
    }
    std::ofstream output;
    std::ostream *of = &std::cout;
    if (!out_path.empty()) {
        output.open(out_path);
        of = &output;
    }
    if (sub == "mssep2ms") {
        if (mask_path.empty() && sup_path.empty()) {
            std::cerr << "Cannot have both superstring and mask redirected from stdin." << std::endl;
            return usage();
        }
        write_log("Started masked superstring joining.");
        std::ifstream mf, sf;
        std::istream *maskf = &std::cin, *supf = &std::cin;
        if (!mask_path.empty()) {
            mf.open(mask_path);
            maskf = &mf;
        }
        if (!sup_path.empty()) {
            sf.open(sup_path);
            supf = &sf;
        }
        std::string superstring, mask;  // join_ms reads one white-space delimited token from each (src/conversions.h:36-38)
        *supf >> superstring;
        *maskf >> mask;
        uint8_t *joined = nullptr;
        uint64_t n = 0;
        if (kc_join_ms(reinterpret_cast<const uint8_t *>(superstring.data()), superstring.size(),
                       reinterpret_cast<const uint8_t *>(mask.data()), mask.size(), &joined, &n) != KC_OK) return 1;
        *of << ">superstring" << std::endl;
        of->write(reinterpret_cast<const char *>(joined), (std::streamsize) n);
        *of << std::endl;
        kc_free(joined);
        write_log("Finished masked superstring joining.");
        return 0;
    }
    if (sub == "ms2mssep" && mask_path.empty()) {
        // src/main.cpp:476-480,493-496: the reference never records that -s was given, so -m is what it insists on
        std::cerr << "Cannot have both superstring and mask redirected to stdout." << std::endl;
        return usage();
    }
    if (sub == "ms2mssep") write_log("Started splitting masked superstring '" + path + "'.");
    else if (sub == "ms2spss") write_log("Started rSPSS computation from masked supertring '" + path + "'.");
    else write_log("Started masked superstring computation corresponding to (r)SPSS '" + path + "'.");
    std::vector<unsigned char> data;
    uint8_t *seq = nullptr;
    uint64_t n_bytes = 0, n_recs = 0, *rec_off = nullptr, *rec_len = nullptr;
    if (!load_framed(path, data, &seq, &n_bytes, &rec_off, &rec_len, &n_recs)) return 1;
    const uint8_t *first = seq + (n_recs ? rec_off[0] : 0);
    const uint64_t first_len = n_recs ? rec_len[0] : 0;
    if (sub == "ms2mssep") {
        uint8_t *sup = nullptr, *mask = nullptr;
        if (kc_split_ms(first, first_len, &sup, &mask) != KC_OK) return 1;
        std::ofstream mf(mask_path), sf;
        std::ostream *supf = &std::cout;
        if (!sup_path.empty()) {
            sf.open(sup_path);
            supf = &sf;
        }
        mf.write(reinterpret_cast<const char *>(mask), (std::streamsize) first_len);
        mf << std::endl;
        supf->write(reinterpret_cast<const char *>(sup), (std::streamsize) first_len);
        *supf << std::endl;
        kc_free(sup);
        kc_free(mask);
        write_log("Finished masked superstring splitting.");
    } else if (sub == "ms2spss") {
        uint8_t *text = nullptr;
        uint64_t n = 0;
        if (kc_ms_to_spss(first, first_len, k, &text, &n) != KC_OK) return 1;
        of->write(reinterpret_cast<const char *>(text), (std::streamsize) n);
        of->flush();
        kc_free(text);
        write_log("Finished computing a rSPSS representing the same set.");
    } else {
        uint8_t *ms = nullptr;
        uint64_t n = 0;
        if (kc_spss_to_ms(seq, rec_off, rec_len, n_recs, k, &ms, &n) != KC_OK) return 1;
        *of << ">superstring " << path << std::endl;
        of->write(reinterpret_cast<const char *>(ms), (std::streamsize) n);
        *of << std::endl;
        kc_free(ms);
        write_log("Finished computing a masked superstring corresponding to the (r)SPSS.");
    }
    kc_free(seq);
    kc_free(rec_off);
    kc_free(rec_len);
    return 0;
}

int main(int argc, char **argv) {
    if (argc < 2) return usage();
    const std::string sub = argv[1];
    if (sub == "-h") {
        usage();
        return 0;
    }
    if (sub == "-v") {
        std::cerr << VERSION << std::endl;
        return 0;
    }
    if (sub == "compute") return camel_compute(argc - 1, argv + 1, false);
    if (sub == "lowerbound") return camel_compute(argc - 1, argv + 1, true);
    if (sub == "maskopt") return camel_optimize(argc - 1, argv + 1);
    if (sub == "verify") return camel_verify(argc - 1, argv + 1);
    if (sub == "ms2mssep" || sub == "mssep2ms" || sub == "ms2spss" || sub == "spss2ms") return camel_convert(sub, argc - 1, argv + 1);
    std::cerr << "Unknown sub-command '" << sub << "'." << std::endl;
    return usage();
}
