/* libkcgpu — C ABI of the B200-native `kmercamel compute` hot path.
 *
 * The reference (OndrejSladky/kmercamel) has no FFI boundary: its compute path is a chain of C++ templates inside
 * one translation unit, src/main.cpp:122-212 kmercamel<kmer_t, kh_wrapper_t>():
 *
 *     ReadKMers / ReadKMersFiltered        src/parser.h:107,123        -> kc_count_kmers   (stage 1 alone)
 *     get_simplitigs | simplitigs_from_fasta  src/simplitigs.h:192,89  \
 *     Global / GlobalSparse                src/global.h:218, src/global_sparse.h:211  -> kc_compute (all stages)
 *     OverlapHamiltonianPath[Sparse]       src/global.h:43, src/global_sparse.h:42     -> kc_overlap_path
 *     kseq_read loop                       src/kseq.h:182-224, src/parser.h:106-118    -> kc_frame_fasta (host only)
 *     Streaming / StreamingFiltered        src/streaming.h:12-107                      -> kc_streaming
 *     Optimize (max-one, min-one)          src/masks.h:240-261                         -> kc_maskopt
 *     split_ms / join_ms / ms_to_spss / spss_to_ms   src/conversions.h:16-91          -> kc_split_ms ... (host only)
 *
 * Conventions: plain C types only; every function returns 0 (KC_OK) or a negative KC_ERR_* code and never throws;
 * one context per process and GPU; calls are synchronous and not thread-safe per context.  There is no CPU
 * fallback: without a CUDA device kc_init fails with KC_ERR_NO_DEVICE.
 *
 * k-mer words cross the boundary as `limbs` little-endian uint64 limbs per k-mer, limbs = 1 (k < 32), 2 (k < 64),
 * 4 (k < 128) — the reference's word widths (src/main.cpp:309-315); base i (0 = leftmost) sits at bits
 * 2(k-1-i)+1..2(k-1-i), A=0 C=1 G=2 T=3 (src/kmers.h:15-32), so integer order is lexicographic order.
 */
#ifndef KCGPU_H
#define KCGPU_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define KC_OK 0
#define KC_ERR_CUDA (-1)
#define KC_ERR_ARG (-2)       /* bad parameter (k outside 1..127, min_frequency outside 1..255, -z with -S, ...) */
#define KC_ERR_OOM (-3)
#define KC_ERR_EMPTY (-4)     /* no k-mer in the input (reference src/main.cpp:155-158) / empty node list (src/global.h:219-221) */
#define KC_ERR_BAD_SEQ (-5)   /* -S record with a non-ACGT byte (reference src/simplitigs.h:82 asserts) or shorter than k */
#define KC_ERR_TOO_LARGE (-6) /* more than 2^32-2 virtual nodes on one GPU, or an input of KC_POS32_BYTES or more that the call
                               * cannot take (see KC_POS32_BYTES); kc_last_error says why */
#define KC_ERR_INTERNAL (-7)
#define KC_ERR_NO_DEVICE (-8)

/* Inputs of KC_POS32_BYTES sequence bytes or more (about 2^32) need 64-bit window positions.  kc_compute, kc_compute_device,
 * kc_lower_bound, kc_streaming and kc_kmer_digest take them on one GPU through the signature-bucket k-mer set construction, which
 * applies with k >= 26, min_frequency 1, no want_maxone and no assume_simplitigs (kc_streaming: any min_frequency, every pass of
 * -z is a first-occurrence construction; kc_kmer_digest ignores assume_simplitigs and want_maxone); outside those conditions, with
 * option sig_set = 0, or when a signature bucket overflows on such an input (heavily repeated sequence), they fail with
 * KC_ERR_TOO_LARGE.  kc_maskopt, kc_count_kmers and groups refuse such inputs with KC_ERR_TOO_LARGE. */
#define KC_POS32_BYTES 0xFFFFFFF0ULL

typedef struct kc_ctx kc_ctx;

/* Flags of `kmercamel compute` (reference src/main.cpp:214-316). */
typedef struct kc_params {
    int k;                 /* -k, 1..127 */
    int complements;       /* 1 = bidirectional (default), 0 = -u */
    int min_frequency;     /* -z, 1..255; k-mers with fewer occurrences are dropped (src/khash_utils.h:143-151) */
    int assume_simplitigs; /* -S: every record is one node, in input order (src/simplitigs.h:89-103) */
    int want_maxone;       /* -M: also produce the max-one mask (src/global.h:185-195) */
} kc_params;

/* Framed input: the record sequences of the FASTA/FASTQ file (what kseq_read yields, src/kseq.h:182-224)
 * concatenated in `seq`, each followed by exactly one '\n'.  rec_off[r] / rec_len[r] delimit record r.
 * kc_frame_fasta produces this from raw file bytes.  For kc_compute the pointers are host pointers, for
 * kc_compute_device they are device pointers (rec_off / rec_len are only read with assume_simplitigs). */
typedef struct kc_input {
    const uint8_t *seq;
    uint64_t n_bytes;
    const uint64_t *rec_off;
    const uint64_t *rec_len;
    uint64_t n_recs;
} kc_input;

typedef struct kc_stage_times { /* device time per stage in milliseconds (CUDA events on the context stream) */
    float extract_ms;           /* bytes -> canonical k-mer occurrences */
    float count_ms;             /* radix sort + dedup + count + -z filter */
    float path_ms;              /* all overlap levels d = k-1..0 */
    float emit_ms;              /* list ranking + character emission (+ max-one) */
    float total_ms;
} kc_stage_times;

typedef struct kc_output {
    uint8_t *ms;           /* the masked superstring, `length` bytes, no newline.  Upper case = mask 1. */
    uint8_t *ms_maxone;    /* same characters with the max-one mask, or NULL without want_maxone */
    uint64_t length;       /* "l=" of the reference log (src/global.h:225) */
    uint64_t n_kmers;      /* distinct (canonical) k-mers kept after -z; 0 with assume_simplitigs unless want_maxone */
    uint64_t n_occurrences;/* k-mer windows seen (M) */
    uint64_t n_nodes;      /* nodes handed to the overlap stage (k-mers, or records with -S) */
    uint64_t n_launches;   /* CUDA kernels launched by this call */
    uint64_t n_simplitigs; /* simplitigs of the d = k-1 level (first-occurrence runs, or records with -S): the count of the
                              reference's "Finished 1. part" log line (src/main.cpp:174).  When 5 * n_simplitigs >= n_kmers the
                              greedy ran on the individual k-mers (src/main.cpp:175-181) and n_nodes == n_kmers. */
    kc_stage_times t;
} kc_output;

/* device = CUDA ordinal; stream = a cudaStream_t to run on (e.g. torch's current stream), or NULL for a private non-blocking
 * one.  To run on the legacy default stream (handle 0) pass cudaStreamLegacy, i.e. (void *) 1. */
int kc_init(int device, void *stream, kc_ctx **out);
void kc_destroy(kc_ctx *ctx);

/* Whole path with HOST buffers: copies the input to the GPU, runs every stage, copies the result back into
 * context-owned pinned buffers (valid until the next call on this context or kc_destroy). */
int kc_compute(kc_ctx *ctx, const kc_params *p, const kc_input *in, kc_output *out);
/* Same with DEVICE buffers in and out (outputs live in the context arena until the next call). */
int kc_compute_device(kc_ctx *ctx, const kc_params *p, const kc_input *in, kc_output *out);

/* `kmercamel lowerbound` (reference src/main.cpp:378-443, LowerBoundLength src/lower_bound.h:9-22): the same path with
 * the cycle and reverse-complement tests of the greedy switched off (src/global.h:95-97), i.e. a cycle cover; returns
 * (sum of node lengths - sum of accepted overlaps) per strand.  Host buffers as kc_compute; want_maxone must be 0.
 * `stats` (may be NULL) receives the counters and stage times, no superstring. */
int kc_lower_bound(kc_ctx *ctx, const kc_params *p, const kc_input *in, uint64_t *lower_bound, kc_output *stats);

/* ---- neighbours of the compute path (SURVEY.md §8f), same conventions as kc_compute (host buffers, pinned result) ---------
 *
 * kc_streaming   `compute -a streaming [-z Z]` (reference src/main.cpp:139-144, Streaming / StreamingFiltered
 *                src/streaming.h:12-107): out->ms = the masked superstring of the one-pass algorithm (the Z-th occurrence
 *                of every k-mer with at least Z occurrences is ON, the k-1 characters after an ON window are kept in
 *                lower case, everything else is dropped); out->n_kmers = k-mers turned ON.  assume_simplitigs and
 *                want_maxone must be 0.  An input without k-mers gives length 0 (the reference prints an empty line).  The
 *                first-occurrence bits of every pass come from the signature construction where it applies (k >= 26), else from
 *                the fixed-slot / exact ones; the output does not depend on which.
 * kc_maskopt     `maskopt -t max-one | min-one` (src/main.cpp:318-376, Optimize / OptimizeOnes src/masks.h:40-78,240-261):
 *                ms = the sequence of the single record (n letters, ACGTacgt only, else KC_ERR_BAD_SEQ); out->ms = the same
 *                letters with the mask that maximises (minimize = 0) or minimises (1) the number of ones while representing
 *                the same k-mer set; out->n_kmers = size of that set.  `-t min-run` needs an ILP solver (GLPK in the
 *                reference) and is not provided. */
int kc_streaming(kc_ctx *ctx, const kc_params *p, const kc_input *in, kc_output *out);
int kc_maskopt(kc_ctx *ctx, const uint8_t *ms, uint64_t n, int k, int complements, int minimize, kc_output *out);

/* Host-only text conversions (reference src/conversions.h:16-91; sub-commands ms2mssep, mssep2ms, ms2spss, spss2ms).
 * Outputs are malloc'ed (NUL-terminated for convenience); release each with kc_free.
 *   kc_split_ms    superstring in upper case + mask as '0'/'1' characters, n bytes each (split_ms, :16-33)
 *   kc_join_ms     letter i of the superstring in the case given by mask[i] == '1' (join_ms, :35-44)
 *   kc_ms_to_spss  the complete FASTA text of the rSPSS (ms_to_spss, :46-72)
 *   kc_spss_to_ms  the masked superstring of framed records (kc_frame_fasta layout): last k-1 letters of each record OFF,
 *                  records shorter than k skipped (spss_to_ms, :74-91)
 *   kc_fasta_first_header  span = {name_off, name_len, has_comment, comment_off, comment_len} of the first record, as
 *                  kseq parses the header line (src/kseq.h:187-194); used to reprint it (src/masks.h:27-37). */
int kc_split_ms(const uint8_t *ms, uint64_t n, uint8_t **superstring, uint8_t **mask);
int kc_join_ms(const uint8_t *superstring, uint64_t n_s, const uint8_t *mask, uint64_t n_m, uint8_t **out, uint64_t *n_out);
int kc_ms_to_spss(const uint8_t *ms, uint64_t n, int k, uint8_t **out, uint64_t *n_out);
int kc_spss_to_ms(const uint8_t *seq, const uint64_t *rec_off, const uint64_t *rec_len, uint64_t n_recs, int k, uint8_t **out,
                  uint64_t *n_out);
int kc_fasta_first_header(const uint8_t *data, uint64_t n, uint64_t *span);

/* Copy n bytes of a kc_compute_device result (or any device buffer) to host memory on the context stream. */
int kc_copy_to_host(kc_ctx *ctx, void *dst_host, const void *src_device, uint64_t n);

/* Stage 1 only (host buffers): sorted distinct k-mers (n * limbs uint64) and min(occurrences-1, 255) per k-mer,
 * after the -z filter.  Outputs are malloc'ed by the library; release with kc_free. */
int kc_count_kmers(kc_ctx *ctx, const kc_params *p, const kc_input *in, uint64_t **keys, uint8_t **counts, uint64_t *n);

/* PartialPreSort of the sparse path (reference src/global_sparse.h:14-35): the k-mers (n * limbs little-endian limbs, host)
 * reordered by a stable counting sort on their top min(2k, 8) bits -> out (host, same size).  kc_compute applies it itself
 * when the sparse switch is taken; this entry point exists for the known-answer tests (tests/global_sparse_unittest.h:11-41). */
int kc_partial_presort(kc_ctx *ctx, const uint64_t *kmers, uint64_t n, int k, uint64_t *out);

/* Stage 1 as an order-independent digest, for sets too large to bring back and compare: digest[0] = n (distinct k-mers kept),
 * digest[1] = sum of h, digest[2] = xor of h, digest[3] = sum of h * c, all mod 2^64, where c = min(occurrences, 256) with
 * min_frequency > 1 (the frequency map of ReadKMersFiltered) and c = 1 otherwise (ReadKMers keeps no counts), and h folds the limbs
 * of a k-mer through the splitmix64 finaliser (h = mix(w0 + C); h = mix(h ^ (w_i + C * (i + 1))), C = 0x9e3779b97f4a7c15).
 * masked = 0: `in` is a framed input as for kc_count_kmers (the digest of ReadKMers / ReadKMersFiltered, src/parser.h:107-141).
 * masked = 1: in->seq is ONE masked superstring of in->n_bytes letters; the set is the k-mers of the windows that start with an
 *             upper-case letter, i.e. the set the superstring REPRESENTS (what the reference's verify.py compares, and
 *             src/parser.h:41-42 case_sensitive); min_frequency must be 1.
 * Without -z and with k >= 26 the set is built as first-occurrence bits by the signature construction and the flagged windows are
 * hashed; otherwise (or after a bucket overflow below KC_POS32_BYTES) the sorted keys are.  The four words do not depend on which.
 * `kmercamel compute` output verifies iff digest(masked = 1, output) == digest(masked = 0, input) (`kmercamel verify`). */
int kc_kmer_digest(kc_ctx *ctx, const kc_params *p, const kc_input *in, int masked, uint64_t *digest);

/* Overlap stage only (host buffers).  first/last: n * limbs limbs.  edge_from: N = n * (1 + complements) entries,
 * -1 = none; overlaps: N entries, 255 = none — the overlapPath of src/global.h:35.  strict = 1 reproduces the
 * reference's tie order exactly; lower_bound = 1 is the cycle-cover mode of src/lower_bound.h. */
int kc_overlap_path(kc_ctx *ctx, const uint64_t *first, const uint64_t *last, uint64_t n, int k, int complements,
                    int lower_bound, int strict, int64_t *edge_from, uint8_t *overlaps);

/* Host-only FASTA/FASTQ framing with kseq semantics (src/kseq.h:182-224 as driven by src/parser.h:106-118).
 * Outputs are malloc'ed; release each with kc_free. */
int kc_frame_fasta(const uint8_t *data, uint64_t n, uint8_t **seq, uint64_t *n_bytes, uint64_t **rec_off,
                   uint64_t **rec_len, uint64_t *n_recs);

/* ---- multi-GPU: hash-range sharded k-mer set construction (SURVEY.md §8e) ----------------------------------------------------
 * The reference is single-threaded; this is the north star's "k-mer counting shards by hash range across the GPUs of one box,
 * the greedy merge on one GPU".  Every rank owns a heap in its HBM that all other ranks address directly (peer pointers over
 * NVLink / NVSwitch); the level-0 partition pass stores each (k-mer, position) item straight into the heap of the GPU that owns
 * the k-mer's hash range, and ranks synchronise through device-side signal words — no collective library and no host round trip
 * on the data path (kmercamel_b200/csrc/group.cuh).  From-FASTA regime only (no -S, no -M); results are identical to kc_compute.
 *
 * (1) One process, one host thread per GPU — what §8(b) calls kc_init(n_gpus, device_ids):
 *       kc_init_multi     contexts on the given devices (an ordinal may repeat: several ranks then share a GPU, which is how the
 *                         single-GPU test box exercises the protocol), peer access enabled between them
 *       kc_group_compute  as kc_compute with HOST buffers: every rank copies in 1 / n of the sequence over its own PCIe link and
 *                         hands it to its peers over NVLink, all ranks build the k-mer set together, every rank repeats the
 *                         (deterministic) greedy stage and emits + copies back its own slice of the superstring into one pinned
 *                         buffer (valid until the next call on the group)
 *       kc_group_ctx      the context of a rank, for kc_set_option / kc_get_stat / kc_profile_* (options must be set on every rank)
 * (2) One process per GPU (torchrun; bench.py, tests): a context from kc_init becomes rank `rank` of `n_ranks`
 *       kc_group_alloc    allocates the rank's heap for inputs of up to n_bytes_cap bytes at word width of k and returns its
 *                         64-byte CUDA IPC handle; the caller all-gathers the handles (any transport: this is set-up, not data path)
 *       kc_group_open     all_handles: n_ranks * 64 bytes in rank order
 *       kc_group_compute_device   one job; in->seq = DEVICE pointer to the whole framed sequence, resident on this GPU.  Every rank
 *                         must make the same call.  out->ms = DEVICE pointer to bytes [*slice_begin, *slice_begin + *slice_len) of
 *                         the superstring (slices are 16-byte aligned and tile the string), out->length = its whole length.
 *       kc_group_close    releases the heap (all ranks must have finished their last job)
 *     kc_group_plan       host only, no GPU: plan[0] = fixed-slot path applies, [1], [2] = the rank's slice of window END positions,
 *                         [3], [4] = its range of level-0 digits (hash range), [5] = level-0 digits, [6] = items per (digit, sender)
 *                         sub-slot, [7] = heap bytes per rank. */
typedef struct kc_group kc_group;
int kc_init_multi(int n_gpus, const int *device_ids, kc_group **out);
void kc_group_destroy(kc_group *g);
int kc_group_size(const kc_group *g);
kc_ctx *kc_group_ctx(kc_group *g, int rank);
int kc_group_compute(kc_group *g, const kc_params *p, const kc_input *in, kc_output *out);
const char *kc_group_last_error(const kc_group *g);

uint64_t kc_shard_granule(int k);  /* window positions per level-0 tile: slices are multiples of it */
int kc_group_alloc(kc_ctx *ctx, int n_ranks, int rank, int k, uint64_t n_bytes_cap, uint8_t *handle_out);
int kc_group_open(kc_ctx *ctx, const uint8_t *all_handles);
int kc_group_compute_device(kc_ctx *ctx, const kc_params *p, const kc_input *in, kc_output *out, uint64_t *slice_begin, uint64_t *slice_len);
int kc_group_close(kc_ctx *ctx);
int kc_group_plan(int n_ranks, int rank, int k, uint64_t n_bytes, uint64_t *plan);

/* Per-kernel-class device timing for roofline reports.  Enable, run kc_compute*, then read the table:
 * names[i], milliseconds, launches, algorithmic bytes (read once + written once, see DESIGN.md). */
int kc_profile_enable(kc_ctx *ctx, int on);
int kc_profile_count(void);
int kc_profile_get(kc_ctx *ctx, int i, const char **name, double *ms, uint64_t *launches, uint64_t *bytes);
int kc_profile_reset(kc_ctx *ctx);

/* CUDA kernels launched through this context since kc_init (every entry point adds its own). */
uint64_t kc_total_launches(const kc_ctx *ctx);

/* Tuning / test knobs.  "sparse_switch" (default 1): hand the individual k-mers to the greedy when 5 * simplitigs >= k-mers.
 * "small_engine" (default 1): run the tail of the overlap levels in the single-CTA kernel.
 * "sig_set" (default 1): try the signature-bucket k-mer set construction first (kmerset_sig.cuh: from-FASTA compute
 * with k >= 26, without -z and -M); "sig_load_pct" (0 = planned from the input size) and "sig_min_items": its plan
 * parameters, exposed so that tests reach the overflow fallback and small inputs.  kc_kmer_digest and kc_streaming try it first as
 * well; an overflow there is counted in "sig_fallbacks" but not remembered by the context.
 * "fast_set" (default 1): then try the histogram-free fixed-slot construction (from-FASTA compute without -M);
 * "fast_leaf_target", "fast_sigmas", "fast_min_items": its plan parameters, exposed so that tests reach the
 * multi-level plan and the overflow fallback with small inputs; "fast_heuristics" (default 1): skip the attempt when
 * duplicates are expected (-z > 1, or the previous call on an input of similar size overflowed).
 * "fast_max_ctas": upper bound of the level >= 1 scatter grid.
 * "tail_spec" (default 1): after the signature-bucket construction, queue the rest of the call sized for a few hundred
 * first-occurrence runs (a genome) with no host round trip before the end; an input with more runs falls back to the
 * ordinary path, and the context skips the attempt for inputs of similar size after that (with "fast_heuristics").
 * Results never depend on these options. */
int kc_set_option(kc_ctx *ctx, const char *name, int value);
/* Counters since kc_init: "sig_runs", "sig_fallbacks", "fast_runs", "fast_fallbacks", "total_launches", "tail_spec_runs",
 * "tail_spec_fallbacks", "read_backs" (synchronising device -> host reads, i.e. host round trips); current value of the
 * option "fast_max_ctas"; device arena: "arena_bytes" (reserved now), "arena_high" (most bytes in use at once since kc_init).
 * Totals of the greedy overlap stage of the LAST call that ran it (kc_compute, kc_lower_bound, kc_overlap_path, a group
 * compute), over the level loop and the single-CTA engine: "path_levels" (overlap levels replayed), "path_ban_rounds" (replays
 * of a level after a cycle was found), "path_bans" (refused edges; with complements each one counts for both strands). */
int kc_get_stat(const kc_ctx *ctx, const char *name, uint64_t *value);

int kc_limbs_for_k(int k);
void kc_free(void *p);
const char *kc_strerror(int code);
const char *kc_last_error(const kc_ctx *ctx); /* file:line detail of the last failure on this context */

#ifdef __cplusplus
}
#endif
#endif
