/* TEST INFRASTRUCTURE ONLY — CPU restatement of the reference's `compute` hot path.
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may load this
 * library, and only as the checker.  The product (libkcgpu.so, host/kmercamel) never links or calls it.
 *
 * Parity status: PINNED.  Every function is checked by tests/test_oracle.py against
 *   (a) the golden vectors of the reference's own unit tests (tests/kmers_unittest.h, parser_unittest.h,
 *       global_unittest.h, global_sparse_unittest.h of /root/reference), and
 *   (b) outputs of the unmodified reference compiled here into oracle/_ref (kmercamel CLI + ref_harness),
 *       committed as fixtures under tests/golden/ together with the script that generated them.
 *
 * k-mer words are `limbs` little-endian uint64 limbs per k-mer: limbs = 1 (k < 32), 2 (k < 64), 4 (k < 128),
 * the word widths picked at reference src/main.cpp:309-315.  Base i (0 = leftmost) occupies bits
 * 2(k-1-i)+1..2(k-1-i), A=0 C=1 G=2 T=3 (src/kmers.h:15-32).
 */
#pragma once
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

int orc_limbs_for_k(int k);

/* k-mer set construction, reference src/parser.h:53-85 (AddKMersWithFrequencies) over framed records.
 * Record r is seq[rec_off[r] .. rec_off[r]+rec_len[r]).  Returns sorted unique canonical k-mers and
 * value = min(occurrences-1, 255).  Outputs are malloc'ed; release with orc_free. */
int orc_count_kmers(const uint8_t *seq, const uint64_t *rec_off, const uint64_t *rec_len, uint64_t n_rec, int k,
                    int complements, uint64_t **keys_out, uint8_t **vals_out, uint64_t *n_out);

/* Reverse complement / prefix / suffix of one k-mer (src/kmers.h:35-44,92-95); in/out are `limbs` limbs. */
void orc_reverse_complement(const uint64_t *in, int k, uint64_t *out);
void orc_bit_prefix(const uint64_t *in, int k, int d, uint64_t *out);
void orc_bit_suffix(const uint64_t *in, int k, int d, uint64_t *out);

/* Greedy overlap Hamiltonian path, reference src/global.h:43-133 (and its k-mer-node twin
 * src/global_sparse.h:42-132, which is the same loop with first == last).
 * first/last: n * limbs limbs (first and last k-mer of every node, ids 0..n-1).
 * edge_from: N = n*(1+complements) entries, -1 = none; overlaps: N entries, 255 = none. */
int orc_overlap_path(const uint64_t *first, const uint64_t *last, uint64_t n, int k, int complements,
                     int lower_bound, int64_t *edge_from, uint8_t *overlaps);

/* The same with `parts` prefix batches instead of the reference's 16 (1..16).  parts = 1 is the tie order of the product's
 * from-FASTA engine (kmercamel_b200/csrc/engine.cuh with strict = false), which puts every prefix into one batch. */
int orc_overlap_path_parts(const uint64_t *first, const uint64_t *last, uint64_t n, int k, int complements,
                           int lower_bound, int parts, int64_t *edge_from, uint8_t *overlaps);

/* The nodes of the product's from-FASTA regime (kmercamel_b200/csrc/runs.cuh), not a reference function: the window end of the
 * first occurrence, in input order, of every canonical k-mer that occurs at least min_frequency times (counted as in
 * orc_count_kmers) is marked, and the maximal runs of consecutive marked ends are returned as (start byte, length) pairs in seq
 * coordinates, in input order.  n_kept_out = number of kept distinct k-mers.  Outputs are malloc'ed; release with orc_free. */
int orc_first_occurrence_runs(const uint8_t *seq, const uint64_t *rec_off, const uint64_t *rec_len, uint64_t n_rec, int k,
                              int complements, int min_frequency, uint64_t **off_out, uint64_t **len_out, uint64_t *n_out,
                              uint64_t *n_kept_out);

/* Superstring emission, reference src/global.h:149-210 (SuperstringFromPath).  Nodes are the framed records
 * (ACGT only, each at least k long).  set_keys (sorted unique canonical-or-not keys, n_set of them) is only
 * read when maxone_out != NULL and plays the role of kMersDict (src/global.h:165-167,185-195).
 * ms_out / maxone_out: malloc'ed, *len_out bytes, no terminator, no newline. */
int orc_superstring(const uint8_t *seq, const uint64_t *rec_off, const uint64_t *rec_len, uint64_t n, int k,
                    int complements, const int64_t *edge_from, const uint8_t *overlaps, const uint64_t *set_keys,
                    uint64_t n_set, uint8_t **ms_out, uint8_t **maxone_out, uint64_t *len_out);

/* `compute -S`: simplitigs_from_fasta + Global (src/main.cpp:171-187, src/global.h:217-226). */
int orc_compute_from_simplitigs(const uint8_t *seq, const uint64_t *rec_off, const uint64_t *rec_len, uint64_t n,
                                int k, int complements, int want_maxone, uint8_t **ms_out, uint8_t **maxone_out,
                                uint64_t *len_out);

/* The check verify.py performs (reference verify.py:41-57 + src/conversions.h:45-72), without jellyfish:
 * sorted unique (canonical if complements) k-mers that start at an upper-case position p with p+k <= len.
 * n_on_out = number of such positions (verify.py's "Total"). */
int orc_ms_kmers(const uint8_t *ms, uint64_t len, int k, int complements, uint64_t **keys_out, uint64_t *n_out,
                 uint64_t *n_on_out);

/* `compute -a streaming [-z]`, reference src/streaming.h:12-107 over framed records (any bytes; non-ACGT restarts the
 * window).  out: malloc'ed, *len_out bytes. */
int orc_streaming(const uint8_t *seq, const uint64_t *rec_off, const uint64_t *rec_len, uint64_t n_rec, int k, int complements,
                  int min_frequency, uint8_t **out, uint64_t *len_out);

/* `maskopt -t max-one` (minimize = 0) / `-t min-one` (1), reference src/masks.h:40-78,240-261 + src/parser.h:22-49
 * (case_sensitive).  out: caller buffer of n bytes.  Returns 1 if a non-ACGT letter was seen (the reference throws). */
int orc_maskopt(const uint8_t *ms, uint64_t n, int k, int complements, int minimize, uint8_t *out);

void orc_free(void *p);

#ifdef __cplusplus
}
#endif
