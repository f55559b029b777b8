// Decoding of the sequence stream shared by the level-0 kernels of the k-mer set constructions, and the node ends of `-S`.
//
// Input is the framed sequence stream: the record sequences concatenated, separated by one non-ACGT byte.  A
// k-mer window is valid iff its k bytes are all ACGT/acgt, which reproduces both the reference's restart on
// N-like bytes (src/parser.h:32-37) and "windows never span records" (one AddKMers call per record,
// src/parser.h:112-114).
//
// A level-0 thread owns a strip of KC_EX_STRIP consecutive window END positions.  Its CTA converts the bytes 4 at a time
// with SIMD-in-register arithmetic (kc_pack4) to 2-bit codes + 1 validity bit, and parks one packed 64-bit code word + one
// 32-bit validity word per strip in shared memory, plus KC_EX_HALO words to the left for the windows that start earlier.
#pragma once
#include "exec.cuh"
#include "kword.cuh"

#ifdef __CUDACC__

static const int KC_EX_STRIP = 32;
static const int KC_EX_HALO = 4;  // halo words: 4 * 32 >= 127 - 1 preceding bases

// 4 ASCII bytes (byte 0 = first base) -> 8 bits of codes (first base in the top 2 bits) and 4 validity bits.
KC_D void kc_pack4(u32 w, u32 &codes, u32 &valid) {
    u32 c = ((w >> 1) ^ (w >> 2)) & 0x03030303u;  // A,a->0 C,c->1 G,g->2 T,t->3
    codes = (c * 0x40100401u) >> 24;
    // valid = the case-folded byte IS the letter its code stands for: A = 0x41, C = A + 2, G = A + 6, T = A + 19, rebuilt for the four bytes
    // at once (three multiply-adds; four emulated __vcmpeq4 cost twice the instructions), then the zero bytes of the difference
    const u32 c0 = c & 0x01010101u, c1 = (c >> 1) & 0x01010101u;
    const u32 expect = 0x41414141u + c0 * 2u + c1 * 6u + (c0 & c1) * 11u;
    const u32 d = (w & 0xDFDFDFDFu) ^ expect;
    const u32 z = ~(((d & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | d) & 0x80808080u;  // bit 7 of every byte that is zero
    valid = (((z >> 7) * 0x08040201u) >> 24) & 0xFu;
}

// First and last k-mer of the node seq[off .. off + len), len >= k.
template <int L> KC_D void kc_node_end_kmers(const u8 *seq, u64 off, u64 len, int k, KWord<L> &first, KWord<L> &last) {
    KWord<L> f = KWord<L>::zero(), l = KWord<L>::zero();
    for (int i = 0; i < k; ++i) {
        f = f.shl(2);
        f.w[0] |= kc_nucleotide_code(seq[off + i]) & 3;
        l = l.shl(2);
        l.w[0] |= kc_nucleotide_code(seq[off + len - k + i]) & 3;
    }
    first = f;
    last = l;
}

// `-S`: first and last k-mer of every record (reference src/simplitigs.h:68-76) and input validation
// (src/simplitigs.h:82 asserts ACGT only; records shorter than k have no k-mer and are rejected here).
template <int L>
void kc_extract_node_ends(CudaExec &ex, const u8 *seq, u64 n_bytes, const u64 *rec_off, const u64 *rec_len, u64 n_recs, int k,
                          KWord<L> *first, KWord<L> *last, u32 *error_flag, bool validate_bytes) {
    ex.for_each(n_recs, [=] __device__(u64 r) {
        u64 off = rec_off[r], len = rec_len[r];
        if (len < (u64) k) {
            *error_flag = 1;
            return;
        }
        kc_node_end_kmers<L>(seq, off, len, k, first[r], last[r]);
    });
    if (!validate_bytes) return;
    // every byte that is not a record separator must be a nucleotide
    ex.for_each(n_bytes, [=] __device__(u64 p) {
        u8 c = seq[p];
        if (c != '\n' && kc_nucleotide_code(c) > 3) *error_flag = 1;
    });
}

#endif  // __CUDACC__
