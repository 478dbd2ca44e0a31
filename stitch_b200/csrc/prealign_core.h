// prealign_core.h — pre-alignment contig selection: the definition shared by the CUDA kernel (kernels_prealign.cuh),
// the host-side index builder and the CPU emulator the tests run (tests/emul).
//
// Reference: Aligners::align runs, per read and per target, a banded local alignment seeded by a k-mer hash of the
// target (fg-stitch-lib/src/align/aligners/mod.rs:246-295 driver, :556-604 prealign_local_banded,
// util/target_seq.rs:50-56 build_target_hash) and keeps the contig-strands whose score reaches pre_align_min_score.
// The banded aligner and the k-mer hash are `bio` 1.1.0 (Cargo.lock:91-94: pairwise::banded::Aligner::
// custom_with_prehash, sparse::hash_kmers), a crate that is not part of the reference checkout and that no reference
// test exercises on this path: PARITY UNPINNED.  What is built here is specified by this file, not by `bio`:
//
//   hits(s)      number of (read position j, strand position p) pairs whose k-mers are equal (k-mers holding a base
//                outside ACGT are skipped), for contig-strand s;
//   candidates   strands with hits(s) >= need, need = max(1, ceil(min_score / match) - K + 1) (a strand with fewer
//                k-mer hits cannot reach the score below); if more than PRE_MAX_CAND strands qualify, need doubles
//                until they fit;
//   chain(s)     max over b of cnt_s[b] + cnt_s[b + 1], cnt_s[b] = hits of s whose diagonal p - j falls into bin b of
//                width W = band_width: the hits inside a band of 2 W diagonals (what bio's band around its seed chain
//                covers);
//   score(s)     match * (chain(s) + K - 1): the bases covered by chain(s) overlapping k-mer hits, each scoring `match`.
//                For an error-free stretch of L bases this is the local alignment score L * match; substitutions and
//                indels inside the band lower it (fewer intact k-mers) roughly as they lower the Smith-Waterman score;
//   selected     strands with score(s) >= min_score; if more than MAX_STRANDS (256, the per-read limit of the aligner),
//                the 256 best by (score descending, strand ascending).
// Everything is a count, so the result does not depend on the order the GPU's atomics happen to run in.
//
// That is the k-mer scoring (STITCH_PREALIGN_KMER, the default).  The banded scoring (STITCH_PREALIGN_BANDED) keeps hits,
// bins and the caps above and changes three things:
//   candidates   hits(s) >= need_b, need_b = max(1, ceil(need / 2)) (pre_need_banded), doubling as above.  `need` bounds
//                a k-mer count, not an alignment score: at 5 % substitutions only about 54 % of the 12-mers of a segment
//                stay intact, so a segment whose alignment reaches min_score can hold far fewer than `need` hits;
//   window       b* = the bin b with the largest cnt_s[b] + cnt_s[b + 1], the LOWEST b on ties; the window is the
//                diagonals d = p - j in [b* W - n, (b* + 2) W - n): the two bins chain(s) covers;
//   score(s)     the best local (Smith-Waterman, floor 0) affine-gap alignment of the read against strand s over the
//                cells whose diagonal lies in the window and inside both sequences (pre_banded_score): match / mismatch
//                by byte equality (N matches N, as in the main DP), a gap of length L costs gap_open + L gap_extend,
//                linear strands (no circular wrap), no clip penalties in any mode.
#pragma once
#include "dp_core.h"

#include <algorithm>
#include <vector>

namespace stitch {

constexpr uint32_t PRE_MAX_CAND = 512;
constexpr uint32_t PRE_DIRECT_K = 12;        // k <= 12: the bucket is the k-mer code itself (4^12 = 16.7 M buckets)
constexpr uint32_t PRE_HASH_BITS = 24;       // k > 12: 2^24 buckets, entries verified against the bases

struct PreHit { uint32_t strand; int32_t score; };

SHD int pre_base2(uint8_t b) { return b == 'A' ? 0 : b == 'C' ? 1 : b == 'G' ? 2 : b == 'T' ? 3 : -1; }

// 2-bit code of the K-mer at s; false when it holds a base outside ACGT.
SHD bool pre_kmer_code(const uint8_t *s, uint32_t K, uint64_t &code) {
    uint64_t c = 0;
    for (uint32_t t = 0; t < K; ++t) {
        const int b = pre_base2(s[t]);
        if (b < 0) return false;
        c = (c << 2) | (uint64_t)b;
    }
    code = c;
    return true;
}
SHD uint32_t pre_n_buckets(uint32_t K) { return K <= PRE_DIRECT_K ? (1u << (2 * K)) : (1u << PRE_HASH_BITS); }
SHD uint32_t pre_bucket(uint64_t code, uint32_t K) {
    return K <= PRE_DIRECT_K ? (uint32_t)code : (uint32_t)((code * 0x9E3779B97F4A7C15ull) >> (64 - PRE_HASH_BITS));
}
SHD bool pre_same_kmer(const uint8_t *a, const uint8_t *b, uint32_t K) {
    for (uint32_t t = 0; t < K; ++t) if (a[t] != b[t]) return false;
    return true;
}
SHD uint32_t pre_need(int32_t min_score, int32_t match, uint32_t K) {
    if (match <= 0) return 1;
    const int64_t bases = ((int64_t)min_score + match - 1) / match;
    const int64_t need = bases - (int64_t)K + 1;
    return need < 1 ? 1u : (uint32_t)need;
}
// Candidate threshold of the banded scoring (see the top of this file).
SHD uint32_t pre_need_banded(int32_t min_score, int32_t match, uint32_t K) { return (pre_need(min_score, match, K) + 1) / 2; }
SHD int32_t pre_score_of(int32_t match, uint32_t chain_hits, uint32_t K) {
    return chain_hits == 0 ? 0 : (int32_t)((int64_t)match * ((int64_t)chain_hits + K - 1));
}
// strand of blob offset p: the last strand whose seq_off <= p (seq_off ascending)
SHD uint32_t pre_strand_of(const uint32_t *seq_off, uint32_t n_strands, uint32_t p) {
    uint32_t lo = 0, hi = n_strands;
    while (hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if (seq_off[mid] <= p) lo = mid; else hi = mid; }
    return lo;
}

// score(s) of the banded scoring: a plain sequential Gotoh over the window's diagonals [dlo, dhi) (d = strand position -
// read position, 0-based).  Row i = read base i - 1, column q = strand base q - 1; H = best local score ending in the cell,
// E / F = best ending in a gap along the strand / along the read.  A cell outside the window or the sequences counts as
// H = 0 and opens gaps from there (o + e <= 0, so such a gap never lifts a cell above the floor): the result is the
// best alignment over the window's cells alone.  The CUDA kernel (kernels_prealign.cuh) computes the same values warp-wide.
inline int32_t pre_banded_score(const uint8_t *read, uint32_t n, const uint8_t *strand, uint32_t m, int32_t dlo, int32_t dhi,
                                const Scoring &sc) {
    const int32_t oe = sc.o + sc.e;
    std::vector<int32_t> H(m + 1, 0), F(m + 1, oe);   // previous row, by column; never-written cells: outside the window
    int32_t best = 0;
    for (int64_t i = 1; i <= (int64_t)n; ++i) {
        const int64_t q0 = std::max<int64_t>(1, i + dlo), q1 = std::min<int64_t>(m, i + dhi - 1);
        if (q0 > q1) continue;
        int32_t diag = H[(size_t)q0 - 1], left = 0, E = oe;   // H(i - 1, q0 - 1); the cell left of q0 is outside
        for (int64_t q = q0; q <= q1; ++q) {
            const int32_t s = read[i - 1] == strand[q - 1] ? sc.match : sc.mismatch;
            const int32_t f = std::max(H[(size_t)q] + oe, F[(size_t)q] + sc.e);
            const int32_t e = q == q0 ? oe : std::max(left + oe, E + sc.e);
            const int32_t h = std::max({0, diag + s, e, f});
            diag = H[(size_t)q]; H[(size_t)q] = h; F[(size_t)q] = f; E = e; left = h;
            best = std::max(best, h);
        }
    }
    return best;
}

}  // namespace stitch
