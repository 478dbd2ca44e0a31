// kernels_prealign.cuh — pre-alignment contig selection on the GPU (definition: prealign_core.h; replaces the per-read,
// per-target banded alignments of Aligners::align, fg-stitch-lib/src/align/aligners/mod.rs:246-295, 556-604).
//
// One persistent CTA per read in flight.  The k-mer index of all contig-strands lives in HBM (bucket offsets + positions,
// built once per context); a read's k-mers are looked up twice:
//   pass 1  every hit adds one to the counter of its contig-strand (per-CTA counters in global memory, L2-resident);
//           the strands with enough hits become candidates (at most PRE_MAX_CAND);
//   pass 2  every hit on a candidate adds one to the bin of its diagonal (width = band width);
//   score   one warp per candidate: the best pair of adjacent bins -> chain hits -> score; the strands reaching the
//           minimum score are written out in ascending order (at most MAX_STRANDS, the best ones);
//   banded  (STITCH_PREALIGN_BANDED) the best pair of bins is only the window: one warp per candidate runs the banded
//           affine-gap local alignment of the read against the strand over it (pre_band_score) and that is the score.
// Memory traffic per read: n bucket look-ups (8 B) + hits x (4 B position + a 12-step binary search in the strand
// table, cached) twice: a few MB against the GBs of the alignment that follows; the kernel is latency-bound gather work.
#pragma once
#include <cuda_runtime.h>

#include "prealign_core.h"

namespace stitch {
namespace gpu {

struct PreKParams {
    const uint32_t *off, *pos;            // k-mer index
    const uint8_t *blob;                  // contig bases (k > 12: hits are verified)
    const uint32_t *seq_off, *strand_len; // per strand
    uint32_t n_strands, K, W, n_bins;     // n_bins per candidate (covers diagonals of the longest read x longest strand)
    int32_t match, min_score;
    uint32_t banded;                      // STITCH_PREALIGN_BANDED: scores from the banded alignment (prealign_core.h)
    int32_t mismatch, gap_open, gap_extend;
    uint32_t band_chunks;                 // chunks of PRE_BAND_CHUNK cells that 2 W diagonals need
    int32_t *band_rows;                   // [grid][PRE_THREADS / 32][2][band_chunks * PRE_BAND_CHUNK]: H and F of the previous
                                          // row per warp, used when a window spans more than one chunk
    const uint8_t *reads; const uint64_t *read_off; const uint32_t *read_len; uint32_t n_reads;
    uint32_t *counter;
    uint32_t *cnt;        // [grid][n_strands]   hits per strand, then candidate slot + 1
    uint32_t *bins;       // [grid][PRE_MAX_CAND][n_bins]
    PreHit *out;          // [n_reads][MAX_STRANDS]
    uint32_t *out_n;      // [n_reads]
};

constexpr int PRE_THREADS = 256;
constexpr int PRE_BAND_CPL = 4;                              // banded DP: contiguous cells per lane and chunk
constexpr uint32_t PRE_BAND_CHUNK = 32u * PRE_BAND_CPL;      // cells of a row one warp-wide step covers

// Calls fn(strand, diagonal + n) for every k-mer hit of the read.
template <typename F>
__device__ __forceinline__ void pre_for_each_hit(const PreKParams &P, const uint8_t *read, uint32_t n, F &&fn) {
    const uint32_t K = P.K;
    if (n < K) return;
    for (uint32_t j = threadIdx.x; j + K <= n; j += PRE_THREADS) {
        uint64_t code;
        if (!pre_kmer_code(read + j, K, code)) continue;
        const uint32_t b = pre_bucket(code, K);
        const uint32_t lo = __ldg(P.off + b), hi = __ldg(P.off + b + 1);
        for (uint32_t e = lo; e < hi; ++e) {
            const uint32_t p = __ldg(P.pos + e);
            if (K > PRE_DIRECT_K && !pre_same_kmer(P.blob + p, read + j, K)) continue;
            const uint32_t s = pre_strand_of(P.seq_off, P.n_strands, p);
            fn(s, (p - __ldg(P.seq_off + s)) + n - j);   // diagonal p_in_strand - j, shifted by n to stay non-negative
        }
    }
}

// One chunk of one row of the banded DP (pre_banded_score's recurrences, warp-wide).  Row i = read base rb; the lane holds
// the window cells t = t0 .. t0 + CPL - 1 (diagonal dlo + t, strand column q = q0 + (t - t0), 1-based) with h / f = H / F
// of the previous row on entry and of this row on exit.
//   diagonal  H(i - 1, t): the lane's own h[k];
//   vertical  H, F(i - 1, t + 1): the next cell of the lane, of lane + 1 (__shfl_down) or, for lane 31, nh / nf (the first
//             cell of the next chunk, or outside the window: H = 0, F = o + e);
//   in-row    E(t) = max over k < t of H'(k) + o + e (t - k), H' = max(0, diagonal, F): per lane sequentially, across the
//             lanes a max-plus scan (__shfl_up + __viaddmax), ec = E entering the chunk (o + e at the window's left edge:
//             a gap opened from outside, never above the floor) and leaving it.
// Cells outside the window or the sequences are forced to H = 0, F = o + e and never count: the Gotoh over the window's
// cells alone, exactly as prealign_core.h states it.
struct PreBandScoring { int32_t match, mismatch, oe, e; };

__device__ __forceinline__ void pre_band_chunk(int32_t (&h)[PRE_BAND_CPL], int32_t (&f)[PRE_BAND_CPL], int32_t nh, int32_t nf,
                                               int32_t &ec, int32_t &best, uint8_t rb, const uint8_t *strand, int32_t q0,
                                               int32_t t0, int32_t width, int32_t m, const PreBandScoring &sc, uint32_t lane) {
    constexpr uint32_t FULL = 0xffffffffu;
    const int32_t dh = __shfl_down_sync(FULL, h[0], 1), df = __shfl_down_sync(FULL, f[0], 1);
    int32_t hp[PRE_BAND_CPL], fn[PRE_BAND_CPL];
    bool in[PRE_BAND_CPL];
    int32_t g = 0;   // E leaving the lane from its own cells
#pragma unroll
    for (int k = 0; k < PRE_BAND_CPL; ++k) {
        const int32_t q = q0 + k;
        in[k] = t0 + k < width && q >= 1 && q <= m;
        const uint8_t sb = in[k] ? __ldg(strand + q - 1) : (uint8_t)0;
        const int32_t vh = k + 1 < PRE_BAND_CPL ? h[k + 1] : (lane == 31 ? nh : dh);
        const int32_t vf = k + 1 < PRE_BAND_CPL ? f[k + 1] : (lane == 31 ? nf : df);
        const int32_t fk = __viaddmax_s32(vf, sc.e, vh + sc.oe);
        const int32_t x = __vimax3_s32(0, h[k] + (rb == sb ? sc.match : sc.mismatch), fk);
        hp[k] = in[k] ? x : 0;
        fn[k] = in[k] ? fk : sc.oe;
        g = k == 0 ? hp[0] + sc.oe : __viaddmax_s32(g, sc.e, hp[k] + sc.oe);
    }
    // inclusive scan: y = E leaving the lane
    int32_t y = lane == 0 ? __viaddmax_s32(ec, PRE_BAND_CPL * sc.e, g) : g;
#pragma unroll
    for (uint32_t s = 1; s < 32; s <<= 1) {
        const int32_t up = __shfl_up_sync(FULL, y, s);
        if (lane >= s) y = __viaddmax_s32(up, (int32_t)s * PRE_BAND_CPL * sc.e, y);
    }
    const int32_t prev = __shfl_up_sync(FULL, y, 1);
    int32_t E = lane == 0 ? ec : prev;
    ec = __shfl_sync(FULL, y, 31);
#pragma unroll
    for (int k = 0; k < PRE_BAND_CPL; ++k) {
        const int32_t hk = in[k] ? max(hp[k], E) : 0;
        best = max(best, hk);
        E = __viaddmax_s32(E, sc.e, hp[k] + sc.oe);
        h[k] = hk; f[k] = fn[k];
    }
}

// score(s) of the banded scoring for one candidate, by one warp: the read against strand s over the window of bin pair
// bstar (prealign_core.h).  Only the diagonals and rows that meet both sequences are swept.  rows: this warp's row buffer
// (2 x band_chunks x PRE_BAND_CHUNK), used when the window needs more than one chunk.
__device__ int32_t pre_band_score(const PreKParams &P, const uint8_t *read, int32_t n, uint32_t s, uint32_t bstar, int32_t *rows,
                                  uint32_t lane) {
    const int32_t m = (int32_t)__ldg(P.strand_len + s);
    const uint8_t *strand = P.blob + __ldg(P.seq_off + s);
    const int32_t dlo = max((int32_t)(bstar * P.W) - n, 1 - n), dhi = min((int32_t)((bstar + 2) * P.W) - n, m);
    if (dlo >= dhi) return 0;
    const int32_t width = dhi - dlo, nch = (width + (int32_t)PRE_BAND_CHUNK - 1) / (int32_t)PRE_BAND_CHUNK;
    const int32_t i_lo = max(1, 2 - dhi), i_hi = min(n, m - dlo);
    const PreBandScoring sc{P.match, P.mismatch, P.gap_open + P.gap_extend, P.gap_extend};
    const int32_t tl = (int32_t)lane * PRE_BAND_CPL;
    int32_t best = 0, rw = 0;
    if (nch == 1) {
        int32_t h[PRE_BAND_CPL], f[PRE_BAND_CPL];
#pragma unroll
        for (int k = 0; k < PRE_BAND_CPL; ++k) { h[k] = 0; f[k] = sc.oe; }
        for (int32_t i = i_lo; i <= i_hi; ++i) {
            const int32_t r = (i - i_lo) & 31;
            if (r == 0) rw = i - 1 + (int32_t)lane < n ? read[i - 1 + lane] : 0;   // read bases once per 32 rows
            const uint8_t rb = (uint8_t)__shfl_sync(0xffffffffu, rw, r);
            int32_t ec = sc.oe;
            pre_band_chunk(h, f, 0, sc.oe, ec, best, rb, strand, i + dlo + tl, tl, width, m, sc, lane);
        }
    } else {
        const int32_t stride = nch * (int32_t)PRE_BAND_CHUNK;
        int32_t *rh = rows, *rf = rows + stride;
        for (int32_t t = (int32_t)lane; t < stride; t += 32) { rh[t] = 0; rf[t] = sc.oe; }
        __syncwarp();
        for (int32_t i = i_lo; i <= i_hi; ++i) {
            const int32_t r = (i - i_lo) & 31;
            if (r == 0) rw = i - 1 + (int32_t)lane < n ? read[i - 1 + lane] : 0;
            const uint8_t rb = (uint8_t)__shfl_sync(0xffffffffu, rw, r);
            int32_t ec = sc.oe;
            for (int32_t c = 0; c < nch; ++c) {
                const int32_t t0 = c * (int32_t)PRE_BAND_CHUNK + tl, tn = (c + 1) * (int32_t)PRE_BAND_CHUNK;
                int32_t h[PRE_BAND_CPL], f[PRE_BAND_CPL];
#pragma unroll
                for (int k = 0; k < PRE_BAND_CPL; ++k) { h[k] = rh[t0 + k]; f[k] = rf[t0 + k]; }
                const int32_t nh = c + 1 < nch ? rh[tn] : 0, nf = c + 1 < nch ? rf[tn] : sc.oe;
                pre_band_chunk(h, f, nh, nf, ec, best, rb, strand, i + dlo + t0, t0, width, m, sc, lane);
#pragma unroll
                for (int k = 0; k < PRE_BAND_CPL; ++k) { rh[t0 + k] = h[k]; rf[t0 + k] = f[k]; }
                __syncwarp();
            }
        }
    }
    for (int d = 16; d >= 1; d >>= 1) best = max(best, __shfl_xor_sync(0xffffffffu, best, d));
    return best;
}

__global__ void __launch_bounds__(PRE_THREADS) prealign_kernel(const PreKParams P) {
    __shared__ uint32_t s_read, s_ncand, s_need;
    __shared__ uint32_t s_cand[PRE_MAX_CAND];
    __shared__ int32_t s_score[PRE_MAX_CAND];
    __shared__ uint32_t s_bstar[PRE_MAX_CAND];   // banded: the lower bin of the best pair (lowest on ties)
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    uint32_t *cnt = P.cnt + (size_t)blockIdx.x * P.n_strands;
    uint32_t *bins = P.bins + (size_t)blockIdx.x * PRE_MAX_CAND * P.n_bins;
    for (;;) {
        __syncthreads();
        if (tid == 0) s_read = atomicAdd(P.counter, 1u);
        __syncthreads();
        const uint32_t r = s_read;
        if (r >= P.n_reads) break;
        const uint8_t *read = P.reads + P.read_off[r];
        const uint32_t n = P.read_len[r];
        // ---- pass 1: hits per strand ----
        for (uint32_t s = tid; s < P.n_strands; s += PRE_THREADS) cnt[s] = 0;
        if (tid == 0) s_need = P.banded ? pre_need_banded(P.min_score, P.match, P.K) : pre_need(P.min_score, P.match, P.K);
        __syncthreads();
        pre_for_each_hit(P, read, n, [&](uint32_t s, uint32_t) { atomicAdd(cnt + s, 1u); });
        __syncthreads();
        // ---- candidates (the threshold doubles until they fit) ----
        for (;;) {
            if (tid == 0) s_ncand = 0;
            __syncthreads();
            const uint32_t need = s_need;
            for (uint32_t s = tid; s < P.n_strands; s += PRE_THREADS)
                if (cnt[s] >= need) { const uint32_t k = atomicAdd(&s_ncand, 1u); if (k < PRE_MAX_CAND) s_cand[k] = s; }
            __syncthreads();
            if (s_ncand <= PRE_MAX_CAND) break;
            __syncthreads();
            if (tid == 0) s_need = need * 2;
            __syncthreads();
        }
        const uint32_t ncand = s_ncand;
        if (ncand == 0) { if (tid == 0) P.out_n[r] = 0; continue; }
        // slot + 1 of every candidate replaces its counter (0 = not a candidate); bins cleared
        for (uint32_t s = tid; s < P.n_strands; s += PRE_THREADS) cnt[s] = 0;
        __syncthreads();
        for (uint32_t k = tid; k < ncand; k += PRE_THREADS) cnt[s_cand[k]] = k + 1;
        for (uint32_t x = tid; x < ncand * P.n_bins; x += PRE_THREADS) bins[x] = 0;
        __syncthreads();
        // ---- pass 2: hits per diagonal bin of the candidates ----
        pre_for_each_hit(P, read, n, [&](uint32_t s, uint32_t dshift) {
            const uint32_t slot = cnt[s];
            if (slot) {
                const uint32_t b = dshift / P.W;
                if (b < P.n_bins) atomicAdd(bins + (size_t)(slot - 1) * P.n_bins + b, 1u);
            }
        });
        __syncthreads();
        // ---- score: one warp per candidate ----
        for (uint32_t k = warp; k < ncand; k += PRE_THREADS / 32) {
            const uint32_t *bk = bins + (size_t)k * P.n_bins;
            uint32_t best = 0, bstar = 0;
            for (uint32_t b = lane; b < P.n_bins; b += 32) {
                const uint32_t v = bk[b] + (b + 1 < P.n_bins ? bk[b + 1] : 0u);
                if (v > best) { best = v; bstar = b; }
            }
            for (int d = 16; d >= 1; d >>= 1) {
                const uint32_t o = __shfl_xor_sync(0xffffffffu, best, d), ob = __shfl_xor_sync(0xffffffffu, bstar, d);
                if (o > best || (o == best && ob < bstar)) { best = o; bstar = ob; }
            }
            if (lane == 0) { s_score[k] = pre_score_of(P.match, best, P.K); s_bstar[k] = bstar; }
        }
        __syncthreads();
        // ---- banded scoring: the alignment over the window replaces the count ----
        if (P.banded) {
            int32_t *rows = P.band_rows ? P.band_rows + ((size_t)blockIdx.x * (PRE_THREADS / 32) + warp) * 2 * P.band_chunks * PRE_BAND_CHUNK
                                        : nullptr;
            for (uint32_t k = warp; k < ncand; k += PRE_THREADS / 32) {
                const int32_t sc = pre_band_score(P, read, (int32_t)n, s_cand[k], s_bstar[k], rows, lane);
                if (lane == 0) s_score[k] = sc;
            }
            __syncthreads();
        }
        // ---- selection, in ascending strand order (thread 0: a few candidates per read) ----
        if (tid == 0) {
            uint32_t nk = 0;
            for (uint32_t k = 0; k < ncand; ++k)
                if (s_score[k] >= P.min_score) { s_cand[nk] = s_cand[k]; s_score[nk] = s_score[k]; ++nk; }
            auto sort = [&](uint32_t cntk, bool by_score) {   // insertion sort of (s_cand, s_score): (score desc, strand asc) or strand asc
                for (uint32_t i = 1; i < cntk; ++i) {
                    const uint32_t c = s_cand[i]; const int32_t sc = s_score[i];
                    uint32_t j = i;
                    while (j > 0) {
                        const bool prev_first = (by_score && s_score[j - 1] != sc) ? s_score[j - 1] > sc : s_cand[j - 1] < c;
                        if (prev_first) break;
                        s_cand[j] = s_cand[j - 1]; s_score[j] = s_score[j - 1]; --j;
                    }
                    s_cand[j] = c; s_score[j] = sc;
                }
            };
            if (nk > MAX_STRANDS) { sort(nk, true); nk = MAX_STRANDS; }
            sort(nk, false);
            for (uint32_t k = 0; k < nk; ++k) { PreHit h; h.strand = s_cand[k]; h.score = s_score[k]; P.out[(size_t)r * MAX_STRANDS + k] = h; }
            P.out_n[r] = nk;
        }
    }
}

}  // namespace gpu
}  // namespace stitch
