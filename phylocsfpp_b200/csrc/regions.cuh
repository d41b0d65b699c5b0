// regions.cuh — six-frame and open-reading-frame regions of score-msa alignments (pcsf_score_regions), sm_100a.
//
// A region is one frame of an alignment, or one ORF inside a frame; it is scored as if the sub-alignment S(r) it stands for had
// been handed to pcsf_score_msa on its own (DESIGN.md §6c has the full contract):
//   frame phi = (sigma, f), f = 0..2, works on W = A (sigma '+') or W = RC(A) (sigma '-'); codon k of the frame is W columns
//   f+3k .. f+3k+2, k < K = max(0, (len - f) / 3).  Minus codon k is codon_minus at original column len-3-f-3k.
//   Codon classes on the reference row: TAA, TAG, TGA stop; ATG start; a codon with a non-ACGT base is neither.
//   asis      one region per frame: W columns [min(f, len), len) (a trailing partial codon included)
//   stopstop  segments s_{j-1}+1 .. s_j (closing stop included), and the open tail s_m+1 .. K-1 if it is not empty
//   atgstop   per segment with an ATG before its stop: first ATG .. stop; the open tail never yields an ORF
//   ORF modes keep regions of at least min_codons codons (stop included).  Order: frame (+1 +2 +3 -1 -2 -3), then codon index.
//
//   k_orf_count / k_orf_emit   one warp per (alignment, frame) unit: reference-row codons classified 32 at a time with ballots,
//                              segments walked in order; count pass -> per-unit region and window counts, emit pass -> region
//                              descriptors at the scanned offsets (k_scan_blocks / k_scan_sums + k_unit_offsets)
//   k_region_windows           (column, strand) of every region's codons, in W codon order
//   k_region_sums              FIXED phylo / anc and the BLS of every region: sequential __dadd_rn sums in S(r)'s order
//   k_region_records           pcsf_region records of all regions
//   k_best_region              one warp per alignment: the region with the largest phylo (NaN never wins, ties: first)
#pragma once

#include "../../include/phylocsf_b200.h"
#include "kernels.cuh"

namespace pcsf {

constexpr uint32_t CODON_ATG = 14, CODON_TAA = 48, CODON_TAG = 50, CODON_TGA = 56;   // 16 b0 + 4 b1 + b2 over A,C,G,T = 0..3

struct RegionUnits {
    const uint8_t *codes;            // packed [nl][ld] of the concatenated batch (run_pack)
    int64_t ld;
    int n_aln, nfr, orf, min_codons;
    const int64_t *col_start, *len;  // [n_aln]
    const int32_t *ref_row;          // [n_aln]
};

struct RegionList {                  // structure of arrays, one entry per region
    int32_t *aln, *fi;               // alignment, frame index 0..5 (+1 +2 +3 -1 -2 -3)
    int64_t *k0, *ncod;              // first codon of the frame, codon count
    int64_t *win_start, *slen;       // first window, length of S(r) in columns
};

__device__ __forceinline__ int64_t frame_codons(int64_t len, int f) { return len > f ? (len - f) / 3 : 0; }

// Walks the frame of unit u (all lanes compute the same state; lane 0 writes).  EMIT = false: *n_reg / *n_win only.
template <bool EMIT>
__device__ void orf_walk(const RegionUnits &U, int64_t u, int64_t reg_base, int64_t win_base, RegionList R, uint32_t *n_reg,
                         uint32_t *n_win) {
    const int lane = threadIdx.x & 31;
    const int aln = (int)(u / U.nfr), fi = (int)(u % U.nfr), f = fi % 3;
    const bool minus = fi >= 3;
    const int64_t len = U.len[aln], K = frame_codons(len, f);
    int64_t nr = 0, nw = 0;
    auto emit = [&](int64_t k0, int64_t n, int64_t slen) {
        if (EMIT && lane == 0) {
            const int64_t r = reg_base + nr;
            R.aln[r] = aln; R.fi[r] = fi; R.k0[r] = k0; R.ncod[r] = n; R.win_start[r] = win_base + nw; R.slen[r] = slen;
        }
        ++nr; nw += n;
    };
    if (U.orf == PCSF_ORF_ASIS) {
        emit(0, K, len - (len < f ? len : f));
    } else {
        const uint8_t *ref = U.codes + (int64_t)U.ref_row[aln] * U.ld + U.col_start[aln];
        int64_t seg = 0, atg = -1;
        for (int64_t b = 0; b < K; b += 32) {
            const int64_t k = b + lane;
            uint32_t c = 64;
            if (k < K) {
                const int64_t o = minus ? len - 3 - f - 3 * k : f + 3 * k;
                c = minus ? codon_minus(ref[o], ref[o + 1], ref[o + 2]) : codon_plus(ref[o], ref[o + 1], ref[o + 2]);
            }
            uint32_t S = __ballot_sync(0xffffffffu, c == CODON_TAA || c == CODON_TAG || c == CODON_TGA);
            uint32_t A = __ballot_sync(0xffffffffu, c == CODON_ATG);
            while (S) {
                const int j = __ffs(S) - 1;
                const uint32_t below = (1u << j) - 1u;
                if (atg < 0 && (A & below)) atg = b + __ffs(A & below) - 1;
                const int64_t s = b + j;
                if (U.orf == PCSF_ORF_STOPSTOP) {
                    if (s - seg + 1 >= U.min_codons) emit(seg, s - seg + 1, 3 * (s - seg + 1));
                } else if (atg >= 0 && s - atg + 1 >= U.min_codons) {
                    emit(atg, s - atg + 1, 3 * (s - atg + 1));
                }
                seg = s + 1;
                atg = -1;
                S &= ~(below | (1u << j));
                A &= ~(below | (1u << j));
            }
            if (atg < 0 && A) atg = b + __ffs(A) - 1;
        }
        if (U.orf == PCSF_ORF_STOPSTOP && K - seg >= 1 && K - seg >= U.min_codons) emit(seg, K - seg, 3 * (K - seg));
    }
    if (!EMIT && lane == 0) { n_reg[u] = (uint32_t)nr; n_win[u] = (uint32_t)nw; }
}

// count pass: per-unit region / window counts and their 64-bit totals (the host checks them before the 32-bit scans are used)
__global__ void __launch_bounds__(256) k_orf_count(RegionUnits U, int64_t n_units, uint32_t *__restrict__ n_reg,
                                                   uint32_t *__restrict__ n_win, unsigned long long *__restrict__ totals) {
    const int64_t u = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (u >= n_units) return;
    orf_walk<false>(U, u, 0, 0, RegionList{}, n_reg, n_win);
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(totals, (unsigned long long)n_reg[u]);
        atomicAdd(totals + 1, (unsigned long long)n_win[u]);
    }
}

// exclusive scans (k_scan_blocks block-local ranks + k_scan_sums block offsets) -> global 64-bit offsets, [n_units] = total
__global__ void k_unit_offsets(int64_t n_units, const uint32_t *__restrict__ rank_r, const uint32_t *__restrict__ bsum_r,
                               const uint32_t *__restrict__ rank_w, const uint32_t *__restrict__ bsum_w,
                               const unsigned long long *__restrict__ totals, int64_t *__restrict__ off_r, int64_t *__restrict__ off_w) {
    const int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (u < n_units) {
        off_r[u] = (int64_t)rank_r[u] + bsum_r[u / SCAN_BLOCK];
        off_w[u] = (int64_t)rank_w[u] + bsum_w[u / SCAN_BLOCK];
    } else if (u == n_units) {
        off_r[u] = (int64_t)totals[0];
        off_w[u] = (int64_t)totals[1];
    }
}

__global__ void __launch_bounds__(256) k_orf_emit(RegionUnits U, int64_t n_units, const int64_t *__restrict__ off_r,
                                                  const int64_t *__restrict__ off_w, RegionList R) {
    const int64_t u = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (u >= n_units) return;
    orf_walk<true>(U, u, off_r[u], off_w[u], R, nullptr, nullptr);
}

// One warp per region (grid-stride): window k of region r is codon k0 + k of its frame, at its column in the batch.  win_strand is
// null when no region lies on the '-' strand.
__global__ void __launch_bounds__(256) k_region_windows(RegionUnits U, int64_t n_reg, RegionList R, uint32_t *__restrict__ win_off,
                                                        uint8_t *__restrict__ win_strand) {
    const int lane = threadIdx.x & 31;
    for (int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < n_reg; r += ((int64_t)gridDim.x * blockDim.x) >> 5) {
        const int aln = R.aln[r], fi = R.fi[r], f = fi % 3;
        const bool minus = fi >= 3;
        const int64_t len = U.len[aln], cs = U.col_start[aln], k0 = R.k0[r], n = R.ncod[r], w0 = R.win_start[r];
        for (int64_t k = lane; k < n; k += 32) {
            const int64_t kk = k0 + k;
            win_off[w0 + k] = (uint32_t)(cs + (minus ? len - 3 - f - 3 * kk : f + 3 * kk));
            if (win_strand) win_strand[w0 + k] = minus ? 1 : 0;
        }
    }
}

// W columns [a, a + slen) of region r (a = f + 3 k0, or min(f, len) for asis), and the same range in the input's columns
__device__ __forceinline__ void region_columns(const RegionUnits &U, const RegionList &R, int64_t r, int64_t *a, int64_t *begin,
                                               int64_t *end) {
    const int aln = R.aln[r], fi = R.fi[r], f = fi % 3;
    const int64_t len = U.len[aln];
    const int64_t w = U.orf == PCSF_ORF_ASIS ? (len < f ? len : f) : f + 3 * R.k0[r];
    *a = w;
    if (fi < 3) { *begin = w; *end = w + R.slen[r]; }
    else { *begin = len - (w + R.slen[r]); *end = len - w; }
}

// Per-region sums, one thread per region, sequential in the reference's order: lpr += log z per codon (fixed_lik.hpp:431-432),
// elpr_anc += ... (:440) in W codon order; bl_total += bl (additional_scores.hpp:71) over S(r)'s columns in S(r)'s order, i.e.
// descending original columns on the '-' strand.  So a region's floats equal pcsf_score_msa's on the extracted S(r).
__global__ void k_region_sums(RegionUnits U, int64_t n_reg, RegionList R, const double *__restrict__ perwin /* [4][nwin] */,
                              int64_t nwin, const double *__restrict__ bl_raw, double bls_all, float *__restrict__ phylo,
                              float *__restrict__ anc, float *__restrict__ bls) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_reg) return;
    const int64_t K = R.slen[r] / 3, w0 = R.win_start[r];
    double lc = 0.0, lnc = 0.0, ac = 0.0, an = 0.0;
    if (phylo || anc) for (int64_t k = 0; k < K; ++k) {
        lc = __dadd_rn(lc, perwin[w0 + k]);
        lnc = __dadd_rn(lnc, perwin[nwin + w0 + k]);
        ac = __dadd_rn(ac, perwin[2 * nwin + w0 + k]);
        an = __dadd_rn(an, perwin[3 * nwin + w0 + k]);
    }
    if (phylo) phylo[r] = (float)(10.0 * (lc - lnc) / log(10.0));
    if (anc) anc[r] = (float)(10.0 * (ac - an) / log(10.0));
    if (bls) {
        int64_t a, c0, c1;
        region_columns(U, R, r, &a, &c0, &c1);
        const double *b = bl_raw + U.col_start[R.aln[r]];
        const int64_t n = R.slen[r];
        double t = 0.0;
        if (R.fi[r] < 3) for (int64_t c = 0; c < n; ++c) t = __dadd_rn(t, b[c0 + c]);
        else for (int64_t c = 0; c < n; ++c) t = __dadd_rn(t, b[c1 - 1 - c]);
        bls[r] = (float)(t / (bls_all * (double)n));
    }
}

__device__ __forceinline__ pcsf_region region_record(const RegionUnits &U, const RegionList &R, int64_t r, const float *phylo,
                                                     const float *anc, const float *bls) {
    pcsf_region o{};
    int64_t a;
    o.aln = R.aln[r];
    o.strand = R.fi[r] < 3 ? 1 : -1;
    o.frame = (int8_t)(R.fi[r] % 3 + 1);
    region_columns(U, R, r, &a, &o.col_begin, &o.col_end);
    o.codons = R.ncod[r];
    o.phylo = phylo[r];
    o.anc = anc ? anc[r] : __int_as_float(0x7fc00000);
    o.bls = bls ? bls[r] : __int_as_float(0x7fc00000);
    return o;
}

__global__ void k_region_records(RegionUnits U, int64_t n_reg, RegionList R, const float *__restrict__ phylo,
                                 const float *__restrict__ anc, const float *__restrict__ bls, pcsf_region *__restrict__ out) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r < n_reg) out[r] = region_record(U, R, r, phylo, anc, bls);
}

// Best-only: one warp per alignment over its regions [off_r[aln * nfr], off_r[(aln + 1) * nfr]).  A candidate beats another if its
// phylo is larger, or equal with a smaller region index; NaN never beats anything.  No finite winner: the first region; no region:
// the "none" record (frame 0, columns -1, NaN scores).
__global__ void __launch_bounds__(256) k_best_region(RegionUnits U, RegionList R, const int64_t *__restrict__ off_r,
                                                     const float *__restrict__ phylo, const float *__restrict__ anc,
                                                     const float *__restrict__ bls, pcsf_region *__restrict__ out) {
    const int64_t aln = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (aln >= U.n_aln) return;
    const int64_t r0 = off_r[aln * U.nfr], r1 = off_r[(aln + 1) * U.nfr];
    float bv = 0.f;
    int64_t bi = -1;
    for (int64_t r = r0 + lane; r < r1; r += 32) {
        const float v = phylo[r];
        if (v == v && (bi < 0 || v > bv)) { bv = v; bi = r; }      // ascending r per lane: an equal later value never replaces
    }
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, d);
        const int64_t oi = __shfl_xor_sync(0xffffffffu, bi, d);
        if (oi >= 0 && (bi < 0 || ov > bv || (ov == bv && oi < bi))) { bv = ov; bi = oi; }
    }
    if (lane != 0) return;
    if (bi < 0 && r1 > r0) bi = r0;
    if (bi >= 0) {
        out[aln] = region_record(U, R, bi, phylo, anc, bls);
    } else {
        pcsf_region o{};
        o.aln = (int32_t)aln;
        o.col_begin = o.col_end = -1;
        o.phylo = o.anc = o.bls = __int_as_float(0x7fc00000);
        out[aln] = o;
    }
}

}  // namespace pcsf
