// mle.cuh — batched maximum-likelihood tree-scale fit: score-msa --strategy mle on the GPU.
//
// Reference: run() MLE branch (src/run.hpp:191-195, 206-209) -> max_lik_lpr_leaves (src/fixed_lik.hpp:511-544)
// -> fit_find_init (:469-509) + gsl_min_fminimizer_brent (GSL 2.x min/brent.c, min/fsolver.c), every function
// evaluation being lpr_leaves(rho) = instantiate_tree(rho) + PhyloModel_make (all P(rho t_b), instance.hpp:449-646)
// + pruning of all codons (fixed_lik.hpp:362-449).
//
// B200 design: the sequential part (Brent's iterate sequence) is a tiny per-alignment state machine
// (k_mle_step, one thread per slot); everything heavy is batched across the alignments that are currently
// being fitted ("slots"):
//     k_mle_step   consumes the previous evaluation (sequential sums of log z / anc in codon order),
//                  advances fit_find_init / Brent exactly as the reference does, emits the next rho; a slot
//                  whose alignment is finished immediately pulls the next alignment from the queue
//     k_mle_plan   tile descriptors (one CTA pass of codons each) of every slot with a pending evaluation
//     k_mle_expm   batched P_b(rho) = S diag(exp(lambda t_b)) S^-1 for every (slot, branch): FP64 DMMA GEMMs,
//                  the reference's clamp / diagonal / row-sum checks, written straight into the DMMA fragment
//                  order (inner edges) or the leaf gather tables (leaf edges) that k_prune consumes
//     k_prune<true> the same pruning kernel as the tracks path, P streams taken per tile
// The coding and the non-coding fit of one alignment run back to back in one slot because they share one
// mt19937(42) stream (score_msa.hpp:115, run.hpp:193-194); the stream's values do not depend on the data, so
// the candidate rho sequence exp(log lo + U_i) is tabulated once on the host with std::mt19937 +
// std::uniform_real_distribution (the reference's own generator).
#pragma once

#include <algorithm>
#include <cmath>
#include <random>
#include <string>
#include <vector>

#include "../../include/phylocsf_b200.h"
#include "kernels.cuh"

namespace pcsf {

constexpr int MLE_MAX_TRIES = 250;
constexpr int MLE_NCAND = 2 * MLE_MAX_TRIES;

struct MleSlot {
    int32_t aln;        // -1: idle
    int32_t model;      // 0 coding, 1 non-coding
    int32_t phase;      // see k_mle_step
    int32_t tries;      // fit_find_init's i
    int32_t rng_pos;    // next candidate index (shared by both models of the alignment)
    int32_t iter;       // Brent iterations left
    int32_t pending;    // 1: an evaluation at x has been requested
    int32_t failed;     // PhyloModel_make check failed at some evaluation (reference throws)
    double x;           // evaluation point
    double lpr, anc;    // results of the last evaluation
    double flo, fhi, fx, xsel;
    double z, fz, xl, xu, v, w, fv, fw, d, e;   // gsl brent state
    double res_lpr[2], res_anc[2];
    int64_t K, win0;
};

// What one mle_run did (pcsf_score_msa_stats): evaluations = lpr_leaves calls, i.e. (alignment, model, rho) triples, each costing
// (n-1) x (2 x 64^3 + 64^2) flop of P(t) construction plus one pruning pass over the alignment's codons.  The per-kernel times are
// CUDA-event times, collected only when pcsf_set_timing is on (the events serialise the rounds a little).
struct MleStats {
    int64_t alignments = 0, evaluations = 0;
    int32_t rounds = 0, slots = 0;
    float ms_step = 0.f, ms_plan = 0.f, ms_expm = 0.f, ms_prune = 0.f;
};

struct MleBatch {
    int n_aln;
    const int64_t *d_win_start, *d_len;
    WinSpace ws;
    int64_t nwin;
    bool want_anc;
    float *d_phylo, *d_anc;
};

// ---------------------------------------------------------------------------------------------------
// gsl brent_iterate, first half: from the state compute the next trial point u (GSL min/brent.c).
__device__ inline double brent_next_u(MleSlot &s) {
    const double golden = 0.3819660;
    const double z = s.z, xl = s.xl, xu = s.xu, v = s.v, w = s.w;
    double d = s.e, e = s.d;   // (sic) GSL loads them swapped
    const double w_lower = z - xl, w_upper = xu - z;
    const double tol = 1.4901161193847656e-08 * fabs(z);
    double p = 0, q = 0, r = 0;
    const double mid = 0.5 * (xl + xu);
    if (fabs(e) > tol) {
        r = (z - w) * (s.fz - s.fv);
        q = (z - v) * (s.fz - s.fw);
        p = (z - v) * q - (z - w) * r;
        q = 2 * (q - r);
        if (q > 0) p = -p; else q = -q;
        r = e;
        e = d;
    }
    double u;
    if (fabs(p) < fabs(0.5 * q * r) && p < q * w_lower && p < q * w_upper) {
        const double t2 = 2 * tol;
        d = p / q;
        u = z + d;
        if ((u - xl) < t2 || (xu - u) < t2) d = (z < mid) ? tol : -tol;
    } else {
        e = (z < mid) ? xu - z : -(z - xl);
        d = golden * e;
    }
    if (fabs(d) >= tol) u = z + d; else u = z + ((d > 0) ? tol : -tol);
    s.e = e;
    s.d = d;
    return u;
}

// gsl brent_iterate, second half: fold f(u) into the bracket.
__device__ inline void brent_update(MleSlot &s, double u, double fu) {
    if (fu <= s.fz) {
        if (u < s.z) s.xu = s.z; else s.xl = s.z;
        s.v = s.w; s.fv = s.fw;
        s.w = s.z; s.fw = s.fz;
        s.z = u; s.fz = fu;
    } else {
        if (u < s.z) s.xl = u; else s.xu = u;
        if (fu <= s.fw || s.w == s.z) {
            s.v = s.w; s.fv = s.fw;
            s.w = u; s.fw = fu;
        } else if (fu <= s.fv || s.v == s.z || s.v == s.w) {
            s.v = u; s.fv = fu;
        }
    }
}

enum : int32_t { PH_LO = 0, PH_HI, PH_TRY, PH_REEVAL, PH_SET_LO, PH_SET_HI, PH_SET_Z, PH_INIT_V, PH_ITER };

// One step of max_lik_lpr_leaves (fixed_lik.hpp:469-544): s.lpr holds the value of the evaluation at s.x that was just
// consumed; sets the next s.x and returns false, or returns true when the fit has ended (s.lpr = the LAST evaluation).
__device__ inline bool fit_advance(MleSlot &s, double lo, double hi, double init, const double *__restrict__ cand) {
    const double F = -s.lpr;   // minimizer_lpr_leaves returns -lpr (fixed_lik.hpp:466)
    switch (s.phase) {
    case PH_LO: s.flo = s.lpr; s.x = hi; s.phase = PH_HI; break;
    case PH_HI: s.fhi = s.lpr; s.x = init; s.tries = 0; s.phase = PH_TRY; break;
    case PH_TRY:
        s.fx = s.lpr;
        if (s.tries < MLE_MAX_TRIES && (s.fx <= s.flo || s.fx <= s.fhi)) {
            s.x = cand[s.rng_pos++];
            ++s.tries;
        } else {
            s.xsel = (s.tries == MLE_MAX_TRIES) ? (s.flo > s.fhi ? lo : hi) : s.x;
            s.x = s.xsel;
            s.phase = PH_REEVAL;
        }
        break;
    case PH_REEVAL:
        if (lo < s.xsel && s.xsel < hi) { s.x = lo; s.phase = PH_SET_LO; }
        else return true;
        break;
    case PH_SET_LO: s.x = hi; s.phase = PH_SET_HI; break;
    case PH_SET_HI: s.x = s.xsel; s.phase = PH_SET_Z; break;
    case PH_SET_Z:
        s.z = s.xsel; s.fz = F; s.xl = lo; s.xu = hi;
        s.v = lo + 0.3819660 * (hi - lo); s.w = s.v; s.d = 0.0; s.e = 0.0;
        s.x = s.v; s.phase = PH_INIT_V;
        break;
    case PH_INIT_V:
        s.fv = F; s.fw = F;
        s.iter = 250;
        s.x = brent_next_u(s);
        s.phase = PH_ITER;
        break;
    case PH_ITER:
        brent_update(s, s.x, F);
        if (((s.xu - s.xl) / s.z) <= 0.01 || --s.iter <= 0) return true;   // fixed_lik.hpp:533-536
        s.x = brent_next_u(s);
        break;
    }
    return false;
}

// One thread per slot.  cand[i] = exp(log(lo) + U_i) (host-tabulated).  queue_head: next alignment to fit.
// Uses __dadd_rn etc. only where the reference's order matters (sequential sums); contraction elsewhere is
// harmless (the iterate sequence is compared at 1e-3 decibans / the reference's own CI tolerance).
__global__ void k_mle_step(MleSlot *slots, int n_slots, int n_aln, int *queue_head, int *n_active, unsigned long long *n_evals,
                           const int64_t *__restrict__ win_start, const int64_t *__restrict__ len,
                           const double *__restrict__ logz, const double *__restrict__ ancw, const int *__restrict__ expm_err,
                           const double *__restrict__ cand, double lo, double hi, double init, int want_anc,
                           float *__restrict__ phylo, float *__restrict__ anc_out) {
    const int si = blockIdx.x * blockDim.x + threadIdx.x;
    if (si >= n_slots) return;
    MleSlot s = slots[si];
    bool have_result = false;
    if (s.aln >= 0 && s.pending) {
        // lpr_leaves: lpr += log z, elpr_anc += ... in codon order (fixed_lik.hpp:431-444)
        double l = 0.0, a = 0.0;
        for (int64_t k = 0; k < s.K; ++k) {
            l = __dadd_rn(l, logz[s.win0 + k]);
            if (want_anc) a = __dadd_rn(a, ancw[s.win0 + k]);
        }
        s.lpr = l;
        s.anc = a;
        s.pending = 0;
        if (expm_err[si]) s.failed = 1;
        have_result = true;
    }
    for (;;) {
        if (s.aln < 0) {
            const int next = atomicAdd(queue_head, 1);
            if (next >= n_aln) { s.aln = -1; break; }
            s = MleSlot{};
            s.aln = next;
            s.K = len[next] / 3;
            s.win0 = win_start[next];
            s.model = 0;
            s.phase = PH_LO;
            s.x = lo;
            s.pending = 1;
            break;
        }
        if (!have_result) break;   // still waiting (cannot happen: every pending slot is evaluated each round)
        have_result = false;
        bool model_done = false;
        if (s.failed) {
            model_done = true;
        } else {
            model_done = fit_advance(s, lo, hi, init, cand);
        }
        if (!model_done) { s.pending = 1; break; }
        // max_lik_lpr_leaves returns the LAST evaluation's lpr / elpr_anc (fixed_lik.hpp:542-543)
        s.res_lpr[s.model] = s.lpr;
        s.res_anc[s.model] = s.anc;
        if (s.model == 0 && !s.failed) {
            s.model = 1; s.phase = PH_LO; s.x = lo; s.tries = 0; s.pending = 1;
            break;
        }
        if (s.failed) {
            if (phylo) phylo[s.aln] = nanf("");
            if (anc_out) anc_out[s.aln] = nanf("");
        } else {
            if (phylo) phylo[s.aln] = (float)(10.0 * (s.res_lpr[0] - s.res_lpr[1]) / log(10.0));
            if (anc_out) anc_out[s.aln] = (float)(10.0 * (s.res_anc[0] - s.res_anc[1]) / log(10.0));
        }
        s.aln = -1;   // loop: pull the next alignment
    }
    slots[si] = s;
    if (s.aln >= 0) atomicAdd(n_active, 1);
    if (s.aln >= 0 && s.pending && n_evals) atomicAdd(n_evals, 1ull);
}

// Single block: tile descriptors for every slot with a pending evaluation.
__global__ void __launch_bounds__(1024) k_mle_plan(const MleSlot *__restrict__ slots, int n_slots, const double *pbase,
                                                    size_t slot_stride /* doubles */, size_t leaf_off /* doubles */, int tw /* windows per tile */,
                                                    TileDesc *__restrict__ tiles, uint32_t *__restrict__ n_tiles,
                                                    const double *pi_slots = nullptr /* [slot][64], OMEGA */) {
    __shared__ uint32_t sh[33];
    const uint32_t per = (n_slots + 1023) / 1024;
    const uint32_t base = threadIdx.x * per;
    uint32_t sum = 0;
    for (uint32_t i = 0; i < per; ++i) {
        const uint32_t si = base + i;
        if (si < (uint32_t)n_slots && slots[si].aln >= 0 && slots[si].pending) sum += (uint32_t)((slots[si].K + tw - 1) / tw);
    }
    uint32_t total;
    uint32_t run = block_excl_scan(sum, &total, sh);
    for (uint32_t i = 0; i < per; ++i) {
        const uint32_t si = base + i;
        if (si >= (uint32_t)n_slots || slots[si].aln < 0 || !slots[si].pending) continue;
        const MleSlot &s = slots[si];
        const uint32_t nt = (uint32_t)((s.K + tw - 1) / tw);
        for (uint32_t t = 0; t < nt; ++t) {
            TileDesc d;
            d.pstream = pbase + (size_t)si * slot_stride;
            d.leafPT = d.pstream + leaf_off;
            d.model = s.model;
            { const int64_t rem = s.K - tw * (int64_t)t; d.count = (int32_t)(rem < tw ? rem : tw); }
            d.win0 = (uint32_t)(s.win0 + tw * (int64_t)t);
            d.pad = 0;
            d.pi = pi_slots ? pi_slots + (size_t)si * 64 : nullptr;
            tiles[run + t] = d;
        }
        run += nt;
    }
    if (threadIdx.x == 0) *n_tiles = total;
}

// ---------------------------------------------------------------------------------------------------
// k_mle_expm: block = (slot, branch), 4 warps x 16 rows.  P = SR * (diag(exp(lambda t)) * SRinv) with FP64 DMMA,
// then PhyloModel_make's row fix-ups (instance.hpp:602-640), then the layouts k_prune reads.
constexpr int EX_BSTRIDE = 68;   // padded row stride of the shared B operand (conflict-free B fragments)

__global__ void __launch_bounds__(128) k_mle_expm(const MleSlot *__restrict__ slots, int n_branches, int nl,
                                                  const float *__restrict__ bl, const double *__restrict__ eig0,
                                                  const double *__restrict__ eig1, const int32_t *__restrict__ edge_to_gemm,
                                                  double *pbase, size_t slot_stride, size_t leaf_off, int *__restrict__ expm_err,
                                                  const double *__restrict__ eig_slots = nullptr /* OMEGA: [slot][64 + 2*4096] */,
                                                  const double *__restrict__ rho_slots = nullptr /* OMEGA: tree scale per slot */) {
    __shared__ double sB[64 * EX_BSTRIDE];
    __shared__ double sEx[64];
    const int si = blockIdx.x / n_branches, b = blockIdx.x % n_branches;
    const MleSlot &s = slots[si];
    if (s.aln < 0 || !s.pending) return;
    const double *eig = eig_slots ? eig_slots + (size_t)si * (64 + 2 * 4096) : (s.model == 0 ? eig0 : eig1);
    const double *lambda = eig, *SR = eig + 64, *SRinv = eig + 64 + 4096;
    // instantiate_tree: float(double(bl) * rho), read back as double (instance.hpp:299-307, :497)
    const double t = (double)(float)((double)bl[b] * (rho_slots ? rho_slots[si] : s.x));
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, q = lane & 3;
    if (tid < 64) sEx[tid] = exp(lambda[tid] * t);
    __syncthreads();
    for (int i = tid; i < 4096; i += 128) {
        const int k = i >> 6, j = i & 63;
        sB[k * EX_BSTRIDE + j] = SRinv[i] * sEx[k];
    }
    __syncthreads();
    double acc[2][16];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int i = 0; i < 16; ++i) acc[mt][i] = 0.0;
    const int row0 = warp * 16;
#pragma unroll 4
    for (int ks = 0; ks < 16; ++ks) {
        const int k = 4 * ks + q;
        const double a0 = __ldg(SR + (row0 + g) * 64 + k), a1 = __ldg(SR + (row0 + 8 + g) * 64 + k);
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            const double bv = sB[k * EX_BSTRIDE + 8 * nt + g];
            dmma(acc[0][2 * nt], acc[0][2 * nt + 1], a0, bv);
            dmma(acc[1][2 * nt], acc[1][2 * nt + 1], a1, bv);
        }
    }
    // thread (g,q) holds rows row0+g (mt 0) and row0+8+g (mt 1), columns 8nt+2q+{0,1}
    bool bad = false;
    double *slot_base = pbase + (size_t)si * slot_stride;
    const int gi = edge_to_gemm[b];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
        const int i = row0 + 8 * mt + g;
        double total = 0.0, off = 0.0;
#pragma unroll
        for (int c = 0; c < 16; ++c) {
            const int j = 8 * (c >> 1) + 2 * q + (c & 1);
            double cell = acc[mt][c];
            total += cell;
            if (cell < 0.0) {
                if (fabs(cell) > 1e-6) bad = true;
                cell = 0.0;
            }
            acc[mt][c] = cell;
            if (j != i) off += cell;
        }
        total += __shfl_xor_sync(0xffffffffu, total, 1); total += __shfl_xor_sync(0xffffffffu, total, 2);
        off += __shfl_xor_sync(0xffffffffu, off, 1); off += __shfl_xor_sync(0xffffffffu, off, 2);
        if (fabs(total - 1.0) > 1e-6) bad = true;
        const double diag = 1.0 - off;
        double rowsum = 0.0;
#pragma unroll
        for (int c = 0; c < 16; ++c) {
            const int j = 8 * (c >> 1) + 2 * q + (c & 1);
            if (j == i) acc[mt][c] = diag;
            rowsum += acc[mt][c];
        }
        rowsum += __shfl_xor_sync(0xffffffffu, rowsum, 1); rowsum += __shfl_xor_sync(0xffffffffu, rowsum, 2);
        if (gi < 0) {
            // leaf table: pt[x][a] = P[a][x]; pt[64][a] = row sum
            double *pt = slot_base + leaf_off + (size_t)b * 65 * 64;
#pragma unroll
            for (int c = 0; c < 16; ++c) {
                const int j = 8 * (c >> 1) + 2 * q + (c & 1);
                pt[j * 64 + i] = acc[mt][c];
            }
            if (q == 0) pt[64 * 64 + i] = rowsum;
        }
    }
    if (gi >= 0) {
        // fragment order: tile[ks][ntp][lane][e] = P[a][bb], a = 8(2ntp+e)+lane/4, bb = 8(ks/2)+2(lane%4)+ks%2.  For this thread's rows
        // (row0 + g and row0 + 8 + g) that is ntp = warp, e = mt, lane = 4g + q = its own lane, ks = c: the two rows of column c are the
        // two halves of ONE 16-byte slot, so a warp writes 512 contiguous bytes per c
        double2 *tile = reinterpret_cast<double2 *>(slot_base + (size_t)gi * 4096);
#pragma unroll
        for (int c = 0; c < 16; ++c) tile[(c * 4 + warp) * 32 + lane] = make_double2(acc[0][c], acc[1][c]);
    }
    if (bad) atomicOr(expm_err + si, 1);
}

// ---------------------------------------------------------------------------------------------------
struct MleSetup {
    std::vector<double> cand;           // candidate rho of fit_find_init's random restarts
    std::vector<int32_t> edge_to_gemm;  // branch id -> index in the P stream, -1 for leaf edges
};

inline MleSetup mle_prepare(const ModelHost &h, double lo, double hi) {
    MleSetup s;
    // fixed_lik.hpp:478-490 with the reference's own generator: std::mt19937 seeded 42 per alignment
    // (score_msa.hpp:115), std::uniform_real_distribution<>(0, width), x = exp(log(lo) + r).
    const double width = std::log(hi) - std::log(lo);
    std::mt19937 gen;
    gen.seed(42);
    std::uniform_real_distribution<> dis(0.0, width);
    s.cand.resize(MLE_NCAND);
    for (int i = 0; i < MLE_NCAND; ++i) s.cand[i] = std::exp(std::log(lo) + dis(gen));
    s.edge_to_gemm.assign(h.n - 1, -1);
    for (size_t g = 0; g < h.gemm_edges.size(); ++g) s.edge_to_gemm[h.gemm_edges[g]] = (int32_t)g;
    return s;
}

#define MCK(call)                                                                   \
    do {                                                                            \
        cudaError_t e_ = (call);                                                    \
        if (e_ != cudaSuccess) {                                                    \
            err = std::string(#call) + ": " + cudaGetErrorString(e_);               \
            return PCSF_ERR_CUDA;                                                   \
        }                                                                           \
    } while (0)

// Runs the whole batch.  d_eig[w]: lambda | SR | SRinv of model w.  scratch: a growable device buffer.
template <class Buf>
inline pcsf_status mle_run(const ModelHost &h, const MleBatch &b, double *const *d_eig, const float *d_bl,
                           const int32_t *d_program, const double *const *d_pi, const double *const *d_logpi, Buf &scratch,
                           int sm_count, size_t prune_smem, int prune_nwarp, cudaStream_t st, std::string &err, int *launches,
                           MleStats *stats = nullptr, bool timing = false) {
    const double lo = 1e-2, hi = 10.0, init = 1.0;   // run.hpp:193-194
    const MleSetup su = mle_prepare(h, lo, hi);
    const int n_br = h.n - 1, n_gemm = (int)h.gemm_edges.size();
    const size_t leaf_off = (size_t)n_gemm * 4096;
    const size_t slot_stride = leaf_off + (size_t)h.nl * 65 * 64;           // doubles
    const size_t budget = (size_t)6 << 30;
    int n_slots = (int)std::min<size_t>((size_t)b.n_aln, std::max<size_t>(1, budget / (slot_stride * 8)));
    n_slots = std::min(n_slots, 8192);
    const int64_t nwin = std::max<int64_t>(b.nwin, 1);
    const int tw = prune_nwarp * 8;
    const size_t max_tiles = (size_t)((b.nwin + tw - 1) / tw) + (size_t)b.n_aln + 1;

    // scratch layout
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    const size_t o_p = take((size_t)n_slots * slot_stride * 8), o_slots = take((size_t)n_slots * sizeof(MleSlot)),
                 o_tiles = take(max_tiles * sizeof(TileDesc)), o_logz = take((size_t)nwin * 8), o_anc = take((size_t)nwin * 8),
                 o_cand = take(su.cand.size() * 8), o_e2g = take(su.edge_to_gemm.size() * 4 + 4), o_err = take((size_t)n_slots * 4),
                 o_ctr = take(64);
    MCK(scratch.reserve(off));
    unsigned char *base = scratch.template as<unsigned char>();
    double *d_p = reinterpret_cast<double *>(base + o_p);
    MleSlot *d_slots = reinterpret_cast<MleSlot *>(base + o_slots);
    TileDesc *d_tiles = reinterpret_cast<TileDesc *>(base + o_tiles);
    double *d_logz = reinterpret_cast<double *>(base + o_logz), *d_ancw = reinterpret_cast<double *>(base + o_anc);
    double *d_cand = reinterpret_cast<double *>(base + o_cand);
    int32_t *d_e2g = reinterpret_cast<int32_t *>(base + o_e2g);
    int *d_err = reinterpret_cast<int *>(base + o_err);
    int *d_ctr = reinterpret_cast<int *>(base + o_ctr);   // [0] queue head, [1] n_active, [2] n_tiles (uint32)

    MCK(cudaMemcpyAsync(d_cand, su.cand.data(), su.cand.size() * 8, cudaMemcpyHostToDevice, st));
    MCK(cudaMemcpyAsync(d_e2g, su.edge_to_gemm.data(), su.edge_to_gemm.size() * 4, cudaMemcpyHostToDevice, st));
    MCK(cudaMemsetAsync(d_slots, 0xFF, (size_t)n_slots * sizeof(MleSlot), st));   // aln = -1 everywhere
    MCK(cudaMemsetAsync(d_err, 0, (size_t)n_slots * 4, st));
    MCK(cudaMemsetAsync(d_ctr, 0, 64, st));

    PruneArgs pa{};
    pa.ws = b.ws;
    pa.tiles = d_tiles;
    pa.n_tiles = reinterpret_cast<uint32_t *>(d_ctr + 2);
    pa.program = d_program;
    pa.n_ops = (int)h.program.size();
    pa.n_gemm = n_gemm;
    pa.max_stack = h.max_stack;
    pa.stagger_ns = 0;
    pa.nwarp = prune_nwarp;
    for (int w = 0; w < 2; ++w) { pa.pi[w] = d_pi[w]; pa.logpi[w] = d_logpi[w]; }
    pa.logz[0] = d_logz;
    pa.anc[0] = b.want_anc ? d_ancw : nullptr;

    cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    if (timing && stats) for (auto &e : ev) MCK(cudaEventCreate(&e));
    struct EvGuard { cudaEvent_t *ev; ~EvGuard() { for (int i = 0; i < 5; ++i) if (ev[i]) cudaEventDestroy(ev[i]); } } ev_guard{ev};
    if (stats) { *stats = MleStats{}; stats->alignments = b.n_aln; stats->slots = n_slots; }
    unsigned long long *d_evals = reinterpret_cast<unsigned long long *>(d_ctr + 4);
    auto finish_stats = [&]() -> cudaError_t {
        if (!stats) return cudaSuccess;
        unsigned long long ne = 0;
        cudaError_t e = cudaMemcpyAsync(&ne, d_evals, 8, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        stats->evaluations = (int64_t)ne;
        return e;
    };
    // every evaluation round: step -> (host reads n_active) -> plan -> expm -> prune
    const int max_rounds = 2 * (3 + MLE_MAX_TRIES + 1 + 4 + 250) * ((b.n_aln + n_slots - 1) / n_slots) + 8;
    for (int round = 0; round < max_rounds; ++round) {
        MCK(cudaMemsetAsync(d_ctr + 1, 0, 4, st));
        if (ev[0]) MCK(cudaEventRecord(ev[0], st));
        k_mle_step<<<(n_slots + 127) / 128, 128, 0, st>>>(d_slots, n_slots, b.n_aln, d_ctr, d_ctr + 1, d_evals, b.d_win_start, b.d_len,
                                                         d_logz, d_ancw, d_err, d_cand, lo, hi, init, b.want_anc ? 1 : 0,
                                                         b.d_phylo, b.d_anc);
        if (ev[0]) MCK(cudaEventRecord(ev[1], st));
        int n_active = 0;
        MCK(cudaMemcpyAsync(&n_active, d_ctr + 1, 4, cudaMemcpyDeviceToHost, st));
        MCK(cudaStreamSynchronize(st));
        if (launches) *launches += 1;
        if (stats) stats->rounds = round;
        if (n_active == 0) { MCK(finish_stats()); return PCSF_OK; }
        MCK(cudaMemsetAsync(d_err, 0, (size_t)n_slots * 4, st));
        k_mle_plan<<<1, 1024, 0, st>>>(d_slots, n_slots, d_p, slot_stride, leaf_off, tw, d_tiles, reinterpret_cast<uint32_t *>(d_ctr + 2));
        if (ev[0]) MCK(cudaEventRecord(ev[2], st));
        k_mle_expm<<<n_slots * n_br, 128, 0, st>>>(d_slots, n_br, h.nl, d_bl, d_eig[0], d_eig[1], d_e2g, d_p, slot_stride, leaf_off, d_err);
        if (ev[0]) MCK(cudaEventRecord(ev[3], st));
        prune_kernel<true>(h.nl)<<<sm_count, (prune_nwarp + 1) * 32, prune_smem, st>>>(pa);
        MCK(cudaGetLastError());
        if (ev[0]) {
            MCK(cudaEventRecord(ev[4], st));
            MCK(cudaEventSynchronize(ev[4]));
            float t;
            MCK(cudaEventElapsedTime(&t, ev[0], ev[1])); stats->ms_step += t;
            MCK(cudaEventElapsedTime(&t, ev[1], ev[2])); stats->ms_plan += t;
            MCK(cudaEventElapsedTime(&t, ev[2], ev[3])); stats->ms_expm += t;
            MCK(cudaEventElapsedTime(&t, ev[3], ev[4])); stats->ms_prune += t;
        }
        if (launches) *launches += 3;
    }
    err = "MLE did not converge within the reference's iteration limits (internal error)";
    return PCSF_ERR_NUMERIC;
}

}  // namespace pcsf
