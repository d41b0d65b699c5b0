// omega.cuh — score-msa --strategy omega on the GPU (SURVEY.md §8 f-1).
//
// Reference: run() OMEGA branch (src/run.hpp:59-182) + src/omega.hpp.  Per alignment: F3x4 codon-position frequencies from
// the alignment (update_f3x4, run.hpp:106-134); two hypotheses (H0: omega = 1, sigma = 1; H1: omega = 0.2, sigma = 0.01), each
// three rounds of { Brent over the tree scale rho in [0.001, 10] with a half-Cauchy log-prior, Brent over kappa in [1, 10]
// with a Gamma log-prior } (max_lik_lpr_leaves, fixed_lik.hpp:511-544); every kappa evaluation rebuilds
// Q(kappa, omega, pi_F3x4), its eigensystem and all P(t); score = 10 (lpr_H1 - lpr_H0) / ln 10 with lpr = the LAST evaluation
// of the respective last fit.  One std::mt19937(42) stream per alignment feeds all twelve fits (score_msa.hpp:115).
//
// B200 design: the batched-Brent machinery of mle.cuh with two additions —
//     k_omega_counts  F3x4 ratios of every alignment (one block per alignment)
//     k_omega_step    the twelve-fit sequence as a per-slot state machine on top of fit_advance()
//     k_omega_eig     batched 64x64 eigensolver, one CTA per slot that needs it: Q is reversible, so the similar symmetric
//                     matrix D^1/2 Q D^-1/2 is diagonalised by a parallel-ordered (round-robin) two-sided Jacobi in shared
//                     memory — 32 disjoint rotations per step, 63 steps per sweep; writes lambda | S | S^-1 and the
//                     equilibrium prior of the slot
// k_mle_expm / k_mle_plan / k_prune<true> then run unchanged with per-slot eigensystems, tree scales and root priors.
// The reference's GSL route (gsl_eigen_nonsymmv + complex LU) and this one give the same P(t) to ~1e-13; Brent trajectories
// that fork on such differences end within the reference's own CI tolerance (squared error <= 0.1, test/tests.sh:46).
#pragma once

#include "mle.cuh"

namespace pcsf {

constexpr int OMEGA_FITS = 12;
constexpr int OMEGA_NCAND = OMEGA_FITS * MLE_MAX_TRIES;
constexpr size_t OMEGA_EIG_STRIDE = 64 + 2 * 4096;          // doubles per slot: lambda | SR | SRinv

struct OmegaExtra {
    int32_t stage;        // 0..11: hypothesis = stage / 6, kind = stage & 1 (0: rho fit, 1: kappa fit)
    int32_t need_eig;     // the pending evaluation needs a new Q and eigensystem
    int32_t force_eig;    // ... because omega/sigma or the alignment changed
    int32_t pad;
    double rho, kappa, omega, sigma;
    double init;          // the current fit's initial point
    double res[2];        // lpr_H0, lpr_H1
};

// translation.hpp: the standard genetic code indexed by 16a+4b+c over A,C,G,T
__device__ inline char omega_aa(int codon) {
    const char *tcag = "FFLLSSSSYY**CC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG";
    const int to_tcag[4] = {2, 1, 3, 0};
    return tcag[16 * to_tcag[codon >> 4] + 4 * to_tcag[(codon >> 2) & 3] + to_tcag[codon & 3]];
}

// omega.hpp:130-141 half-Cauchy(mode 1, scale 0.5) log-density; :143-149 log Gamma(7, 0.25) density at kappa - 1 + eps
__device__ inline double omega_lpr_rho(double rho) {
    const double mode = 1.0, scale = 0.5, pi = 3.14159265358979323846;
    const double numer = 1.0 / (pi * scale * (1.0 + pow(((rho - mode) / scale), 2.0)));
    const double cauchy_cdf = atan((0.0 - mode) / scale) / pi + 0.5;
    return log(numer) - log(1.0 - cauchy_cdf);
}
__device__ inline double omega_lpr_kappa(double kappa) {
    const double k = kappa - 1.0 + 2.2204460492503131e-16;
    const double a = 7.0, b = 0.25;
    const double g = (k <= 0) ? 0.0 : exp((a - 1) * log(k / b) - k / b - lgamma(a)) / b;
    return log(g);
}

// update_f3x4 (run.hpp:106-134): pseudo-count 1, certain codons of all species; ratios to the T count.
__global__ void __launch_bounds__(256) k_omega_counts(WinSpace ws, int n_aln, const int64_t *__restrict__ win_start,
                                                     const int64_t *__restrict__ len, double *__restrict__ f3x4) {
    __shared__ unsigned int cnt[12];
    const int aln = blockIdx.x;
    if (aln >= n_aln) return;
    if (threadIdx.x < 12) cnt[threadIdx.x] = 0;
    __syncthreads();
    const int64_t K = len[aln] / 3, w0 = win_start[aln];
    unsigned int loc[12] = {0};
    for (int64_t i = threadIdx.x; i < K * ws.nl; i += blockDim.x) {
        const int sp = (int)(i / K);
        const int64_t k = i - (int64_t)sp * K;
        const uint8_t *c = ws.codes + (size_t)sp * ws.ld + ws.win_off[w0 + k];
        int a = c[0], b = c[1], d = c[2];
        if (ws.win_strand && ws.win_strand[w0 + k] && a < 4 && b < 4 && d < 4) {   // '-' window: the complemented, reversed codon
            const int t = a; a = 3 - d; b = 3 - b; d = 3 - t;
        }
        if (a < 4 && b < 4 && d < 4) { ++loc[a]; ++loc[4 + b]; ++loc[8 + d]; }
    }
    for (int j = 0; j < 12; ++j) if (loc[j]) atomicAdd(&cnt[j], loc[j]);
    __syncthreads();
    if (threadIdx.x < 9) {
        const int i = threadIdx.x / 3, j = threadIdx.x % 3;
        f3x4[(size_t)aln * 9 + threadIdx.x] = (1.0 + (double)cnt[4 * i + j]) / (1.0 + (double)cnt[4 * i + 3]);
    }
}

// One thread per slot: consumes the evaluation that just finished and advances the alignment's twelve-fit sequence.
__global__ void k_omega_step(MleSlot *slots, OmegaExtra *extra, double *__restrict__ rho_slots, int n_slots, int n_aln,
                             int *queue_head, int *n_active, const int64_t *__restrict__ win_start, const int64_t *__restrict__ len,
                             const double *__restrict__ logz, const int *__restrict__ expm_err,
                             const double *__restrict__ cand_rho, const double *__restrict__ cand_kappa, float *__restrict__ phylo) {
    const int si = blockIdx.x * blockDim.x + threadIdx.x;
    if (si >= n_slots) return;
    const double LO[2] = {0.001, 1.0}, HI[2] = {10.0, 10.0};          // run.hpp:150,153
    MleSlot s = slots[si];
    OmegaExtra e = extra[si];
    bool have_result = false;
    if (s.aln >= 0 && s.pending) {
        double l = 0.0;                                              // lpr_leaves_omega: lpr += log z in codon order (omega.hpp:200)
        for (int64_t k = 0; k < s.K; ++k) l = __dadd_rn(l, logz[s.win0 + k]);
        l += (e.stage & 1) ? omega_lpr_kappa(s.x) : omega_lpr_rho(s.x);
        s.lpr = l;
        s.pending = 0;
        if (expm_err[si]) s.failed = 1;
        have_result = true;
    }
    for (;;) {
        bool start_fit = false;
        if (s.aln < 0) {
            const int next = atomicAdd(queue_head, 1);
            if (next >= n_aln) { s.aln = -1; break; }
            s = MleSlot{};
            e = OmegaExtra{};
            s.aln = next;
            s.K = len[next] / 3;
            s.win0 = win_start[next];
            e.rho = 1.0; e.kappa = 2.5; e.omega = 1.0; e.sigma = 1.0;      // run.hpp:75-82
            e.stage = 0;
            e.force_eig = 1;
            start_fit = true;
        } else {
            if (!have_result) break;
            have_result = false;
            const int kind = e.stage & 1;
            const bool done = s.failed ? true : fit_advance(s, LO[kind], HI[kind], e.init, kind ? cand_kappa : cand_rho);
            if (done) {
                if (s.failed) {
                    if (phylo) phylo[s.aln] = nanf("");
                    s.aln = -1;
                    continue;
                }
                if (e.stage == 5) e.res[0] = s.lpr;
                if (e.stage == OMEGA_FITS - 1) {
                    e.res[1] = s.lpr;
                    if (phylo) phylo[s.aln] = (float)(10.0 * (e.res[1] - e.res[0]) / log(10.0));
                    s.aln = -1;
                    continue;
                }
                ++e.stage;
                if (e.stage == 6) { e.omega = 0.2; e.sigma = 0.01; e.force_eig = 1; }          // run.hpp:161-166
                start_fit = true;
            }
        }
        const int kind = e.stage & 1;
        if (start_fit) {
            e.init = kind ? e.kappa : e.rho;          // run.hpp:149-154: the values the previous fit left behind
            s.phase = PH_LO;
            s.x = LO[kind];
            s.tries = 0;
        }
        // issue the evaluation at s.x (omega.hpp:205-233)
        if (kind) { e.kappa = s.x; e.need_eig = 1; }
        else { e.rho = s.x; e.need_eig = e.force_eig; }
        e.force_eig = 0;
        s.pending = 1;
        break;
    }
    slots[si] = s;
    extra[si] = e;
    rho_slots[si] = e.rho;
    if (s.aln >= 0) atomicAdd(n_active, 1);
}

// Batched eigensystem: one CTA (256 threads) per slot whose pending evaluation needs a new Q.
// Shared memory: A[64][64] | V[64][64] | pi[64] | sq[64] | c[32] | s[32] | pairs.
constexpr size_t OMEGA_EIG_SMEM = (2 * 4096 + 64 + 64 + 64) * 8 + 64 * 4 + 64;

__global__ void __launch_bounds__(256) k_omega_eig(const MleSlot *__restrict__ slots, const OmegaExtra *__restrict__ extra,
                                                   const double *__restrict__ f3x4, double *__restrict__ eig_slots,
                                                   double *__restrict__ pi_slots) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int si = blockIdx.x;
    const MleSlot &sl = slots[si];
    if (sl.aln < 0 || !sl.pending || !extra[si].need_eig) return;
    double *A = reinterpret_cast<double *>(smem_raw), *V = A + 4096, *pi = V + 4096, *sq = pi + 64, *rc = sq + 64, *rs = rc + 32;
    int *pp = reinterpret_cast<int *>(rs + 32), *qq = pp + 32;
    __shared__ double s_factor, s_off, s_diag;
    const int tid = threadIdx.x;
    const OmegaExtra &ex = extra[si];
    const double kappa = ex.kappa, omega = ex.omega, sigma = ex.sigma;
    const double *f = f3x4 + (size_t)sl.aln * 9;
    // pi_expr (omega.hpp:8-36)
    const auto pi_sc = [&](int codon) {
        const int i1 = codon >> 4, i2 = (codon >> 2) & 3, i3 = codon & 3;
        const double f1 = ((i1 == 3) ? 1.0 : f[i1]) / (1.0 + f[0] + f[1] + f[2]);
        const double f2 = ((i2 == 3) ? 1.0 : f[3 + i2]) / (1.0 + f[3] + f[4] + f[5]);
        const double f3 = ((i3 == 3) ? 1.0 : f[6 + i3]) / (1.0 + f[6] + f[7] + f[8]);
        return f1 * f2 * f3;
    };
    if (tid < 64) {
        const double denom = 1.0 - ((1.0 - sigma) * (pi_sc(48) + pi_sc(50) + pi_sc(56)));          // TAA, TAG, TGA
        pi[tid] = pi_sc(tid) / denom;
        sq[tid] = sqrt(pi[tid]);
    }
    __syncthreads();
    // comp_q_p14n (omega.hpp:38-95), unscaled
    for (int idx = tid; idx < 4096; idx += 256) {
        const int i = idx >> 6, j = idx & 63;
        const int i1 = i >> 4, i2 = (i >> 2) & 3, i3 = i & 3, j1 = j >> 4, j2 = (j >> 2) & 3, j3 = j & 3;
        double val = 0.0;
        if ((i1 != j1) + (i2 != j2) + (i3 != j3) == 1) {
            bool ts = false;
            if (i1 != j1 && (i1 + j1 == 2 || i1 + j1 == 4)) ts = true;
            if (i2 != j2 && (i2 + j2 == 2 || i2 + j2 == 4)) ts = true;
            if (i3 != j3 && (i3 + j3 == 2 || i3 + j3 == 4)) ts = true;
            val = ts ? kappa : 1.0;
            const char ia = omega_aa(i), ja = omega_aa(j);
            val *= (ia != '*' && ja != '*' && ia != ja) ? omega : 1.0;
            val *= pi[j];
        }
        A[idx] = val;
        V[idx] = (i == j) ? 1.0 : 0.0;
    }
    __syncthreads();
    if (tid < 64) {
        double val = 0.0;
        for (int j = 0; j < 64; ++j) if (j != tid) val -= A[tid * 64 + j];
        A[tid * 64 + tid] = val;
    }
    __syncthreads();
    if (tid == 0) {
        double factor = 0.0;                                          // comp_q_scale (omega.hpp:97-103)
        for (int i = 0; i < 64; ++i) factor -= pi[i] * A[i * 64 + i];
        s_factor = factor;
    }
    __syncthreads();
    // D^1/2 (Q / scale) D^-1/2, then the exact symmetrisation of its rounding noise
    for (int idx = tid; idx < 4096; idx += 256) {
        const int i = idx >> 6, j = idx & 63;
        A[idx] = sq[i] * (A[idx] / s_factor) / sq[j];
    }
    __syncthreads();
    for (int idx = tid; idx < 4096; idx += 256) {
        const int i = idx >> 6, j = idx & 63;
        if (i < j) {
            const double m = 0.5 * (A[i * 64 + j] + A[j * 64 + i]);
            A[i * 64 + j] = m;
            A[j * 64 + i] = m;
        }
    }
    __syncthreads();
    for (int sweep = 0; sweep < 40; ++sweep) {
        // convergence: off-diagonal mass against the diagonal's
        if (tid < 32) {
            double off = 0.0, dg = 0.0;
            for (int r = tid; r < 64; r += 32) {
                for (int c = 0; c < 64; ++c) { const double v = A[r * 64 + c]; if (c == r) dg += v * v; else off += v * v; }
            }
            for (int o = 16; o; o >>= 1) { off += __shfl_xor_sync(0xffffffffu, off, o); dg += __shfl_xor_sync(0xffffffffu, dg, o); }
            if (tid == 0) { s_off = off; s_diag = dg; }
        }
        __syncthreads();
        if (s_off <= 1e-34 * s_diag || s_off < 1e-300) break;
        for (int r = 0; r < 63; ++r) {
            if (tid < 32) {
                int a, b;
                if (tid == 0) { a = 63; b = r; }
                else { a = (r + tid) % 63; b = (r + 63 - tid) % 63; }
                const int p = a < b ? a : b, q = a < b ? b : a;
                const double apq = A[p * 64 + q];
                double c = 1.0, s = 0.0;
                if (fabs(apq) >= 1e-310) {
                    const double app = A[p * 64 + p], aqq = A[q * 64 + q];
                    const double theta = (aqq - app) / (2.0 * apq);
                    const double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
                    c = 1.0 / sqrt(t * t + 1.0);
                    s = t * c;
                }
                pp[tid] = p; qq[tid] = q; rc[tid] = c; rs[tid] = s;
            }
            __syncthreads();
            // columns p, q of A and of V  (x J)
            for (int idx = tid; idx < 2048; idx += 256) {
                const int k = idx & 31, i = idx >> 5;
                const int p = pp[k], q = qq[k];
                const double c = rc[k], s = rs[k];
                const double aip = A[i * 64 + p], aiq = A[i * 64 + q];
                A[i * 64 + p] = c * aip - s * aiq;
                A[i * 64 + q] = s * aip + c * aiq;
                const double vip = V[i * 64 + p], viq = V[i * 64 + q];
                V[i * 64 + p] = c * vip - s * viq;
                V[i * 64 + q] = s * vip + c * viq;
            }
            __syncthreads();
            // rows p, q of A  (J^T x)
            for (int idx = tid; idx < 2048; idx += 256) {
                const int j = idx & 63, k = idx >> 6;
                const int p = pp[k], q = qq[k];
                const double c = rc[k], s = rs[k];
                const double apj = A[p * 64 + j], aqj = A[q * 64 + j];
                A[p * 64 + j] = c * apj - s * aqj;
                A[q * 64 + j] = s * apj + c * aqj;
            }
            __syncthreads();
        }
    }
    // lambda | SR (right eigenvectors in columns) | SRinv (left eigenvectors in rows)
    double *eig = eig_slots + (size_t)si * OMEGA_EIG_STRIDE;
    if (tid < 64) eig[tid] = A[tid * 64 + tid];
    for (int idx = tid; idx < 4096; idx += 256) {
        const int i = idx >> 6, k = idx & 63;
        const double u = V[i * 64 + k];
        eig[64 + i * 64 + k] = u / sq[i];
        eig[64 + 4096 + k * 64 + i] = u * sq[i];
    }
    __syncthreads();
    // equilibrium prior (fixed_lik.hpp:323-346): the row of S^-1 at the smallest |lambda|, normalised
    if (tid == 0) {
        double minL = fabs(A[0]);
        int minp = 0;
        for (int i = 1; i < 64; ++i) { const double m = fabs(A[i * 64 + i]); if (m < minL) { minL = m; minp = i; } }
        double mass = 0.0;
        for (int j = 0; j < 64; ++j) mass += V[j * 64 + minp] * sq[j];
        for (int j = 0; j < 64; ++j) pi_slots[(size_t)si * 64 + j] = (V[j * 64 + minp] * sq[j]) / mass;
    }
}

struct OmegaBatch {
    int n_aln;
    const int64_t *d_win_start, *d_len;
    WinSpace ws;
    int64_t nwin;
    float *d_phylo;
};

// Runs the whole batch (see mle_run for the round structure).
template <class Buf>
inline pcsf_status omega_run(const ModelHost &h, const OmegaBatch &b, const float *d_bl, const int32_t *d_program,
                             const double *const *d_pi, const double *const *d_logpi, Buf &scratch, int sm_count, size_t prune_smem,
                             int prune_nwarp, cudaStream_t st, std::string &err, int *launches) {
    const double lo[2] = {0.001, 1.0}, hi[2] = {10.0, 10.0};
    // candidate points of fit_find_init's random restarts: draw i of the alignment's std::mt19937(42) stream, mapped with the
    // reference's own expression (fixed_lik.hpp:478-490) for either interval
    std::vector<double> cand[2];
    for (int k = 0; k < 2; ++k) {
        const double width = std::log(hi[k]) - std::log(lo[k]);
        std::mt19937 gen;
        gen.seed(42);
        std::uniform_real_distribution<> dis(0.0, width);
        cand[k].resize(OMEGA_NCAND + 1);
        for (int i = 0; i <= OMEGA_NCAND; ++i) cand[k][i] = std::exp(std::log(lo[k]) + dis(gen));
    }
    std::vector<int32_t> edge_to_gemm(h.n - 1, -1);
    for (size_t g = 0; g < h.gemm_edges.size(); ++g) edge_to_gemm[h.gemm_edges[g]] = (int32_t)g;
    const int n_br = h.n - 1, n_gemm = (int)h.gemm_edges.size();
    const size_t leaf_off = (size_t)n_gemm * 4096;
    const size_t slot_stride = leaf_off + (size_t)h.nl * 65 * 64;
    const size_t budget = (size_t)6 << 30;
    int n_slots = (int)std::min<size_t>((size_t)b.n_aln, std::max<size_t>(1, budget / ((slot_stride + OMEGA_EIG_STRIDE) * 8)));
    n_slots = std::min(n_slots, 4096);
    const int64_t nwin = std::max<int64_t>(b.nwin, 1);
    const int tw = prune_nwarp * 8;
    const size_t max_tiles = (size_t)((b.nwin + tw - 1) / tw) + (size_t)b.n_aln + 1;

    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    const size_t o_p = take((size_t)n_slots * slot_stride * 8), o_eig = take((size_t)n_slots * OMEGA_EIG_STRIDE * 8),
                 o_pi = take((size_t)n_slots * 64 * 8), o_rho = take((size_t)n_slots * 8), o_slots = take((size_t)n_slots * sizeof(MleSlot)),
                 o_extra = take((size_t)n_slots * sizeof(OmegaExtra)), o_tiles = take(max_tiles * sizeof(TileDesc)),
                 o_logz = take((size_t)nwin * 8), o_f = take((size_t)b.n_aln * 9 * 8), o_cr = take(cand[0].size() * 8),
                 o_ck = take(cand[1].size() * 8), o_e2g = take(edge_to_gemm.size() * 4 + 4), o_err = take((size_t)n_slots * 4),
                 o_ctr = take(64);
    MCK(scratch.reserve(off));
    unsigned char *base = scratch.template as<unsigned char>();
    double *d_p = reinterpret_cast<double *>(base + o_p), *d_eig = reinterpret_cast<double *>(base + o_eig);
    double *d_pis = reinterpret_cast<double *>(base + o_pi), *d_rho = reinterpret_cast<double *>(base + o_rho);
    MleSlot *d_slots = reinterpret_cast<MleSlot *>(base + o_slots);
    OmegaExtra *d_extra = reinterpret_cast<OmegaExtra *>(base + o_extra);
    TileDesc *d_tiles = reinterpret_cast<TileDesc *>(base + o_tiles);
    double *d_logz = reinterpret_cast<double *>(base + o_logz), *d_f = reinterpret_cast<double *>(base + o_f);
    double *d_cr = reinterpret_cast<double *>(base + o_cr), *d_ck = reinterpret_cast<double *>(base + o_ck);
    int32_t *d_e2g = reinterpret_cast<int32_t *>(base + o_e2g);
    int *d_err = reinterpret_cast<int *>(base + o_err), *d_ctr = reinterpret_cast<int *>(base + o_ctr);

    MCK(cudaMemcpyAsync(d_cr, cand[0].data(), cand[0].size() * 8, cudaMemcpyHostToDevice, st));
    MCK(cudaMemcpyAsync(d_ck, cand[1].data(), cand[1].size() * 8, cudaMemcpyHostToDevice, st));
    MCK(cudaMemcpyAsync(d_e2g, edge_to_gemm.data(), edge_to_gemm.size() * 4, cudaMemcpyHostToDevice, st));
    MCK(cudaMemsetAsync(d_slots, 0xFF, (size_t)n_slots * sizeof(MleSlot), st));
    MCK(cudaMemsetAsync(d_extra, 0, (size_t)n_slots * sizeof(OmegaExtra), st));
    MCK(cudaMemsetAsync(d_err, 0, (size_t)n_slots * 4, st));
    MCK(cudaMemsetAsync(d_ctr, 0, 64, st));
    MCK(cudaFuncSetAttribute(k_omega_eig, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)OMEGA_EIG_SMEM));
    k_omega_counts<<<b.n_aln, 256, 0, st>>>(b.ws, b.n_aln, b.d_win_start, b.d_len, d_f);
    MCK(cudaGetLastError());
    if (launches) *launches += 1;

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
    for (int w = 0; w < 2; ++w) { pa.pi[w] = d_pi[w]; pa.logpi[w] = d_logpi[w]; }          // unused: every tile carries its own prior
    pa.logz[0] = d_logz;
    pa.anc[0] = nullptr;

    const int max_rounds = OMEGA_FITS * (3 + MLE_MAX_TRIES + 1 + 4 + 250) * ((b.n_aln + n_slots - 1) / n_slots) + 8;
    for (int round = 0; round < max_rounds; ++round) {
        MCK(cudaMemsetAsync(d_ctr + 1, 0, 4, st));
        k_omega_step<<<(n_slots + 127) / 128, 128, 0, st>>>(d_slots, d_extra, d_rho, n_slots, b.n_aln, d_ctr, d_ctr + 1, b.d_win_start,
                                                           b.d_len, d_logz, d_err, d_cr, d_ck, b.d_phylo);
        int n_active = 0;
        MCK(cudaMemcpyAsync(&n_active, d_ctr + 1, 4, cudaMemcpyDeviceToHost, st));
        MCK(cudaStreamSynchronize(st));
        if (launches) *launches += 1;
        if (n_active == 0) return PCSF_OK;
        MCK(cudaMemsetAsync(d_err, 0, (size_t)n_slots * 4, st));
        k_omega_eig<<<n_slots, 256, OMEGA_EIG_SMEM, st>>>(d_slots, d_extra, d_f, d_eig, d_pis);
        k_mle_plan<<<1, 1024, 0, st>>>(d_slots, n_slots, d_p, slot_stride, leaf_off, tw, d_tiles, reinterpret_cast<uint32_t *>(d_ctr + 2), d_pis);
        k_mle_expm<<<n_slots * n_br, 128, 0, st>>>(d_slots, n_br, h.nl, d_bl, nullptr, nullptr, d_e2g, d_p, slot_stride, leaf_off, d_err,
                                                  d_eig, d_rho);
        prune_kernel<true>(h.nl)<<<sm_count, (prune_nwarp + 1) * 32, prune_smem, st>>>(pa);
        MCK(cudaGetLastError());
        if (launches) *launches += 4;
    }
    err = "OMEGA did not converge within the reference's iteration limits (internal error)";
    return PCSF_ERR_NUMERIC;
}

}  // namespace pcsf
