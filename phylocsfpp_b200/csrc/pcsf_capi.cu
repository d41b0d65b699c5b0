// pcsf_capi.cu — C-ABI (include/phylocsf_b200.h) over the sm_100a kernels in kernels.cuh.
//
// Replaces the reference's call seam run_tracks / run / compute_bls_score (src/run.hpp:35,57,
// src/additional_scores.hpp:44).  No CPU fallback: every compute entry point needs a CUDA device.
#include "../../include/phylocsf_b200.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <string>
#include <vector>

#include "kernels.cuh"
#include "mle.cuh"
#include "omega.cuh"
#include "prune_tc5.cuh"
#include "regions.cuh"
#include <nvtx3/nvToolsExt.h>

using namespace pcsf;

static thread_local std::string g_err;
static pcsf_status fail(pcsf_status st, const std::string &msg) { g_err = msg; return st; }

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(PCSF_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));        \
    } while (0)

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    // Grows with 25 % headroom (2 MiB granularity): callers such as the command line host pass batches whose sizes differ by a few
    // columns from call to call, and an exact-size policy turned every slightly larger batch into a cudaFree + cudaMalloc of all
    // scratch buffers (measured: 60-1100 ms of allocation churn per 10 M columns, against 104 ms of pruning).
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 4;
        want = (want + ((size_t)2 << 20) - 1) & ~(((size_t)2 << 20) - 1);
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { cudaGetLastError(); want = bytes; e = cudaMalloc(&p, want); }          // no room for headroom: exact size
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T *as() const { return reinterpret_cast<T *>(p); }
};

// NVTX range around the host-side enqueue of one stage (nsys / ncu --nvtx group the launches by it)
struct NvtxRange {
    explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};

struct pcsf_model {
    int device = 0;
    int sm_count = 148;
    cudaStream_t own_stream = nullptr;   // the host-buffer entry points run here (non-blocking: handles on one GPU overlap)
    cudaStream_t copy_stream = nullptr;  // results of a finished dedup chunk go home while the next chunk is pruned
    cudaEvent_t ev_chunk = nullptr;
    // host destinations of the call in flight (pcsf_tracks only; null for the device-pointer entry point)
    double *h_plus = nullptr, *h_minus = nullptr, *h_bls = nullptr;
    uint32_t *h_pat = nullptr;
    const uint8_t *h_seqs = nullptr;     // non-null: the input is still on the host and arrives segment by segment (one per dedup chunk)
    int64_t h_ld = 0;
    cudaStream_t h2d_stream = nullptr;
    std::vector<cudaEvent_t> ev_h2d;
    ModelHost host;
    // device blob
    double *d_pstream[2] = {nullptr, nullptr}, *d_leafPT[2] = {nullptr, nullptr};
    double *d_pi[2] = {nullptr, nullptr}, *d_logpi[2] = {nullptr, nullptr};
    double *d_eig[2] = {nullptr, nullptr};   // lambda[64] | SR[4096] | SRinv[4096]
    float *d_pstream_tc5[2] = {nullptr, nullptr};
    float *d_rowtab_tc5[2] = {nullptr, nullptr};   // [tc5_rows][64] leaf and cherry message tables in program order (k_build_rows)
    Tc5Src *d_tc5_srcs = nullptr;
    uint32_t *d_tc5_steps = nullptr;
    float *d_tc5_scratch = nullptr;      // stack spill of k_prune_tc5: [sm_count][2][max_stack][T5_STACK_ENTRY_FLOATS]
    size_t prune_tc5_smem = 0;
    int tc5_nstage = 2, tc5_nids = 1;
    MleStats msa_stats;                  // of the last MLE score-msa call
    uint8_t *h_msa = nullptr;            // page-locked staging of pcsf_score_msa's concatenated [nl][Ltot] matrix (grows with 25 % headroom)
    size_t h_msa_cap = 0;
    DevBuf tc5_ids;                      // codon ids of the unique windows, [pairs][2][nl][128] (k_tc5_ids)
    int32_t *d_program = nullptr;
    void *d_bls_prog = nullptr;          // BlsInnerDev<2> (trees of at most SMALL_TREE_MAX_LEAVES leaves) or BlsInnerDev<8>
    double *d_bls_tables = nullptr;
    float *d_bl = nullptr;
    int32_t *d_gemm_edges = nullptr;
    // scratch
    DevBuf codes, klo, khi, slot, flag, uniq, pidx, table, bsums, logz, anc, io_in, io_out, perwin, mle;
    DevBuf rg_units, rg_regions, rg_win;      // score-msa (both entry points): per-(alignment, frame) counts, region lists, region windows
    std::vector<pcsf_region> regions;         // records of the last pcsf_score_regions call
    int *d_bad = nullptr;
    uint32_t *d_nuniq = nullptr;       // [max chunks]
    int64_t chunk_cols = (int64_t)1 << 21;          // 2 Mi columns: calls of 4 Mi columns and more are pipelined (H2D | compute | D2H per chunk)
    bool timing = false;
    uint32_t stagger_ns = 1000;
    pcsf_tracks_stats last{};
    int64_t last_nwin = 0;
    int launches = 0;
    int last_chunks = 0;
    int64_t codes_ld = 0;
    size_t prune_smem = 0;
    int prune_nwarp = 8;
    cudaEvent_t ev[8] = {};
};

static const int MAX_CHUNKS = 4096;

extern "C" const char *pcsf_last_error(void) { return g_err.c_str(); }
extern "C" int pcsf_abi_version(void) { return PCSF_ABI_VERSION; }

static pcsf_status upload(const void *src, size_t bytes, void **dst) {
    CK(cudaMalloc(dst, bytes ? bytes : 16));
    if (bytes) CK(cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice));
    return PCSF_OK;
}

extern "C" pcsf_status pcsf_model_create(const pcsf_model_desc *d, int device, pcsf_model **out) {
    if (!d || !out || d->nl < 2 || !d->child1 || !d->child2 || !d->branch_len || !d->branch_len_f64 || !d->ecm_c ||
        !d->freq_c || !d->ecm_nc || !d->freq_nc)
        return fail(PCSF_ERR_INVALID, "pcsf_model_create: null argument or fewer than 2 leaves");
    if (d->nl > PCSF_MAX_LEAVES)
        return fail(PCSF_ERR_UNSUPPORTED, "tree of " + std::to_string(d->nl) + " leaves: at most " + std::to_string(PCSF_MAX_LEAVES) +
                                              " leaves (PCSF_MAX_LEAVES) are supported");
    pcsf_model *m = new pcsf_model;
    struct Guard {                       // every early return below releases the handle and what it already owns on the device
        pcsf_model *m;
        ~Guard() { if (m) pcsf_model_destroy(m); }
    } guard{m};
    const double *S[2] = {d->ecm_c, d->ecm_nc}, *f[2] = {d->freq_c, d->freq_nc};
    const std::string err = prepare_model(m->host, d->nl, d->child1, d->child2, d->branch_len, d->branch_len_f64, S, f);
    if (!err.empty()) {
        return fail(err.find("substition_matrix") != std::string::npos ? PCSF_ERR_NUMERIC : PCSF_ERR_INVALID, err);
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0 || device < 0 || device >= ndev) {
        guard.m = nullptr;
        delete m;                        // nothing on a device yet (and pcsf_model_destroy would call cudaSetDevice)
        return fail(PCSF_ERR_CUDA, "no CUDA device available (this library has no CPU fallback)");
    }
    m->device = device;
    if (const char *e = getenv("PCSF_STAGGER_NS")) m->stagger_ns = (uint32_t)atoi(e);
    CK(cudaSetDevice(device));
    CK(cudaDeviceGetAttribute(&m->sm_count, cudaDevAttrMultiProcessorCount, device));
    {
        uint8_t lut[256];
        memset(lut, 255, sizeof lut);
        lut['A'] = lut['a'] = 0; lut['C'] = lut['c'] = 1; lut['G'] = lut['g'] = 2; lut['T'] = lut['t'] = 3;
        lut['.'] = lut['-'] = lut['N'] = lut['n'] = 4;
        CK(cudaMemcpyToSymbol(c_dna_lut, lut, sizeof lut));
    }
    pcsf_status st;
    for (int w = 0; w < 2; ++w) {
        const EcmHost &e = m->host.ecm[w];
        if ((st = upload(e.pstream.data(), e.pstream.size() * 8, (void **)&m->d_pstream[w]))) return st;
        if ((st = upload(e.leafPT.data(), e.leafPT.size() * 8, (void **)&m->d_leafPT[w]))) return st;
        if ((st = upload(e.pstream_tc5.data(), e.pstream_tc5.size() * 4, (void **)&m->d_pstream_tc5[w]))) return st;
        if ((st = upload(e.pi, 64 * 8, (void **)&m->d_pi[w]))) return st;
        if ((st = upload(e.logpi, 64 * 8, (void **)&m->d_logpi[w]))) return st;
        std::vector<double> eig(64 + 2 * 4096);
        memcpy(eig.data(), e.lambda, 64 * 8);
        memcpy(eig.data() + 64, e.SR, 4096 * 8);
        memcpy(eig.data() + 64 + 4096, e.SRinv, 4096 * 8);
        if ((st = upload(eig.data(), eig.size() * 8, (void **)&m->d_eig[w]))) return st;
    }
    if ((st = upload(m->host.program.data(), m->host.program.size() * 4, (void **)&m->d_program))) return st;
    // Trees above SMALL_TREE_MAX_LEAVES leaves have no tcgen05 program (model_prep.hpp): no row tables, and pcsf_tracks_device refuses
    // PCSF_TRACKS_TC5 for them.
    if (m->host.nl <= SMALL_TREE_MAX_LEAVES) {
        if ((st = upload(m->host.tc5_steps.data(), m->host.tc5_steps.size() * 4, (void **)&m->d_tc5_steps))) return st;
        CK(cudaMalloc(&m->d_tc5_scratch, (size_t)m->sm_count * 2 * std::max(1, m->host.tc5_max_stack) * T5_STACK_ENTRY_FLOATS * 4));
        // row tables (leaf columns and cherry messages): FP64 on the device from the leaves' columns and the cherry nodes' P, FP32 rows
        const int ns = (int)m->host.tc5_srcs.size();
        if ((st = upload(m->host.tc5_srcs.data(), (size_t)ns * sizeof(Tc5Src), (void **)&m->d_tc5_srcs))) return st;
        for (int w = 0; w < 2; ++w) {
            double *d_cp = nullptr;
            if ((st = upload(m->host.ecm[w].cherry_P.data(), m->host.ecm[w].cherry_P.size() * 8, (void **)&d_cp))) return st;
            cudaError_t e = cudaMalloc(&m->d_rowtab_tc5[w], (size_t)m->host.tc5_rows * 64 * 4);
            if (e == cudaSuccess) {
                k_build_rows<<<dim3(65, ns), 64>>>(m->d_tc5_srcs, d_cp, m->d_leafPT[w], m->d_rowtab_tc5[w]);
                e = cudaGetLastError();
                if (e == cudaSuccess) e = cudaDeviceSynchronize();
            }
            cudaFree(d_cp);
            CK(e);
        }
        prune_tc5_pick_stages(m->host.nl, (int)m->host.tc5_steps.size(), (int)m->host.tc5_srcs.size(), &m->tc5_nstage, &m->tc5_nids);
        if (const char *e = getenv("PCSF_TC5_NSTAGE")) m->tc5_nstage = std::max(2, std::min(m->tc5_nstage, atoi(e)));
        if (const char *e = getenv("PCSF_TC5_NIDS")) m->tc5_nids = std::max(1, std::min(m->tc5_nids, atoi(e)));
        m->prune_tc5_smem = prune_tc5_smem_bytes(m->host.nl, (int)m->host.tc5_steps.size(), (int)m->host.tc5_srcs.size(), m->tc5_nstage, m->tc5_nids);
        // Trees above the tcgen05 path's budget (127 and 128 leaves always, 124 to 126 depending on the shape) still get a model: the FP64
        // path and score-msa do not need k_prune_tc5, and pcsf_tracks_device refuses PCSF_TRACKS_TC5 for them with PCSF_ERR_UNSUPPORTED.
        if (m->prune_tc5_smem <= 227 * 1024)
            CK(cudaFuncSetAttribute(k_prune_tc5, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)m->prune_tc5_smem));
        const std::vector<BlsInnerDev<2>> prog = bls_device_program<2>(m->host.bls_short);
        if ((st = upload(prog.data(), prog.size() * sizeof(prog[0]), &m->d_bls_prog))) return st;
    } else {
        const std::vector<BlsInnerDev<8>> prog = bls_device_program<8>(m->host.bls_short);
        if ((st = upload(prog.data(), prog.size() * sizeof(prog[0]), &m->d_bls_prog))) return st;
    }
    if ((st = upload(m->host.bls_tables.data(), std::max<size_t>(m->host.bls_tables.size(), 1) * sizeof(double), (void **)&m->d_bls_tables))) return st;
    if ((st = upload(m->host.bl.data(), m->host.bl.size() * 4, (void **)&m->d_bl))) return st;
    {
        std::vector<int32_t> ge(m->host.gemm_edges.begin(), m->host.gemm_edges.end());
        if ((st = upload(ge.data(), ge.size() * 4, (void **)&m->d_gemm_edges))) return st;
    }
    CK(cudaMalloc(&m->d_bad, sizeof(int)));
    CK(cudaMemset(m->d_bad, 0, sizeof(int)));
    if (!getenv("PCSF_LEGACY_STREAM")) {
        CK(cudaStreamCreateWithFlags(&m->own_stream, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&m->copy_stream, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&m->h2d_stream, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&m->ev_chunk, cudaEventDisableTiming));
    }
    CK(cudaMalloc(&m->d_nuniq, sizeof(uint32_t) * MAX_CHUNKS));
    for (auto &e : m->ev) CK(cudaEventCreate(&e));
    m->prune_nwarp = PR_MAX_NWARP;
    if (const char *e = getenv("PCSF_PRUNE_NWARP")) m->prune_nwarp = std::max(1, std::min(PR_MAX_NWARP, atoi(e)));
    while (m->prune_nwarp > 4 &&
           prune_smem_bytes(m->host.nl, (int)m->host.program.size(), m->host.max_stack, m->prune_nwarp) > 227 * 1024)
        m->prune_nwarp -= 4;
    m->prune_smem = prune_smem_bytes(m->host.nl, (int)m->host.program.size(), m->host.max_stack, m->prune_nwarp);
    if (m->prune_smem > 227 * 1024) {
        return fail(PCSF_ERR_UNSUPPORTED, "tree needs more shared memory than one SM has (stack depth " +
                                              std::to_string(m->host.max_stack) + ")");
    }
    CK(cudaFuncSetAttribute(prune_kernel<false>(m->host.nl), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)m->prune_smem));
    CK(cudaFuncSetAttribute(prune_kernel<true>(m->host.nl), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)m->prune_smem));
    CK(cudaFuncSetAttribute(m->host.nl <= SMALL_TREE_MAX_LEAVES ? (const void *)k_bls<2> : (const void *)k_bls<8>,
                            cudaFuncAttributeMaxDynamicSharedMemorySize, std::max(1, m->host.bls_short_depth) * BLS_THREADS * BLS_COLS * 8));
    guard.m = nullptr;
    *out = m;
    return PCSF_OK;
}

extern "C" void pcsf_model_destroy(pcsf_model *m) {
    if (!m) return;
    cudaSetDevice(m->device);
    for (int w = 0; w < 2; ++w) {
        cudaFree(m->d_pstream[w]); cudaFree(m->d_leafPT[w]); cudaFree(m->d_rowtab_tc5[w]); cudaFree(m->d_pstream_tc5[w]); cudaFree(m->d_pi[w]); cudaFree(m->d_logpi[w]);
        cudaFree(m->d_eig[w]);
    }
    cudaFree(m->d_program); cudaFree(m->d_bls_prog); cudaFree(m->d_bls_tables); cudaFree(m->d_bl); cudaFree(m->d_gemm_edges);
    cudaFree(m->d_bad); cudaFree(m->d_nuniq); cudaFree(m->d_tc5_steps); cudaFree(m->d_tc5_scratch); cudaFree(m->d_tc5_srcs);
    if (m->h_msa) cudaFreeHost(m->h_msa);
    if (m->own_stream) cudaStreamDestroy(m->own_stream);
    if (m->copy_stream) cudaStreamDestroy(m->copy_stream);
    if (m->h2d_stream) cudaStreamDestroy(m->h2d_stream);
    for (cudaEvent_t e : m->ev_h2d) cudaEventDestroy(e);
    if (m->ev_chunk) cudaEventDestroy(m->ev_chunk);
    DevBuf *bufs[] = {&m->codes, &m->klo, &m->khi, &m->slot, &m->flag, &m->uniq, &m->pidx, &m->table,
                      &m->bsums, &m->logz, &m->anc, &m->io_in, &m->io_out, &m->perwin, &m->mle, &m->tc5_ids,
                      &m->rg_units, &m->rg_regions, &m->rg_win};
    for (DevBuf *b : bufs) b->release();
    for (auto &e : m->ev) if (e) cudaEventDestroy(e);
    delete m;
}

extern "C" pcsf_status pcsf_score_msa_stats(const pcsf_model *m, pcsf_msa_stats *stats) {
    if (!m || !stats) return fail(PCSF_ERR_INVALID, "pcsf_score_msa_stats: null argument");
    const MleStats &s = m->msa_stats;
    *stats = pcsf_msa_stats{s.alignments, s.evaluations, s.rounds, s.slots, s.ms_step, s.ms_plan, s.ms_expm, s.ms_prune};
    return PCSF_OK;
}

extern "C" pcsf_status pcsf_model_get(const pcsf_model *m, int which, double *lambda, double *pi, double *P) {
    if (!m || which < 0 || which > 1) return fail(PCSF_ERR_INVALID, "pcsf_model_get: bad argument");
    const EcmHost &e = m->host.ecm[which];
    if (lambda) memcpy(lambda, e.lambda, 64 * 8);
    if (pi) memcpy(pi, e.pi, 64 * 8);
    if (P) memcpy(P, e.P.data(), e.P.size() * 8);
    return PCSF_OK;
}

extern "C" pcsf_status pcsf_set_chunk_columns(pcsf_model *m, int64_t columns) {
    if (!m || columns < 0) return fail(PCSF_ERR_INVALID, "pcsf_set_chunk_columns: bad argument");
    if (columns == 0) columns = (int64_t)1 << 21;
    if (columns > ((int64_t)1 << 23)) columns = (int64_t)1 << 23;   // window ids are 32-bit, scan is 2-level
    m->chunk_cols = columns;
    return PCSF_OK;
}

extern "C" pcsf_status pcsf_set_timing(pcsf_model *m, int enabled) {
    if (!m) return fail(PCSF_ERR_INVALID, "null model");
    m->timing = enabled != 0;
    return PCSF_OK;
}

static inline uint32_t next_pow2(uint64_t x) {
    uint64_t p = 1;
    while (p < x) p <<= 1;
    return (uint32_t)p;
}

// dedup + prune for one window space of `nwin` local windows; results land in m->pidx (pattern id per
// window), m->logz / m->anc (per pattern); *d_nuniq_slot receives the pattern count.
static pcsf_status dedup_and_prune(pcsf_model *m, const WinSpace &ws, uint32_t nwin, bool dedup, bool want_anc, int prec /* 0 FP64 DMMA, 2 tcgen05 */,
                                   uint32_t *d_nuniq_slot, uint32_t *d_pattern_out, int64_t out_base,
                                   cudaStream_t st, float *ms_hash, float *ms_dedup, float *ms_prune) {
    NvtxRange nvtx_("pcsf: keys + dedup + prune");
    const int TB = 256;
    const uint32_t nblk = (nwin + TB - 1) / TB;
    CK(m->uniq.reserve((size_t)nwin * 4));
    CK(m->pidx.reserve((size_t)nwin * 4));
    CK(m->logz.reserve((size_t)nwin * 16));
    if (want_anc) CK(m->anc.reserve((size_t)nwin * 16));
    if (m->timing) CK(cudaEventRecord(m->ev[0], st));
    if (dedup) {
        CK(m->klo.reserve((size_t)nwin * 8));
        CK(m->khi.reserve((size_t)nwin * 8));
        if (ws.mode == 0) {
            const int64_t ncols = nwin / 2;
            m->launches++;
            if ((ws.c0 & 3) == 0 && (ws.ld & 3) == 0 && (reinterpret_cast<uintptr_t>(ws.codes) & 3) == 0) {
                const int64_t nthr = (ncols + 3) / 4;
                k_keys_tracks<<<(unsigned)((nthr + TB - 1) / TB), TB, 0, st>>>(ws, ncols, m->klo.as<ulonglong2>(), m->khi.as<ulonglong2>());
            } else {
                k_keys_tracks_unaligned<<<(unsigned)((ncols + TB - 1) / TB), TB, 0, st>>>(ws, ncols, m->klo.as<ulonglong2>(), m->khi.as<ulonglong2>());
            }
        } else {
            m->launches++; k_keys_list<<<nblk, TB, 0, st>>>(ws, nwin, m->klo.as<uint64_t>(), m->khi.as<uint64_t>());
        }
        CK(cudaGetLastError());
        if (m->timing) CK(cudaEventRecord(m->ev[1], st));
        const uint32_t T = next_pow2((uint64_t)nwin * 2 < 1024 ? 1024 : (uint64_t)nwin * 2);
        const uint32_t nsb = (nwin + SCAN_BLOCK - 1) / SCAN_BLOCK;
        CK(m->table.reserve((size_t)T * 4));
        CK(m->slot.reserve((size_t)nwin * 4));
        CK(m->flag.reserve((size_t)nwin * 4));
        CK(m->bsums.reserve((size_t)(nsb + 1) * 4));
        CK(cudaMemsetAsync(m->table.p, 0xFF, (size_t)T * 4, st));
        m->launches += 5; k_insert<<<nblk, TB, 0, st>>>(ws, m->klo.as<uint64_t>(), m->khi.as<uint64_t>(), nwin, m->table.as<uint32_t>(), T - 1,
                                      m->slot.as<uint32_t>());
        k_resolve<<<nblk, TB, 0, st>>>(nwin, m->slot.as<uint32_t>(), m->table.as<uint32_t>(), m->flag.as<uint32_t>());
        k_scan_blocks<<<nsb, SCAN_THREADS, 0, st>>>(m->flag.as<uint32_t>(), nwin, m->bsums.as<uint32_t>());
        k_scan_sums<<<1, 1024, 0, st>>>(m->bsums.as<uint32_t>(), nsb, d_nuniq_slot);
        k_finalize<<<nblk, TB, 0, st>>>(nwin, m->slot.as<uint32_t>(), m->flag.as<uint32_t>(), m->bsums.as<uint32_t>(),
                                        m->uniq.as<uint32_t>(), m->pidx.as<uint32_t>(), d_pattern_out, out_base);
        CK(cudaGetLastError());
    } else {
        if (m->timing) CK(cudaEventRecord(m->ev[1], st));
        m->launches++; k_identity<<<nblk, TB, 0, st>>>(nwin, m->uniq.as<uint32_t>(), m->pidx.as<uint32_t>(), d_nuniq_slot, d_pattern_out,
                                        out_base);
        CK(cudaGetLastError());
    }
    if (m->timing) CK(cudaEventRecord(m->ev[2], st));
    if (prec == 2) {
        // codon ids of the unique windows in the producers' layout, one 2 x nl x 128-byte block per pair of tiles
        const uint32_t mp = (nwin + 255) / 256;
        CK(m->tc5_ids.reserve((size_t)mp * 2 * m->host.nl * 128));
        m->launches++;
        k_tc5_ids<<<std::min<uint32_t>(mp, (uint32_t)m->sm_count * 16), 128, 0, st>>>(ws, m->uniq.as<uint32_t>(), d_nuniq_slot, m->tc5_ids.as<uint8_t>());
        CK(cudaGetLastError());
        PruneTc5Args ta{};
        ta.ids = m->tc5_ids.as<uint8_t>();
        ta.nl = m->host.nl;
        ta.nids = m->tc5_nids;
        ta.n_unique = d_nuniq_slot;
        ta.steps = m->d_tc5_steps;
        ta.n_steps = (int)m->host.tc5_steps.size();
        ta.max_stack = m->host.tc5_max_stack;
        ta.n_src = (int)m->host.tc5_srcs.size();
        ta.srcs = m->d_tc5_srcs;
        ta.nstage = m->tc5_nstage;
        ta.scratch = m->d_tc5_scratch;
        for (int w = 0; w < 2; ++w) {
            ta.pstream[w] = m->d_pstream_tc5[w];
            ta.rowtab[w] = m->d_rowtab_tc5[w];
            ta.pi[w] = m->d_pi[w];
            ta.logz[w] = m->logz.as<double>() + (size_t)w * nwin;
        }
        const unsigned gridt = std::min<uint32_t>((uint32_t)m->sm_count, std::max<uint32_t>(1u, mp));
        m->launches++;
        k_prune_tc5<<<gridt, T5_THREADS, m->prune_tc5_smem, st>>>(ta);
        CK(cudaGetLastError());
        if (m->timing) {
            CK(cudaEventRecord(m->ev[3], st));
            CK(cudaEventSynchronize(m->ev[3]));
            float t;
            CK(cudaEventElapsedTime(&t, m->ev[0], m->ev[1])); *ms_hash += t;
            CK(cudaEventElapsedTime(&t, m->ev[1], m->ev[2])); *ms_dedup += t;
            CK(cudaEventElapsedTime(&t, m->ev[2], m->ev[3])); *ms_prune += t;
        }
        return PCSF_OK;
    }
    PruneArgs pa{};
    pa.ws = ws;
    pa.uniq = m->uniq.as<uint32_t>();
    pa.n_unique = d_nuniq_slot;
    pa.program = m->d_program;
    pa.n_ops = (int)m->host.program.size();
    pa.n_gemm = (int)m->host.gemm_edges.size();
    pa.max_stack = m->host.max_stack;
    pa.stagger_ns = m->stagger_ns;
    pa.nwarp = m->prune_nwarp;
    for (int w = 0; w < 2; ++w) {
        pa.pstream[w] = m->d_pstream[w];
        pa.leafPT[w] = m->d_leafPT[w];
        pa.pi[w] = m->d_pi[w];
        pa.logpi[w] = m->d_logpi[w];
        pa.logz[w] = m->logz.as<double>() + (size_t)w * nwin;
        pa.anc[w] = want_anc ? m->anc.as<double>() + (size_t)w * nwin : nullptr;
    }
    const uint32_t tile_w = (uint32_t)m->prune_nwarp * 8;
    const uint32_t max_tiles = (nwin + tile_w - 1) / tile_w;
    const unsigned grid = std::min<uint32_t>((uint32_t)m->sm_count, std::max<uint32_t>(1u, max_tiles));
    m->launches++; prune_kernel<false>(m->host.nl)<<<grid, (m->prune_nwarp + 1) * 32, m->prune_smem, st>>>(pa);
    CK(cudaGetLastError());
    if (m->timing) {
        CK(cudaEventRecord(m->ev[3], st));
        CK(cudaEventSynchronize(m->ev[3]));
        float t;
        CK(cudaEventElapsedTime(&t, m->ev[0], m->ev[1])); *ms_hash += t;
        CK(cudaEventElapsedTime(&t, m->ev[1], m->ev[2])); *ms_dedup += t;
        CK(cudaEventElapsedTime(&t, m->ev[2], m->ev[3])); *ms_prune += t;
    }
    return PCSF_OK;
}

static pcsf_status run_pack(pcsf_model *m, const uint8_t *d_seqs, int64_t L, int64_t ld, cudaStream_t st) {
    const int nl = m->host.nl;
    m->codes_ld = ((L + 16 + 15) / 16) * 16;
    CK(m->codes.reserve((size_t)m->codes_ld * nl));
    CK(cudaMemsetAsync(m->d_bad, 0, sizeof(int), st));
    const int64_t nvec = m->codes_ld / 16;
    // a few fat blocks per SM with grid-stride loops (four vectors in flight per thread) instead of one block per 4 KB of a row
    dim3 grid((unsigned)std::max<int64_t>(1, std::min<int64_t>((nvec + 255) / 256, ((int64_t)m->sm_count * 16 + nl - 1) / nl)), nl);
    NvtxRange nvtx_("pcsf: pack");
    m->launches++; k_pack<<<grid, 256, 0, st>>>(d_seqs, L, ld, nl, m->codes.as<uint8_t>(), m->codes_ld, m->codes_ld, m->d_bad);
    CK(cudaGetLastError());
    return PCSF_OK;
}

// k_bls over columns [s0, s0 + n) of m->codes, with the mask width of the tree
static pcsf_status launch_bls(pcsf_model *m, int64_t s0, int64_t n, int raw, double *d_out, cudaStream_t st) {
    const size_t sh = (size_t)std::max(1, m->host.bls_short_depth) * BLS_THREADS * BLS_COLS * 8;
    const unsigned grid = (unsigned)((n + BLS_THREADS * BLS_COLS - 1) / (BLS_THREADS * BLS_COLS));
    m->launches++;
    if (m->host.nl <= SMALL_TREE_MAX_LEAVES)
        k_bls<2><<<grid, BLS_THREADS, sh, st>>>(m->codes.as<uint8_t>() + s0, m->codes_ld, m->host.nl, n,
                                                static_cast<const BlsInnerDev<2> *>(m->d_bls_prog), (int)m->host.bls_short.size(),
                                                m->host.bls_short_depth, m->d_bls_tables, m->host.bls_all, raw, d_out);
    else
        k_bls<8><<<grid, BLS_THREADS, sh, st>>>(m->codes.as<uint8_t>() + s0, m->codes_ld, m->host.nl, n,
                                                static_cast<const BlsInnerDev<8> *>(m->d_bls_prog), (int)m->host.bls_short.size(),
                                                m->host.bls_short_depth, m->d_bls_tables, m->host.bls_all, raw, d_out);
    CK(cudaGetLastError());
    return PCSF_OK;
}

static pcsf_status run_bls(pcsf_model *m, int64_t L, int raw, double *d_out, cudaStream_t st) {
    if (L <= 0) return PCSF_OK;
    NvtxRange nvtx_("pcsf: bls");
    return launch_bls(m, 0, L, raw, d_out, st);
}

// Columns [s0, s1) only (s0 a multiple of 16): the pieces of run_pack / run_bls for an input that arrives in segments.
static pcsf_status run_pack_segment(pcsf_model *m, const uint8_t *d_seqs, int64_t ld, int64_t s0, int64_t s1, bool last, cudaStream_t st) {
    const int nl = m->host.nl;
    const int64_t out_cols = last ? m->codes_ld - s0 : s1 - s0;
    dim3 grid((unsigned)std::min<int64_t>((out_cols / 16 + 255) / 256 + 1, 65535), nl);
    m->launches++; k_pack<<<grid, 256, 0, st>>>(d_seqs + s0, s1 - s0, ld, nl, m->codes.as<uint8_t>() + s0, m->codes_ld, out_cols, m->d_bad);
    CK(cudaGetLastError());
    return PCSF_OK;
}
static pcsf_status run_bls_segment(pcsf_model *m, int64_t s0, int64_t s1, double *d_out, cudaStream_t st) {
    if (s1 <= s0) return PCSF_OK;
    return launch_bls(m, s0, s1 - s0, 0, d_out + s0, st);
}

extern "C" pcsf_status pcsf_tracks_device(pcsf_model *m, const uint8_t *d_seqs, int64_t L, int64_t ld, uint32_t flags,
                                          double *d_plus, double *d_minus, double *d_bls, uint32_t *d_pattern_index,
                                          void *cuda_stream) {
    if (!m || L < 0 || ld < L || (L > 0 && !d_seqs)) return fail(PCSF_ERR_INVALID, "pcsf_tracks: bad argument");
    if ((flags & PCSF_TRACKS_SCORES) && L > 2 && (!d_plus || !d_minus)) return fail(PCSF_ERR_INVALID, "plus/minus required");
    if ((flags & PCSF_TRACKS_BLS) && L > 0 && !d_bls) return fail(PCSF_ERR_INVALID, "bls required");
    if ((flags & PCSF_TRACKS_TC5) && m->host.nl > SMALL_TREE_MAX_LEAVES)
        return fail(PCSF_ERR_UNSUPPORTED, "the tcgen05 path (PCSF_TRACKS_TC5) does not support trees of more than " +
                                              std::to_string(SMALL_TREE_MAX_LEAVES) + " leaves (this one has " + std::to_string(m->host.nl) +
                                              "); the FP64 path scores them");
    if ((flags & PCSF_TRACKS_TC5) && m->prune_tc5_smem > 227 * 1024)
        return fail(PCSF_ERR_UNSUPPORTED, "tree too large for the tcgen05 path's shared-memory budget");
    CK(cudaSetDevice(m->device));
    cudaStream_t st = (cudaStream_t)cuda_stream;
    m->last = pcsf_tracks_stats{};
    m->last_nwin = 0;
    m->last_chunks = 0;
    m->launches = 0;
    if (L == 0) return PCSF_OK;
    pcsf_status rc;
    // Segmented input (pcsf_tracks with two or more dedup chunks): d_seqs is the device staging buffer that the h2d stream fills
    // segment by segment from the caller's host matrix; every chunk packs (and BLS-scores) its own segment right before it is keyed
    // and pruned, so the copy of segment c+1 runs under the pruning of chunk c.  Segment c = columns [s0, s1): s1 = the chunk's last
    // window + 2 columns of halo, rounded up to 16; the last one ends at L and also writes the padding.
    const bool seg = m->h_seqs != nullptr;
    const int64_t W_all = L - 2;
    const int64_t nchunks_all = W_all > 0 ? (W_all + m->chunk_cols - 1) / m->chunk_cols : 0;
    auto seg_end = [&](int64_t c) {
        if (c + 1 >= nchunks_all) return L;
        const int64_t c1 = std::min(W_all, (c + 1) * m->chunk_cols);
        return std::min<int64_t>(L, ((c1 + 2 + 15) / 16) * 16);
    };
    NvtxRange nvtx_("pcsf_tracks_device");
    if (seg) {
        NvtxRange nvtx_h2d("pcsf: H2D segments");
        m->codes_ld = ((L + 16 + 15) / 16) * 16;
        CK(m->codes.reserve((size_t)m->codes_ld * m->host.nl));
        CK(cudaMemsetAsync(m->d_bad, 0, sizeof(int), st));
        while ((int64_t)m->ev_h2d.size() < nchunks_all) {
            cudaEvent_t e;
            CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            m->ev_h2d.push_back(e);
        }
        for (int64_t c = 0; c < nchunks_all; ++c) {
            const int64_t s0 = c == 0 ? 0 : seg_end(c - 1), s1 = seg_end(c);
            if (s1 > s0)
                CK(cudaMemcpy2DAsync(const_cast<uint8_t *>(d_seqs) + s0, (size_t)ld, m->h_seqs + s0, (size_t)m->h_ld, (size_t)(s1 - s0),
                                     (size_t)m->host.nl, cudaMemcpyHostToDevice, m->h2d_stream));
            CK(cudaEventRecord(m->ev_h2d[c], m->h2d_stream));
        }
    }
    if (m->timing) CK(cudaEventRecord(m->ev[4], st));
    if (!seg && (rc = run_pack(m, d_seqs, L, ld, st))) return rc;
    if (m->timing) CK(cudaEventRecord(m->ev[5], st));
    if ((flags & PCSF_TRACKS_BLS) && !seg) {
        if ((rc = run_bls(m, L, 0, d_bls, st))) return rc;
        if (m->h_bls && m->copy_stream) {          // host-buffer call: the BLS vector goes home under the pruning
            CK(cudaEventRecord(m->ev_chunk, st));
            CK(cudaStreamWaitEvent(m->copy_stream, m->ev_chunk, 0));
            CK(cudaMemcpyAsync(m->h_bls, d_bls, (size_t)L * 8, cudaMemcpyDeviceToHost, m->copy_stream));
        }
    }
    if (m->timing) {
        CK(cudaEventRecord(m->ev[6], st));
        CK(cudaEventSynchronize(m->ev[6]));
        CK(cudaEventElapsedTime(&m->last.ms_pack, m->ev[4], m->ev[5]));
        CK(cudaEventElapsedTime(&m->last.ms_bls, m->ev[5], m->ev[6]));
    }
    const int64_t W = L - 2;
    if ((flags & PCSF_TRACKS_SCORES) && W > 0) {
        const int64_t nchunks = (W + m->chunk_cols - 1) / m->chunk_cols;
        if (nchunks > MAX_CHUNKS) return fail(PCSF_ERR_INVALID, "too many chunks; raise pcsf_set_chunk_columns");
        for (int64_t c = 0; c < nchunks; ++c) {
            const int64_t c0 = c * m->chunk_cols, c1 = std::min(W, c0 + m->chunk_cols);
            const uint32_t nwin = (uint32_t)(2 * (c1 - c0));
            if (seg) {
                const int64_t s0 = c == 0 ? 0 : seg_end(c - 1), s1 = seg_end(c);
                CK(cudaStreamWaitEvent(st, m->ev_h2d[c], 0));
                // An empty segment (s1 == s0: the previous chunk's halo already reached L) has nothing to pack: the segment that
                // reached L ran with last = true and wrote the padding columns.  Packing again from s0 = L would start at an
                // address that is not 16-byte aligned whenever L % 16 != 0 and run into the next species' row.
                if (s1 > s0) {
                    if ((rc = run_pack_segment(m, d_seqs, ld, s0, s1, s1 == L, st))) return rc;
                    if (flags & PCSF_TRACKS_BLS) {
                        if ((rc = run_bls_segment(m, s0, s1, d_bls, st))) return rc;
                        if (m->h_bls) {
                            CK(cudaEventRecord(m->ev_chunk, st));
                            CK(cudaStreamWaitEvent(m->copy_stream, m->ev_chunk, 0));
                            CK(cudaMemcpyAsync(m->h_bls + s0, d_bls + s0, (size_t)(s1 - s0) * 8, cudaMemcpyDeviceToHost, m->copy_stream));
                        }
                    }
                }
            }
            WinSpace ws{m->codes.as<uint8_t>(), m->codes_ld, m->host.nl, 0, c0, nullptr};
            if ((rc = dedup_and_prune(m, ws, nwin, !(flags & PCSF_TRACKS_NO_DEDUP), false, (flags & PCSF_TRACKS_TC5) ? 2 : 0, m->d_nuniq + c, d_pattern_index,
                                      2 * c0, st, &m->last.ms_hash, &m->last.ms_dedup, &m->last.ms_prune)))
                return rc;
            if (m->timing) CK(cudaEventRecord(m->ev[0], st));
            NvtxRange nvtx_sc("pcsf: scatter + D2H");
            m->launches++; k_scatter_tracks<<<(nwin + 255) / 256, 256, 0, st>>>(nwin, m->pidx.as<uint32_t>(), m->logz.as<double>(),
                                                                 m->logz.as<double>() + nwin, c0, d_plus, d_minus);
            CK(cudaGetLastError());
            if (m->timing) {
                CK(cudaEventRecord(m->ev[1], st));
                CK(cudaEventSynchronize(m->ev[1]));
                float t;
                CK(cudaEventElapsedTime(&t, m->ev[0], m->ev[1]));
                m->last.ms_scatter += t;
            }
            if (m->h_plus && m->copy_stream) {          // host-buffer call: this chunk's scores go home while the next one is pruned
                CK(cudaEventRecord(m->ev_chunk, st));
                CK(cudaStreamWaitEvent(m->copy_stream, m->ev_chunk, 0));
                CK(cudaMemcpyAsync(m->h_plus + c0, d_plus + c0, (size_t)(c1 - c0) * 8, cudaMemcpyDeviceToHost, m->copy_stream));
                CK(cudaMemcpyAsync(m->h_minus + c0, d_minus + c0, (size_t)(c1 - c0) * 8, cudaMemcpyDeviceToHost, m->copy_stream));
                if (m->h_pat && d_pattern_index)
                    CK(cudaMemcpyAsync(m->h_pat + 2 * c0, d_pattern_index + 2 * c0, (size_t)(c1 - c0) * 8, cudaMemcpyDeviceToHost, m->copy_stream));
            }
        }
        m->last_chunks = (int)nchunks;
        m->last_nwin = 2 * W;
    }
    return PCSF_OK;
}

extern "C" pcsf_status pcsf_tracks_device_finish(pcsf_model *m, void *cuda_stream, pcsf_tracks_stats *stats) {
    if (!m) return fail(PCSF_ERR_INVALID, "null model");
    CK(cudaSetDevice(m->device));
    cudaStream_t st = (cudaStream_t)cuda_stream;
    int bad = 0;
    CK(cudaMemcpyAsync(&bad, m->d_bad, sizeof(int), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    m->last.n_windows = m->last_nwin;
    m->last.n_chunks = m->last_chunks;
    m->last.n_launches = m->launches;
    m->last.n_unique = 0;
    if (m->last_chunks > 0) {
        std::vector<uint32_t> nu(m->last_chunks);
        CK(cudaMemcpyAsync(nu.data(), m->d_nuniq, sizeof(uint32_t) * m->last_chunks, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        for (uint32_t v : nu) m->last.n_unique += v;
    }
    if (stats) *stats = m->last;
    if (bad) return fail(PCSF_ERR_BAD_CHAR, "alignment contains a character outside ACGTacgt.-Nn (reference: exit(37))");
    return PCSF_OK;
}

extern "C" pcsf_status pcsf_tracks(pcsf_model *m, const uint8_t *seqs, int64_t L, int64_t ld, uint32_t flags, double *plus,
                                   double *minus, double *bls, uint32_t *pattern_index, pcsf_tracks_stats *stats) {
    if (!m || L < 0 || ld < L || (L > 0 && !seqs)) return fail(PCSF_ERR_INVALID, "pcsf_tracks: bad argument");
    NvtxRange nvtx_("pcsf_tracks (host buffers)");
    CK(cudaSetDevice(m->device));
    if (stats) *stats = pcsf_tracks_stats{};
    if (L == 0) return PCSF_OK;
    const int nl = m->host.nl;
    const int64_t W = std::max<int64_t>(L - 2, 0);
    const int64_t ldd = ((L + 15) / 16) * 16;
    CK(m->io_in.reserve((size_t)ldd * nl));
    const size_t out_bytes = (size_t)W * 16 + (size_t)L * 8 + (pattern_index ? (size_t)W * 8 : 0) + 64;
    CK(m->io_out.reserve(out_bytes));
    // everything on the handle's own non-blocking stream: the copies of one handle overlap the kernels of another on the same GPU, and
    // with pinned host buffers (pcsf_alloc_pinned) they are plain DMA
    cudaStream_t st = m->own_stream;
    const int64_t nchunks = W > 0 ? (W + m->chunk_cols - 1) / m->chunk_cols : 0;
    const bool segmented = m->copy_stream != nullptr && !m->timing && (flags & PCSF_TRACKS_SCORES) && nchunks >= 2 && nchunks <= MAX_CHUNKS;
    if (!segmented) CK(cudaMemcpy2DAsync(m->io_in.p, (size_t)ldd, seqs, (size_t)ld, (size_t)L, (size_t)nl, cudaMemcpyHostToDevice, st));
    m->h_seqs = segmented ? seqs : nullptr;
    m->h_ld = ld;
    double *d_plus = m->io_out.as<double>(), *d_minus = d_plus + W, *d_bls = d_minus + W;
    uint32_t *d_pat = pattern_index ? reinterpret_cast<uint32_t *>(d_bls + L) : nullptr;
    const bool piped = m->copy_stream != nullptr;
    m->h_plus = ((flags & PCSF_TRACKS_SCORES) && W > 0 && piped) ? plus : nullptr;
    m->h_minus = m->h_plus ? minus : nullptr;
    m->h_pat = m->h_plus ? pattern_index : nullptr;
    m->h_bls = ((flags & PCSF_TRACKS_BLS) && piped) ? bls : nullptr;
    pcsf_status rc = pcsf_tracks_device(m, m->io_in.as<uint8_t>(), L, ldd, flags, d_plus, d_minus, d_bls, d_pat, st);
    m->h_plus = m->h_minus = m->h_bls = nullptr;
    m->h_pat = nullptr;
    m->h_seqs = nullptr;
    if (rc) { if (piped) { cudaStreamSynchronize(m->h2d_stream); cudaStreamSynchronize(m->copy_stream); } return rc; }
    if (!piped) {
        if ((flags & PCSF_TRACKS_SCORES) && W > 0) {
            CK(cudaMemcpyAsync(plus, d_plus, (size_t)W * 8, cudaMemcpyDeviceToHost, st));
            CK(cudaMemcpyAsync(minus, d_minus, (size_t)W * 8, cudaMemcpyDeviceToHost, st));
            if (pattern_index) CK(cudaMemcpyAsync(pattern_index, d_pat, (size_t)W * 8, cudaMemcpyDeviceToHost, st));
        }
        if (flags & PCSF_TRACKS_BLS) CK(cudaMemcpyAsync(bls, d_bls, (size_t)L * 8, cudaMemcpyDeviceToHost, st));
    }
    rc = pcsf_tracks_device_finish(m, st, stats);
    if (piped && cudaStreamSynchronize(m->copy_stream) != cudaSuccess && rc == PCSF_OK) rc = fail(PCSF_ERR_CUDA, "copy stream failed");
    return rc;
}

extern "C" void *pcsf_alloc_pinned(size_t bytes) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) { g_err = "cudaHostAlloc failed"; return nullptr; }
    return p;
}
extern "C" void pcsf_free_pinned(void *p) { if (p) cudaFreeHost(p); }
extern "C" pcsf_status pcsf_register_host(void *p, size_t bytes) {
    if (!p || !bytes) return fail(PCSF_ERR_INVALID, "pcsf_register_host: null argument");
    if (cudaHostRegister(p, bytes, cudaHostRegisterPortable) != cudaSuccess) { cudaGetLastError(); return fail(PCSF_ERR_CUDA, "cudaHostRegister failed"); }
    return PCSF_OK;
}
extern "C" pcsf_status pcsf_unregister_host(void *p) {
    if (!p) return PCSF_OK;
    if (cudaHostUnregister(p) != cudaSuccess) { cudaGetLastError(); return fail(PCSF_ERR_CUDA, "cudaHostUnregister failed"); }
    return PCSF_OK;
}
extern "C" int pcsf_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

// ---- score-msa -------------------------------------------------------------------------------------
// The batch side by side ([nl][Ltot], alignment i at col_start[i], two N pad columns behind each) in the handle's page-locked staging
// (allocated once, re-used by every call: plain DMA, no fresh 100 MB vector per call), copied to the device and packed into m->codes;
// only the pad columns and the tail are filled with N.
static pcsf_status stage_and_pack(pcsf_model *m, int32_t n_aln, const uint8_t *seqs, const int64_t *offset, const int64_t *len,
                                  const int64_t *col_start, int64_t Ltot, cudaStream_t st) {
    const int nl = m->host.nl;
    const int64_t ldd = ((Ltot + 15) / 16) * 16;
    const size_t h_bytes = (size_t)ldd * nl;
    if (h_bytes > m->h_msa_cap) {
        if (m->h_msa) cudaFreeHost(m->h_msa);
        m->h_msa = nullptr;
        m->h_msa_cap = h_bytes + h_bytes / 4 + 4096;
        CK(cudaHostAlloc(reinterpret_cast<void **>(&m->h_msa), m->h_msa_cap, cudaHostAllocPortable));
    }
    uint8_t *h = m->h_msa;
    for (int s = 0; s < nl; ++s) {
        uint8_t *row = h + (size_t)s * ldd;
        for (int i = 0; i < n_aln; ++i) {
            memcpy(row + col_start[i], seqs + offset[i] + (size_t)s * len[i], (size_t)len[i]);
            row[col_start[i] + len[i]] = 'N';
            row[col_start[i] + len[i] + 1] = 'N';
        }
        memset(row + Ltot, 'N', (size_t)(ldd - Ltot));
    }
    CK(m->io_in.reserve(h_bytes));
    CK(cudaMemcpyAsync(m->io_in.p, h, h_bytes, cudaMemcpyHostToDevice, st));
    return run_pack(m, m->io_in.as<uint8_t>(), Ltot, ldd, st);
}

// One scoring path for reading frames / ORFs (pcsf_score_regions); pcsf_score_msa is its frame +1 as is, one region per alignment.
static_assert(sizeof(pcsf_region) == 48, "pcsf_region layout is part of the ABI");

// What score_regions_core leaves on the device for its caller (in m->rg_units / m->rg_regions).
struct ScoredRegions {
    int64_t nreg = 0;
    RegionUnits U{};
    RegionList R{};
    const int64_t *off_r = nullptr;                           // [n_aln * frames + 1]: first region of each (alignment, frame) unit
    float *phylo = nullptr, *anc = nullptr, *bls = nullptr;   // [nreg]; phylo if fit, anc / bls if asked for, else null
    pcsf_region *rec = nullptr;                               // room for max(nreg, n_aln) records
};

// The scoring path of both entry points: stage and pack the batch, enumerate its regions, score every region as an item of the
// dedup + prune (FIXED), MLE or OMEGA machinery, synchronise and check for bad characters.  fit = false skips the likelihoods and
// computes the BLS only.  ref_row may be null for PCSF_ORF_ASIS, which never reads it.
static pcsf_status score_regions_core(pcsf_model *m, pcsf_strategy strategy, int32_t n_aln, const uint8_t *seqs, const int64_t *offset,
                                      const int64_t *len, const int64_t *col_start, int64_t Ltot, const int32_t *ref_row, int32_t frames,
                                      pcsf_orf_mode orf, int32_t min_codons, bool fit, bool want_anc, bool want_bls, ScoredRegions *out) {
    const int nl = m->host.nl;
    cudaStream_t st = m->own_stream;
    pcsf_status rc;
    if ((rc = stage_and_pack(m, n_aln, seqs, offset, len, col_start, Ltot, st))) return rc;

    // per-unit buffers: col_start | len | ref_row | totals | n_reg | n_win | bsums x 2 | off_r | off_w
    const int64_t n_units = (int64_t)n_aln * frames;
    const uint32_t nsb = (uint32_t)((n_units + SCAN_BLOCK - 1) / SCAN_BLOCK);
    size_t o = 0;
    auto take = [&](size_t bytes) { const size_t r = o; o += (bytes + 255) / 256 * 256; return r; };
    const size_t o_cs = take((size_t)n_aln * 8), o_len = take((size_t)n_aln * 8), o_ref = take((size_t)n_aln * 4), o_tot = take(16),
                 o_nr = take((size_t)n_units * 4), o_nw = take((size_t)n_units * 4), o_br = take((size_t)(nsb + 1) * 4),
                 o_bw = take((size_t)(nsb + 1) * 4), o_or = take((size_t)(n_units + 1) * 8), o_ow = take((size_t)(n_units + 1) * 8);
    CK(m->rg_units.reserve(o));
    unsigned char *ub = m->rg_units.as<unsigned char>();
    CK(cudaMemcpyAsync(ub + o_cs, col_start, (size_t)n_aln * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(ub + o_len, len, (size_t)n_aln * 8, cudaMemcpyHostToDevice, st));
    if (ref_row) CK(cudaMemcpyAsync(ub + o_ref, ref_row, (size_t)n_aln * 4, cudaMemcpyHostToDevice, st));
    CK(cudaMemsetAsync(ub + o_tot, 0, 16, st));
    unsigned long long *d_tot = reinterpret_cast<unsigned long long *>(ub + o_tot);
    uint32_t *d_nr = reinterpret_cast<uint32_t *>(ub + o_nr), *d_nw = reinterpret_cast<uint32_t *>(ub + o_nw);
    uint32_t *d_br = reinterpret_cast<uint32_t *>(ub + o_br), *d_bw = reinterpret_cast<uint32_t *>(ub + o_bw);
    int64_t *d_or = reinterpret_cast<int64_t *>(ub + o_or), *d_ow = reinterpret_cast<int64_t *>(ub + o_ow);
    RegionUnits U{m->codes.as<uint8_t>(), m->codes_ld, n_aln, frames, (int)orf, min_codons, reinterpret_cast<const int64_t *>(ub + o_cs),
                  reinterpret_cast<const int64_t *>(ub + o_len), ref_row ? reinterpret_cast<const int32_t *>(ub + o_ref) : nullptr};
    const unsigned warp_blocks = (unsigned)((n_units * 32 + 255) / 256);
    {
        NvtxRange nvtx_e("pcsf: region enumeration");
        m->launches += 6;
        k_orf_count<<<warp_blocks, 256, 0, st>>>(U, n_units, d_nr, d_nw, d_tot);
        k_scan_blocks<<<nsb, SCAN_THREADS, 0, st>>>(d_nr, (uint32_t)n_units, d_br);
        k_scan_sums<<<1, 1024, 0, st>>>(d_br, nsb, d_br + nsb);
        k_scan_blocks<<<nsb, SCAN_THREADS, 0, st>>>(d_nw, (uint32_t)n_units, d_bw);
        k_scan_sums<<<1, 1024, 0, st>>>(d_bw, nsb, d_bw + nsb);
        k_unit_offsets<<<(unsigned)((n_units + 1 + 255) / 256), 256, 0, st>>>(n_units, d_nr, d_br, d_nw, d_bw, d_tot, d_or, d_ow);
        CK(cudaGetLastError());
    }
    unsigned long long tot[2] = {0, 0};
    CK(cudaMemcpyAsync(tot, d_tot, 16, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    // the 32-bit scans above are exact only below 2^32; the window lists (uint32 ids, int counts in the fits) need < 2^31
    if (tot[0] >= (1ull << 31) || tot[1] >= (1ull << 31)) return fail(PCSF_ERR_INVALID, "too many regions or region codons: split the call");
    const int64_t nreg = (int64_t)tot[0], nwin = (int64_t)tot[1];

    // per-region buffers: aln | fi | k0 | ncod | win_start | slen | phylo | anc | bls | records
    o = 0;
    const size_t nr1 = (size_t)std::max<int64_t>(nreg, 1);
    const size_t o_ra = take(nr1 * 4), o_rf = take(nr1 * 4), o_rk = take(nr1 * 8), o_rn = take(nr1 * 8), o_rw = take(nr1 * 8),
                 o_rl = take(nr1 * 8), o_ph = take(nr1 * 4), o_an = take(nr1 * 4), o_bl = take(nr1 * 4),
                 o_rec = take((size_t)std::max<int64_t>({nreg, n_aln, 1}) * sizeof(pcsf_region));
    CK(m->rg_regions.reserve(o));
    unsigned char *rb = m->rg_regions.as<unsigned char>();
    RegionList R{reinterpret_cast<int32_t *>(rb + o_ra), reinterpret_cast<int32_t *>(rb + o_rf), reinterpret_cast<int64_t *>(rb + o_rk),
                 reinterpret_cast<int64_t *>(rb + o_rn), reinterpret_cast<int64_t *>(rb + o_rw), reinterpret_cast<int64_t *>(rb + o_rl)};
    float *d_phylo = reinterpret_cast<float *>(rb + o_ph), *d_anc = reinterpret_cast<float *>(rb + o_an),
          *d_bls = reinterpret_cast<float *>(rb + o_bl);
    CK(m->rg_win.reserve((size_t)std::max<int64_t>(nwin, 1) * 5 + 16));
    uint32_t *d_woff = m->rg_win.as<uint32_t>();
    // only the minus frames (-1 -2 -3, in six-frame calls) have '-' windows: otherwise the window consumers read no strand at all
    uint8_t *d_wstr = frames == 6 ? m->rg_win.as<uint8_t>() + (size_t)std::max<int64_t>(nwin, 1) * 4 : nullptr;
    if (nreg > 0) {
        NvtxRange nvtx_w("pcsf: region windows");
        m->launches += 2;
        k_orf_emit<<<warp_blocks, 256, 0, st>>>(U, n_units, d_or, d_ow, R);
        k_region_windows<<<(unsigned)std::min<int64_t>((nreg * 32 + 255) / 256, (int64_t)m->sm_count * 32), 256, 0, st>>>(U, nreg, R, d_woff,
                                                                                                                           d_wstr);
        CK(cudaGetLastError());
    }
    double *d_blraw = nullptr;
    if (want_bls && nreg > 0) {
        CK(m->io_out.reserve((size_t)Ltot * 8 + 64));
        d_blraw = m->io_out.as<double>();
        if ((rc = run_bls(m, Ltot, 1, d_blraw, st))) return rc;
    }
    const unsigned rgrid = (unsigned)((nreg + 127) / 128);
    WinSpace ws{m->codes.as<uint8_t>(), m->codes_ld, nl, 1, 0, d_woff, d_wstr};
    if (nreg > 0 && fit && strategy == PCSF_STRATEGY_FIXED) {
        CK(m->perwin.reserve((size_t)std::max<int64_t>(nwin, 1) * 32));
        if (nwin > 0) {
            float t0 = 0, t1 = 0, t2 = 0;
            if ((rc = dedup_and_prune(m, ws, (uint32_t)nwin, true, want_anc, 0, m->d_nuniq, nullptr, 0, st, &t0, &t1, &t2))) return rc;
            k_scatter_list<<<(unsigned)((nwin + 255) / 256), 256, 0, st>>>(
                (uint32_t)nwin, m->pidx.as<uint32_t>(), m->logz.as<double>(), m->logz.as<double>() + nwin,
                want_anc ? m->anc.as<double>() : nullptr, want_anc ? m->anc.as<double>() + nwin : nullptr, m->perwin.as<double>());
            CK(cudaGetLastError());
        }
        k_region_sums<<<rgrid, 128, 0, st>>>(U, nreg, R, m->perwin.as<double>(), nwin, d_blraw, m->host.bls_all, d_phylo,
                                             want_anc ? d_anc : nullptr, want_bls ? d_bls : nullptr);
        CK(cudaGetLastError());
    } else if (nreg > 0) {
        if (fit && strategy == PCSF_STRATEGY_OMEGA) {
            OmegaBatch b{};
            b.n_aln = (int)nreg;
            b.d_win_start = R.win_start;
            b.d_len = R.slen;
            b.ws = ws;
            b.nwin = nwin;
            b.d_phylo = d_phylo;
            if ((rc = omega_run(m->host, b, m->d_bl, m->d_program, m->d_pi, m->d_logpi, m->mle, m->sm_count, m->prune_smem, m->prune_nwarp, st,
                                g_err, &m->launches)))
                return rc;
        } else if (fit) {
            MleBatch b{};
            b.n_aln = (int)nreg;
            b.d_win_start = R.win_start;
            b.d_len = R.slen;
            b.ws = ws;
            b.nwin = nwin;
            b.want_anc = want_anc;
            b.d_phylo = d_phylo;
            b.d_anc = want_anc ? d_anc : nullptr;
            if ((rc = mle_run(m->host, b, m->d_eig, m->d_bl, m->d_program, m->d_pi, m->d_logpi, m->mle, m->sm_count, m->prune_smem,
                              m->prune_nwarp, st, g_err, &m->launches, &m->msa_stats, m->timing)))
                return rc;
        }
        if (want_bls) {
            k_region_sums<<<rgrid, 128, 0, st>>>(U, nreg, R, nullptr, 0, d_blraw, m->host.bls_all, nullptr, nullptr, d_bls);
            CK(cudaGetLastError());
        }
    }
    CK(cudaStreamSynchronize(st));
    int bad = 0;
    CK(cudaMemcpy(&bad, m->d_bad, sizeof(int), cudaMemcpyDeviceToHost));
    if (bad) return fail(PCSF_ERR_BAD_CHAR, "alignment contains a character outside ACGTacgt.-Nn (reference: exit(37))");
    *out = ScoredRegions{nreg, U, R, d_or, fit ? d_phylo : nullptr, want_anc ? d_anc : nullptr, want_bls ? d_bls : nullptr,
                         reinterpret_cast<pcsf_region *>(rb + o_rec)};
    return PCSF_OK;
}

extern "C" pcsf_status pcsf_score_msa(pcsf_model *m, pcsf_strategy strategy, int32_t n_aln, const uint8_t *seqs,
                                      const int64_t *offset, const int64_t *len, float *phylo, float *anc, float *bls) {
    if (!m || n_aln < 0 || (n_aln > 0 && (!seqs || !offset || !len)))
        return fail(PCSF_ERR_INVALID, "pcsf_score_msa: bad argument");
    if (strategy != PCSF_STRATEGY_FIXED && strategy != PCSF_STRATEGY_MLE && strategy != PCSF_STRATEGY_OMEGA)
        return fail(PCSF_ERR_INVALID, "pcsf_score_msa: unknown strategy");
    NvtxRange nvtx_("pcsf_score_msa");
    CK(cudaSetDevice(m->device));
    if (n_aln == 0) return PCSF_OK;
    // concatenate the alignments along the columns into one [nl][Ltot] matrix (2 pad columns between them)
    std::vector<int64_t> col_start(n_aln);
    int64_t Ltot = 0, nwin = 0;
    for (int i = 0; i < n_aln; ++i) {
        if (len[i] < 0) return fail(PCSF_ERR_INVALID, "negative alignment length");
        col_start[i] = Ltot;
        Ltot += len[i] + 2; nwin += len[i] / 3;
    }
    if (Ltot >= ((int64_t)1 << 32) || nwin >= ((int64_t)1 << 31))
        return fail(PCSF_ERR_INVALID, "batch too large: split the call");
    // Frame +1 as is: region i is alignment i.  With nothing but the branch length score asked for, the reference does not call run()
    // at all (score_msa.hpp:112), whatever the strategy — no fit, and no way for a failing fit to turn the batch into an error.
    ScoredRegions r;
    pcsf_status rc = score_regions_core(m, strategy, n_aln, seqs, offset, len, col_start.data(), Ltot, nullptr, 1, PCSF_ORF_ASIS, 1,
                                        phylo || anc, anc && strategy != PCSF_STRATEGY_OMEGA, bls != nullptr, &r);
    if (rc) return rc;
    if (phylo) CK(cudaMemcpy(phylo, r.phylo, (size_t)n_aln * 4, cudaMemcpyDeviceToHost));
    if (anc && strategy == PCSF_STRATEGY_OMEGA) { for (int i = 0; i < n_aln; ++i) anc[i] = nanf(""); }
    else if (anc) CK(cudaMemcpy(anc, r.anc, (size_t)n_aln * 4, cudaMemcpyDeviceToHost));
    if (bls) CK(cudaMemcpy(bls, r.bls, (size_t)n_aln * 4, cudaMemcpyDeviceToHost));
    return PCSF_OK;
}

extern "C" pcsf_status pcsf_score_regions(pcsf_model *m, pcsf_strategy strategy, int32_t n_aln, const uint8_t *seqs, const int64_t *offset,
                                          const int64_t *len, const int32_t *ref_row, int32_t frames, pcsf_orf_mode orf, int32_t min_codons,
                                          int32_t best_only, int32_t want_anc, int32_t want_bls, int64_t *n_regions) {
    if (!m || !n_regions || n_aln < 0 || (n_aln > 0 && (!seqs || !offset || !len || !ref_row)))
        return fail(PCSF_ERR_INVALID, "pcsf_score_regions: bad argument");
    *n_regions = 0;
    m->regions.clear();
    if (strategy != PCSF_STRATEGY_FIXED && strategy != PCSF_STRATEGY_MLE && strategy != PCSF_STRATEGY_OMEGA)
        return fail(PCSF_ERR_INVALID, "pcsf_score_regions: unknown strategy");
    if (frames != 1 && frames != 3 && frames != 6) return fail(PCSF_ERR_INVALID, "pcsf_score_regions: frames must be 1, 3 or 6");
    if (orf != PCSF_ORF_ASIS && orf != PCSF_ORF_STOPSTOP && orf != PCSF_ORF_ATGSTOP)
        return fail(PCSF_ERR_INVALID, "pcsf_score_regions: unknown ORF mode");
    if (min_codons < 1) return fail(PCSF_ERR_INVALID, "pcsf_score_regions: min_codons must be >= 1");
    if (want_anc && strategy == PCSF_STRATEGY_OMEGA)
        return fail(PCSF_ERR_INVALID, "pcsf_score_regions: OMEGA has no ancestral score");
    const int nl = m->host.nl;
    std::vector<int64_t> col_start(n_aln);
    int64_t Ltot = 0;
    for (int i = 0; i < n_aln; ++i) {
        if (len[i] < 0) return fail(PCSF_ERR_INVALID, "negative alignment length");
        if (ref_row[i] < 0 || ref_row[i] >= nl) return fail(PCSF_ERR_INVALID, "pcsf_score_regions: ref_row out of range");
        col_start[i] = Ltot;
        Ltot += len[i] + 2;
    }
    const int64_t n_units = (int64_t)n_aln * frames;
    if (Ltot >= ((int64_t)1 << 32) || n_units >= ((int64_t)1 << 31)) return fail(PCSF_ERR_INVALID, "batch too large: split the call");
    NvtxRange nvtx_("pcsf_score_regions");
    CK(cudaSetDevice(m->device));
    if (n_aln == 0) return PCSF_OK;
    ScoredRegions r;
    pcsf_status rc = score_regions_core(m, strategy, n_aln, seqs, offset, len, col_start.data(), Ltot, ref_row, frames, orf, min_codons,
                                        true, want_anc != 0, want_bls != 0, &r);
    if (rc) return rc;
    cudaStream_t st = m->own_stream;
    const int64_t n_out = best_only ? n_aln : r.nreg;
    if (best_only) {
        k_best_region<<<(unsigned)(((int64_t)n_aln * 32 + 255) / 256), 256, 0, st>>>(r.U, r.R, r.off_r, r.phylo, r.anc, r.bls, r.rec);
        CK(cudaGetLastError());
    } else if (r.nreg > 0) {
        k_region_records<<<(unsigned)((r.nreg + 127) / 128), 128, 0, st>>>(r.U, r.nreg, r.R, r.phylo, r.anc, r.bls, r.rec);
        CK(cudaGetLastError());
    }
    m->regions.resize((size_t)n_out);
    if (n_out > 0) CK(cudaMemcpyAsync(m->regions.data(), r.rec, (size_t)n_out * sizeof(pcsf_region), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    *n_regions = n_out;
    return PCSF_OK;
}

extern "C" pcsf_status pcsf_score_regions_get(const pcsf_model *m, pcsf_region *out, int64_t n) {
    if (!m || n < 0 || (n > 0 && !out) || n > (int64_t)m->regions.size())
        return fail(PCSF_ERR_INVALID, "pcsf_score_regions_get: bad argument (n exceeds the records of the last call)");
    if (n > 0) memcpy(out, m->regions.data(), (size_t)n * sizeof(pcsf_region));
    return PCSF_OK;
}
