// kernel_harness.cu — thin C entry points around the score-msa kernels of phylocsfpp_b200/csrc/omega.cuh (and, through it,
// mle.cuh), so that tests/test_gpu_msa_kernels.py can check each kernel on its own against high-precision references.
// Each entry point packs flat host arrays into the kernel's structs, copies them in, launches once, synchronises, copies the
// results out and frees.  Return value: 0, or the CUDA error code.
#include <cstdint>
#include <cstring>
#include <vector>

#include "../phylocsfpp_b200/csrc/omega.cuh"

using namespace pcsf;

namespace {

struct DevBufs {
    std::vector<void *> p;
    ~DevBufs() { for (void *q : p) cudaFree(q); }
    template <class T> T *alloc(size_t n) {
        void *q = nullptr;
        if (cudaMalloc(&q, n * sizeof(T) + 16) != cudaSuccess) return nullptr;
        p.push_back(q);
        return static_cast<T *>(q);
    }
    template <class T> T *upload(const T *h, size_t n) {
        T *d = alloc<T>(n);
        if (d && n) cudaMemcpy(d, h, n * sizeof(T), cudaMemcpyHostToDevice);
        return d;
    }
};

#define HCK(call)                                       \
    do {                                                \
        cudaError_t e_ = (call);                        \
        if (e_ != cudaSuccess) return (int)e_;          \
    } while (0)

std::vector<MleSlot> make_slots(int n, const int32_t *aln, const int32_t *pending, const int32_t *model, const double *x,
                                const int64_t *K, const int64_t *win0) {
    std::vector<MleSlot> s(n);
    std::memset(s.data(), 0, s.size() * sizeof(MleSlot));
    for (int i = 0; i < n; ++i) {
        s[i].aln = aln[i];
        s[i].pending = pending ? pending[i] : 1;
        s[i].model = model ? model[i] : 0;
        s[i].x = x ? x[i] : 0.0;
        s[i].K = K ? K[i] : 0;
        s[i].win0 = win0 ? win0[i] : 0;
    }
    return s;
}

}  // namespace

extern "C" {

int h_eig_stride() { return (int)OMEGA_EIG_STRIDE; }

// k_omega_eig on n slots: slot i is idle when aln[i] < 0, else it diagonalises Q(kso[i]) with the F3x4 ratios f3x4[aln[i]].
// kso: [n][3] kappa, omega, sigma.  eig: [n][64 + 2 * 4096] lambda | SR | SRinv, pi: [n][64]; both copied in first and back
// after the launch, so slots the kernel skips keep what the caller put there.
int h_omega_eig(int n, const int32_t *aln, const double *kso, const double *f3x4, int n_f3x4, double *eig, double *pi) {
    DevBufs B;
    std::vector<MleSlot> s = make_slots(n, aln, nullptr, nullptr, nullptr, nullptr, nullptr);
    std::vector<OmegaExtra> ex(n);
    std::memset(ex.data(), 0, ex.size() * sizeof(OmegaExtra));
    for (int i = 0; i < n; ++i) {
        ex[i].need_eig = 1;
        ex[i].kappa = kso[3 * i];
        ex[i].omega = kso[3 * i + 1];
        ex[i].sigma = kso[3 * i + 2];
    }
    MleSlot *d_s = B.upload(s.data(), n);
    OmegaExtra *d_ex = B.upload(ex.data(), n);
    double *d_f = B.upload(f3x4, (size_t)n_f3x4 * 9);
    double *d_eig = B.upload(eig, (size_t)n * OMEGA_EIG_STRIDE), *d_pi = B.upload(pi, (size_t)n * 64);
    if (!d_s || !d_ex || !d_f || !d_eig || !d_pi) return (int)cudaErrorMemoryAllocation;
    HCK(cudaFuncSetAttribute(k_omega_eig, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)OMEGA_EIG_SMEM));
    k_omega_eig<<<n, 256, OMEGA_EIG_SMEM>>>(d_s, d_ex, d_f, d_eig, d_pi);
    HCK(cudaGetLastError());
    HCK(cudaDeviceSynchronize());
    HCK(cudaMemcpy(eig, d_eig, (size_t)n * OMEGA_EIG_STRIDE * 8, cudaMemcpyDeviceToHost));
    HCK(cudaMemcpy(pi, d_pi, (size_t)n * 64 * 8, cudaMemcpyDeviceToHost));
    return 0;
}

// k_mle_expm on n slots x n_br branches.  Slot i: aln[i] (< 0 idle), pending[i], model[i] (0: eig0, 1: eig1), x[i] (its tree
// scale on the ECM route).  With eig_slots ([n][64 + 2 * 4096]) the OMEGA route runs instead: per-slot eigensystems and the
// tree scales rho_slots[i].  p: [n][slot_stride] doubles (n_gemm GEMM tiles, then nl leaf tables of 65 x 64), copied in first;
// err: [n] expm_err, copied in first.
int h_mle_expm(int n, const int32_t *aln, const int32_t *pending, const int32_t *model, const double *x, int n_br, int nl,
               const float *bl, const double *eig0, const double *eig1, const int32_t *edge_to_gemm, int n_gemm,
               const double *eig_slots, const double *rho_slots, double *p, int32_t *err) {
    DevBufs B;
    const size_t leaf_off = (size_t)n_gemm * 4096, slot_stride = leaf_off + (size_t)nl * 65 * 64;
    std::vector<MleSlot> s = make_slots(n, aln, pending, model, x, nullptr, nullptr);
    MleSlot *d_s = B.upload(s.data(), n);
    float *d_bl = B.upload(bl, n_br);
    int32_t *d_e2g = B.upload(edge_to_gemm, n_br);
    double *d_e0 = eig0 ? B.upload(eig0, OMEGA_EIG_STRIDE) : nullptr, *d_e1 = eig1 ? B.upload(eig1, OMEGA_EIG_STRIDE) : nullptr;
    double *d_es = eig_slots ? B.upload(eig_slots, (size_t)n * OMEGA_EIG_STRIDE) : nullptr;
    double *d_rho = rho_slots ? B.upload(rho_slots, n) : nullptr;
    double *d_p = B.upload(p, (size_t)n * slot_stride);
    int32_t *d_err = B.upload(err, n);
    if (!d_s || !d_bl || !d_e2g || !d_p || !d_err) return (int)cudaErrorMemoryAllocation;
    k_mle_expm<<<n * n_br, 128>>>(d_s, n_br, nl, d_bl, d_e0, d_e1, d_e2g, d_p, slot_stride, leaf_off, d_err, d_es, d_rho);
    HCK(cudaGetLastError());
    HCK(cudaDeviceSynchronize());
    HCK(cudaMemcpy(p, d_p, (size_t)n * slot_stride * 8, cudaMemcpyDeviceToHost));
    HCK(cudaMemcpy(err, d_err, (size_t)n * 4, cudaMemcpyDeviceToHost));
    return 0;
}

// k_mle_plan on n slots.  The P stream base and the per-slot prior base are the addresses pbase and pi_base (never
// dereferenced by the kernel; pi_base 0 = no per-slot priors).  desc: [max_tiles][7] int64 per tile: pstream - pbase,
// leafPT - pbase (both in doubles), model, count, win0, pad, pi - pi_base in doubles (-1 for a null pi).
int h_mle_plan(int n, const int32_t *aln, const int32_t *pending, const int32_t *model, const int64_t *K, const int64_t *win0,
               int tw, uint64_t slot_stride, uint64_t leaf_off, uint64_t pbase, uint64_t pi_base, int max_tiles, int64_t *desc,
               uint32_t *n_tiles) {
    DevBufs B;
    std::vector<MleSlot> s = make_slots(n, aln, pending, model, nullptr, K, win0);
    MleSlot *d_s = B.upload(s.data(), n);
    TileDesc *d_t = B.alloc<TileDesc>(max_tiles);
    uint32_t *d_n = B.alloc<uint32_t>(1);
    if (!d_s || !d_t || !d_n) return (int)cudaErrorMemoryAllocation;
    HCK(cudaMemset(d_t, 0, (size_t)max_tiles * sizeof(TileDesc)));
    k_mle_plan<<<1, 1024>>>(d_s, n, reinterpret_cast<const double *>(pbase), slot_stride, leaf_off, tw, d_t, d_n,
                            reinterpret_cast<const double *>(pi_base));
    HCK(cudaGetLastError());
    HCK(cudaDeviceSynchronize());
    HCK(cudaMemcpy(n_tiles, d_n, 4, cudaMemcpyDeviceToHost));
    std::vector<TileDesc> t(max_tiles);
    HCK(cudaMemcpy(t.data(), d_t, (size_t)max_tiles * sizeof(TileDesc), cudaMemcpyDeviceToHost));
    for (int i = 0; i < max_tiles; ++i) {
        int64_t *o = desc + 7 * (size_t)i;
        o[0] = (int64_t)(reinterpret_cast<uint64_t>(t[i].pstream) - pbase) / 8;
        o[1] = (int64_t)(reinterpret_cast<uint64_t>(t[i].leafPT) - pbase) / 8;
        o[2] = t[i].model;
        o[3] = t[i].count;
        o[4] = t[i].win0;
        o[5] = t[i].pad;
        o[6] = t[i].pi ? (int64_t)(reinterpret_cast<uint64_t>(t[i].pi) - pi_base) / 8 : -1;
    }
    return 0;
}

// k_omega_counts: codes [nl][ld] base codes (0..3 ACGT, 4 anything else), win_off [nwin] column of window w, win_start / len
// [n_aln]; f3x4 [n_aln][9].
int h_omega_counts(int nl, const uint8_t *codes, int64_t ld, const uint32_t *win_off, int64_t nwin, int n_aln,
                   const int64_t *win_start, const int64_t *len, double *f3x4) {
    DevBufs B;
    uint8_t *d_c = B.upload(codes, (size_t)nl * ld);
    uint32_t *d_w = B.upload(win_off, (size_t)(nwin > 0 ? nwin : 1));
    int64_t *d_ws = B.upload(win_start, n_aln), *d_len = B.upload(len, n_aln);
    double *d_f = B.alloc<double>((size_t)n_aln * 9);
    if (!d_c || !d_w || !d_ws || !d_len || !d_f) return (int)cudaErrorMemoryAllocation;
    WinSpace ws{d_c, ld, nl, 1, 0, d_w};
    k_omega_counts<<<n_aln, 256>>>(ws, n_aln, d_ws, d_len, d_f);
    HCK(cudaGetLastError());
    HCK(cudaDeviceSynchronize());
    HCK(cudaMemcpy(f3x4, d_f, (size_t)n_aln * 9 * 8, cudaMemcpyDeviceToHost));
    return 0;
}

}  // extern "C"
