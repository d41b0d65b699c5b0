// prune_tc5.cuh — k_prune_tc5: Felsenstein pruning on the 5th-generation tensor cores (tcgen05.mma kind::tf32,
// accumulators and the A operand in TMEM, P tiles streamed by bulk TMA, leaf and cherry messages gathered from L2-resident
// row tables by dedicated producer warps).  FP32-class arithmetic with per-window log-scaling; the FP64 DMMA kernel (k_prune)
// stays the parity anchor.
//
// Formulation (ensure_alpha, fixed_lik.hpp:125-164).  For 128 codon windows at a time every edge above a NON-CHERRY inner
// node c is one GEMM  D[w][a] = sum_b A[w][b] * P_c[a][b]  on the tensor core (M = 128 windows, K = 64 child states):
// A = alpha_c split into TF32 hi + lo (per-window power-of-two normalised, the exponent kept as an integer);
// B = [hi(P_c) | lo(P_c)] side by side (N = 128): per k-step one N = 128 MMA with hi(A) gives hi*hi | hi*lo and one
// N = 64 MMA with lo(A) adds lo*hi, in FP32 accumulators; msg = D[:, 0:64] + D[:, 64:128] (~2^-21 per product).  A TS-form MMA
// reads its 4 KB A slab from TMEM at 64 B/clk, i.e. ~64 cycles whatever its N <= 128 (tools/tc5_probe.cu), so the
// side-by-side layout is what makes two instructions per k-step enough.
// LEAF edges are not GEMMs: the message of a leaf with codon x is column x of P_l (all ones for a gap/N codon, the row
// sums of fixed_lik.hpp:111-118): one row of a 65-row table.
// CHERRY edges are not GEMMs either (round 2): the message of the edge above a node whose two children are leaves depends only on
// the two codons, P_c . (P_l[:, x] * P_r[:, y]): 65 x 65 rows of 64 floats tabulated once per model in FP64 (k_build_rows).  That
// removes 17 of 56 GEMMs, 34 of 58 leaf factors and half of the stack pushes for 58mammals (28 of 98, 56 of 100 for 100vertebrates).
// Both kinds are ROW SOURCES of one row table per ECM in global memory (19 MB for 58mammals: L2 resident), consumed in program
// order.  Six PRODUCER warps copy the rows of the 128 windows of a chain with 16-byte cp.async (sixteen lanes per 256-byte row: full
// sectors; jobs of 32 rows dealt round-robin) into one of the chain's two XOR-swizzled 32 KB staging buffers, two sources ahead
// of the program, and signal a full mbarrier (cp.async.mbarrier.arrive); every epilogue thread then reads its own row with
// conflict-free LDS.128 and releases the buffer through an empty mbarrier.  The epilogue warps — the critical path of the
// kernel — neither compute a row index nor issue a copy.  (Round 1 streamed whole leaf tables through a shared-memory ring and
// gathered from them with 2.6-way bank conflicts, 1000-2000 cycles per gather; letting the epilogue warps issue the cp.async
// themselves cost ~1000 cycles per step on the critical path.)
// (Round 2, measured and dropped: one 256-byte bulk TMA copy per row issued by the lane that owns the window, rows padded to 272 bytes:
// ptxas serialises the 32 UBLKCP of a warp, 104 M against 122 M columns/s.)
// The codon ids the row indices are computed from come from k_tc5_ids: one pass that writes, per pair of 128-window tiles, the
// [chain][leaf][window] byte block the producers want in shared memory, so that a single bulk TMA copy brings it in (the
// epilogue threads used to gather 3 bytes per leaf and window from the code matrix: 18 k cycles per pair with the tensor pipe idle).
//
// One persistent CTA per SM works on a PAIR of 128-window tiles (chains X and Y) that share the tile ring: while the
// tensor core runs chain Y's GEMM of step g, chain X's epilogue turns D_g into A_{g+1} (and vice versa).
//   warps 0-3   epilogue of chain X: thread = window = TMEM lane; the 64-state partial lives in registers
//   warps 4-7   epilogue of chain Y        TMEM columns 256c..256c+255: two 128-column regions, A_g in one, D_g in the
//   warp  8     MMA issue (one elected lane)    other; A_{g+1} overwrites D_g in place
//   warp  9     TMA producer, inner-edge tiles (32 KB each, 2- or 3-stage full/empty mbarrier ring)
//   warps 10-15 row producers (warp 10 also issues the bulk copy of the next pair's codon ids)
// The producer warpgroups give their registers to the epilogue warpgroups (setmaxnreg 40 / 216).
// Waiting sibling partials (stack depth = Strahler number over the non-cherry inner nodes - 1) spill to an L2-resident scratch
// in global memory, every thread only ever touching its own column: the push is issued after the next A has been handed to
// the tensor core, the pop is prefetched while the GEMM runs, so neither is on the critical path.
#pragma once

#include "kernels.cuh"
#include "tc5.cuh"

namespace pcsf {

constexpr int T5_MAX_NSTAGE = 3;         // inner-edge tile ring (stages chosen at model creation: what fits)
constexpr int T5_TILE_BYTES = 32768;
constexpr int T5_THREADS = 512;
constexpr int T5_NPROD = 6;              // row producer warps (10..15)
constexpr int T5_STACK_ENTRY_FLOATS = 64 * 128 + 128;   // 128 windows x 64 states + 128 exponents
constexpr int T5_ROW_PITCH = 256;                       // XOR-swizzled 16-byte chunks, no padding
constexpr int T5_ROW_STAGE_BYTES = 128 * T5_ROW_PITCH;  // one staging buffer of one chain: the rows of its 128 windows

struct PruneTc5Args {
    const uint32_t *n_unique;
    const uint32_t *steps;
    int nl, n_steps, max_stack;
    int n_src;                   // row sources per ECM pass, in consumption order
    int nstage;                  // tile ring depth
    int nids;                    // codon-id ring depth (2 when it fits, else 1)
    const uint8_t *ids;          // [pairs][2 chains][nl][128] codon ids (k_tc5_ids)
    const float *pstream[2];     // [n_steps][8192]
    const float *rowtab[2];      // [rows][64]: leaf and cherry message tables (Tc5Src::row_base)
    const Tc5Src *srcs;          // [n_src]
    const double *pi[2];
    double *logz[2];
    float *scratch;              // [grid][2][max_stack][T5_STACK_ENTRY_FLOATS]
};

__host__ __device__ inline size_t prune_tc5_smem_bytes(int nl, int n_steps, int n_src, int nstage, int nids) {
    size_t b = (size_t)nstage * T5_TILE_BYTES;
    b += (size_t)2 * 2 * T5_ROW_STAGE_BYTES;                // row staging: 2 chains x 2 buffers
    b += (size_t)T5_NPROD * 256;                            // row index exchange, 2 x 32 x 4 bytes per producer warp
    b += (size_t)nids * 2 * nl * 128;                       // codon ids of both tiles
    b += (size_t)(((n_steps + 1) * 4 + 15) / 16) * 16;      // steps
    b += (size_t)(n_src + 1) * sizeof(Tc5Src);              // sources
    b += 2 * 64 * 8;                                        // pi
    b += 32 * 8;                                            // mbarriers + TMEM base
    return b;
}
// Deepest rings that fit into one SM's shared memory: the codon ids double-buffered first (a single buffer exposes the bulk
// copy's latency once per pair), then a third tile stage.
inline void prune_tc5_pick_stages(int nl, int n_steps, int n_src, int *nstage, int *nids) {
    *nstage = 2; *nids = 1;
    if (prune_tc5_smem_bytes(nl, n_steps, n_src, 2, 2) <= 227 * 1024) *nids = 2;
    if (prune_tc5_smem_bytes(nl, n_steps, n_src, 3, *nids) <= 227 * 1024) *nstage = 3;
}

// Codon ids of the unique windows in the layout the producers of k_prune_tc5 read: block (pair, chain) = [leaf][128 windows].
// Windows past n_unique repeat the last one (their results are never stored).
__global__ void __launch_bounds__(128) k_tc5_ids(const WinSpace ws, const uint32_t *__restrict__ uniq, const uint32_t *__restrict__ n_unique_p,
                                                 uint8_t *__restrict__ ids) {
    const uint32_t n_unique = *n_unique_p;
    const uint32_t npairs = (n_unique + 255) / 256;
    // Thread t owns ranks 2t and 2t+1 of the pair: in window order these are usually the '+' and the '-' window of ONE column offset
    // (the unique list is in order of first occurrence), which share their three bytes per species: one set of loads, both codons,
    // one 16-bit store.  Anything else (a duplicate removed in between, the tracks of a window list) takes the two-window path.
    for (uint32_t pair = blockIdx.x; pair < npairs; pair += gridDim.x) {
        const uint32_t u0 = pair * 256 + 2 * threadIdx.x, u1 = u0 + 1;
        const uint32_t lw0 = uniq[u0 < n_unique ? u0 : n_unique - 1], lw1 = uniq[u1 < n_unique ? u1 : n_unique - 1];
        uint8_t *out = ids + (size_t)pair * 2 * ws.nl * 128 + (size_t)(threadIdx.x >> 6) * ws.nl * 128 + ((2 * threadIdx.x) & 127);
        if (ws.mode == 0 && (lw0 & 1) == 0 && lw1 == lw0 + 1) {
            const uint8_t *p = ws.codes + ws.c0 + (lw0 >> 1);
            for (int s0 = 0; s0 < ws.nl; s0 += 16) {
                uint32_t v[16][3];
#pragma unroll
                for (int k = 0; k < 16; ++k) {
                    const uint8_t *q = p + (int64_t)(s0 + k < ws.nl ? s0 + k : s0) * ws.ld;
                    v[k][0] = __ldg(q); v[k][1] = __ldg(q + 1); v[k][2] = __ldg(q + 2);
                }
#pragma unroll
                for (int k = 0; k < 16; ++k)
                    if (s0 + k < ws.nl)
                        *reinterpret_cast<uint16_t *>(out + (size_t)(s0 + k) * 128) =
                            (uint16_t)(codon_plus(v[k][0], v[k][1], v[k][2]) | (codon_minus(v[k][0], v[k][1], v[k][2]) << 8));
            }
            continue;
        }
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const uint32_t lw = h ? lw1 : lw0;
            uint32_t strand;
            const int64_t o = win_column(ws, lw, &strand);
            const uint8_t *p = ws.codes + o;
            for (int s0 = 0; s0 < ws.nl; s0 += 16) {
                uint32_t v[16][3];
#pragma unroll
                for (int k = 0; k < 16; ++k) {
                    const uint8_t *q = p + (int64_t)(s0 + k < ws.nl ? s0 + k : s0) * ws.ld;
                    v[k][0] = __ldg(q); v[k][1] = __ldg(q + 1); v[k][2] = __ldg(q + 2);
                }
#pragma unroll
                for (int k = 0; k < 16; ++k)
                    if (s0 + k < ws.nl)
                        out[(size_t)(s0 + k) * 128 + h] = (uint8_t)(strand ? codon_minus(v[k][0], v[k][1], v[k][2]) : codon_plus(v[k][0], v[k][1], v[k][2]));
            }
        }
    }
}

// Row table of one ECM.  grid (65, n_src), 64 threads (thread = parent state a).
//   leaf source    row x = P_l[:, x] for x < 64, all ones for x = 64 (the gap/N codon)                    [block x writes row x]
//   cherry source  row x * 65 + y = sum_b P_c[a][b] * u_x[b] * v_y[b], u_x = the left leaf's row x, v_y the right leaf's row y,
//                  FP64 accumulation, FP32 storage                                                          [block x writes 65 rows]
__global__ void __launch_bounds__(64) k_build_rows(const Tc5Src *__restrict__ srcs, const double *__restrict__ cherry_P,
                                                   const double *__restrict__ leafPT, float *__restrict__ tab) {
    __shared__ double u[64];
    __shared__ double v[65][64];
    const Tc5Src d = srcs[blockIdx.y];
    const int x = blockIdx.x, a = threadIdx.x;
    if (d.l2 == 0xff) {
        tab[((size_t)d.row_base + x) * 64 + a] = x < 64 ? (float)leafPT[((size_t)d.l1 * 65 + x) * 64 + a] : 1.0f;
        return;
    }
    u[a] = x < 64 ? leafPT[((size_t)d.l1 * 65 + x) * 64 + a] : 1.0;
    for (int y = 0; y < 65; ++y) v[y][a] = y < 64 ? leafPT[((size_t)d.l2 * 65 + y) * 64 + a] : 1.0;
    __syncthreads();
    double pa[64];
#pragma unroll
    for (int b = 0; b < 64; ++b) pa[b] = cherry_P[(size_t)d.cherry * 4096 + a * 64 + b] * u[b];
    float *out = tab + ((size_t)d.row_base + (size_t)x * 65) * 64 + a;
    for (int y = 0; y < 65; ++y) {
        double s = 0.0;
#pragma unroll
        for (int b = 0; b < 64; ++b) s += pa[b] * v[y][b];
        out[(size_t)y * 64] = (float)s;
    }
}

__device__ __forceinline__ void cp_async_16(uint32_t dst_smem, const void *src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst_smem), "l"(src) : "memory");
}
// the same copy allocating in L1: the 65 rows of a LEAF source (16.6 KB) are fetched ~4 times each per pair of tiles
__device__ __forceinline__ void cp_async_16_ca(uint32_t dst_smem, const void *src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst_smem), "l"(src) : "memory");
}
#ifndef PCSF_TC5_ROWS_CA
#define PCSF_TC5_ROWS_CA 2          // 0: every row copy bypasses L1, 1: all allocate in L1, 2: only the leaf sources' (measured 124.1 / 125.4 / 126.7 M columns/s)
#endif
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__global__ void __launch_bounds__(T5_THREADS, 1) k_prune_tc5(const PruneTc5Args a) {
    extern __shared__ __align__(1024) unsigned char smem[];
    unsigned char *sp_ = smem;
    const uint32_t T5_NSTAGE = a.nstage;
    unsigned char *stage_buf = sp_; sp_ += (size_t)T5_NSTAGE * T5_TILE_BYTES;
    unsigned char *row_buf = sp_; sp_ += (size_t)2 * 2 * T5_ROW_STAGE_BYTES;       // [chain][buffer][128 rows][256 B]
    uint32_t *row_xchg = reinterpret_cast<uint32_t *>(sp_); sp_ += (size_t)T5_NPROD * 256;
    uint8_t *ids = sp_; sp_ += (size_t)a.nids * 2 * a.nl * 128;                    // [slot][chain][leaf][128]
    uint32_t *steps = reinterpret_cast<uint32_t *>(sp_); sp_ += (size_t)(((a.n_steps + 1) * 4 + 15) / 16) * 16;
    Tc5Src *srcs = reinterpret_cast<Tc5Src *>(sp_); sp_ += (size_t)(a.n_src + 1) * sizeof(Tc5Src);
    double *s_pi = reinterpret_cast<double *>(sp_); sp_ += 2 * 64 * 8;
    uint64_t *full = reinterpret_cast<uint64_t *>(sp_);
    uint64_t *empty = full + T5_MAX_NSTAGE;
    uint64_t *a_ready = empty + T5_MAX_NSTAGE;     // [2 chains][2 halves] epilogue -> MMA: states 0..31 / 32..63 of the step's A are in TMEM
    uint64_t *d_ready = a_ready + 4;               // [2] MMA -> epilogue: D of the step is complete
    uint64_t *row_full = d_ready + 2;              // [2 chains][2 buffers] producers -> epilogue: the 128 rows of a source have landed
    uint64_t *row_empty = row_full + 4;            // [2][2] epilogue -> producers: every thread of the chain has read its row
    uint64_t *ids_full = row_empty + 4;            // [2 slots] bulk copy of a pair's codon ids has landed
    uint64_t *ids_empty = ids_full + 2;            // [2] every producer warp has computed its last row index of the pair
    uint32_t *tmem_base_slot = reinterpret_cast<uint32_t *>(ids_empty + 2);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
#ifdef PCSF_TC5_TRACE
    __shared__ long long trace[3][64][4];
    __shared__ long long ptrace[T5_NPROD][56][3];       // row producers: per job [before row_empty wait, after it, copies issued]
    __shared__ unsigned short pjob[T5_NPROD][56];
#define T5_TRACE(who, s, i) do { if (blockIdx.x == 0 && first_seq && (s) < 64) trace[who][s][i] = clock64(); } while (0)
#else
#define T5_TRACE(who, s, i) do { } while (0)
#endif
    if (tid == 0) {
        for (int s = 0; s < T5_MAX_NSTAGE; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, 1); }
        for (int c = 0; c < 2; ++c) { for (int k = 0; k < 2; ++k) mbar_init(a_ready + 2 * c + k, 128); mbar_init(d_ready + c, 1); }
        for (int i = 0; i < 4; ++i) { mbar_init(row_full + i, 128); mbar_init(row_empty + i, 128); }   // 4 jobs (x 32 lanes) / 128 readers
        for (int i = 0; i < 2; ++i) { mbar_init(ids_full + i, 1); mbar_init(ids_empty + i, T5_NPROD); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 8) { tc5::tmem_alloc(tmem_base_slot, 512); tc5::tmem_relinquish(); }
    for (int i = tid; i < a.n_steps; i += blockDim.x) steps[i] = a.steps[i];
    for (int i = tid; i < a.n_src; i += blockDim.x) srcs[i] = a.srcs[i];
    for (int i = tid; i < 128; i += blockDim.x) s_pi[i] = (i >> 6 ? a.pi[1] : a.pi[0])[i & 63];
    tc5::fence_before_sync();
    __syncthreads();
    tc5::fence_after_sync();
    const uint32_t tmem = *tmem_base_slot;

    const uint32_t n_unique = *a.n_unique;
    const uint32_t npairs = (n_unique + 255) / 256;
    const int n_src2 = 2 * a.n_src;                 // sources of a pair: both ECM passes

    if (warp >= 8) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
        if (warp == 9) {
            // ---- TMA producer: inner-edge tiles
            if (lane == 0) {
                uint32_t use = 0;
                for (uint32_t pair = blockIdx.x; pair < npairs; pair += gridDim.x)
                    for (int m = 0; m < 2; ++m)
                        for (int s = 0; s < a.n_steps; ++s, ++use) {
                            const uint32_t st = use % T5_NSTAGE;
                            mbar_wait(empty + st, ((use / T5_NSTAGE) & 1) ^ 1);
                            mbar_arrive_expect_tx(full + st, T5_TILE_BYTES);
                            tma_bulk_g2s(stage_buf + (size_t)st * T5_TILE_BYTES, (m ? a.pstream[1] : a.pstream[0]) + (size_t)s * 8192, T5_TILE_BYTES, full + st);
                        }
            }
        } else if (warp == 8) {
            // ---- MMA issue: warp-uniform control flow, one elected lane issues
            const uint32_t idesc = tc5::idesc_tf32(128, 128), idesc_hi = tc5::idesc_tf32(128, 64);
            uint32_t use = 0;
            for (uint32_t pair = blockIdx.x; pair < npairs; pair += gridDim.x)
                for (int m = 0; m < 2; ++m)
                    for (int s = 0; s < a.n_steps; ++s, ++use) {
                        const uint32_t st = use % T5_NSTAGE;
#ifdef PCSF_TC5_TRACE
                        const bool first_seq = pair == blockIdx.x + 4 * gridDim.x && m == 0 && lane == 0;
#endif
                        mbar_wait(full + st, (use / T5_NSTAGE) & 1);
                        const uint32_t sb = tc5::smem_addr(stage_buf + (size_t)st * T5_TILE_BYTES);
                        for (int c = 0; c < 2; ++c) {
                            // k-steps 0..3 only need states 0..31 of A: they are issued while the epilogue threads still split and store
                            // the other half (measured: 101.2 -> 95.8 ms per 8 Mi columns; four quarters: 98.6 ms, the extra
                            // tcgen05.wait::st round trips cost more than the earlier start gains)
                            const uint32_t ta = tmem + c * 256 + (use & 1) * 128, td = tmem + c * 256 + ((use & 1) ^ 1) * 128;
#pragma unroll
                            for (int k = 0; k < 2; ++k) {
                                mbar_wait(a_ready + 2 * c + k, use & 1);
                                if (k == 0) T5_TRACE(2, s, 2 * c);
                                tc5::fence_after_sync();
                                if (tc5::elect_one()) {
#pragma unroll
                                    for (int j = 4 * k; j < 4 * k + 4; ++j) {
                                        const uint64_t bd = tc5::smem_desc(sb + j * 4096, 128, 256);
                                        tc5::mma_tf32_ts(td, ta + 8 * j, bd, idesc, j > 0);
                                        tc5::mma_tf32_ts(td, ta + 64 + 8 * j, bd, idesc_hi, 1);      // lo(A) x hi(B) only
                                    }
                                    if (k == 1) {
                                        tc5::commit(d_ready + c);
                                        if (c == 1) tc5::commit(empty + st);
                                    }
                                }
                                __syncwarp();
                            }
                            __syncwarp();
                            T5_TRACE(2, s, 2 * c + 1);
                        }
                    }
        } else {
            // ---- row producers.  Job j of a pair = (source g, chain c, quarter q) with j = (g * 2 + c) * 4 + q: the rows of windows
            // 32q..32q+31 of chain c for source g (g = ECM * n_src + k, consumed in this order) go to the chain's staging buffer g & 1.
            // The jobs are dealt round-robin over the six warps; every warp works through its jobs in order, so the lowest
            // unfinished job never waits for a higher one (no deadlock).  Chunk ch (16 bytes) of row rr sits at chunk position
            // (ch & 8) | ((ch ^ rr) & 7): the sixteen lanes that copy one row write two full 128-byte lines, and the eight threads of a
            // quarter warp that later read chunk j of their OWN rows (LDS.128) hit eight different bank groups.
            const int pw = warp - 10;
            uint32_t *xchg = row_xchg + pw * 64;
            const uint32_t row_s = tc5::smem_addr(row_buf);
            const int jobs_per_pair = n_src2 * 8;
            const int half = lane >> 4, ch = lane & 15;
            const size_t ids_slot_bytes = (size_t)2 * a.nl * 128;
            uint32_t it = 0;                               // pair iteration of this CTA
            uint32_t J = pw;                               // global job counter of this warp (over all pairs of the CTA)
            const uint32_t my_pairs = npairs > blockIdx.x ? (npairs - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
            // warp 10, lane 0: bulk copy of the codon ids of pair iteration k into slot k % nids
            auto load_ids = [&](uint32_t k) {
                const uint32_t slot = k % a.nids, round = k / a.nids;
                mbar_wait_sleepy(ids_empty + slot, (round & 1) ^ 1);
                mbar_arrive_expect_tx(ids_full + slot, (uint32_t)ids_slot_bytes);
                tma_bulk_g2s(ids + slot * ids_slot_bytes, a.ids + ((size_t)blockIdx.x + (size_t)k * gridDim.x) * ids_slot_bytes,
                             (uint32_t)ids_slot_bytes, ids_full + slot);
            };
            if (pw == 0 && lane == 0)
                for (uint32_t k = 0; k < (uint32_t)a.nids - 1 && k < my_pairs; ++k) load_ids(k);
            for (; it < my_pairs; ++it) {
                if (pw == 0 && lane == 0 && it + a.nids - 1 < my_pairs) load_ids(it + a.nids - 1);
                __syncwarp();
                const uint32_t slot = it % a.nids;
                mbar_wait_sleepy(ids_full + slot, (it / a.nids) & 1);
                const uint8_t *pids = ids + slot * ids_slot_bytes;
                const uint32_t jend = (it + 1) * (uint32_t)jobs_per_pair;
                for (; J < jend; J += T5_NPROD) {
                    const uint32_t j = J - it * (uint32_t)jobs_per_pair;
                    const uint32_t q = j & 3, c = (j >> 2) & 1, g = j >> 3;
                    const uint32_t G = it * (uint32_t)n_src2 + g;                    // running source number of the chain
                    const int m = g >= (uint32_t)a.n_src ? 1 : 0;
                    const Tc5Src d = srcs[g - m * a.n_src];
                    const uint8_t *wid = pids + (size_t)c * a.nl * 128 + q * 32 + lane;
                    const uint32_t x = wid[(uint32_t)d.l1 * 128];
#if defined(PCSF_TC5_EXP) && PCSF_TC5_EXP == 2
                    const uint32_t myrow = d.row_base + (x & 0u) + q * 32 + lane;          // timing experiment: 32 consecutive rows (wrong results)
#else
                    const uint32_t myrow = d.row_base + (d.l2 == 0xff ? x : x * 65u + wid[(uint32_t)d.l2 * 128]);
#endif
                    // every lane copies one 16-byte chunk of sixteen rows (lanes 0-15: the even windows, lanes 16-31: the odd ones): the row
                    // indices change hands through 128 bytes of shared memory, even windows first.  The exchange area is double-buffered
                    // per warp (the __syncwarp of job J+1 orders the reads of job J before the writes of job J+2), and the indices are read
                    // back four at a time right before their copies: an LDGSTS keeps its address registers until the LSU has taken the
                    // request, and with the 40 registers of a producer warp ptxas used ONE register pair for all sixteen addresses, every
                    // copy waiting for the previous one (~50 cycles each, 800-1000 per job: the rows arrived late, ncu source page).
                    uint32_t *xb = xchg + (((J / T5_NPROD) & 1u) << 5);
                    xb[(lane & 1) * 16 + (lane >> 1)] = myrow;
                    __syncwarp();
                    const uint32_t b = c * 2 + (G & 1);
#ifdef PCSF_TC5_TRACE
                    const uint32_t pj = (J - it * (uint32_t)jobs_per_pair) / T5_NPROD;
                    const bool ptr_on = blockIdx.x == 0 && it == 4 && pj < 56 && lane == 0;
                    if (ptr_on) { ptrace[pw][pj][0] = clock64(); pjob[pw][pj] = (unsigned short)j; }
#endif
                    mbar_wait(row_empty + b, ((G >> 1) & 1) ^ 1);
#ifdef PCSF_TC5_TRACE
                    if (ptr_on) ptrace[pw][pj][1] = clock64();
#endif
                    const float *tab = (m ? a.rowtab[1] : a.rowtab[0]) + ch * 4;
                    const uint32_t dst = row_s + b * T5_ROW_STAGE_BYTES + q * 32 * 256;
                    const bool use_l1 = PCSF_TC5_ROWS_CA == 1 || (PCSF_TC5_ROWS_CA == 2 && d.l2 == 0xff);
#if defined(PCSF_TC5_EXP) && PCSF_TC5_EXP == 1
                    mbar_arrive(row_full + b);          // timing experiment: no copies at all (wrong results)
                    (void)tab; (void)dst; (void)use_l1;
                    continue;
#endif
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const uint4 v = reinterpret_cast<const uint4 *>(xb + half * 16)[k];
                        const float *s0 = tab + (size_t)v.x * 64, *s1 = tab + (size_t)v.y * 64, *s2 = tab + (size_t)v.z * 64, *s3 = tab + (size_t)v.w * 64;
                        const int r0 = 2 * (4 * k) + half, r1 = r0 + 2, r2 = r0 + 4, r3 = r0 + 6;          // the windows (rows of the quarter) of these four copies
                        const uint32_t d0 = dst + r0 * 256 + (((ch & 8) | ((ch ^ r0) & 7)) << 4), d1 = dst + r1 * 256 + (((ch & 8) | ((ch ^ r1) & 7)) << 4),
                                       d2 = dst + r2 * 256 + (((ch & 8) | ((ch ^ r2) & 7)) << 4), d3 = dst + r3 * 256 + (((ch & 8) | ((ch ^ r3) & 7)) << 4);
                        if (use_l1) { cp_async_16_ca(d0, s0); cp_async_16_ca(d1, s1); cp_async_16_ca(d2, s2); cp_async_16_ca(d3, s3); }
                        else { cp_async_16(d0, s0); cp_async_16(d1, s1); cp_async_16(d2, s2); cp_async_16(d3, s3); }
                    }
                    // the lane's arrival on the full barrier is triggered when all of its copies above have landed
                    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(tc5::smem_addr(row_full + b)) : "memory");
#ifdef PCSF_TC5_TRACE
                    if (ptr_on) ptrace[pw][pj][2] = clock64();
#endif
                }
                __syncwarp();
                if (lane == 0) { tc5::fence_proxy_async_smem(); mbar_arrive(ids_empty + slot); }   // the slot is refilled by TMA (async proxy)
            }
        }
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 216;");
        // ---- epilogue warps: chain c, thread = window t = TMEM lane t
        const int c = warp >> 2, t = tid & 127;
        const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16) + c * 256;
        float *stk = a.scratch + ((size_t)blockIdx.x * 2 + c) * (size_t)(a.max_stack > 0 ? a.max_stack : 1) * T5_STACK_ENTRY_FLOATS;
        uint32_t use = 0;
        uint32_t taken = 0;           // running source number of this chain (over all pairs of the CTA)
        const unsigned char *rstage = row_buf + (size_t)c * 2 * T5_ROW_STAGE_BYTES + (size_t)t * T5_ROW_PITCH;
        // L (= or *=) the staged message of this thread's window from the next source of the program
        auto take_row = [&](float (&L)[64], bool mul) {
            const uint32_t b = taken & 1;
            mbar_wait(row_full + c * 2 + b, (taken >> 1) & 1);
            const float4 *row = reinterpret_cast<const float4 *>(rstage + b * T5_ROW_STAGE_BYTES);
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const float4 v = row[(j & 8) | ((j ^ t) & 7)];
                if (mul) { L[4 * j] *= v.x; L[4 * j + 1] *= v.y; L[4 * j + 2] *= v.z; L[4 * j + 3] *= v.w; }
                else { L[4 * j] = v.x; L[4 * j + 1] = v.y; L[4 * j + 2] = v.z; L[4 * j + 3] = v.w; }
            }
            mbar_arrive(row_empty + c * 2 + b);
            ++taken;
        };

#ifdef PCSF_TC5_TRACE
        long long t_seq = 0, t_pro = 0, t_begin = clock64();
#endif
        for (uint32_t pair = blockIdx.x; pair < npairs; pair += gridDim.x) {
            const uint32_t u = pair * 256 + c * 128 + t;
            for (int m = 0; m < 2; ++m) {
                float R[64];
                int E = 0, sp = 0;
#ifdef PCSF_TC5_TRACE
                long long tt1 = clock64();
#endif
                take_row(R, false);
                take_row(R, true);
#ifdef PCSF_TC5_TRACE
                long long tt2 = clock64();
                t_pro += tt2 - tt1;
#endif
                // A = split(alpha): per-window normalisation by an exact power of two, then TF32 hi + lo (hi = the 19 bits
                // the tensor core reads, lo = the exact remainder); hands the step to the MMA warp
                float amax_prev = 0.f;          // largest entry of the A that was handed over last (in [1, 2), or 0)
                // normalise(V): V *= 2^-e with e the exponent of V's largest entry (a tree of 3-input maxima, not a 64-long chain);
                // returns e and leaves the new maximum (in [1, 2), or 0) in vmax
                auto normalise = [&](float (&V)[64], float &vmax) {
                    float m4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                    for (int i = 0; i < 64; i += 8) {
#pragma unroll
                        for (int k = 0; k < 4; ++k) m4[k] = fmaxf(m4[k], fmaxf(V[i + 2 * k], V[i + 2 * k + 1]));
                    }
                    const float mx = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
                    const int e = mx > 0.f ? (int)((__float_as_uint(mx) >> 23) & 0xff) - 127 : 0;
                    const float sc = __uint_as_float((uint32_t)(127 - e) << 23);
                    const float2 sc2 = make_float2(sc, sc);
#pragma unroll
                    for (int i = 0; i < 64; i += 2) {
                        const float2 r = __fmul2_rn(make_float2(V[i], V[i + 1]), sc2);
                        V[i] = r.x; V[i + 1] = r.y;
                    }
                    vmax = mx * sc;
                    return e;
                };
                // store_A(V, areg): TF32 hi + lo of the (normalised) partial into TMEM, states 0..31 handed to the MMA warp first
                auto store_A = [&](const float (&V)[64], uint32_t areg) {
#pragma unroll
                    for (int h = 0; h < 4; ++h) {
                        uint32_t hi[16], lo[16];
#pragma unroll
                        for (int i = 0; i < 16; i += 2) {
                            hi[i] = __float_as_uint(V[16 * h + i]) & 0xffffe000u;
                            hi[i + 1] = __float_as_uint(V[16 * h + i + 1]) & 0xffffe000u;
                            const float2 l = __fadd2_rn(make_float2(V[16 * h + i], V[16 * h + i + 1]),
                                                        make_float2(-__uint_as_float(hi[i]), -__uint_as_float(hi[i + 1])));
                            lo[i] = __float_as_uint(l.x);
                            lo[i + 1] = __float_as_uint(l.y);
                        }
                        if (h == 2) {
                            // states 0..31 are on their way: hand them to the MMA warp before storing the rest
                            tc5::wait_st();
                            tc5::fence_before_sync();
                            mbar_arrive(a_ready + 2 * c);
                        }
                        tc5::st16(areg + 16 * h, hi);
                        tc5::st16(areg + 64 + 16 * h, lo);
                    }
                    tc5::wait_st();
                    tc5::fence_before_sync();
                    mbar_arrive(a_ready + 2 * c + 1);
                };
                if (a.n_steps > 0) {
                    E += normalise(R, amax_prev);
                    store_A(R, lane_base + (use & 1) * 128);
                }

                for (int s = 0; s < a.n_steps; ++s, ++use) {
                    const uint32_t step = steps[s];
                    const uint32_t post = (step >> 16) & 3u;           // MUL, PUSH_START or POP_MUL (prepare_tc5_program admits nothing else)
#ifdef PCSF_TC5_TRACE
                    const bool first_seq = pair == blockIdx.x + 4 * gridDim.x && m == 0 && (t == 0);
#endif
                    T5_TRACE(c, s, 0);
                    // ---- while the GEMM runs: what the program multiplies in before the next GEMM — leaf / cherry messages from
                    // the staged table rows, or the waiting sibling partial from the stack
                    float L[64];
                    int Epop = 0;                  // exponent that comes with L: of the popped partial / of the new chain's start
                    float amax_start = 0.f;
                    if (post == T5_MUL) {
                        take_row(L, false);
                    } else if (post == T5_PUSH_START) {
                        // the start of a new chain does not depend on the running GEMM: it is normalised here, in the GEMM's shadow
                        take_row(L, false);
                        take_row(L, true);
                        Epop = normalise(L, amax_start);
                    } else {
                        --sp;
                        const float4 *e4 = reinterpret_cast<const float4 *>(stk + (size_t)sp * T5_STACK_ENTRY_FLOATS);
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            const float4 v = __ldcg(e4 + j * 128 + t);
                            L[4 * j] = v.x; L[4 * j + 1] = v.y; L[4 * j + 2] = v.z; L[4 * j + 3] = v.w;
                        }
                        Epop = __ldcg(reinterpret_cast<const int *>(stk + (size_t)sp * T5_STACK_ENTRY_FLOATS + 8192) + t);
                    }
                    uint32_t dreg = lane_base + ((use & 1) ^ 1) * 128;           // D_s; A_{s+1} overwrites it in place
                    asm volatile("" : "+r"(dreg));                               // in a register before the wait, not after it
                    T5_TRACE(c, s, 1);
                    mbar_wait(d_ready + c, use & 1);
                    T5_TRACE(c, s, 2);
                    tc5::fence_after_sync();
                    // Any power of two is an exact scale, so the normalisation does not have to wait for this message's own maximum:
                    // every entry is <= the largest entry of the A it was computed from (rows of P sum to <= 1), hence the exponent of
                    // that previous maximum brings the message back to O(1), and how far below 1 the factors multiplied in push it is
                    // corrected one step later.  The scale goes in BEFORE anything small is multiplied in: two lagging factors (a cherry
                    // row is the product of two leaf columns) must not meet below FP32's range.
                    const int e = amax_prev > 0.f ? (int)((__float_as_uint(amax_prev) >> 23) & 0xff) - 127 : 0;
                    const float sc = __uint_as_float((uint32_t)(127 - e) << 23);
                    const float2 sc2 = make_float2(sc, sc);
                    E += e;
                    if (post == T5_PUSH_START) {
                        // The message is pushed onto the stack (brought back to O(1) first) and the new chain's start (already normalised,
                        // in L) becomes the next GEMM's input.  D_s is read in two halves, each pushed straight from the registers it
                        // was loaded into: with L live, all four tcgen05.ld at once would not fit into the register file (the second
                        // wait::ld round trip costs ~150 cycles on 9 of 39 steps of 58mammals; the spills it replaces cost more)
                        float4 *e4 = reinterpret_cast<float4 *>(stk + (size_t)sp * T5_STACK_ENTRY_FLOATS);
#pragma unroll
                        for (int hh = 0; hh < 2; ++hh) {
                            uint32_t x0[32], y0[32];
                            tc5::ld32(dreg + 32 * hh, x0);
                            tc5::ld32(dreg + 64 + 32 * hh, y0);
                            tc5::wait_ld();
#pragma unroll
                            for (int i = 0; i < 32; i += 4) {
                                const float2 v0 = __fmul2_rn(__fadd2_rn(make_float2(__uint_as_float(x0[i]), __uint_as_float(x0[i + 1])),
                                                                        make_float2(__uint_as_float(y0[i]), __uint_as_float(y0[i + 1]))), sc2);
                                const float2 v1 = __fmul2_rn(__fadd2_rn(make_float2(__uint_as_float(x0[i + 2]), __uint_as_float(x0[i + 3])),
                                                                        make_float2(__uint_as_float(y0[i + 2]), __uint_as_float(y0[i + 3]))), sc2);
                                __stcg(e4 + (8 * hh + i / 4) * 128 + t, make_float4(v0.x, v0.y, v1.x, v1.y));
                            }
                        }
                        __stcg(reinterpret_cast<int *>(stk + (size_t)sp * T5_STACK_ENTRY_FLOATS + 8192) + t, E);
                        ++sp;
                        E = Epop;
                        amax_prev = amax_start;
                        store_A(L, dreg);
                    } else if (s + 1 == a.n_steps) {
                        // the root: alpha_root = msg * L stays in R for the dot product with pi
                        uint32_t x0[32], y0[32], x1[32], y1[32];
                        tc5::ld32(dreg, x0);
                        tc5::ld32(dreg + 64, y0);
                        tc5::ld32(dreg + 32, x1);
                        tc5::ld32(dreg + 96, y1);
                        tc5::wait_ld();
#pragma unroll
                        for (int i = 0; i < 32; i += 2) {
                            float2 v0 = __fmul2_rn(__fadd2_rn(make_float2(__uint_as_float(x0[i]), __uint_as_float(x0[i + 1])),
                                                              make_float2(__uint_as_float(y0[i]), __uint_as_float(y0[i + 1]))), sc2);
                            float2 v1 = __fmul2_rn(__fadd2_rn(make_float2(__uint_as_float(x1[i]), __uint_as_float(x1[i + 1])),
                                                              make_float2(__uint_as_float(y1[i]), __uint_as_float(y1[i + 1]))), sc2);
                            v0 = __fmul2_rn(v0, make_float2(L[i], L[i + 1]));
                            v1 = __fmul2_rn(v1, make_float2(L[32 + i], L[32 + i + 1]));
                            R[i] = v0.x; R[i + 1] = v0.y; R[32 + i] = v1.x; R[32 + i + 1] = v1.y;
                        }
                        E += Epop;
                    } else {
                        // Streamed hand-over: alpha_parent = msg * L becomes A_{s+1} without a separate max pass (one tcgen05.wait::ld
                        // round trip; streaming the TMEM loads in two halves was measured slower, 114 against 97 ms)
                        E += Epop;
                        float amax = 0.f;
                        float V[64];
                        {
                            uint32_t x0[32], y0[32], x1[32], y1[32];
                            tc5::ld32(dreg, x0);
                            tc5::ld32(dreg + 64, y0);
                            tc5::ld32(dreg + 32, x1);
                            tc5::ld32(dreg + 96, y1);
                            tc5::wait_ld();
#pragma unroll
                            for (int i = 0; i < 32; i += 2) {
                                float2 v0 = __fadd2_rn(make_float2(__uint_as_float(x0[i]), __uint_as_float(x0[i + 1])),
                                                       make_float2(__uint_as_float(y0[i]), __uint_as_float(y0[i + 1])));
                                float2 v1 = __fadd2_rn(make_float2(__uint_as_float(x1[i]), __uint_as_float(x1[i + 1])),
                                                       make_float2(__uint_as_float(y1[i]), __uint_as_float(y1[i + 1])));
                                v0 = __fmul2_rn(v0, sc2);
                                v1 = __fmul2_rn(v1, sc2);
                                v0 = __fmul2_rn(v0, make_float2(L[i], L[i + 1]));
                                v1 = __fmul2_rn(v1, make_float2(L[32 + i], L[32 + i + 1]));
                                amax = fmaxf(amax, fmaxf(fmaxf(v0.x, v0.y), fmaxf(v1.x, v1.y)));
                                V[i] = v0.x; V[i + 1] = v0.y; V[32 + i] = v1.x; V[32 + i + 1] = v1.y;
                            }
                        }
                        store_A(V, dreg);
                        amax_prev = amax;
                    }
                    T5_TRACE(c, s, 3);
                }
                // z = pi . alpha_root (fixed_lik.hpp:159-163), log z with the exponents taken out so far
                {
                    const double *pi = s_pi + m * 64;
                    double z = 0.0;
#pragma unroll
                    for (int i = 0; i < 64; ++i) z += pi[i] * (double)R[i];
                    if (u < n_unique) (m ? a.logz[1] : a.logz[0])[u] = log(z) + (double)E * 0.6931471805599453;
                }
#ifdef PCSF_TC5_TRACE
                t_seq += clock64() - tt2;
#endif
            }
        }
#ifdef PCSF_TC5_TRACE
        if ((blockIdx.x == 0 || blockIdx.x == 77) && t == 0)
            printf("T5 cta %d chain %d: total %lld cycles, prologue gathers %lld, steps+END %lld, pairs %u\n", blockIdx.x, c,
                   clock64() - t_begin, t_pro, t_seq, (npairs - blockIdx.x + gridDim.x - 1) / gridDim.x);
#endif
    }
#ifdef PCSF_TC5_TRACE
    __syncwarp();
    __syncthreads();
    if (blockIdx.x == 0 && tid == 0) {
        const long long t0 = trace[0][0][0];
        for (int w = 0; w < T5_NPROD; ++w)
            for (int k = 0; k < 56 && k * T5_NPROD + w < a.n_src * 8; ++k) {
                const int j = pjob[w][k];
                printf("T5P warp %d job %3d src %2d chain %d q %d | start %7lld got-buffer %7lld (+%5lld) issued +%4lld\n", w, j, j >> 3, (j >> 2) & 1, j & 3,
                       ptrace[w][k][0] - t0, ptrace[w][k][1] - t0, ptrace[w][k][1] - ptrace[w][k][0], ptrace[w][k][2] - ptrace[w][k][1]);
            }
        for (int s = 0; s < a.n_steps && s < 64; ++s)
            printf("T5 s=%3d post=%u | X: A-ready %7lld gather %5lld wait-D %5lld combine %5lld | Y: A-ready %7lld gather %5lld wait-D %5lld combine %5lld | MMA: aX %7lld issX %4lld aY %7lld issY %4lld\n",
                   s, (steps[s] >> 16) & 3u, trace[0][s][0] - t0, trace[0][s][1] - trace[0][s][0], trace[0][s][2] - trace[0][s][1],
                   trace[0][s][3] - trace[0][s][2], trace[1][s][0] - t0, trace[1][s][1] - trace[1][s][0], trace[1][s][2] - trace[1][s][1],
                   trace[1][s][3] - trace[1][s][2], trace[2][s][0] - t0, trace[2][s][1] - trace[2][s][0], trace[2][s][2] - t0,
                   trace[2][s][3] - trace[2][s][2]);
    }
#endif
    // teardown: every tcgen05.ld has completed and every MMA was waited for by its epilogue
    tc5::fence_before_sync();
    __syncthreads();
    if (warp == 8) tc5::tmem_dealloc(tmem, 512);
}

}  // namespace pcsf
