// kernels.cuh — sm_100a kernels of the PhyloCSF++ hot path.
//
//   k_pack      ASCII -> nucleotide codes 0..4 (translation.hpp:29-53), bad-character flag      [HBM]
//   k_keys      128-bit site-pattern key of every codon window, both strands
//               (get_amino_acid_id, translation.hpp:80-88; '-' strand = update_seqs on the
//               reverse complement, parallel_file_reader.hpp:86-112, build_tracks.hpp:219-226)    [HBM]
//   k_insert / k_resolve / k_scan* / k_finalize   site-pattern dedup: first-occurrence rank          [HBM/L2]
//   k_prune     Felsenstein pruning of the unique patterns, both ECMs (ensure_alpha + lpr_leaves,
//               fixed_lik.hpp:125-164, 395-445): register-chained FP64 DMMA, P tiles streamed by TMA  [FP64 pipe]
//   k_scatter   deciban epilogue 10*(log zC - log zNC)/ln 10 (run.hpp:51-54) back to all windows   [HBM]
//   k_bls       per-base branch length score (additional_scores.hpp:5-84)                          [HBM]
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "model_prep.hpp"

namespace pcsf {

__constant__ uint8_t c_dna_lut[256];

// ---------------------------------------------------------------------------------------------------
// k_pack: codes[s][i] = get_dna_id(seqs[s][i]); columns [L, cols_out) are filled with 4 ("N").
// 16 bytes per thread when rows are 16-byte aligned, scalar otherwise.
__global__ void k_pack(const uint8_t *__restrict__ seqs, int64_t L, int64_t ld_in, int nl,
                       uint8_t *__restrict__ codes, int64_t ld_out, int64_t cols_out, int *__restrict__ bad) {
    const int s = blockIdx.y;
    const uint8_t *src = seqs + (int64_t)s * ld_in;
    uint8_t *dst = codes + (int64_t)s * ld_out;          // ld_out: row stride; cols_out: columns written (>= L, a multiple of 16)
    const bool vec = ((reinterpret_cast<uintptr_t>(src) & 15) == 0);
    int local_bad = 0;
    // main part: four 16-byte vectors per thread and iteration, all four loads in flight before the first compare (one load per
    // iteration left the kernel latency-bound at 2.5 TB/s)
    const int64_t stride = (int64_t)gridDim.x * blockDim.x * 16;
    int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 16;
    if (vec) {
        for (; i + 3 * stride + 16 <= L; i += 4 * stride) {
            uint4 v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) v[u] = __ldg(reinterpret_cast<const uint4 *>(src + i + u * stride));
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const uint32_t in[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
                uint32_t o4[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const uint32_t w = in[k], lc = w | 0x20202020u;
                    const uint32_t isc = __vcmpeq4(lc, 0x63636363u), isg = __vcmpeq4(lc, 0x67676767u), ist = __vcmpeq4(lc, 0x74747474u);
                    const uint32_t acgt = __vcmpeq4(lc, 0x61616161u) | isc | isg | ist;
                    const uint32_t gap = __vcmpeq4(lc, 0x6e6e6e6eu) | __vcmpeq4(w, 0x2e2e2e2eu) | __vcmpeq4(w, 0x2d2d2d2du);
                    local_bad |= (~(acgt | gap)) != 0u;
                    o4[k] = (isc & 0x01010101u) | (isg & 0x02020202u) | (ist & 0x03030303u) | (~acgt & 0x04040404u);
                }
                *reinterpret_cast<uint4 *>(dst + i + u * stride) = make_uint4(o4[0], o4[1], o4[2], o4[3]);
            }
        }
    }
    for (; i < cols_out; i += stride) {
        uint32_t out[4];
        if (vec && i + 16 <= L) {
            // four bytes per SIMD-in-register step: a data-dependent index into the constant-memory table would serialise the
            // warp (32 different addresses per load); byte-wise compares do not
            const uint4 v = __ldg(reinterpret_cast<const uint4 *>(src + i));
            const uint32_t in[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const uint32_t w = in[k], u = w | 0x20202020u;          // lower case (translation.hpp:29-53 accepts both)
                const uint32_t isc = __vcmpeq4(u, 0x63636363u), isg = __vcmpeq4(u, 0x67676767u), ist = __vcmpeq4(u, 0x74747474u);
                const uint32_t acgt = __vcmpeq4(u, 0x61616161u) | isc | isg | ist;
                const uint32_t gap = __vcmpeq4(u, 0x6e6e6e6eu) | __vcmpeq4(w, 0x2e2e2e2eu) | __vcmpeq4(w, 0x2d2d2d2du);   // N n . -
                local_bad |= (~(acgt | gap)) != 0u;
                out[k] = (isc & 0x01010101u) | (isg & 0x02020202u) | (ist & 0x03030303u) | (~acgt & 0x04040404u);
            }
        } else {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                uint32_t r = 0;
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    const int64_t p = i + 4 * k + b;
                    uint32_t c = 4;
                    if (p < L) {
                        c = c_dna_lut[src[p]];
                        local_bad |= (c == 255);
                        if (c == 255) c = 4;
                    }
                    r |= c << (8 * b);
                }
                out[k] = r;
            }
        }
        *reinterpret_cast<uint4 *>(dst + i) = make_uint4(out[0], out[1], out[2], out[3]);
    }
    if (local_bad) atomicOr(bad, 1);
}

// ---------------------------------------------------------------------------------------------------
// Window enumeration.  mode 0 (tracks): local window lw of a chunk starting at column c0 is
// (o = c0 + lw/2, strand = lw&1).  mode 1 (score-msa): o = win_off[lw], strand = win_strand[lw] (0 '+', 1 '-'), or '+' for every
// window when win_strand is null.  A '-' window at o is the codon comp(x[o+2]) comp(x[o+1]) comp(x[o]) (codon_minus).
struct WinSpace {
    const uint8_t *codes;
    int64_t ld;
    int nl;
    int mode;
    int64_t c0;
    const uint32_t *win_off;
    const uint8_t *win_strand;   // mode 1 only, nullable
};

// (column offset, strand) of local window lw
__device__ __forceinline__ int64_t win_column(const WinSpace &ws, uint32_t lw, uint32_t *strand) {
    if (ws.mode == 0) { *strand = lw & 1; return ws.c0 + (lw >> 1); }
    *strand = ws.win_strand ? ws.win_strand[lw] : 0u;
    return ws.win_off[lw];
}

__device__ __forceinline__ uint32_t codon_plus(uint32_t b0, uint32_t b1, uint32_t b2) {
    return ((b0 | b1 | b2) & 4u) ? 64u : 16u * b0 + 4u * b1 + b2;
}
__device__ __forceinline__ uint32_t codon_minus(uint32_t b0, uint32_t b1, uint32_t b2) {
    // complement(x) = 3 - x for A,C,G,T = 0..3 (translation.hpp:55-78); reading direction reversed
    return ((b0 | b1 | b2) & 4u) ? 64u : 16u * (3u - b2) + 4u * (3u - b1) + (3u - b0);
}

__device__ __forceinline__ uint64_t fmix64(uint64_t k) {
    k ^= k >> 33; k *= 0xff51afd7ed558ccdULL; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ULL; k ^= k >> 33;
    return k;
}

// 128-bit site-pattern key of one window: the nl codon ids (7 bits each) are packed nine to a 64-bit word and every full word is
// folded into two independent multiply-xor lanes — two 64-bit multiplies per nine species instead of per species (the kernel is bound
// by these integer multiplies, not by bytes).  Pattern identity = equality of the (fmix64(h1), fmix64(h2)) pair.
struct PatternHash {
    uint64_t h1 = 0x9E3779B97F4A7C15ULL, h2 = 0xC2B2AE3D27D4EB4FULL, acc = 0;
    __device__ __forceinline__ void fold() {
        h1 = (h1 ^ acc) * 0x100000001B3ULL;
        h1 ^= h1 >> 32;
        h2 = (h2 + acc + 1) * 0xFF51AFD7ED558CCDULL;
        h2 ^= h2 >> 29;
        acc = 0;
    }
    __device__ __forceinline__ void add(uint32_t codon) { acc = (acc << 7) | codon; }
};

// k_keys mode 0: both strands of FOUR consecutive column offsets per thread (two aligned 32-bit loads per species give the six
// bytes they share).  Needs rows and c0 that are multiples of four (rows are padded to 16, chunk starts are multiples of four).
__global__ void k_keys_tracks(WinSpace ws, int64_t ncols, ulonglong2 *__restrict__ klo, ulonglong2 *__restrict__ khi) {
    const int64_t t4 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (t4 >= ncols) return;
    const uint8_t *p = ws.codes + ws.c0 + t4;
    PatternHash hp[4], hm[4];
    int inword = 0;
    for (int s = 0; s < ws.nl; ++s, p += ws.ld) {
        const uint32_t w0 = *reinterpret_cast<const uint32_t *>(p), w1 = *reinterpret_cast<const uint32_t *>(p + 4);   // bytes t4 .. t4+7
        const uint32_t b[6] = {w0 & 0xff, (w0 >> 8) & 0xff, (w0 >> 16) & 0xff, w0 >> 24, w1 & 0xff, (w1 >> 8) & 0xff};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            hp[j].add(codon_plus(b[j], b[j + 1], b[j + 2]));
            hm[j].add(codon_minus(b[j], b[j + 1], b[j + 2]));
        }
        if (++inword == 9) {
            inword = 0;
#pragma unroll
            for (int j = 0; j < 4; ++j) { hp[j].fold(); hm[j].fold(); }
        }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        hp[j].fold(); hm[j].fold();
        if (t4 + j < ncols) {
            klo[t4 + j] = make_ulonglong2(fmix64(hp[j].h1), fmix64(hm[j].h1));
            khi[t4 + j] = make_ulonglong2(fmix64(hp[j].h2), fmix64(hm[j].h2));
        }
    }
}

// The same keys, one thread per column offset, for a window space whose first column is not a multiple of four.
__global__ void k_keys_tracks_unaligned(WinSpace ws, int64_t ncols, ulonglong2 *__restrict__ klo, ulonglong2 *__restrict__ khi) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= ncols) return;
    const uint8_t *p = ws.codes + ws.c0 + t;
    PatternHash hp, hm;
    int inword = 0;
    for (int s = 0; s < ws.nl; ++s, p += ws.ld) {
        const uint32_t x0 = p[0], x1 = p[1], x2 = p[2];
        hp.add(codon_plus(x0, x1, x2));
        hm.add(codon_minus(x0, x1, x2));
        if (++inword == 9) { inword = 0; hp.fold(); hm.fold(); }
    }
    hp.fold(); hm.fold();
    klo[t] = make_ulonglong2(fmix64(hp.h1), fmix64(hm.h1));
    khi[t] = make_ulonglong2(fmix64(hp.h2), fmix64(hm.h2));
}

// k_keys mode 1: one thread per listed window (the '-' codon id for a '-' window).
__global__ void k_keys_list(WinSpace ws, int64_t nwin, uint64_t *__restrict__ klo, uint64_t *__restrict__ khi) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nwin) return;
    const bool minus = ws.win_strand && ws.win_strand[t];
    const uint8_t *p = ws.codes + ws.win_off[t];
    uint64_t a1 = 0x9E3779B97F4A7C15ULL, a2 = 0xC2B2AE3D27D4EB4FULL;
    for (int s = 0; s < ws.nl; ++s, p += ws.ld) {
        const uint64_t cp = minus ? codon_minus(p[0], p[1], p[2]) : codon_plus(p[0], p[1], p[2]);
        a1 = (a1 ^ cp) * 0x100000001B3ULL;
        a2 = (a2 + cp + 1) * 0xFF51AFD7ED558CCDULL; a2 ^= a2 >> 29;
    }
    klo[t] = fmix64(a1);
    khi[t] = fmix64(a2);
}

// ---------------------------------------------------------------------------------------------------
// Dedup: open-addressing table of window ids keyed by the 128-bit pattern key; a key match is confirmed on the codon columns.
constexpr uint32_t EMPTY = 0xFFFFFFFFu;

// The nl codon ids of two windows, compared one by one.  Only windows whose 128-bit keys are equal get here (i.e. duplicates pay
// for it, nl x 6 byte loads), and it makes pattern identity exact instead of "equal up to a 128-bit hash collision".
__device__ __forceinline__ bool same_pattern(const WinSpace &ws, uint32_t w1, uint32_t w2) {
    uint32_t s1, s2;
    const int64_t o1 = win_column(ws, w1, &s1), o2 = win_column(ws, w2, &s2);
    const uint8_t *p = ws.codes + o1, *q = ws.codes + o2;
    for (int s = 0; s < ws.nl; ++s, p += ws.ld, q += ws.ld) {
        const uint32_t a = s1 ? codon_minus(p[0], p[1], p[2]) : codon_plus(p[0], p[1], p[2]);
        const uint32_t b = s2 ? codon_minus(q[0], q[1], q[2]) : codon_plus(q[0], q[1], q[2]);
        if (a != b) return false;
    }
    return true;
}

// table[slot] ends up holding the SMALLEST window id of the pattern that owns the slot: the first window of a pattern claims an empty
// slot with a CAS, every later one lowers the entry with atomicMin.  Whoever sits in a slot at any moment has the slot's pattern (entries
// only change from EMPTY to a window, or to a smaller window of the same pattern), so a probe may compare with whatever it reads.
__global__ void k_insert(WinSpace ws, const uint64_t *__restrict__ klo, const uint64_t *__restrict__ khi, uint32_t nwin,
                         uint32_t *table, uint32_t tmask, uint32_t *__restrict__ slot_of) {
    const uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= nwin) return;
    const uint64_t a = klo[w], b = khi[w];
    uint32_t slot = (uint32_t)(a ^ (a >> 32)) & tmask;
    while (true) {
        uint32_t cur = __ldcg(table + slot);
        if (cur == EMPTY) {
            const uint32_t prev = atomicCAS(table + slot, EMPTY, w);
            if (prev == EMPTY) break;
            cur = prev;
        }
        if (cur == w) break;
        if (klo[cur] == a && khi[cur] == b && same_pattern(ws, w, cur)) {
            if (w < cur) atomicMin(table + slot, w);
            break;
        }
        slot = (slot + 1) & tmask;
    }
    slot_of[w] = slot;
}

// rep[w] = smallest window id with the same pattern; flag[w] = (rep[w] == w).  rep overwrites slot_of.
__global__ void k_resolve(uint32_t nwin, uint32_t *__restrict__ slot_of_rep, const uint32_t *__restrict__ table,
                          uint32_t *__restrict__ flag) {
    const uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= nwin) return;
    const uint32_t rep = table[slot_of_rep[w]];
    slot_of_rep[w] = rep;
    flag[w] = (rep == w);
}

// Exclusive scan of flag[] in place (flag -> rank), 3 kernels, up to SCAN_BLOCK*SCAN_BLOCK... elements.
constexpr int SCAN_THREADS = 512;
constexpr int SCAN_ITEMS = 8;
constexpr int SCAN_BLOCK = SCAN_THREADS * SCAN_ITEMS;  // 4096 elements per block

__device__ __forceinline__ uint32_t block_excl_scan(uint32_t v, uint32_t *total, uint32_t *sh /*[33]*/) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t n = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += n;
    }
    if (lane == 31) sh[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        uint32_t x = lane < nw ? sh[lane] : 0, xi = x;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t n = __shfl_up_sync(0xffffffffu, xi, d);
            if (lane >= d) xi += n;
        }
        if (lane < nw) sh[lane] = xi - x;
        if (lane == 31) sh[32] = xi;
    }
    __syncthreads();
    const uint32_t res = inc - v + sh[warp];
    *total = sh[32];
    __syncthreads();
    return res;
}

__global__ void __launch_bounds__(SCAN_THREADS) k_scan_blocks(uint32_t *__restrict__ data, uint32_t n,
                                                             uint32_t *__restrict__ block_sums) {
    __shared__ uint32_t sh[33];
    const uint32_t base = blockIdx.x * SCAN_BLOCK + threadIdx.x * SCAN_ITEMS;
    uint32_t v[SCAN_ITEMS], sum = 0;
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
        v[i] = (base + i < n) ? data[base + i] : 0;
        sum += v[i];
    }
    uint32_t total;
    uint32_t run = block_excl_scan(sum, &total, sh);
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
        if (base + i < n) data[base + i] = run;
        run += v[i];
    }
    if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}

// single block: exclusive scan of up to 1024*32 block sums; writes the grand total to *n_total
__global__ void __launch_bounds__(1024) k_scan_sums(uint32_t *__restrict__ block_sums, uint32_t nblocks,
                                                    uint32_t *__restrict__ n_total) {
    __shared__ uint32_t sh[33];
    const uint32_t per = (nblocks + 1023) / 1024;
    const uint32_t base = threadIdx.x * per;
    uint32_t sum = 0;
    for (uint32_t i = 0; i < per; ++i)
        if (base + i < nblocks) sum += block_sums[base + i];
    uint32_t total;
    uint32_t run = block_excl_scan(sum, &total, sh);
    for (uint32_t i = 0; i < per; ++i)
        if (base + i < nblocks) {
            const uint32_t v = block_sums[base + i];
            block_sums[base + i] = run;
            run += v;
        }
    if (threadIdx.x == 0) *n_total = total;
}

// rank[w] (block-local) + block offset -> pattern index; unique list; optional pattern_index output.
__global__ void k_finalize(uint32_t nwin, const uint32_t *__restrict__ rep, const uint32_t *__restrict__ rank_local,
                           const uint32_t *__restrict__ block_sums, uint32_t *__restrict__ uniq,
                           uint32_t *__restrict__ pidx /* [nwin] chunk-local, always written */,
                           uint32_t *__restrict__ pattern_out /* nullable, global [2*(L-2)] */, int64_t out_base) {
    const uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= nwin) return;
    const uint32_t r = rep[w];
    const uint32_t pr = rank_local[r] + block_sums[r / SCAN_BLOCK];
    pidx[w] = pr;
    if (r == w) uniq[pr] = w;
    if (pattern_out) pattern_out[out_base + w] = pr;
}

__global__ void k_identity(uint32_t nwin, uint32_t *__restrict__ uniq, uint32_t *__restrict__ pidx,
                           uint32_t *__restrict__ n_total, uint32_t *__restrict__ pattern_out, int64_t out_base) {
    const uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w == 0) *n_total = nwin;
    if (w >= nwin) return;
    uniq[w] = w;
    pidx[w] = w;
    if (pattern_out) pattern_out[out_base + w] = w;
}

// ---------------------------------------------------------------------------------------------------
// PTX helpers: mbarrier + 1-D bulk TMA (cp.async.bulk -> UBLKCP) + FP64 DMMA.
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// The same wait with a suspend-time hint: the thread sleeps in hardware until the phase completes (or the hint expires) instead of
// spinning through the issue slots of its scheduler — for producer warps that share a scheduler with latency-critical warps.
__device__ __forceinline__ void mbar_wait_sleepy(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP_S:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n"
        "@p bra WAIT_DONE_S;\n"
        "bra WAIT_LOOP_S;\n"
        "WAIT_DONE_S:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity), "r"(20000u) : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void dmma(double &d0, double &d1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ---------------------------------------------------------------------------------------------------
// k_prune.  One persistent CTA per SM: 8 compute warps + 1 TMA producer warp.
//
// Formulation.  For one inner edge c -> parent the reference computes, per codon window w and parent
// state a,  msg[a] = sum_b P_c[a][b] * alpha_c[b]   (dot_with_alpha, fixed_lik.hpp:105-123; ensure_alpha
// :135-157).  Batched over windows that is D[w][a] = sum_b A[w][b] * B[b][a] with A = alpha_c^T and
// B = P_c^T: an (8 windows) x (64 states) x (64 states) FP64 GEMM per warp, done as 16 k-steps x 8 n-tiles of
// mma.sync.m8n8k4.f64.  With the k-steps permuted as b = 8*(ks/2) + 2*(lane%4) + (ks%2), the accumulator
// fragment of one GEMM (thread (g,q) holds states 8*nt + 2q + {0,1} of window g) IS the A fragment of the
// next GEMM: partials never leave registers between a node and its parent; leaf messages are gathered
// straight into the same layout (P_l[:, x] for a certain codon x, row sums for x = 64); sibling partials
// wait in a per-warp shared-memory stack (depth = Strahler number - 1 of the tree).
// B fragments (the P_c tiles, pre-ordered on the host so a warp's LDS.128 is 512 contiguous bytes) are
// streamed global -> shared by 1-D bulk TMA in program order through a 2-stage full/empty mbarrier ring.
constexpr int PR_MAX_NWARP = 12;            // compute warps: 12 (3 per SMSP) when shared memory allows, else 8
constexpr int PR_THREADS = (PR_MAX_NWARP + 1) * 32;   // launch bound; the launch uses (nwarp + 1) * 32
constexpr int PR_NSTAGE = 2;
constexpr int PR_TILE_BYTES = NS * NS * 8;  // 32 KB

// Per-tile descriptor (MLE): every alignment has its own P(rho) stream during the Brent search.
struct TileDesc {
    const double *pstream;   // [n_gemm][4096] of this tile's (alignment, model)
    const double *leafPT;    // [nl][65][64]
    int32_t model;           // 0 coding / 1 non-coding (selects pi)
    int32_t count;           // windows in this tile (<= 8 * nwarp)
    uint32_t win0;           // first window (index into ws.win_off) == output index
    uint32_t pad;
    const double *pi;        // nullable: this tile's own root prior (OMEGA: the equilibrium of the slot's current Q)
};

struct PruneArgs {
    WinSpace ws;
    const TileDesc *tiles;       // per-tile mode only
    const uint32_t *n_tiles;     // per-tile mode only (device scalar)
    const uint32_t *uniq;        // [n_unique] local window ids
    const uint32_t *n_unique;    // device scalar
    const int32_t *program;
    int n_ops, n_gemm, max_stack;
    int nwarp;                   // compute warps per CTA (8 windows each)
    const double *pstream[2];    // [n_gemm][4096] fragment-ordered
    const double *leafPT[2];     // [nl][65][64]
    const double *pi[2];
    const double *logpi[2];
    double *logz[2];             // [capacity]
    double *anc[2];              // nullable
    uint32_t stagger_ns;         // phase offset between the two warps of an SMSP (see k_prune)
};

__host__ __device__ inline size_t prune_smem_bytes(int nl, int n_ops, int max_stack, int nwarp) {
    size_t b = (size_t)PR_NSTAGE * PR_TILE_BYTES;            // P stages
    b += (size_t)nwarp * (max_stack > 0 ? max_stack : 1) * 4096;  // stacks
    b += (size_t)((nl * nwarp * 8 + 15) / 16) * 16;          // leaf codon ids
    b += (size_t)nwarp * 8 * 8;                              // window offsets
    b += (size_t)((n_ops * 4 + 15) / 16) * 16;               // program
    b += 4 * 64 * 8;                                         // pi, logpi x 2 models
    b += 2 * PR_NSTAGE * 8;                                  // mbarriers
    if (nl > SMALL_TREE_MAX_LEAVES) b += (size_t)nwarp * (max_stack > 0 ? max_stack : 1) * 32 * 4;   // exponents of the stack (k_prune_scaled)
    return b;
}

// k_prune_scaled (trees above SMALL_TREE_MAX_LEAVES leaves): an unscaled FP64 likelihood of a few hundred species can fall below the
// double range.  Every window carries an integer exponent e with true partial = R * 2^-e.  After each step that can shrink the partial
// (GEMM, leaf or stack Hadamard product), a window whose largest entry is below 2^-512 is multiplied by an exact power of two that brings
// that entry to [1, 2).  A window that never falls below the threshold keeps e = 0 and the unscaled arithmetic, bit for bit.
constexpr int PR_RESCALE_BIASED_EXP = 1023 - 512;

__device__ __forceinline__ void prune_rescale(double (&R)[16], int &e) {
    double mx = R[0];
#pragma unroll
    for (int i = 1; i < 16; ++i) mx = fmax(mx, R[i]);
    mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, 1));      // the four lanes of a window
    mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
    const int be = (int)((__double_as_longlong(mx) >> 52) & 0x7ff);   // partials are >= 0: biased exponent of the largest
    if (be < PR_RESCALE_BIASED_EXP && mx > 0.0) {
        const int k = min(1023 - be, 1022);
        const double f = __longlong_as_double((long long)(1023 + k) << 52);   // 2^k
#pragma unroll
        for (int i = 0; i < 16; ++i) R[i] *= f;
        e += k;
    }
}

template <bool PER_TILE, bool SCALED>
__device__ __forceinline__ void prune_body(const PruneArgs &a, unsigned char *smem) {
    unsigned char *sp_ = smem;
    const int PR_NWARP = a.nwarp, PR_TILE_W = a.nwarp * 8;
    double *stage_buf = reinterpret_cast<double *>(sp_); sp_ += (size_t)PR_NSTAGE * PR_TILE_BYTES;
    double2 *stack = reinterpret_cast<double2 *>(sp_); sp_ += (size_t)PR_NWARP * (a.max_stack > 0 ? a.max_stack : 1) * 4096;
    uint8_t *ids = sp_; sp_ += (size_t)((a.ws.nl * PR_TILE_W + 15) / 16) * 16;
    int64_t *s_woff = reinterpret_cast<int64_t *>(sp_); sp_ += (size_t)PR_TILE_W * 8;
    int32_t *prog = reinterpret_cast<int32_t *>(sp_); sp_ += (size_t)((a.n_ops * 4 + 15) / 16) * 16;
    double *s_pi = reinterpret_cast<double *>(sp_); sp_ += 4 * 64 * 8;   // [model][pi 64 | logpi 64]
    uint64_t *full = reinterpret_cast<uint64_t *>(sp_);
    uint64_t *empty = full + PR_NSTAGE;
    int *estack = reinterpret_cast<int *>(empty + PR_NSTAGE);   // SCALED: [warp][max_stack][lane] exponents of the stacked partials

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
        for (int s = 0; s < PR_NSTAGE; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, PR_NWARP); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int i = tid; i < a.n_ops; i += blockDim.x) prog[i] = a.program[i];
    for (int i = tid; i < 256; i += blockDim.x) {
        const int m = i >> 7, r = i & 127;
        s_pi[i] = r < 64 ? a.pi[m][r] : a.logpi[m][r - 64];
    }
    __syncthreads();

    const uint32_t n_unique = PER_TILE ? 0u : *a.n_unique;
    const uint32_t ntiles = PER_TILE ? *a.n_tiles : (n_unique + PR_TILE_W - 1) / PR_TILE_W;
    constexpr int NMODEL = PER_TILE ? 1 : 2;

    if (warp == PR_NWARP) {
        // ---- TMA producer: P tiles in program order, for every (tile, model) this CTA processes
        if (lane == 0) {
            uint32_t use = 0;
            for (uint32_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x)
                for (int m = 0; m < NMODEL; ++m) {
                    const double *ps = PER_TILE ? a.tiles[tile].pstream : a.pstream[m];
                    for (int g = 0; g < a.n_gemm; ++g, ++use) {
                        const uint32_t st = use % PR_NSTAGE;
                        mbar_wait(empty + st, ((use / PR_NSTAGE) & 1) ^ 1);
                        mbar_arrive_expect_tx(full + st, PR_TILE_BYTES);
                        tma_bulk_g2s(stage_buf + (size_t)st * NS * NS, ps + (size_t)g * NS * NS, PR_TILE_BYTES, full + st);
                    }
                }
        }
        return;
    }

    // ---- compute warps
    const int g = lane >> 2, q = lane & 3;
    const int mywin = warp * 8 + g;
    double2 *mystack = stack + (size_t)warp * (a.max_stack > 0 ? a.max_stack : 1) * 256;
    int *myestack = estack + (size_t)warp * (a.max_stack > 0 ? a.max_stack : 1) * 32 + lane;
    uint32_t use = 0;
    for (uint32_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        // leaf codon ids of this tile's 64 windows
        TileDesc td{};
        if (PER_TILE) td = a.tiles[tile];
        named_bar_sync(1, PR_NWARP * 32);
        // window -> (column offset, strand) once per window, then species-major byte gathers with independent loads
        if (tid < PR_TILE_W) {
            uint32_t lw;
            if (PER_TILE) {
                lw = td.win0 + (uint32_t)(tid < td.count ? tid : td.count - 1);
            } else {
                uint32_t u = tile * PR_TILE_W + tid;
                if (u >= n_unique) u = n_unique - 1;
                lw = a.uniq[u];
            }
            uint32_t strand;
            const int64_t o = win_column(a.ws, lw, &strand);
            s_woff[tid] = (o << 1) | strand;
        }
        named_bar_sync(1, PR_NWARP * 32);
#pragma unroll 4
        for (int i = tid; i < a.ws.nl * PR_TILE_W; i += PR_NWARP * 32) {
            const int s = i / PR_TILE_W, wi = i - s * PR_TILE_W;
            const int64_t ow = s_woff[wi];
            const uint8_t *p = a.ws.codes + (int64_t)s * a.ws.ld + (ow >> 1);
            const uint32_t x0 = p[0], x1 = p[1], x2 = p[2];
            ids[i] = (uint8_t)((ow & 1) ? codon_minus(x0, x1, x2) : codon_plus(x0, x1, x2));
        }
        named_bar_sync(1, PR_NWARP * 32);
        // Warps w and w+4 share an SMSP and would otherwise run the program in lockstep: both in the DMMA phase,
        // then both in the gather/stack phase with the tensor pipe idle.  A one-off phase offset per tile makes one
        // warp's non-DMMA phase overlap the other's DMMA phase.
        if (warp >= PR_NWARP / 2 && a.stagger_ns) __nanosleep(a.stagger_ns);

        // score-msa tiles belong to one alignment each and are rarely full (config 5: 68 % of the warps have windows): a warp without
        // windows only keeps the tile ring's barriers in step, its SMSP's DMMA pipe is left to the warp it shares it with
        const bool idle_warp = PER_TILE && (uint32_t)(warp * 8) >= td.count;
        for (int mm = 0; mm < NMODEL; ++mm) {
            const int m = PER_TILE ? td.model : mm;
            const double *leafPT = PER_TILE ? td.leafPT : a.leafPT[m];
            double R[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) R[i] = 0.0;
            int sp = 0;
            int e2 = 0;                       // SCALED: exponent of R
            if (idle_warp) {
                for (int pc = 0; pc < a.n_ops; ++pc) {
                    if ((prog[pc] >> 16) != OP_GEMM) continue;
                    const uint32_t st = use % PR_NSTAGE;
                    mbar_wait(full + st, (use / PR_NSTAGE) & 1);
                    __syncwarp();
                    if (lane == 0) mbar_arrive(empty + st);
                    ++use;
                }
                continue;
            }
            for (int pc = 0; pc < a.n_ops; ++pc) {
                const int32_t op = prog[pc];
                const int code = op >> 16, arg = op & 0xffff;
                if (code == OP_GATHER_SET || code == OP_GATHER_MUL) {
                    const int x = ids[arg * PR_TILE_W + mywin];
                    const double2 *row = reinterpret_cast<const double2 *>(leafPT + ((size_t)arg * 65 + x) * NS);
                    double2 v[8];
#pragma unroll
                    for (int nt = 0; nt < 8; ++nt) v[nt] = __ldg(row + nt * 4 + q);
                    if (code == OP_GATHER_SET) {
#pragma unroll
                        for (int nt = 0; nt < 8; ++nt) { R[2 * nt] = v[nt].x; R[2 * nt + 1] = v[nt].y; }
                        if (SCALED) e2 = 0;
                    } else {
#pragma unroll
                        for (int nt = 0; nt < 8; ++nt) { R[2 * nt] *= v[nt].x; R[2 * nt + 1] *= v[nt].y; }
                        if (SCALED) prune_rescale(R, e2);
                    }
                } else if (code == OP_GEMM) {
                    const uint32_t st = use % PR_NSTAGE;
                    mbar_wait(full + st, (use / PR_NSTAGE) & 1);
                    const double2 *bt = reinterpret_cast<const double2 *>(stage_buf + (size_t)st * NS * NS) + lane;
                    double acc[16];
#pragma unroll
                    for (int i = 0; i < 16; ++i) acc[i] = 0.0;
#pragma unroll
                    for (int ks = 0; ks < 16; ++ks) {
                        const double av = R[ks];   // R[2*(ks/2) + (ks%2)]
#pragma unroll
                        for (int ntp = 0; ntp < 4; ++ntp) {
                            const double2 b = bt[(ks * 4 + ntp) * 32];
                            dmma(acc[4 * ntp], acc[4 * ntp + 1], av, b.x);
                            dmma(acc[4 * ntp + 2], acc[4 * ntp + 3], av, b.y);
                        }
                    }
                    __syncwarp();
                    if (lane == 0) mbar_arrive(empty + st);
                    ++use;
#pragma unroll
                    for (int i = 0; i < 16; ++i) R[i] = acc[i];
                    if (SCALED) prune_rescale(R, e2);
                } else if (code == OP_PUSH) {
#pragma unroll
                    for (int nt = 0; nt < 8; ++nt) mystack[(sp * 8 + nt) * 32 + lane] = make_double2(R[2 * nt], R[2 * nt + 1]);
                    if (SCALED) myestack[sp * 32] = e2;
                    ++sp;
                } else if (code == OP_POP_MUL) {
                    --sp;
#pragma unroll
                    for (int nt = 0; nt < 8; ++nt) {
                        const double2 v = mystack[(sp * 8 + nt) * 32 + lane];
                        R[2 * nt] *= v.x; R[2 * nt + 1] *= v.y;
                    }
                    if (SCALED) {
                        e2 += myestack[sp * 32];
                        prune_rescale(R, e2);
                    }
                } else {  // OP_END: z = pi . alpha_root; log z; optional ancestral term
                    const double *pi = (PER_TILE && td.pi != nullptr) ? td.pi : s_pi + m * 128, *lpi = s_pi + m * 128 + 64;
                    double z = 0.0;
#pragma unroll
                    for (int nt = 0; nt < 8; ++nt) {
                        z += pi[8 * nt + 2 * q] * R[2 * nt];
                        z += pi[8 * nt + 2 * q + 1] * R[2 * nt + 1];
                    }
                    z += __shfl_xor_sync(0xffffffffu, z, 1);
                    z += __shfl_xor_sync(0xffffffffu, z, 2);
                    double e = 0.0;
                    if (a.anc[PER_TILE ? 0 : m] != nullptr) {
                        if (z != 0.0) {
#pragma unroll
                            for (int nt = 0; nt < 8; ++nt) {
                                e += lpi[8 * nt + 2 * q] * (R[2 * nt] * pi[8 * nt + 2 * q] / z);
                                e += lpi[8 * nt + 2 * q + 1] * (R[2 * nt + 1] * pi[8 * nt + 2 * q + 1] / z);
                            }
                        }
                        e += __shfl_xor_sync(0xffffffffu, e, 1);
                        e += __shfl_xor_sync(0xffffffffu, e, 2);
                    }
                    // the ancestral term is a ratio of the scaled partials: the scale cancels in it, and only log z is corrected
                    double lz = log(z);
                    if (SCALED && e2 != 0) lz -= (double)e2 * 0.6931471805599453094;
                    if (PER_TILE) {
                        if (q == 0 && mywin < td.count) {
                            a.logz[0][td.win0 + mywin] = lz;
                            if (a.anc[0] != nullptr) a.anc[0][td.win0 + mywin] = e;
                        }
                    } else {
                        const uint32_t u = tile * PR_TILE_W + mywin;
                        if (q == 0 && u < n_unique) {
                            a.logz[m][u] = lz;
                            if (a.anc[m] != nullptr) a.anc[m][u] = e;
                        }
                    }
                }
            }
        }
    }
}

template <bool PER_TILE>
__global__ void __launch_bounds__(PR_THREADS, 1) k_prune(const PruneArgs a) {
    extern __shared__ __align__(128) unsigned char smem[];
    prune_body<PER_TILE, false>(a, smem);
}
template <bool PER_TILE>
__global__ void __launch_bounds__(PR_THREADS, 1) k_prune_scaled(const PruneArgs a) {
    extern __shared__ __align__(128) unsigned char smem[];
    prune_body<PER_TILE, true>(a, smem);
}

// The pruning kernel of a tree of nl leaves: unscaled up to SMALL_TREE_MAX_LEAVES leaves (what the reference computes), rescaled above.
using PruneKernel = void (*)(PruneArgs);
template <bool PER_TILE>
inline PruneKernel prune_kernel(int nl) { return nl > SMALL_TREE_MAX_LEAVES ? k_prune_scaled<PER_TILE> : k_prune<PER_TILE>; }

// ---------------------------------------------------------------------------------------------------
// k_scatter (tracks): decibans of every window from its pattern's two log-likelihoods (run.hpp:51-54).
__global__ void k_scatter_tracks(uint32_t nwin, const uint32_t *__restrict__ pidx, const double *__restrict__ lc,
                                 const double *__restrict__ lnc, int64_t c0, double *__restrict__ plus,
                                 double *__restrict__ minus) {
    const uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= nwin) return;
    const uint32_t p = pidx[w];
    const double score = 10.0 * (lc[p] - lnc[p]) / log(10.0);
    const int64_t o = c0 + (w >> 1);
    if (w & 1) minus[o] = score; else plus[o] = score;
}

// k_scatter (score-msa): per-window log-likelihoods and ancestral terms of both models.
__global__ void k_scatter_list(uint32_t nwin, const uint32_t *__restrict__ pidx, const double *__restrict__ lc,
                               const double *__restrict__ lnc, const double *__restrict__ ac,
                               const double *__restrict__ anc, double *__restrict__ out /* [4][nwin] */) {
    const uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= nwin) return;
    const uint32_t p = pidx[w];
    out[w] = lc[p];
    out[(size_t)nwin + w] = lnc[p];
    out[2 * (size_t)nwin + w] = ac ? ac[p] : 0.0;
    out[3 * (size_t)nwin + w] = anc ? anc[p] : 0.0;
}

// ---------------------------------------------------------------------------------------------------
// k_bls: per-base branch length score.  One thread per column: presence mask of the species with A/C/G/T (get_dna_id <= 3,
// additional_scores.hpp:63) in NW 64-bit words (2 for trees of at most 128 leaves, 8 up to 512), then the post-order BLS program
// with a per-thread stack in shared memory; summation order (own + left) + right as in newick_sum_branch_lengths
// (additional_scores.hpp:5-41) => bit-identical doubles.
// raw != 0: write bl(S) itself (score-msa sums it, :71), else bl(S)/bl(all) (:73-74).
constexpr int BLS_THREADS = 128;
constexpr int BLS_COLS = 4;            // columns per thread: one 32-bit load per species, four independent evaluations in flight

template <int NW>
__global__ void __launch_bounds__(BLS_THREADS) k_bls(const uint8_t *__restrict__ codes, int64_t ld, int nl, int64_t L,
                                                    const BlsInnerDev<NW> *__restrict__ prog, int n_prog, int depth,
                                                    const double *__restrict__ tables, double all, int raw, double *__restrict__ out) {
    extern __shared__ double bls_stack[];  // [depth][BLS_COLS][BLS_THREADS]
    const int64_t i0 = ((int64_t)blockIdx.x * BLS_THREADS + threadIdx.x) * BLS_COLS;
    if (i0 >= L) return;
    // presence masks of four consecutive columns (rows are padded with N up to a multiple of 16 columns, so the word load is safe)
    uint64_t msk[NW][BLS_COLS];
#pragma unroll
    for (int i = 0; i < NW; ++i)
#pragma unroll
        for (int j = 0; j < BLS_COLS; ++j) msk[i][j] = 0;
    if constexpr (NW == 2) {
        for (int s = 0; s < nl; ++s) {
            const uint32_t w = __ldg(reinterpret_cast<const uint32_t *>(codes + (int64_t)s * ld + i0));
            const uint32_t present = ~(w >> 2) & 0x01010101u;          // code <= 3 (A, C, G, T): bit 2 clear
            if (s < 64) {
#pragma unroll
                for (int j = 0; j < BLS_COLS; ++j) msk[0][j] |= (uint64_t)((present >> (8 * j)) & 1u) << s;
            } else {
#pragma unroll
                for (int j = 0; j < BLS_COLS; ++j) msk[1][j] |= (uint64_t)((present >> (8 * j)) & 1u) << (s - 64);
            }
        }
    } else {
        // one word at a time into registers, then a static store into its place: the masks never leave registers
        for (int s0 = 0; s0 < nl; s0 += 64) {
            uint64_t word[BLS_COLS] = {0, 0, 0, 0};
            for (int s = s0; s < min(nl, s0 + 64); ++s) {
                const uint32_t w = __ldg(reinterpret_cast<const uint32_t *>(codes + (int64_t)s * ld + i0));
                const uint32_t present = ~(w >> 2) & 0x01010101u;
#pragma unroll
                for (int j = 0; j < BLS_COLS; ++j) word[j] |= (uint64_t)((present >> (8 * j)) & 1u) << (s - s0);
            }
#pragma unroll
            for (int i = 0; i < NW; ++i)
                if (64 * i == s0) {
#pragma unroll
                    for (int j = 0; j < BLS_COLS; ++j) msk[i][j] = word[j];
                }
        }
    }
    // inner nodes in post-order; a leaf child contributes its own branch length (no stack traffic), an inner child the value on
    // top of the stack (right child first: it was evaluated last).  Summation order = the reference's: (own + left) + right.
    // A TABLE entry (model_prep.hpp: bls_build_tables) pushes the tabulated value of a whole subtree of <= 12 leaves.
    double *st = bls_stack + threadIdx.x;
    int sp = 0;
    double v[BLS_COLS] = {0.0, 0.0, 0.0, 0.0};
    for (int k = 0; k < n_prog; ++k) {
        const BlsInnerDev<NW> e = prog[k];
        if (e.flags & 4) {
            const int nbits = (e.flags >> 16) & 0xff;
#pragma unroll
            for (int j = 0; j < BLS_COLS; ++j) {
                uint64_t out_of = 0;
#pragma unroll
                for (int i = 0; i < NW; ++i) out_of |= msk[i][j] & ~e.self[i];
                const bool arrived = out_of != 0;
                uint64_t bits;
                if constexpr (NW == 2) {
                    const int shift = (e.flags >> 8) & 0xff;
                    if (shift >= 64) bits = msk[1][j] >> (shift - 64);
                    else bits = (msk[0][j] >> shift) | (shift ? msk[1][j] << (64 - shift) : 0ull);
                } else {
                    // first leaf: bits 0-7 in flag bits 8-15, bits 8-15 in flag bits 24-31 (model_prep.hpp: bls_table_flags).  Every
                    // word shifts its part into place (no indexed access: the masks stay in registers)
                    const int shift = ((e.flags >> 8) & 0xff) | ((e.flags >> 16) & 0xff00);
                    bits = 0;
#pragma unroll
                    for (int i = 0; i < NW; ++i) {
                        const int d = 64 * i - shift;   // where word i starts, relative to the first leaf
                        if (d <= 0 && d > -64) bits |= msk[i][j] >> -d;
                        else if (d > 0 && d < 64) bits |= msk[i][j] << d;
                    }
                }
                bits &= (1ull << nbits) - 1;
                v[j] = __ldg(tables + e.tab_off + 2 * bits + (arrived ? 1 : 0));
            }
        } else {
            double r[BLS_COLS], l[BLS_COLS];
            if (e.flags & 2) {
#pragma unroll
                for (int j = 0; j < BLS_COLS; ++j) r[j] = e.right_bl;
            } else {
                --sp;
#pragma unroll
                for (int j = 0; j < BLS_COLS; ++j) r[j] = st[(sp * BLS_COLS + j) * BLS_THREADS];
            }
            if (e.flags & 1) {
#pragma unroll
                for (int j = 0; j < BLS_COLS; ++j) l[j] = e.left_bl;
            } else {
                --sp;
#pragma unroll
                for (int j = 0; j < BLS_COLS; ++j) l[j] = st[(sp * BLS_COLS + j) * BLS_THREADS];
            }
#pragma unroll
            for (int j = 0; j < BLS_COLS; ++j) {
                uint64_t out_of = 0, in_l = 0, in_r = 0;
#pragma unroll
                for (int i = 0; i < NW; ++i) {
                    out_of |= msk[i][j] & ~e.self[i];
                    in_l |= msk[i][j] & e.left[i];
                    in_r |= msk[i][j] & e.self[i] & ~e.left[i];
                }
                double x = out_of != 0 ? e.bl : 0.0;
                if (in_l != 0) x = __dadd_rn(x, l[j]);
                if (in_r != 0) x = __dadd_rn(x, r[j]);
                v[j] = x;
            }
        }
#pragma unroll
        for (int j = 0; j < BLS_COLS; ++j) st[(sp * BLS_COLS + j) * BLS_THREADS] = v[j];
        ++sp;
    }
#pragma unroll
    for (int j = 0; j < BLS_COLS; ++j) {
        if (i0 + j >= L) break;
        int present = 0;
#pragma unroll
        for (int i = 0; i < NW; ++i) present += __popcll(msk[i][j]);
        double res = 0.0;
        if (present >= 2) {          // fewer than two species with a base: 0 (additional_scores.hpp:66-69)
            res = v[j];
            if (!raw) res = __ddiv_rn(res, all);
        }
        out[i0 + j] = res;
    }
}

}  // namespace pcsf
