// model_prep.hpp — one-off host preparation of the device model blob.
//
// What the reference recomputes on every run_tracks()/run() call (PhyloCSFModel_make,
// src/instance.hpp:687-712: Q from the ECM, eigendecomposition, all P(t_b); lpr_leaves rebuilding
// every P again, src/fixed_lik.hpp:370-372; get_prior, :281-360) is done here ONCE per model:
//   * Q (instance.hpp:648-685), its real eigensystem (instance.hpp:309-434; symmetrised Jacobi instead
//     of gsl_eigen_nonsymmv — Q is reversible, so D^{1/2} Q D^{-1/2} is symmetric), pi (equilibrium row
//     of S^-1 at argmin|lambda|), P_b = S diag(exp(lambda t_b)) S^-1 with the reference's clamp /
//     diagonal fix-up / error checks (instance.hpp:487-640), t_b = double(float(double(bl_b) * rho))
//     (instance.hpp:299-307; newick_elem::branch_length is a float);
//   * the pruning program: a children-first traversal that finishes the subtree needing more live
//     partials first (values are order independent, fixed_lik.hpp:135-157), flattened into
//     GATHER/PUSH/POP/GEMM ops, plus the P matrices of the GEMM edges re-ordered into DMMA fragment order;
//   * the BLS program: post-order node list with "species below" masks (up to 512 bits) and the pointer tree's
//     double branch lengths (additional_scores.hpp:5-41).
#pragma once

#include <cmath>
#include <cstdint>
#include <cstring>
#include <string>
#include <vector>

namespace pcsf {

constexpr int NS = 64;

// Trees of up to this many leaves run the unscaled FP64 pruning (k_prune), the two-word BLS masks (k_bls<2>) and have a tcgen05
// program; larger ones (up to PCSF_MAX_LEAVES = 512) run k_prune_scaled and k_bls<8> and have no tcgen05 program (its leaf and
// source ids are 8-bit, and the tcgen05 kernel's shared memory holds no tree above 126 leaves anyway).
constexpr int SMALL_TREE_MAX_LEAVES = 128;
constexpr int BLS_MAX_WORDS = 8;   // 64-bit words of a leaf set: 512 leaves

// A set of leaves (bit l = leaf l), as wide as the largest tree.  The device programs carry only the words their tree needs.
struct LeafSet {
    uint64_t w[BLS_MAX_WORDS] = {};
    LeafSet operator|(const LeafSet &o) const { LeafSet r; for (int i = 0; i < BLS_MAX_WORDS; ++i) r.w[i] = w[i] | o.w[i]; return r; }
    LeafSet operator&(const LeafSet &o) const { LeafSet r; for (int i = 0; i < BLS_MAX_WORDS; ++i) r.w[i] = w[i] & o.w[i]; return r; }
    LeafSet operator~() const { LeafSet r; for (int i = 0; i < BLS_MAX_WORDS; ++i) r.w[i] = ~w[i]; return r; }
    bool any() const { uint64_t x = 0; for (int i = 0; i < BLS_MAX_WORDS; ++i) x |= w[i]; return x != 0; }
    int count() const { int c = 0; for (int i = 0; i < BLS_MAX_WORDS; ++i) c += __builtin_popcountll(w[i]); return c; }
    int first() const { for (int i = 0; i < BLS_MAX_WORDS; ++i) if (w[i]) return 64 * i + __builtin_ctzll(w[i]); return -1; }
    void set(int l) { w[l >> 6] |= 1ull << (l & 63); }
    static LeafSet all(int nl) { LeafSet r; for (int l = 0; l < nl; ++l) r.set(l); return r; }
    uint64_t bits(int shift, int nbits) const {   // nbits <= 63 bits starting at leaf `shift`
        const int i = shift >> 6, o = shift & 63;
        uint64_t v = w[i] >> o;
        if (o && i + 1 < BLS_MAX_WORDS) v |= w[i + 1] << (64 - o);
        return v & ((1ull << nbits) - 1);
    }
};

// ---- pruning program ops (int32: code << 16 | arg) -------------------------------------------------
enum : int32_t { OP_GATHER_SET = 1, OP_GATHER_MUL = 2, OP_PUSH = 3, OP_POP_MUL = 4, OP_GEMM = 5, OP_END = 6 };
inline int32_t mk_op(int code, int arg) { return (code << 16) | (arg & 0xffff); }

struct BlsNode {            // one post-order entry of the BLS program
    double bl;              // newick_node::branch_length (double)
    LeafSet self;           // leaves below this node
    LeafSet left;           // leaves below the left child (empty for leaves)
    int32_t is_leaf;
};

struct BlsInner {           // one INNER node of the BLS program, post-order; leaf children are folded in (their value is their own
    double bl;              // branch length, whatever the presence mask): half of the stack traffic of the node-per-entry program
    double left_bl, right_bl;    // the child's branch length if it is a leaf
    LeafSet self, left;
    int32_t flags;          // bit 0: left child is a leaf, bit 1: right child is a leaf;
                            // bit 2: TABLE entry — the value of this node for every presence pattern of its (<= BLS_TABLE_BITS, consecutively
                            // numbered) leaves and for arrived = 0 / 1 was tabulated on the host with the very same additions: the device
                            // pushes tables[tab_off + 2 * pattern + arrived]; number of the first leaf: bits 0-7 in bits 8-15, bits 8-15 in
                            // bits 24-31; bits 16-23: leaf count
    int32_t tab_off;
};
inline int bls_table_shift(int32_t flags) { return ((flags >> 8) & 0xff) | ((flags >> 16) & 0xff00); }
inline int32_t bls_table_flags(int shift, int nbits) { return 4 | ((shift & 0xff) << 8) | (nbits << 16) | ((shift >> 8) << 24); }

// The entry k_bls<NW> reads: the BlsInner with its masks cut to NW words (NW = 2 for trees of at most 128 leaves, 8 above).
template <int NW>
struct BlsInnerDev {
    double bl;
    double left_bl, right_bl;
    uint64_t self[NW], left[NW];
    int32_t flags;
    int32_t tab_off;
};
template <int NW>
inline std::vector<BlsInnerDev<NW>> bls_device_program(const std::vector<BlsInner> &prog) {
    std::vector<BlsInnerDev<NW>> out(prog.size());
    for (size_t k = 0; k < prog.size(); ++k) {
        const BlsInner &e = prog[k];
        BlsInnerDev<NW> &d = out[k];
        d.bl = e.bl; d.left_bl = e.left_bl; d.right_bl = e.right_bl;
        for (int i = 0; i < NW; ++i) { d.self[i] = e.self.w[i]; d.left[i] = e.left.w[i]; }
        d.flags = e.flags; d.tab_off = e.tab_off;
    }
    return out;
}

struct EcmHost {
    double lambda[NS], SR[NS * NS], SRinv[NS * NS], pi[NS], logpi[NS];
    std::vector<double> P;        // (n-1) x 64 x 64 at rho = 1, row-major P[a][b]
    std::vector<double> pstream;  // n_gemm tiles of 4096 doubles, DMMA fragment order, program order
    std::vector<double> leafPT;   // nl x 65 x 64: leafPT[l][x][a] = P_l[a][x], x = 64 -> row sums
    // tcgen05 path: one 32 KB tile per inner NON-CHERRY edge in step order (UMMA K-major no-swizzle B layout, N = 128 =
    // [hi | lo]) and, per cherry in program order, the cherry node's own P (row-major FP64) from which k_build_rows tabulates
    // the message of the edge above it (the leaves' columns come from leafPT)
    std::vector<float> pstream_tc5;
    std::vector<double> cherry_P;   // n_cherry x 64 x 64
};

// One row source of the tcgen05 program, in the order the program consumes them: the message table of a direct leaf (65 rows:
// codon x -> P_l[:, x], row 64 = all ones) or of a cherry (65 x 65 rows: x * 65 + y), rows of 64 floats at row_base of the
// ECM's row table.
struct Tc5Src {
    uint32_t row_base;
    uint8_t l1, l2;      // leaf ids whose codons select the row; l2 = 0xff for a leaf source
    uint8_t cherry;      // cherry number (index into cherry_P) for a cherry source
    uint8_t pad;
};

struct ModelHost {
    int nl = 0, n = 0;
    std::vector<int16_t> child1, child2;
    std::vector<float> bl;
    std::vector<double> bl64;
    EcmHost ecm[2];
    std::vector<int32_t> program;
    std::vector<int> gemm_edges;  // node id of the g-th GEMM op
    int max_stack = 0;
    // tcgen05 path (prepare_tc5_program): one step per GEMM (non-cherry inner edge) + what follows it up to the next GEMM
    std::vector<uint32_t> tc5_steps;   // src1 | src2 << 8 | post-op << 16 | END << 20
    std::vector<int> tc5_edges;        // node id of the edge of step s
    std::vector<int> tc5_leaf_order;   // direct leaves in the order the program gathers them (the leaf-table ring)
    std::vector<int> tc5_cherries;     // cherry node ids in the order the program consumes their tables
    std::vector<uint16_t> tc5_cherry_leaves;   // left leaf | right leaf << 8 of cherry k
    std::vector<Tc5Src> tc5_srcs;      // every source, in consumption order
    uint32_t tc5_rows = 0;             // rows of one ECM's row table
    uint32_t tc5_start = 0;            // src1 | src2 << 8 of the chain start the program begins with
    int tc5_max_stack = 0;             // pushes alive at once (depth of the global-memory stack)
    std::vector<BlsNode> bls_prog;
    std::vector<BlsInner> bls_inner;
    std::vector<BlsInner> bls_short;      // the program k_bls runs: subtrees of <= BLS_TABLE_BITS leaves collapsed into TABLE entries
    std::vector<double> bls_tables;
    int bls_short_depth = 0;
    int bls_depth = 0;
    double bls_all = 0.0;         // all_species_branch_length (additional_scores.hpp:56)
};

// instance.hpp:648-685
inline void build_q(const double *S, const double *f, double *Q) {
    double scale = 0.0;
    for (int i = 0; i < NS; ++i) {
        double rowsum = 0.0;
        for (int j = 0; j < NS; ++j) {
            const double v = S[i * NS + j] * f[j];
            Q[i * NS + j] = v;
            rowsum -= v;
        }
        Q[i * NS + i] = rowsum;
        scale -= rowsum * f[i];
    }
    for (int i = 0; i < NS * NS; ++i) Q[i] /= scale;
}

// Symmetric eigenproblem by cyclic Jacobi rotations.  A is overwritten; V's columns are eigenvectors.
inline void jacobi64(std::vector<double> &A, std::vector<double> &V, double *w) {
    for (int i = 0; i < NS; ++i)
        for (int j = 0; j < NS; ++j) V[i * NS + j] = (i == j);
    for (int sweep = 0; sweep < 128; ++sweep) {
        double off = 0.0;
        for (int p = 0; p < NS; ++p)
            for (int q = p + 1; q < NS; ++q) off += A[p * NS + q] * A[p * NS + q];
        if (off < 1e-300) break;
        for (int p = 0; p + 1 < NS; ++p)
            for (int q = p + 1; q < NS; ++q) {
                const double apq = A[p * NS + q];
                if (std::fabs(apq) < 1e-310) continue;
                const double theta = (A[q * NS + q] - A[p * NS + p]) / (2.0 * apq);
                const double t = std::copysign(1.0, theta) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
                const double c = 1.0 / std::sqrt(t * t + 1.0), s = t * c;
                for (int k = 0; k < NS; ++k) {
                    const double x = A[k * NS + p], y = A[k * NS + q];
                    A[k * NS + p] = c * x - s * y;
                    A[k * NS + q] = s * x + c * y;
                }
                for (int k = 0; k < NS; ++k) {
                    const double x = A[p * NS + k], y = A[q * NS + k];
                    A[p * NS + k] = c * x - s * y;
                    A[q * NS + k] = s * x + c * y;
                }
                for (int k = 0; k < NS; ++k) {
                    const double x = V[k * NS + p], y = V[k * NS + q];
                    V[k * NS + p] = c * x - s * y;
                    V[k * NS + q] = s * x + c * y;
                }
            }
    }
    for (int i = 0; i < NS; ++i) w[i] = A[i * NS + i];
}

// instance.hpp:309-434 (real spectrum) + fixed_lik.hpp:323-346 (equilibrium)
inline bool eigen_and_prior(const double *Q, const double *f, EcmHost &e, std::string &err) {
    double sq[NS];
    for (int i = 0; i < NS; ++i) {
        if (!(f[i] > 0.0)) { err = "codon frequencies must be strictly positive"; return false; }
        sq[i] = std::sqrt(f[i]);
    }
    std::vector<double> A(NS * NS), U(NS * NS);
    for (int i = 0; i < NS; ++i)
        for (int j = 0; j < NS; ++j) A[i * NS + j] = sq[i] * Q[i * NS + j] / sq[j];
    for (int i = 0; i < NS; ++i)
        for (int j = i + 1; j < NS; ++j) A[i * NS + j] = A[j * NS + i] = 0.5 * (A[i * NS + j] + A[j * NS + i]);
    jacobi64(A, U, e.lambda);
    for (int i = 0; i < NS; ++i)
        for (int k = 0; k < NS; ++k) {
            e.SR[i * NS + k] = U[i * NS + k] / sq[i];
            e.SRinv[k * NS + i] = U[i * NS + k] * sq[i];
        }
    int kmin = 0;
    double best = std::fabs(e.lambda[0]);
    for (int k = 1; k < NS; ++k)
        if (std::fabs(e.lambda[k]) < best) { best = std::fabs(e.lambda[k]); kmin = k; }
    double mass = 0.0;
    for (int j = 0; j < NS; ++j) mass += e.SRinv[kmin * NS + j];
    for (int j = 0; j < NS; ++j) {
        e.pi[j] = e.SRinv[kmin * NS + j] / mass;
        e.logpi[j] = std::log(e.pi[j]);
    }
    return true;
}

inline double branch_time(float bl, double rho) { return (double)(float)((double)bl * rho); }

// instance.hpp:487-640, one branch.  0 ok, 1 negative entry beyond tolerance, 2 row sum off.
inline int pmatrix(const EcmHost &e, double t, double *P) {
    double ex[NS];
    std::vector<double> B(NS * NS);
    for (int k = 0; k < NS; ++k) ex[k] = std::exp(e.lambda[k] * t);
    for (int k = 0; k < NS; ++k)
        for (int j = 0; j < NS; ++j) B[k * NS + j] = e.SRinv[k * NS + j] * ex[k];
    for (int i = 0; i < NS; ++i) {
        double *row = P + i * NS;
        for (int j = 0; j < NS; ++j) row[j] = 0.0;
        for (int k = 0; k < NS; ++k) {
            const double a = e.SR[i * NS + k];
            for (int j = 0; j < NS; ++j) row[j] += a * B[k * NS + j];
        }
    }
    for (int i = 0; i < NS; ++i) {
        double total = 0.0, diag = 1.0;
        for (int j = 0; j < NS; ++j) {
            const double cell = P[i * NS + j];
            total += cell;
            if (cell < 0.0) {
                if (std::fabs(cell) > 1e-6) return 1;
                P[i * NS + j] = 0.0;
            }
            if (i != j) diag -= P[i * NS + j];
        }
        if (std::fabs(total - 1.0) > 1e-6) return 2;
        P[i * NS + i] = diag;
    }
    return 0;
}

// DMMA m8n8k4 fragment order of one 64x64 P for the chained, K-permuted GEMM of k_prune:
//   tile[ks][ntp][lane][e] = P[a][b],  a = 8*(2*ntp+e) + lane/4,  b = 8*(ks/2) + 2*(lane%4) + (ks%2)
inline void to_fragment_order(const double *P, double *tile) {
    for (int ks = 0; ks < 16; ++ks)
        for (int ntp = 0; ntp < 4; ++ntp)
            for (int lane = 0; lane < 32; ++lane)
                for (int e = 0; e < 2; ++e) {
                    const int a = 8 * (2 * ntp + e) + lane / 4;
                    const int b = 8 * (ks / 2) + 2 * (lane % 4) + (ks % 2);
                    tile[((ks * 4 + ntp) * 32 + lane) * 2 + e] = P[a * NS + b];
                }
}

// cvt.rna.tf32.f32 on the host: round to 10 explicit mantissa bits, ties away from zero.
inline float tf32_rna(float x) {
    uint32_t u;
    std::memcpy(&u, &x, 4);
    u = (u + 0x1000u) & 0xffffe000u;
    float r;
    std::memcpy(&r, &u, 4);
    return r;
}

// ---- tcgen05 path ------------------------------------------------------------------------------------------
// Sources of a factor that is not a GEMM result.  A LEAF's message is column x of P_l (gathered from a shared-memory table);
// a CHERRY's message (the edge above a node whose two children are leaves) depends only on the two leaves' codons, so it is
// tabulated once per model: T_c[x][y][a] = sum_b P_c[a][b] P_l[b][x] P_r[b][y], x, y in 0..64 (64 = gap/N: all ones),
// 4225 rows of 64 floats in global memory (L2), and GATHERED — no GEMM, no leaf gathers, no stack push for that edge.
//   source byte: bit 7 = cherry, bits 0-6 = leaf id (leaf) / cherry number in program order (cherry)
// Step word: bits 0-7 src1, 8-15 src2, 16-17 post-op (what the program does between this GEMM and the next), bit 20 END.
//   T5_MUL         alpha_parent = msg * src1
//   T5_PUSH_START  push msg; alpha of a new chain = src1 * src2 (a node whose two children are leaves / cherries)
//   T5_POP_MUL     alpha_parent = msg * pop
enum : uint32_t { T5_NONE = 0, T5_MUL = 1, T5_PUSH_START = 2, T5_POP_MUL = 3, T5_END = 1u << 20, T5_SRC_CHERRY = 0x80u };
constexpr int T5_CHERRY_ROWS = 65 * 65;
// One inner edge as the B operand of tcgen05.mma kind::tf32 (K-major, no swizzle): B[n][k], n = 0..127, k = 0..63 with
// B[n][k] = hi(P[n][k]) for n < 64 and lo(P[n-64][k]) for n >= 64, so that D[w][0:64] + D[w][64:128] = sum_k A[w][k] P[.][k].
// Chunk j (k = 8j..8j+7) is 4 KB contiguous; inside a chunk 8-row x 16-byte core matrices: 8-row group stride 256 B
// (SBO), the two K halves 128 B apart (LBO).
inline void to_tc5_tile(const double *P, float *tile /* 8192 floats */) {
    for (int n = 0; n < 128; ++n)
        for (int k = 0; k < NS; ++k) {
            const double p = P[(n & 63) * NS + k];
            const float hi = tf32_rna((float)p);
            const float v = n < 64 ? hi : tf32_rna((float)(p - (double)hi));
            tile[(k / 8) * 1024 + (n / 8) * 64 + ((k % 8) / 4) * 32 + (n % 8) * 4 + (k % 4)] = v;
        }
}
inline void to_leaf_table(const double *P, double *pt /* 65 x 64 */) {
    for (int a = 0; a < NS; ++a) {
        double rs = 0.0;
        for (int x = 0; x < NS; ++x) {
            pt[x * NS + a] = P[a * NS + x];
            rs += P[a * NS + x];   // fixed_lik.hpp:116-118: sum over j ascending
        }
        pt[64 * NS + a] = rs;
    }
}

namespace detail {
inline int strahler(const ModelHost &m, int i, std::vector<int> &need) {
    if (m.child1[i] < 0) return need[i] = 0;
    const int a = strahler(m, m.child1[i], need), b = strahler(m, m.child2[i], need);
    int r = (a == b) ? (a == 0 ? 1 : a + 1) : (a > b ? a : b);
    return need[i] = r;
}
// emits ops leaving alpha_i (the partial of node i) in R
inline void emit_partial(ModelHost &m, int i, const std::vector<int> &need, int &sp);
// emits ops leaving the message of child c to its parent in R (inner child) — or a gather (leaf child)
inline void emit_msg(ModelHost &m, int c, const std::vector<int> &need, int &sp, bool first) {
    if (m.child1[c] < 0) {
        m.program.push_back(mk_op(first ? OP_GATHER_SET : OP_GATHER_MUL, c));
    } else {
        emit_partial(m, c, need, sp);
        m.program.push_back(mk_op(OP_GEMM, (int)m.gemm_edges.size()));
        m.gemm_edges.push_back(c);
    }
}
inline void emit_partial(ModelHost &m, int i, const std::vector<int> &need, int &sp) {
    const int c1 = m.child1[i], c2 = m.child2[i];
    const bool l1 = m.child1[c1] < 0, l2 = m.child1[c2] < 0;
    if (l1 && l2) {
        emit_msg(m, c1, need, sp, true);
        emit_msg(m, c2, need, sp, false);
    } else if (l1 != l2) {
        const int inner = l1 ? c2 : c1, leaf = l1 ? c1 : c2;
        emit_msg(m, inner, need, sp, true);
        emit_msg(m, leaf, need, sp, false);
    } else {
        const int first = need[c1] >= need[c2] ? c1 : c2, second = first == c1 ? c2 : c1;
        emit_msg(m, first, need, sp, true);
        m.program.push_back(mk_op(OP_PUSH, 0));
        ++sp;
        if (sp > m.max_stack) m.max_stack = sp;
        emit_msg(m, second, need, sp, true);
        m.program.push_back(mk_op(OP_POP_MUL, 0));
        --sp;
    }
}
// ---- tcgen05 path program (cherry tables) -------------------------------------------------------------------------
// Node kinds: 'L' leaf, 'C' cherry (both children leaves; not the root: its message is tabulated), 'I' every other
// inner node.  Only edges above 'I' nodes are GEMMs.
struct Tc5Emit {
    ModelHost &m;
    std::vector<char> kind;
    std::vector<int> need;                // live partials needed to evaluate the subtree (Strahler number over 'I' nodes)
    std::vector<uint32_t> ops;            // (code << 16) | a | b << 8: 1 START(a, b), 2 GEMM, 3 MUL(a), 4 PUSH, 5 POP_MUL
    std::vector<int> op_edge;             // node id for GEMM ops
    int sp = 0;
    explicit Tc5Emit(ModelHost &mm) : m(mm), kind(mm.n), need(mm.n, 0) {}
    void classify(int i) {
        if (m.child1[i] < 0) { kind[i] = 'L'; return; }
        classify(m.child1[i]); classify(m.child2[i]);
        const bool cherry = kind[m.child1[i]] == 'L' && kind[m.child2[i]] == 'L' && i != m.n - 1;
        kind[i] = cherry ? 'C' : 'I';
        if (kind[i] == 'I') {
            const int a = need[m.child1[i]], b = need[m.child2[i]];
            need[i] = (a == 0 && b == 0) ? 1 : (a == b ? a + 1 : (a > b ? a : b));
        }
    }
    uint32_t src(int c) {                 // c is 'L' or 'C': registers its table in program order
        Tc5Src d{};
        d.row_base = m.tc5_rows;
        if (kind[c] == 'L') {
            m.tc5_leaf_order.push_back(c);
            d.l1 = (uint8_t)c; d.l2 = 0xff;
            m.tc5_rows += 65;
            m.tc5_srcs.push_back(d);
            return (uint32_t)c;
        }
        const uint32_t k = (uint32_t)m.tc5_cherries.size();
        m.tc5_cherries.push_back(c);
        m.tc5_cherry_leaves.push_back((uint16_t)(m.child1[c] | (m.child2[c] << 8)));
        d.l1 = (uint8_t)m.child1[c]; d.l2 = (uint8_t)m.child2[c]; d.cherry = (uint8_t)k;
        m.tc5_rows += T5_CHERRY_ROWS;
        m.tc5_srcs.push_back(d);
        return T5_SRC_CHERRY | k;
    }
    void alpha(int i) {                   // leaves alpha_i as the running partial
        const int c1 = m.child1[i], c2 = m.child2[i];
        const bool i1 = kind[c1] == 'I', i2 = kind[c2] == 'I';
        if (!i1 && !i2) {
            const uint32_t a = src(c1), b = src(c2);
            ops.push_back((1u << 16) | a | (b << 8)); op_edge.push_back(-1);
        } else if (i1 != i2) {
            const int inner = i1 ? c1 : c2, other = i1 ? c2 : c1;
            msg(inner);
            ops.push_back((3u << 16) | src(other)); op_edge.push_back(-1);
        } else {
            const int first = need[c1] >= need[c2] ? c1 : c2, second = first == c1 ? c2 : c1;
            msg(first);
            ops.push_back(4u << 16); op_edge.push_back(-1);
            if (++sp > m.tc5_max_stack) m.tc5_max_stack = sp;
            msg(second);
            ops.push_back(5u << 16); op_edge.push_back(-1);
            --sp;
        }
    }
    void msg(int c) { alpha(c); ops.push_back(2u << 16); op_edge.push_back(c); }
};

// Returns nullptr on success.
inline const char *prepare_tc5_program(ModelHost &m) {
    m.tc5_steps.clear(); m.tc5_edges.clear(); m.tc5_leaf_order.clear(); m.tc5_cherries.clear(); m.tc5_cherry_leaves.clear();
    m.tc5_max_stack = 0; m.tc5_start = 0; m.tc5_srcs.clear(); m.tc5_rows = 0;
    Tc5Emit e(m);
    e.classify(m.n - 1);
    e.alpha(m.n - 1);
    const std::vector<uint32_t> &ops = e.ops;
    auto code = [&](size_t i) { return i < ops.size() ? ops[i] >> 16 : 0u; };
    if (code(0) != 1) return "internal error: tcgen05 program does not begin with a chain start";
    m.tc5_start = ops[0] & 0xffffu;
    size_t i = 1;
    while (code(i) == 2) {
        uint32_t w = 0;
        m.tc5_edges.push_back(e.op_edge[i]);
        ++i;
        if (code(i) == 3) { w = (ops[i] & 0xffu) | (T5_MUL << 16); ++i; }
        else if (code(i) == 4) {
            if (code(i + 1) != 1) return "internal error: tcgen05 program: PUSH not followed by a chain start";
            w = (ops[i + 1] & 0xffffu) | (T5_PUSH_START << 16);
            i += 2;
        } else if (code(i) == 5) { w = T5_POP_MUL << 16; ++i; }
        else return "internal error: tcgen05 program: a message is neither multiplied nor pushed";
        m.tc5_steps.push_back(w);
    }
    if (!m.tc5_steps.empty()) m.tc5_steps.back() |= T5_END;
    int n_inner_edges = 0;
    for (int v = m.nl; v < m.n - 1; ++v) n_inner_edges += e.kind[v] == 'I';
    if (i != ops.size() || (int)m.tc5_steps.size() != n_inner_edges ||
        (int)m.tc5_leaf_order.size() + 2 * (int)m.tc5_cherries.size() != m.nl || m.tc5_cherries.size() > 127)
        return "internal error: tcgen05 step list";
    return nullptr;
}

inline void bls_walk(ModelHost &m, int i, LeafSet &below, int &depth_out) {
    BlsNode e{};
    e.bl = m.bl64[i];
    if (m.child1[i] < 0) {
        e.is_leaf = 1;
        e.self.set(i);
        below = e.self;
        depth_out = 1;
        m.bls_prog.push_back(e);
        return;
    }
    LeafSet l, r;
    int dl, dr;
    bls_walk(m, m.child1[i], l, dl);
    bls_walk(m, m.child2[i], r, dr);
    e.left = l;
    e.self = l | r;
    below = e.self;
    depth_out = dl > dr + 1 ? dl : dr + 1;
    m.bls_prog.push_back(e);
    BlsInner in{};
    in.bl = e.bl;
    const int cl = m.child1[i], cr = m.child2[i];
    in.left_bl = m.bl64[cl]; in.right_bl = m.bl64[cr];
    in.self = e.self; in.left = l;
    in.flags = (m.child1[cl] < 0 ? 1 : 0) | (m.child1[cr] < 0 ? 2 : 0);
    m.bls_inner.push_back(in);
}
}  // namespace detail

// Host restatement of newick_sum_branch_lengths over the BLS program (also what k_bls executes).
inline double bls_eval_host(const ModelHost &m, const LeafSet &mask) {
    std::vector<double> st(m.bls_depth + 2);
    int sp = 0;
    for (const BlsNode &e : m.bls_prog) {
        if (e.is_leaf) { st[sp++] = e.bl; continue; }
        const double r = st[--sp], l = st[--sp];
        const bool ol = (mask & e.left).any();
        const bool orr = (mask & e.self & ~e.left).any();
        const bool arrived = (mask & ~e.self).any();
        double v = arrived ? e.bl : 0.0;
        if (ol) v += l;
        if (orr) v += r;
        st[sp++] = v;
    }
    return st[0];
}

// The inner-node program (what k_bls executed before the tables): value on top of the stack right after entry `upto`.
inline double bls_eval_inner_host(const std::vector<BlsInner> &prog, int depth, const LeafSet &mask, int upto) {
    std::vector<double> st(depth + 2);
    int sp = 0;
    double v = 0.0;
    for (int k = 0; k <= upto; ++k) {
        const BlsInner &e = prog[k];
        double r, l;
        if (e.flags & 2) r = e.right_bl; else r = st[--sp];
        if (e.flags & 1) l = e.left_bl; else l = st[--sp];
        const bool ol = (mask & e.left).any();
        const bool orr = (mask & e.self & ~e.left).any();
        const bool arrived = (mask & ~e.self).any();
        v = arrived ? e.bl : 0.0;
        if (ol) v += l;
        if (orr) v += r;
        st[sp++] = v;
    }
    return v;
}

constexpr int BLS_TABLE_BITS = 12;

// Collapses every maximal subtree of <= BLS_TABLE_BITS leaves into one TABLE entry.  A node's value depends only on which of ITS leaves
// are present and on whether any leaf outside is (arrived): 2^k x 2 doubles, computed by the inner-node program itself, so the
// device reads exactly the doubles it would have summed (58mammals: 16 entries instead of 57, 113 KB of tables).
inline void bls_build_tables(ModelHost &m) {
    m.bls_short.clear();
    m.bls_tables.clear();
    const int n_inner = (int)m.bls_inner.size();
    // post-order program: the subtree of entry k is a contiguous run of entries ending at k; find its first entry by counting
    std::vector<int> first(n_inner);
    {
        std::vector<int> stack;          // start index of the run of every value currently on the stack
        for (int k = 0; k < n_inner; ++k) {
            const BlsInner &e = m.bls_inner[k];
            int f = k;
            if (!(e.flags & 2)) { f = std::min(f, stack.back()); stack.pop_back(); }
            if (!(e.flags & 1)) { f = std::min(f, stack.back()); stack.pop_back(); }
            first[k] = f;
            stack.push_back(f);
        }
    }
    std::vector<char> is_root(n_inner, 0);
    for (int k = n_inner - 1; k >= 0; --k) {
        const BlsInner &e = m.bls_inner[k];
        if (e.self.count() > BLS_TABLE_BITS) continue;
        bool inside = false;             // already inside a collapsed subtree?
        for (int r = k + 1; r < n_inner && !inside; ++r) inside = is_root[r] && first[r] <= k;
        if (!inside) is_root[k] = 1;
    }
    const LeafSet all = LeafSet::all(m.nl);
    for (int k = 0; k < n_inner; ++k) {
        bool dropped = false;
        for (int r = k + 1; r < n_inner && !dropped; ++r) dropped = is_root[r] && first[r] <= k;
        if (dropped) continue;
        BlsInner e = m.bls_inner[k];
        if (is_root[k]) {
            const int nbits = e.self.count();
            const int shift = e.self.first();
            // one leaf outside the subtree stands for "arrived" (none exists when the subtree is the whole tree: arrived is never set)
            const int outside = (all & ~e.self).first();
            e.flags = bls_table_flags(shift, nbits);
            e.tab_off = (int32_t)m.bls_tables.size();
            for (uint64_t pat = 0; pat < (1ull << nbits); ++pat)
                for (int arrived = 0; arrived < 2; ++arrived) {
                    LeafSet mask;
                    for (int b = 0; b < nbits; ++b)
                        if ((pat >> b) & 1) mask.set(shift + b);
                    if (arrived && outside >= 0) mask.set(outside);
                    m.bls_tables.push_back(bls_eval_inner_host(m.bls_inner, m.bls_depth, mask, k));
                }
        }
        m.bls_short.push_back(e);
    }
    // stack depth of the short program
    int sp = 0, depth = 1;
    for (const BlsInner &e : m.bls_short) {
        if (!(e.flags & 4)) { if (!(e.flags & 2)) --sp; if (!(e.flags & 1)) --sp; }
        ++sp;
        depth = std::max(depth, sp);
    }
    m.bls_short_depth = depth;
    if (m.bls_tables.empty()) m.bls_tables.push_back(0.0);
}

// What k_bls executes, on the host (self-check at model creation).
inline double bls_eval_short_host(const ModelHost &m, const LeafSet &mask) {
    std::vector<double> st(m.bls_short_depth + 2);
    int sp = 0;
    double v = 0.0;
    for (const BlsInner &e : m.bls_short) {
        const bool arrived = (mask & ~e.self).any();
        if (e.flags & 4) {
            const uint64_t bits = mask.bits(bls_table_shift(e.flags), (e.flags >> 16) & 0xff);
            v = m.bls_tables[(size_t)e.tab_off + 2 * bits + (arrived ? 1 : 0)];
        } else {
            double r, l;
            if (e.flags & 2) r = e.right_bl; else r = st[--sp];
            if (e.flags & 1) l = e.left_bl; else l = st[--sp];
            const bool ol = (mask & e.left).any();
            const bool orr = (mask & e.self & ~e.left).any();
            v = arrived ? e.bl : 0.0;
            if (ol) v += l;
            if (orr) v += r;
        }
        st[sp++] = v;
    }
    return v;
}

// Returns "" on success.
inline std::string prepare_model(ModelHost &m, int nl, const int16_t *c1, const int16_t *c2, const float *bl,
                                 const double *bl64, const double *const S[2], const double *const f[2]) {
    m.nl = nl;
    m.n = 2 * nl - 1;
    m.child1.assign(c1, c1 + m.n);
    m.child2.assign(c2, c2 + m.n);
    m.bl.assign(bl, bl + m.n);
    m.bl64.assign(bl64, bl64 + m.n);
    for (int i = 0; i < m.n; ++i) {
        const bool leaf = i < nl;
        if (leaf != (c1[i] < 0) || leaf != (c2[i] < 0)) return "tree is not in newick_flatten order (leaves first)";
        if (!leaf && (c1[i] >= i || c2[i] >= i || c1[i] < 0 || c2[i] < 0)) return "inner nodes must follow their children";
    }
    // pruning program
    std::vector<int> need(m.n);
    detail::strahler(m, m.n - 1, need);
    int sp = 0;
    m.program.clear(); m.gemm_edges.clear(); m.max_stack = 0;
    detail::emit_partial(m, m.n - 1, need, sp);
    m.program.push_back(mk_op(OP_END, 0));
    if ((int)m.gemm_edges.size() != nl - 2) return "internal error: GEMM count";
    // the tcgen05 program only for trees it can hold (8-bit leaf and source ids; k_prune_tc5 refuses every tree above 126 leaves)
    if (nl <= SMALL_TREE_MAX_LEAVES)
        if (const char *terr = detail::prepare_tc5_program(m)) return terr;
    // BLS program
    LeafSet below;
    m.bls_prog.clear();
    m.bls_inner.clear();
    detail::bls_walk(m, m.n - 1, below, m.bls_depth);
    const LeafSet all = LeafSet::all(nl);
    m.bls_all = bls_eval_host(m, all);
    bls_build_tables(m);
    {   // the collapsed program must give the node-by-node program's doubles, bit for bit
        uint64_t x = 0x9E3779B97F4A7C15ull;
        auto next = [&x]() { x ^= x << 13; x ^= x >> 7; x ^= x << 17; return x; };
        for (int t = 0; t < 2000; ++t) {
            LeafSet mask;
            for (int i = 0; i < BLS_MAX_WORDS; ++i) {
                mask.w[i] = next();
                if (t % 3 == 1) mask.w[i] &= next();   // sparse masks
                if (t % 3 == 2) mask.w[i] |= next();   // dense masks
            }
            mask = mask & all;
            const double a = bls_eval_host(m, mask), b = bls_eval_short_host(m, mask);
            if (memcmp(&a, &b, 8) != 0) return "internal error: BLS tables disagree with the node-by-node program";
        }
    }
    // the two ECMs
    for (int w = 0; w < 2; ++w) {
        EcmHost &e = m.ecm[w];
        std::vector<double> Q(NS * NS);
        std::string err;
        build_q(S[w], f[w], Q.data());
        if (!eigen_and_prior(Q.data(), f[w], e, err)) return err;
        e.P.resize((size_t)(m.n - 1) * NS * NS);
        for (int b = 0; b < m.n - 1; ++b) {
            const int rc = pmatrix(e, branch_time(m.bl[b], 1.0), e.P.data() + (size_t)b * NS * NS);
            if (rc) return std::string("CamlPaml.Q.substition_matrix check failed for branch ") + std::to_string(b) +
                           (rc == 1 ? " (entry < 0)" : " (row sum != 1)");
        }
        e.pstream.resize(m.gemm_edges.size() * (size_t)NS * NS);
        for (size_t g = 0; g < m.gemm_edges.size(); ++g)
            to_fragment_order(e.P.data() + (size_t)m.gemm_edges[g] * NS * NS, e.pstream.data() + g * NS * NS);
        e.leafPT.resize((size_t)nl * 65 * NS);
        for (int l = 0; l < nl; ++l) to_leaf_table(e.P.data() + (size_t)l * NS * NS, e.leafPT.data() + (size_t)l * 65 * NS);
        e.pstream_tc5.resize(m.tc5_edges.size() * (size_t)8192);
        for (size_t st = 0; st < m.tc5_edges.size(); ++st)
            to_tc5_tile(e.P.data() + (size_t)m.tc5_edges[st] * NS * NS, e.pstream_tc5.data() + st * 8192);
        e.cherry_P.resize(m.tc5_cherries.size() * (size_t)NS * NS);
        for (size_t k = 0; k < m.tc5_cherries.size(); ++k)
            std::memcpy(e.cherry_P.data() + k * NS * NS, e.P.data() + (size_t)m.tc5_cherries[k] * NS * NS, sizeof(double) * NS * NS);
    }
    return "";
}

}  // namespace pcsf
