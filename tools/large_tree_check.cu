// large_tree_check.cu — CPU check of what a model of up to 512 leaves gets at creation (csrc/model_prep.hpp, csrc/kernels.cuh).
//
// Prints the FP64 pruning program's size and stack depth, the shared memory k_prune needs for it at 4, 8 and 12 compute warps, and
// the BLS program k_bls runs.  With a masks file (one line per column: nl characters '0' / '1', leaf l present = character l), it
// also evaluates the per-base branch length score of each column through the device BLS program (BlsInnerDev<NW> with the tree's
// word count, interpreted here exactly as k_bls<NW> does it) and prints it as a hexadecimal double.  Host code only: no GPU needed.
//
// build: nvcc -gencode arch=compute_100a,code=sm_100a -std=c++17 -O2 -o /tmp/large_tree_check tools/large_tree_check.cu
// usage: large_tree_check <model> [masks-file]
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <fstream>
#include <string>

#include "../phylocsfpp_b200/host/util.hpp"
#include "../phylocsfpp_b200/host/model.hpp"
#include "../phylocsfpp_b200/csrc/kernels.cuh"

using namespace pcsf;

// k_bls<NW> on one column, on the host: same masks, same word shifts of a TABLE entry, same additions in the same order
template <int NW>
static double bls_column(const ModelHost &m, const std::vector<BlsInnerDev<NW>> &prog, const uint64_t *msk) {
    std::vector<double> st(m.bls_short_depth + 2);
    int sp = 0;
    double v = 0.0;
    for (const BlsInnerDev<NW> &e : prog) {
        uint64_t out_of = 0, in_l = 0, in_r = 0;
        for (int i = 0; i < NW; ++i) {
            out_of |= msk[i] & ~e.self[i];
            in_l |= msk[i] & e.left[i];
            in_r |= msk[i] & e.self[i] & ~e.left[i];
        }
        if (e.flags & 4) {
            const int nbits = (e.flags >> 16) & 0xff, shift = ((e.flags >> 8) & 0xff) | ((e.flags >> 16) & 0xff00);
            uint64_t bits = 0;
            for (int i = 0; i < NW; ++i) {
                const int d = 64 * i - shift;
                if (d <= 0 && d > -64) bits |= msk[i] >> -d;
                else if (d > 0 && d < 64) bits |= msk[i] << d;
            }
            bits &= (1ull << nbits) - 1;
            v = m.bls_tables[(size_t)e.tab_off + 2 * bits + (out_of != 0 ? 1 : 0)];
        } else {
            const double r = (e.flags & 2) ? e.right_bl : st[--sp];
            const double l = (e.flags & 1) ? e.left_bl : st[--sp];
            v = out_of != 0 ? e.bl : 0.0;
            if (in_l != 0) v += l;
            if (in_r != 0) v += r;
        }
        st[sp++] = v;
    }
    int present = 0;
    for (int i = 0; i < NW; ++i) present += __builtin_popcountll(msk[i]);
    return present >= 2 ? v / m.bls_all : 0.0;
}

template <int NW>
static void bls_file(const ModelHost &m, const char *path) {
    const std::vector<BlsInnerDev<NW>> prog = bls_device_program<NW>(m.bls_short);
    std::ifstream in(path);
    std::string line;
    while (std::getline(in, line)) {
        if ((int)line.size() != m.nl) host::die("mask line of %zu characters for %d leaves", line.size(), m.nl);
        uint64_t msk[NW] = {};
        for (int l = 0; l < m.nl; ++l)
            if (line[l] == '1') msk[l >> 6] |= 1ull << (l & 63);
        printf("%a\n", bls_column<NW>(m, prog, msk));
    }
}

int main(int argc, char **argv) {
    if (argc < 2) host::die("usage: large_tree_check <model> [masks-file]");
    host::Model hm;
    host::load_model(hm, argv[1], "", "");
    ModelHost m;
    const double *S[2] = {hm.c.S.data(), hm.nc.S.data()}, *f[2] = {hm.c.f.data(), hm.nc.f.data()};
    const std::string err = prepare_model(m, hm.tree.nl, hm.tree.child1.data(), hm.tree.child2.data(), hm.tree.bl.data(), hm.tree.bl64.data(), S, f);
    if (!err.empty()) host::die("%s", err.c_str());
    const int ops = (int)m.program.size();
    int n_tab = 0;
    for (const BlsInner &e : m.bls_short) n_tab += (e.flags & 4) != 0;
    printf("nl %d, program ops %d, max_stack %d, smem 4 warps %zu, 8 warps %zu, 12 warps %zu, tc5 steps %zu, "
           "bls entries %zu, bls tables %d, bls depth %d\n",
           m.nl, ops, m.max_stack, prune_smem_bytes(m.nl, ops, m.max_stack, 4), prune_smem_bytes(m.nl, ops, m.max_stack, 8),
           prune_smem_bytes(m.nl, ops, m.max_stack, 12), m.tc5_steps.size(), m.bls_short.size(), n_tab, m.bls_short_depth);
    if (argc > 2) {
        if (m.nl <= SMALL_TREE_MAX_LEAVES) bls_file<2>(m, argv[2]);
        else bls_file<8>(m, argv[2]);
    }
    return 0;
}
