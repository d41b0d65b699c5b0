/*
 * phylocsf_b200.h — C-ABI of the B200-native PhyloCSF++ likelihood hot path.
 *
 * The reference (cpockrandt/PhyloCSFpp, header-only C++) has no FFI; its hot path is reached through
 * three C++ entry points.  This ABI is what a binding for that seam would bind (file:line relative to
 * the reference repo):
 *
 *   run_tracks(Data&, const Model&, const alignment_t&, std::vector<double>&)          src/run.hpp:35
 *       called 6x per alignment from src/phylocsf++build_tracks.hpp:172 after
 *       alignment_t::update_seqs (src/parallel_file_reader.hpp:61)               -> pcsf_tracks*
 *   compute_bls_score<bool>(const newick_node*, const alignment_t&, const Model&, std::vector<double>&)
 *       src/additional_scores.hpp:44, called from build_tracks.hpp:136, score_msa.hpp:132,141
 *                                                                                 -> pcsf_tracks* (bls[]),
 *                                                                                    pcsf_score_msa (bls[])
 *   run(Data&, const Model&, const alignment_t&, algorithm_t, std::mt19937&, bool)       src/run.hpp:57
 *       FIXED and MLE branches (:183-210), called from src/phylocsf++score_msa.hpp:116 -> pcsf_score_msa
 *   PhyloCSFModel_make / instantiate_qs / PhyloModel_make (src/instance.hpp:687,309,449): redone by the
 *       reference on every call; here once per model                               -> pcsf_model_create
 *
 * Conventions: plain C, no exceptions cross the boundary, every function returns a pcsf_status.
 * Numerical failures of one item (the reference's std::runtime_error from PhyloModel_make,
 * instance.hpp:618,635, caught at score_msa.hpp:124) yield NaN in that item's outputs.  A character
 * outside "ACGTacgt.-Nn" (the reference's exit(37), src/translation.hpp:46-51) yields PCSF_ERR_BAD_CHAR.
 * There is no CPU fallback: without a CUDA device every compute call returns PCSF_ERR_CUDA.
 * Thread safety: one pcsf_model may be used from one host thread at a time; create one per worker.
 */
#ifndef PHYLOCSF_B200_H
#define PHYLOCSF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PCSF_ABI_VERSION 1

typedef enum {
    PCSF_OK = 0,
    PCSF_ERR_INVALID = 1,      /* bad argument */
    PCSF_ERR_CUDA = 2,         /* CUDA runtime error / no device */
    PCSF_ERR_NUMERIC = 3,      /* model matrices violate PhyloModel_make's checks at rho = 1 */
    PCSF_ERR_UNSUPPORTED = 4,  /* e.g. more than PCSF_MAX_LEAVES leaves */
    PCSF_ERR_BAD_CHAR = 37     /* mirrors the reference's exit(37) */
} pcsf_status;

/* Largest species tree pcsf_model_create accepts.  At 512 leaves the FP64 pruning kernel's per-warp stack of sibling partials still
 * fits one SM's shared memory for every tree shape (a balanced tree is the deepest).  Trees of more than 128 leaves are pruned with
 * an exact power-of-two rescaling per window, so their likelihoods do not underflow where the reference's unscaled product does, and
 * they have no tcgen05 path (PCSF_TRACKS_TC5 returns PCSF_ERR_UNSUPPORTED). */
#define PCSF_MAX_LEAVES 512

/* Flattened species tree + the two empirical codon models: what `struct Model` (src/models.hpp:1742)
 * holds after load_model.  Node ids follow newick_flatten (src/newick.hpp:218): leaves 0..nl-1 in DFS
 * order, inner nodes nl..n-1 in post-order, root = n-1, n = 2*nl-1. */
typedef struct {
    int32_t nl;
    const int16_t *child1;          /* [n], -1 for leaves */
    const int16_t *child2;          /* [n] */
    const float *branch_len;        /* [n] newick_elem::branch_length (float; likelihood) */
    const double *branch_len_f64;   /* [n] newick_node::branch_length (double; BLS) */
    const double *ecm_c;            /* [64*64] symmetric exchangeabilities, zero diagonal (coding) */
    const double *freq_c;           /* [64] codon frequencies (coding) */
    const double *ecm_nc;           /* [64*64] (non-coding) */
    const double *freq_nc;          /* [64] */
} pcsf_model_desc;

typedef struct pcsf_model pcsf_model;

/* Builds Q, its eigensystem, pi and all P(t_b) at rho = 1 for both ECMs (instance.hpp:648-712,
 * fixed_lik.hpp:281-360), the pruning program, the BLS masks, and uploads them to `device`. */
pcsf_status pcsf_model_create(const pcsf_model_desc *desc, int device, pcsf_model **out);
void pcsf_model_destroy(pcsf_model *m);

/* Page-locked host memory for the buffers handed to pcsf_tracks / pcsf_score_msa (optional: any host pointer works; pinned ones are
 * copied by DMA without staging — bench.py's e2e leg uses pinned buffers).  The reference's caller owns Data / alignment_t / the output
 * vectors (build_tracks.hpp:60, 74-79); here the caller owns these buffers.  Pinning costs ~0.4 ms per MB: worth it for buffers that
 * are reused across many calls (measured: the command line host on a 10 M-column file is faster with pageable vectors). */
void *pcsf_alloc_pinned(size_t bytes);
void pcsf_free_pinned(void *p);
/* Page-locks memory the caller already owns (and may already be using), e.g. long-lived staging buffers of a driver: calls made before
 * a buffer is pinned work, their copies are just staged by the driver.  p and bytes should be multiples of the page size. */
pcsf_status pcsf_register_host(void *p, size_t bytes);
pcsf_status pcsf_unregister_host(void *p);

/* CUDA devices visible to the process (0 without a driver or device).  The command line host deals chain groups to all of them by
 * default, as the reference uses all cores by default (build_tracks.hpp:88, --threads). */
int pcsf_device_count(void);

/* Thread-local description of the last error returned on this thread. */
const char *pcsf_last_error(void);
int pcsf_abi_version(void);

/* ---- build-tracks path ------------------------------------------------------------------------- */

#define PCSF_TRACKS_SCORES   0x1u  /* plus[]/minus[] decibans */
#define PCSF_TRACKS_BLS      0x2u  /* bls[] */
#define PCSF_TRACKS_NO_DEDUP 0x4u  /* prune every window, do not deduplicate site patterns */
/* 0x8u was PCSF_TRACKS_FP32 (split-TF32 on mma.sync, round 1): superseded by the tcgen05 path and removed from the library */
#define PCSF_TRACKS_TC5      0x10u /* FP32-class arithmetic on tcgen05/TMEM (5th-gen tensor cores): split TF32 + per-window log-scaling, |delta| <= 1e-3 decibans */
/* The tcgen05 path holds the tree's codon ids, step program and row sources in one SM's shared memory: every tree of at most 123
 * leaves fits, trees of 124 to 126 leaves fit depending on their shape (a caterpillar is the largest program for its leaf count),
 * trees of 127 and 128 leaves never fit.  For a tree that does not fit, pcsf_model_create still succeeds (the FP64 path and score-msa
 * run on it) and a call with PCSF_TRACKS_TC5 returns PCSF_ERR_UNSUPPORTED. */

typedef struct {
    int64_t n_windows;        /* 2 * max(L-2, 0) */
    int64_t n_unique;         /* prunings actually executed per model (after site-pattern dedup) */
    int32_t n_chunks;         /* dedup domains */
    int32_t n_launches;       /* kernels launched by the call */
    float ms_pack, ms_hash, ms_dedup, ms_prune, ms_scatter, ms_bls; /* device times (CUDA events); 0 unless timing enabled */
} pcsf_tracks_stats;

/*
 * One matrix of L alignment columns (one alignment, or several concatenated along the columns: windows
 * that straddle two alignments are computed but meaningless, the caller ignores them).
 *   seqs           ASCII nucleotides [nl][ld], row s = species s (alignment_t::seqs[s]), ld >= L
 *   plus, minus    [max(L-2,0)] decibans 10*(log zC - log zNC)/ln 10 of the '+' codon seq[o..o+2] and of
 *                  the '-' codon comp(seq[o+2]) comp(seq[o+1]) comp(seq[o])   (run.hpp:51-54)
 *   bls            [L] per-base branch length score (additional_scores.hpp:57-79)
 *   pattern_index  [2*max(L-2,0)] or NULL: site-pattern index of window (o, strand) at [2*o + strand]
 *                  (strand 0 = '+'): rank of the first occurrence of its leaf-state column, in index
 *                  order, within its dedup chunk
 * pcsf_tracks takes HOST pointers and includes H2D/D2H copies; pcsf_tracks_device takes DEVICE pointers
 * (same device as the model) and enqueues all work on `cuda_stream` (a cudaStream_t) without
 * synchronising; `stats` is then filled from device counters only after pcsf_tracks_device_finish.
 */
pcsf_status pcsf_tracks(pcsf_model *m, const uint8_t *seqs, int64_t L, int64_t ld, uint32_t flags,
                        double *plus, double *minus, double *bls, uint32_t *pattern_index,
                        pcsf_tracks_stats *stats);
pcsf_status pcsf_tracks_device(pcsf_model *m, const uint8_t *d_seqs, int64_t L, int64_t ld, uint32_t flags,
                               double *d_plus, double *d_minus, double *d_bls, uint32_t *d_pattern_index,
                               void *cuda_stream);
/* Synchronises the stream, checks the bad-character flag and fills stats. */
pcsf_status pcsf_tracks_device_finish(pcsf_model *m, void *cuda_stream, pcsf_tracks_stats *stats);

/* Maximum number of columns per dedup chunk (default 1<<21); 0 restores the default. */
pcsf_status pcsf_set_chunk_columns(pcsf_model *m, int64_t columns);
/* Enable/disable per-stage CUDA-event timing in pcsf_tracks (adds synchronisation). */
pcsf_status pcsf_set_timing(pcsf_model *m, int enabled);

/* ---- score-msa path ---------------------------------------------------------------------------- */

typedef enum { PCSF_STRATEGY_MLE = 0, PCSF_STRATEGY_FIXED = 1, PCSF_STRATEGY_OMEGA = 2 } pcsf_strategy;

/*
 * n_aln alignments, each scored on its own in frame +1 from offset 0 (score_msa.hpp:102-116).
 *   seqs      host ASCII; alignment i is the [nl][len[i]] row-major matrix at seqs + offset[i]
 *   phylo     [n_aln] float(10*(lprC - lprNC)/ln 10)        (run.hpp:206)   NaN on numerical failure
 *   anc       [n_aln] float(10*(ancC - ancNC)/ln 10) or NULL (run.hpp:207)
 *   bls       [n_aln] float(compute_bls_score<false>)  or NULL (score_msa.hpp:132)
 * MLE replays mt19937(42) per alignment (score_msa.hpp:115) and GSL's Brent minimiser
 * (fixed_lik.hpp:469-544).
 * OMEGA (run.hpp:59-182, omega.hpp): phylo = float(10*(lpr_H1 - lpr_H0)/ln 10) from the alternating rho / kappa fits of the
 * two dN/dS hypotheses on a Q(kappa, omega, F3x4) built per alignment; there is no ancestral score for it (the reference
 * returns NaN, run.hpp:181): anc, if given, is filled with NaN.
 */
pcsf_status pcsf_score_msa(pcsf_model *m, pcsf_strategy strategy, int32_t n_aln, const uint8_t *seqs,
                           const int64_t *offset, const int64_t *len, float *phylo, float *anc, float *bls);

/* ---- six-frame / open-reading-frame scoring (score-msa --frames, --orf) --------------------------- */

typedef enum { PCSF_ORF_ASIS = 0, PCSF_ORF_STOPSTOP = 1, PCSF_ORF_ATGSTOP = 2 } pcsf_orf_mode;

/* One scored region.  strand +1/-1 and frame 1..3 name the reading frame (0 and 0: the "none" record of an alignment without a
 * region in best-only mode, with columns -1 and NaN scores).  [col_begin, col_end) are columns of the input alignment; codons counts
 * the region's full codons (for PCSF_ORF_ATGSTOP / STOPSTOP including the closing stop). */
typedef struct {
    int32_t aln;
    int8_t strand;
    int8_t frame;
    int16_t pad;
    int64_t col_begin, col_end, codons;
    float phylo, anc, bls;
} pcsf_region;

/*
 * Scores the reading frames, or the open reading frames, of n_aln alignments (the inputs of pcsf_score_msa) on the device.
 *   ref_row     [n_aln] model row of each alignment's reference species: its codons define stops (TAA TAG TGA) and starts (ATG)
 *   frames      1 (+1), 3 (+1 +2 +3) or 6 (+1 +2 +3 -1 -2 -3); a '-' frame reads the reverse complement of the whole alignment
 *   orf         ASIS: one region per frame, from the frame's offset to the alignment's end (frame +1 = the whole alignment);
 *               STOPSTOP: every stop-delimited segment of a frame (closing stop included) and its non-empty open tail;
 *               ATGSTOP: per segment, its first ATG through its stop (the open tail never yields one)
 *   min_codons  >= 1; the ORF modes keep regions of at least this many codons
 *   best_only   0: every region, by alignment, frame (+1 +2 +3 -1 -2 -3) and codon; 1: one region per alignment, the largest phylo
 *               (NaN never wins, ties go to the earlier region; all NaN: the first; none: the "none" record)
 * A region's (phylo, anc, bls) are bit for bit what pcsf_score_msa returns for its sub-alignment extracted on the host (reverse
 * complemented for '-').  anc / bls are NaN unless want_anc / want_bls.  FP64 throughout.  *n_regions receives the number of
 * records; pcsf_score_regions_get copies the first n of them (n <= *n_regions) from the handle.
 */
pcsf_status pcsf_score_regions(pcsf_model *m, pcsf_strategy strategy, int32_t n_aln, const uint8_t *seqs, const int64_t *offset,
                               const int64_t *len, const int32_t *ref_row, int32_t frames, pcsf_orf_mode orf, int32_t min_codons,
                               int32_t best_only, int32_t want_anc, int32_t want_bls, int64_t *n_regions);
pcsf_status pcsf_score_regions_get(const pcsf_model *m, pcsf_region *out, int64_t n);   /* records of the last pcsf_score_regions call on this handle */

/* ---- introspection (used by the parity tests) -------------------------------------------------- */

/* What the last pcsf_score_msa call with PCSF_STRATEGY_MLE did on this handle: `evaluations` counts lpr_leaves calls — (alignment,
 * ECM, rho) triples, each one (n-1) x (2 x 64^3 + 64^2) flop of P(t) = exp(Qt) construction (PhyloModel_make, instance.hpp:449-646)
 * plus one pruning pass over the alignment's codons.  The per-kernel CUDA-event times are filled only with pcsf_set_timing on. */
typedef struct {
    int64_t alignments, evaluations;
    int32_t rounds, slots;
    float ms_step, ms_plan, ms_expm, ms_prune;
} pcsf_msa_stats;
pcsf_status pcsf_score_msa_stats(const pcsf_model *m, pcsf_msa_stats *stats);

/* Copies the model's host-side matrices: which in {0 coding, 1 non-coding}.
 * lambda[64], pi[64], P[(n-1)*64*64] row-major P_b[a][c] at rho = 1; any pointer may be NULL. */
pcsf_status pcsf_model_get(const pcsf_model *m, int which, double *lambda, double *pi, double *P);

#ifdef __cplusplus
}
#endif
#endif /* PHYLOCSF_B200_H */
