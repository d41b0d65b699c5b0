"""Parity of the CUDA score-msa path (pcsf_score_msa) against the reference's golden .scores files."""
import os

import numpy as np
import pytest

from oracle import oracle as orc
from phylocsfpp_b200 import capi
from phylocsfpp_b200.maf import MafReader
from phylocsfpp_b200.models import load_model
from tests.util import random_alignment

pytestmark = pytest.mark.gpu


def golden_rows(path):
    rows = [ln.rstrip("\n").split("\t") for ln in open(path)]
    return rows[1:]


@pytest.mark.parametrize("maf,scores", [("chr22.50alignments.maf", "chr22.50alignments.fixed.scores"),
                                        ("chr22.516alignments.maf.gz", "chr22.516alignments.maf.fixed.scores")])
def test_fixed_golden(golden_dir, maf, scores):
    """Config 2: score-msa --strategy fixed --comp-anc 1 with 100vertebrates (test/tests.sh:35-37)."""
    G = os.path.join(golden_dir, "score-msa")
    model = load_model("100vertebrates")
    alns = list(MafReader(os.path.join(G, maf), model.seqid_to_phyloid, model.nl, False, warn=False))
    gold = golden_rows(os.path.join(G, scores))
    assert len(alns) == len(gold)
    dm = capi.DeviceModel(model)
    phylo, anc, bls = dm.score_msa([a.seqs for a in alns], capi.STRATEGY_FIXED)
    mism = 0
    for a, g, p, an, b in zip(alns, gold, phylo, anc, bls):
        # older golden files have no strand column (SURVEY.md section 4)
        vals = g[4:] if len(g) == 7 else g[3:]
        assert g[0] == a.chrom and int(g[1]) == a.start_pos and int(g[2]) == a.start_pos + a.L - 1
        ours = ["%.6f" % p, "%.6f" % an, "%.6f" % b]
        assert ours[2] == vals[2], "BLS must be exact"
        for x, y in zip(ours[:2], vals[:2]):
            assert abs(float(x) - float(y)) <= 1e-3 * max(1.0, abs(float(y)) * 1e-3)
            mism += x != y
    print(f"{scores}: {mism} printed values differ in the last digit")
    assert mism <= len(gold) // 50
    dm.close()


def test_fixed_vs_oracle_random():
    model = load_model("29mammals")
    dm = capi.DeviceModel(model)
    alns = [random_alignment(model.nl, L, seed=100 + L) for L in (0, 1, 2, 3, 5, 30, 31, 32, 299, 300, 1201)]
    phylo, anc, bls = dm.score_msa(alns, capi.STRATEGY_FIXED)
    mc = orc.OracleModel(model.tree, model.S_c, model.f_c)
    mnc = orc.OracleModel(model.tree, model.S_nc, model.f_nc)
    for a, p, an, b in zip(alns, phylo, anc, bls):
        rp, ra = orc.run_fixed(mc, mnc, orc.translate(a), True)
        assert abs(float(p) - float(rp)) <= 1e-3 and abs(float(an) - float(ra)) <= 1e-3
        if a.shape[1] > 0:
            assert np.float32(orc.bls(model.tree, a, per_base=False)[0]) == b
    dm.close()


def test_mle_golden_small(golden_dir):
    """score-msa --strategy mle --comp-anc 1, 100vertebrates, against the reference's own output with the
    reference's own CI tolerance (squared error <= 0.001 per score, test/tests.sh:40-42); most rows agree
    to 1e-3 (rows that do not are Brent trajectories that fork on ~1e-13 differences in P(t), see DESIGN.md)."""
    G = os.path.join(golden_dir, "score-msa")
    model = load_model("100vertebrates")
    alns = list(MafReader(os.path.join(G, "chr22.50alignments.maf"), model.seqid_to_phyloid, model.nl, False, warn=False))
    gold = golden_rows(os.path.join(G, "chr22.50alignments.mle.scores"))
    dm = capi.DeviceModel(model)
    phylo, anc, bls = dm.score_msa([a.seqs for a in alns], capi.STRATEGY_MLE)
    tight = 0
    for a, g, p, an, b in zip(alns, gold, phylo, anc, bls):
        assert g[0] == a.chrom and int(g[1]) == a.start_pos and int(g[2]) == a.start_pos + a.L - 1
        assert (float(p) - float(g[4])) ** 2 <= 0.001, (g, p)
        assert (float(an) - float(g[5])) ** 2 <= 0.001, (g, an)
        assert "%.6f" % b == g[6]
        tight += abs(float(p) - float(g[4])) <= 1e-3 and abs(float(an) - float(g[5])) <= 1e-3
    print(f"MLE golden: {tight}/{len(gold)} rows within 1e-3 of the reference output")
    assert tight >= len(gold) - 1          # observed: 49/50, row 5 is the documented Brent fork (DESIGN.md section 7)
    dm.close()


def test_mle_golden_516(golden_dir, tmp_path):
    """The reference's medium MLE input (test/maf-file-medium, 516 alignments, 100vertebrates).  Pinned against what the reference's
    UNMODIFIED current sources write for it (tests/golden/ref-generated/chr22.516alignments.mle.refbuilt.scores, made by
    tests/golden/make_ref_fixtures.py with oracle/_ref): coordinates and BLS text exact, every row inside the reference's CI tolerance
    (squared error <= 0.001, test/tests.sh:40-42) except Brent forks, whose number is pinned at what was observed and each of which
    must agree with the CPU restatement instead.  The SHIPPED golden of this input predates v1.2.0: 135 of its rows are not
    reproduced by the unmodified sources either; where the two files agree the device has to agree with both."""
    import gzip
    import shutil
    G = os.path.join(golden_dir, "score-msa")
    maf = os.path.join(str(tmp_path), "chr22.516alignments.maf")
    with gzip.open(os.path.join(G, "chr22.516alignments.maf.gz"), "rb") as fi, open(maf, "wb") as fo:
        shutil.copyfileobj(fi, fo)
    model = load_model("100vertebrates")
    alns = list(MafReader(maf, model.seqid_to_phyloid, model.nl, False, warn=False))
    shipped = golden_rows(os.path.join(G, "chr22.516alignments.maf.mle.scores"))
    built = [ln.rstrip("\n").split("\t") for ln in open(os.path.join(golden_dir, "ref-generated", "chr22.516alignments.mle.refbuilt.scores"))
             if ln.startswith("chr")]
    assert len(shipped) == len(built) == len(alns) == 516
    dm = capi.DeviceModel(model)
    phylo, anc, bls = dm.score_msa([a.seqs for a in alns], capi.STRATEGY_MLE)
    forked, drift = [], 0
    for i, (a, g, r, p, an, b) in enumerate(zip(alns, shipped, built, phylo, anc, bls)):
        assert g[0] == r[0] == a.chrom and int(g[1]) == int(r[1]) == a.start_pos and int(g[2]) == int(r[2]) == a.start_pos + a.L - 1
        assert "%.6f" % b == g[6] == r[6]
        if "nan" in (r[4], r[5]):
            assert np.isnan(p) or np.isnan(an), (i, r, p, an)
            continue
        close = lambda row: abs(float(p) - float(row[4])) <= 1e-3 and abs(float(an) - float(row[5])) <= 1e-3
        if not close(r):
            forked.append(i)
        agree = abs(float(g[4]) - float(r[4])) <= 1e-3 and abs(float(g[5]) - float(r[5])) <= 1e-3
        drift += not agree
        if agree and not close(g) and i not in forked:
            forked.append(i)
    print(f"MLE 516: {516 - len(forked)}/516 rows within 1e-3 of the reference built from its current sources; forked rows: {forked}; "
          f"{drift} rows of the shipped golden differ from that build")
    mc = orc.OracleModel(model.tree, model.S_c, model.f_c)
    mnc = orc.OracleModel(model.tree, model.S_nc, model.f_nc)
    for i in forked:          # a legitimate fork: the CPU restatement (same eigensolver family as the device) lands within the CI tolerance of the device
        rp, ra, info = orc.run_mle(mc, mnc, orc.translate(alns[i].seqs), True)
        assert (float(phylo[i]) - float(rp)) ** 2 <= 0.001 and (float(anc[i]) - float(ra)) ** 2 <= 0.001, (i, phylo[i], rp, anc[i], ra, info)
    assert len(forked) <= 8
    dm.close()


def _tiny_branch_model(neg: float):
    """12flies with all branches shortened 1000-fold and one negative exchangeability: P(t) = exp(Qt) then has a negative entry of
    about neg * pi * t, inside PhyloModel_make's 1e-6 tolerance at the fixed tree for a small |neg| and outside it once the MLE
    search scales the tree up (instance.hpp:612-636 -> runtime_error -> NaN row, score_msa.hpp:124)."""
    import copy
    model = copy.deepcopy(load_model("12flies"))
    t = model.tree
    t.branch_len = (np.asarray(t.branch_len, np.float64) * 1e-3).astype(np.float32)
    t.branch_len_f64 = np.asarray(t.branch_len_f64, np.float64) * 1e-3
    for S in (model.S_c, model.S_nc):
        S[5, 9] = S[9, 5] = neg
    return model


def test_numeric_violation_gives_nan_rows_and_model_error():
    """a6 failure path.  (i) A violation that only appears at scaled branch lengths marks that alignment NaN (as the reference's
    runtime_error does) while the call succeeds, and the oracle restatement agrees; (ii) a violation at the fixed tree makes
    pcsf_model_create fail with PCSF_ERR_NUMERIC."""
    model = _tiny_branch_model(-0.02)
    dm = capi.DeviceModel(model)          # the fixed tree is inside the tolerance
    alns = [random_alignment(model.nl, L, seed=40 + L, gap=0.1, conserve=0.8) for L in (30, 90)]
    phylo_f, anc_f, _ = dm.score_msa(alns, capi.STRATEGY_FIXED)
    assert np.isfinite(phylo_f).all() and np.isfinite(anc_f).all()
    phylo, anc, bls = dm.score_msa(alns, capi.STRATEGY_MLE)
    mc = orc.OracleModel(model.tree, model.S_c, model.f_c)
    mnc = orc.OracleModel(model.tree, model.S_nc, model.f_nc)
    for a, p, an in zip(alns, phylo, anc):
        rp, ra, info = orc.run_mle(mc, mnc, orc.translate(a), True)
        assert np.isnan(rp) and np.isnan(ra), info          # the reference path throws on this input
        assert np.isnan(p) and np.isnan(an)
    assert np.isfinite(bls).all()
    dm.close()
    with pytest.raises(capi.PcsfError) as ei:
        capi.DeviceModel(_tiny_branch_model(-2.0))
    assert ei.value.status == capi.PCSF_ERR_NUMERIC


@pytest.mark.parametrize("strategy", [capi.STRATEGY_FIXED, capi.STRATEGY_MLE, capi.STRATEGY_OMEGA])
def test_bls_only_call(strategy):
    """phylo = anc = NULL: the call succeeds without a fit (the reference does not call run() then, score_msa.hpp:112) and its BLS
    equals the full call's bit for bit."""
    model = load_model("12flies")
    dm = capi.DeviceModel(model)
    alns = [random_alignment(model.nl, L, seed=500 + L, gap=0.2) for L in (0, 1, 2, 3, 5, 30, 61, 150)]
    phylo, anc, bls = dm.score_msa(alns, strategy, comp_phylo=False, comp_anc=False)
    assert phylo is None and anc is None
    _, _, full = dm.score_msa(alns, strategy)
    assert np.array_equal(bls.view(np.uint32), full.view(np.uint32))
    dm.close()


def test_mle_vs_oracle_random():
    model = load_model("29mammals", "Human,Chimp,Mouse,Dog,Cow,Horse,Elephant,Armadillo,Rat,Rabbit,Cat,Megabat")
    dm = capi.DeviceModel(model)
    alns = [random_alignment(model.nl, L, seed=900 + L, gap=0.2, conserve=c)
            for L, c in ((0, .7), (2, .7), (3, .7), (30, .9), (61, .5), (150, .8), (299, .95), (600, .6), (900, .85))]
    phylo, anc, bls = dm.score_msa(alns, capi.STRATEGY_MLE)
    mc = orc.OracleModel(model.tree, model.S_c, model.f_c)
    mnc = orc.OracleModel(model.tree, model.S_nc, model.f_nc)
    tight = 0
    for a, p, an in zip(alns, phylo, anc):
        rp, ra, info = orc.run_mle(mc, mnc, orc.translate(a), True)
        assert (float(p) - float(rp)) ** 2 <= 0.001 and (float(an) - float(ra)) ** 2 <= 0.001, (a.shape, p, rp, an, ra, info)
        tight += abs(float(p) - float(rp)) <= 1e-3 and abs(float(an) - float(ra)) <= 1e-3
    assert tight >= len(alns) - 1
    dm.close()


def test_omega_vs_oracle_random():
    """pcsf_score_msa(OMEGA) against the oracle's restatement of run.hpp:59-182 on random alignments, incl. L < 3 (prior-only
    fits: both hypotheses see the same function, score 0) — the same 1 %-bracket tolerance as against the reference."""
    model = load_model("12flies")
    dm = capi.DeviceModel(model)
    alns = [random_alignment(model.nl, L, seed=300 + L, gap=0.2) for L in (2, 30, 61, 150, 333)]
    phylo, anc, bls = dm.score_msa(alns, capi.STRATEGY_OMEGA, comp_anc=False)
    d = []
    for a, p, b in zip(alns, phylo, bls):
        s, info = orc.run_omega(model.tree, orc.translate(a))
        print(a.shape[1], float(p), float(s), info["evals"])
        d.append(abs(float(p) - float(s)))
        assert np.float32(orc.bls(model.tree, a, per_base=False)[0]) == b
    assert max(d) ** 2 <= 0.1 and min(d) <= 1e-3
    assert abs(float(phylo[0])) < 1e-6
    dm.close()
