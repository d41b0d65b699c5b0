"""pcsf_score_regions (score-msa --frames / --orf / --all-scores) on the device: its region lists against the plain-Python mirror
phylocsfpp_b200.orf, its scores bit for bit against pcsf_score_msa on the host-extracted sub-alignments, against the oracle, the
best-only rule, the error statuses, and the command line on the reference's 516-alignment fixture."""
import copy
import gzip
import os
import shutil
import subprocess

import numpy as np
import pytest

from oracle import oracle as orc
from phylocsfpp_b200 import capi, orf
from phylocsfpp_b200.maf import MafReader
from phylocsfpp_b200.models import load_model
from tests.util import random_alignment

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "phylocsfpp_b200", "bin", "phylocsf_b200")
LENGTHS = (0, 1, 2, 3, 4, 5, 299, 300, 301, 3000)
MODES = (orf.ASIS, orf.STOPSTOP, orf.ATGSTOP)


def planted(nl: int, L: int, seed: int, ref: int, conserve: float = 0.8) -> np.ndarray:
    """A random alignment whose reference row is built from codon-sized pieces rich in ATG and stops on both strands (CAT, TTA, CTA
    and TCA are their reverse complements) at arbitrary offsets, so every one of the six frames sees starts and stops."""
    a = random_alignment(nl, L, seed, gap=0.2, conserve=conserve)
    rng = np.random.default_rng(seed + 17)
    pieces = [b"ATG", b"TAA", b"TAG", b"TGA", b"CAT", b"TTA", b"CTA", b"TCA", b"GCC", b"AAG", b"CTG", b"C", b"GT", b"atg", b"tga",
              b"N", b"-"]
    w = np.array([3, 1, 1, 1, 3, 1, 1, 1, 6, 6, 6, 2, 2, 1, 1, 1, 1], float)
    row = b"".join(pieces[i] for i in rng.choice(len(pieces), size=L, p=w / w.sum()))[:L]
    a[ref] = np.frombuffer(row, np.uint8)
    return a


def expected_regions(alns, refs, frames, mode, min_codons):
    out = []
    for i, (a, r) in enumerate(zip(alns, refs)):
        out += [(i, reg) for reg in orf.regions(a[r], a.shape[1], frames, mode, min_codons)]
    return out


def as_tuples(rec):
    return [(int(x["aln"]), int(x["strand"]), int(x["frame"]), int(x["col_begin"]), int(x["col_end"]), int(x["codons"])) for x in rec]


def same_bits(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(a[~np.isnan(a)].view(np.uint32), b[~np.isnan(b)].view(np.uint32))


def same_record(x, y):
    """Field by field (the 4 tail bytes of pcsf_region are padding), floats bit for bit with NaN equal to NaN."""
    ints = ("aln", "strand", "frame", "col_begin", "col_end", "codons")
    return all(int(x[k]) == int(y[k]) for k in ints) and all(same_bits([x[k]], [y[k]]) for k in ("phylo", "anc", "bls"))


def _batch(model, seed0, conserve=0.8):
    refs = [(7 * i) % model.nl for i in range(len(LENGTHS))]
    alns = [planted(model.nl, L, seed0 + L, r, conserve) for L, r in zip(LENGTHS, refs)]
    return alns, refs


@pytest.mark.parametrize("name", ["29mammals", "100vertebrates"])
def test_region_lists_equal_mirror(name):
    model = load_model(name)
    dm = capi.DeviceModel(model)
    alns, refs = _batch(model, 50)
    for mode in MODES:
        for frames in (1, 3, 6):
            for mc in (1, 25):
                rec = dm.score_regions(alns, refs, capi.STRATEGY_FIXED, frames, mode, mc, comp_anc=False, comp_bls=False)
                exp = expected_regions(alns, refs, frames, mode, mc)
                assert as_tuples(rec) == [(i, r.strand, r.frame, r.col_begin, r.col_end, r.codons) for i, r in exp], (mode, frames, mc)
                if mode != orf.ASIS and frames == 6 and mc == 1:
                    assert len({(r.strand, r.frame) for _, r in exp}) == 6     # the planted patterns reach every frame
    dm.close()


def test_region_lists_across_scan_blocks():
    """900 alignments x 6 frames = 5400 (alignment, frame) units: the offsets cross a 4096-element block of the scans."""
    model = load_model("12flies")
    dm = capi.DeviceModel(model)
    rng = np.random.default_rng(5)
    alns = [planted(model.nl, int(L), 2000 + i, i % model.nl) for i, L in enumerate(rng.integers(0, 90, size=900))]
    refs = [i % model.nl for i in range(900)]
    for mode, best in ((orf.STOPSTOP, False), (orf.ATGSTOP, False), (orf.ATGSTOP, True)):
        rec = dm.score_regions(alns, refs, capi.STRATEGY_FIXED, 6, mode, 2)
        exp = expected_regions(alns, refs, 6, mode, 2)
        assert as_tuples(rec) == [(i, r.strand, r.frame, r.col_begin, r.col_end, r.codons) for i, r in exp]
        if best:
            _check_best(dm.score_regions(alns, refs, capi.STRATEGY_FIXED, 6, mode, 2, best_only=True), rec, len(alns))
    dm.close()


def _extract(alns, rec):
    out = []
    for x in rec:
        r = orf.Region(int(x["strand"]), int(x["frame"]), 0, int(x["codons"]), int(x["col_begin"]), int(x["col_end"]))
        out.append(orf.sub_alignment(alns[int(x["aln"])], r))
    return out


@pytest.mark.parametrize("strategy", [capi.STRATEGY_FIXED, capi.STRATEGY_MLE])
def test_scores_bit_identical_to_score_msa(strategy):
    model = load_model("29mammals")
    dm = capi.DeviceModel(model)
    alns, refs = _batch(model, 80)
    if strategy == capi.STRATEGY_MLE:
        alns, refs = alns[:-1], refs[:-1]            # MLE: without the 3000-column alignment (its ~100 regions add nothing new)
    for mode, mc in ((orf.ASIS, 25), (orf.ATGSTOP, 2), (orf.STOPSTOP, 3)):
        rec = dm.score_regions(alns, refs, strategy, 6, mode, mc)
        subs = _extract(alns, rec)
        phylo, anc, bls = dm.score_msa(subs, strategy)
        assert same_bits(rec["phylo"], phylo), mode
        assert same_bits(rec["anc"], anc), mode
        assert same_bits(rec["bls"], bls), mode
        print(f"strategy {strategy} mode {mode}: {len(rec)} regions bit-identical")
    dm.close()


def test_omega_bit_identical_to_score_msa():
    model = load_model("12flies")
    dm = capi.DeviceModel(model)
    alns = [planted(model.nl, L, 300 + L, 0) for L in (61, 150, 333)]
    rec = dm.score_regions(alns, [0, 0, 0], capi.STRATEGY_OMEGA, 6, orf.STOPSTOP, 8, comp_anc=False)
    assert len(rec) >= 14, len(rec)
    rec = rec[:14]
    phylo, _, bls = dm.score_msa(_extract(alns, rec), capi.STRATEGY_OMEGA, comp_anc=False)
    assert same_bits(rec["phylo"], phylo) and same_bits(rec["bls"], bls)
    assert np.isnan(rec["anc"]).all()
    with pytest.raises(capi.PcsfError) as ei:
        dm.score_regions(alns, [0, 0, 0], capi.STRATEGY_OMEGA, 6, orf.STOPSTOP, 8, comp_anc=True)
    assert ei.value.status == capi.PCSF_ERR_INVALID
    dm.close()


def test_fixed_and_mle_against_oracle():
    model = load_model("29mammals", "Human,Chimp,Mouse,Dog,Cow,Horse,Elephant,Armadillo,Rat,Rabbit,Cat,Megabat")
    dm = capi.DeviceModel(model)
    alns = [planted(model.nl, L, 700 + L, 0, conserve=c) for L, c in ((150, .9), (301, .6), (600, .85))]
    mc = orc.OracleModel(model.tree, model.S_c, model.f_c)
    mnc = orc.OracleModel(model.tree, model.S_nc, model.f_nc)
    rec = dm.score_regions(alns, [0, 0, 0], capi.STRATEGY_FIXED, 6, orf.STOPSTOP, 4)
    for x, s in zip(rec, _extract(alns, rec)):
        rp, ra = orc.run_fixed(mc, mnc, orc.translate(s), True)
        assert abs(float(x["phylo"]) - rp) <= 1e-3 and abs(float(x["anc"]) - ra) <= 1e-3
        if s.shape[1]:
            assert np.float32(orc.bls(model.tree, s, per_base=False)[0]) == x["bls"]
    # MLE on the six frames of alignments whose rows all descend from one ancestor, as test_mle_vs_oracle_random (DESIGN.md §6c: on
    # the planted rows above, pcsf_score_msa's own fit of the 600-column alignment differs from the oracle's)
    alns = [random_alignment(model.nl, L, seed=900 + L, gap=0.2, conserve=c) for L, c in ((150, .8), (301, .95), (600, .6))]
    rec = dm.score_regions(alns, [0, 0, 0], capi.STRATEGY_MLE, 6, orf.ASIS, 25)
    tight = 0
    for x, s in zip(rec, _extract(alns, rec)):
        rp, ra, info = orc.run_mle(mc, mnc, orc.translate(s), True)
        p, an = float(x["phylo"]), float(x["anc"])
        assert (p - rp) ** 2 <= 0.001 and (an - ra) ** 2 <= 0.001, (x, rp, ra, info)
        tight += abs(p - rp) <= 1e-3 and abs(an - ra) <= 1e-3
    assert tight >= len(rec) - 2
    dm.close()


@pytest.mark.parametrize("strategy", [capi.STRATEGY_FIXED, capi.STRATEGY_MLE])
def test_frame1_asis_equals_score_msa(strategy):
    model = load_model("29mammals")
    dm = capi.DeviceModel(model)
    alns, refs = _batch(model, 120)
    rec = dm.score_regions(alns, refs, strategy, 1, orf.ASIS, 25)
    phylo, anc, bls = dm.score_msa(alns, strategy)
    assert list(rec["aln"]) == list(range(len(alns)))
    assert list(rec["col_begin"]) == [0] * len(alns) and list(rec["col_end"]) == [a.shape[1] for a in alns]
    assert same_bits(rec["phylo"], phylo) and same_bits(rec["anc"], anc) and same_bits(rec["bls"], bls)
    dm.close()


def _best_from_all(rec_all, n_aln):
    out = []
    for i in range(n_aln):
        mine = rec_all[rec_all["aln"] == i]
        b = orf.best_index([float(v) for v in mine["phylo"]])
        out.append(None if b < 0 else mine[b])
    return out


def _check_best(best, rec_all, n_aln):
    assert len(best) == n_aln
    for i, (x, want) in enumerate(zip(best, _best_from_all(rec_all, n_aln))):
        assert int(x["aln"]) == i
        if want is None:
            assert (int(x["strand"]), int(x["frame"]), int(x["col_begin"]), int(x["col_end"])) == (0, 0, -1, -1)
            assert np.isnan(x["phylo"]) and np.isnan(x["anc"]) and np.isnan(x["bls"])
        else:
            assert same_record(x, want)


def test_best_only_rule_and_none_records():
    model = load_model("29mammals")
    dm = capi.DeviceModel(model)
    alns, refs = _batch(model, 160)
    alns.append(np.frombuffer(b"CCC" * 40, np.uint8)[None, :].repeat(model.nl, 0).copy())   # no stop, no ATG: no ORF at all
    refs.append(3)
    n = len(alns)
    for strategy in (capi.STRATEGY_FIXED, capi.STRATEGY_MLE):
        for mode, mc in ((orf.ATGSTOP, 25), (orf.ATGSTOP, 2), (orf.STOPSTOP, 5), (orf.ASIS, 25)):
            rec_all = dm.score_regions(alns, refs, strategy, 6, mode, mc)
            best = dm.score_regions(alns, refs, strategy, 6, mode, mc, best_only=True)
            _check_best(best, rec_all, n)
            if mode == orf.ATGSTOP and mc == 25:
                assert (best["frame"] == 0).sum() >= 7        # the short alignments and the ORF-free one
    dm.close()


def _tiny_branch_model(neg: float):
    """12flies with all branches shortened 1000-fold and one negative exchangeability: P(t) = exp(Qt) then has a negative entry of
    about neg * pi * t, inside PhyloModel_make's 1e-6 tolerance at the fixed tree for a small |neg| and outside it once the MLE
    search scales the tree up (instance.hpp:612-636 -> runtime_error -> NaN row, score_msa.hpp:124)."""
    model = copy.deepcopy(load_model("12flies"))
    t = model.tree
    t.branch_len = (np.asarray(t.branch_len, np.float64) * 1e-3).astype(np.float32)
    t.branch_len_f64 = np.asarray(t.branch_len_f64, np.float64) * 1e-3
    for S in (model.S_c, model.S_nc):
        S[5, 9] = S[9, 5] = neg
    return model


def test_best_only_with_nan_regions():
    model = _tiny_branch_model(-0.02)
    dm = capi.DeviceModel(model)
    alns = [planted(model.nl, L, 40 + L, 0) for L in (30, 90, 2)]
    rec_all = dm.score_regions(alns, [0, 0, 0], capi.STRATEGY_MLE, 6, orf.ASIS, 25)
    assert np.isnan(rec_all["phylo"]).any()
    best = dm.score_regions(alns, [0, 0, 0], capi.STRATEGY_MLE, 6, orf.ASIS, 25, best_only=True)
    _check_best(best, rec_all, len(alns))
    dm.close()


def test_error_statuses():
    model = load_model("12flies")
    dm = capi.DeviceModel(model)
    alns = [random_alignment(model.nl, 30, 1)]

    def status(**kw):
        args = dict(strategy=capi.STRATEGY_FIXED, frames=6, orf=orf.ATGSTOP, min_codons=25)
        args.update(kw)
        refs = args.pop("refs", [0])
        a = args.pop("alns", alns)
        try:
            dm.score_regions(a, refs, **args)
        except capi.PcsfError as e:
            return e.status
        return capi.PCSF_OK

    assert status(frames=2) == capi.PCSF_ERR_INVALID
    assert status(frames=0) == capi.PCSF_ERR_INVALID
    assert status(min_codons=0) == capi.PCSF_ERR_INVALID
    assert status(refs=[-1]) == capi.PCSF_ERR_INVALID
    assert status(refs=[model.nl]) == capi.PCSF_ERR_INVALID
    assert status(orf=3) == capi.PCSF_ERR_INVALID
    assert status(strategy=7) == capi.PCSF_ERR_INVALID
    assert status(strategy=capi.STRATEGY_OMEGA, comp_anc=True) == capi.PCSF_ERR_INVALID
    bad = alns[0].copy()
    bad[2, 5] = ord("X")
    assert status(alns=[bad]) == capi.PCSF_ERR_BAD_CHAR
    assert len(dm.score_regions([], [], capi.STRATEGY_MLE, 6, orf.ATGSTOP, 25)) == 0
    assert status() == capi.PCSF_OK
    dm.close()


def _scores(path):
    return [ln.rstrip("\n").split("\t") for ln in open(path)]


def test_cli_516(golden_dir, tmp_path):
    src = os.path.join(golden_dir, "score-msa", "chr22.516alignments.maf.gz")
    maf = str(tmp_path / "chr22.516alignments.maf")
    with gzip.open(src, "rb") as fi, open(maf, "wb") as fo:
        shutil.copyfileobj(fi, fo)
    model = load_model("100vertebrates")
    alns = list(MafReader(maf, model.seqid_to_phyloid, model.nl, False, warn=False))
    alns = [a for a in alns if a.ref_row >= 0]
    assert len(alns) == 516

    def run(tag, *opts):
        out = str(tmp_path / tag)
        subprocess.run([BIN, "score-msa", "--strategy", "fixed", "--comp-anc", "1", *opts, "--output", out, "100vertebrates", maf],
                       check=True, capture_output=True)
        return open(os.path.join(out, "chr22.516alignments.maf.scores"), "rb").read()

    # default options: the plain score-msa path and format, byte for byte
    plain = run("plain")
    assert run("explicit", "--frames", "1", "--orf", "AsIs", "--min-codons", "25", "--all-scores", "0") == plain
    dm = capi.DeviceModel(model)
    phylo, anc, bls = dm.score_msa([a.seqs for a in alns], capi.STRATEGY_FIXED)
    lines = plain.decode().splitlines()
    assert lines[1] == "seq\tstart\tend\tstrand\tphylocsf-score\tanc-score\tbls-score"
    want = ["%s\t%d\t%d\t%s\t%.6f\t%.6f\t%.6f" % (a.chrom, a.start_pos, a.start_pos + a.L - 1, a.strand, p, an, b)
            for a, p, an, b in zip(alns, phylo, anc, bls)]
    assert lines[2:] == want

    # all scores: one row per region, the capi records formatted with %.6f, ORF columns mapped onto start / end
    all_txt = run("all", "--frames", "6", "--orf", "ATGStop", "--all-scores", "1").decode().splitlines()
    assert all_txt[1] == "seq\tstart\tend\tstrand\tframe\torf-start\torf-end\tphylocsf-score\tanc-score\tbls-score"
    rec = dm.score_regions([a.seqs for a in alns], [a.ref_row for a in alns], capi.STRATEGY_FIXED, 6, orf.ATGSTOP, 25)
    assert len(rec) == len(all_txt) - 2 > 0
    for x, ln in zip(rec, all_txt[2:]):
        a = alns[int(x["aln"])]
        fr = "%s%d" % ("+" if x["strand"] > 0 else "-", x["frame"])
        assert ln == "%s\t%d\t%d\t%s\t%s\t%d\t%d\t%.6f\t%.6f\t%.6f" % (
            a.chrom, a.start_pos, a.start_pos + a.L - 1, a.strand, fr, a.start_pos + x["col_begin"], a.start_pos + x["col_end"] - 1,
            x["phylo"], x["anc"], x["bls"])
        assert (int(x["col_end"]) - int(x["col_begin"])) == 3 * int(x["codons"])

    # best only: one row per block, the per-block maximum of the all-scores rows (NaN never wins, ties: the first row)
    best_txt = run("best", "--frames", "6", "--orf", "ATGStop").decode().splitlines()[2:]
    assert len(best_txt) == 516
    rows_all = [ln.split("\t") for ln in all_txt[2:]]
    by_block = {}
    for r in rows_all:
        by_block.setdefault((r[0], r[1], r[2], r[3]), []).append(r)
    for ln in best_txt:
        r = ln.split("\t")
        cand = by_block.get(tuple(r[:4]), [])
        if not cand:
            assert r[4:7] == [".", ".", "."] and r[7:] in (["nan"] * 3, ["-nan"] * 3), r
            continue
        b = orf.best_index([float(c[7]) for c in cand])
        assert r == cand[b] or float(r[7]) == float(cand[b][7]), (r, cand[b])
    dm.close()
