"""Species trees of 129 to 512 leaves (tests/large_tree_shapes.py) on the GPU: model creation and the leaf limit, the rescaled FP64
pruning (k_prune_scaled) against the C oracle and an extended-precision pruning, windows on which the reference's unscaled product
underflows, bit-for-bit invariances, score-msa (FIXED, MLE, OMEGA, reading frames) and the command line on large models."""
import functools
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import oracle as orc
from phylocsfpp_b200 import capi, orf, tracks
from phylocsfpp_b200.maf import MafReader
from phylocsfpp_b200.models import load_model
from tests import large_tree_shapes as lt
from tests.util import pattern_index_reference, prune_longdouble, random_alignment

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "phylocsfpp_b200", "bin", "phylocsf_b200")
TOL64 = 1e-6            # decibans, FP64 path against the oracle where the oracle's likelihoods are normal doubles
REL_LOGZ = 1e-12        # relative error of log z against the extended-precision pruning, on every window
LOG_DBL_MIN = np.log(np.finfo(np.float64).tiny)
DB = 10.0 / np.log(10.0)


@pytest.fixture(scope="module")
def tree_dir(tmp_path_factory):
    d = str(tmp_path_factory.mktemp("large_trees"))
    for t in lt.ALL:
        lt.write_model(d, t.spec)
    lt.write_model(d, lt.TOO_LARGE)
    return d


@functools.lru_cache(maxsize=None)
def _load(prefix):
    return load_model(prefix)


def model_of(tree_dir, name):
    return _load(os.path.join(tree_dir, name))


def window_codons(seqs, idx):
    plus, minus = orc.window_codons(seqs)
    o, s = idx // 2, idx % 2
    return np.where(s[None, :] == 0, plus[:, o], minus[:, o])


def interleave(res):
    out = np.empty(2 * len(res["plus"]))
    out[0::2], out[1::2] = res["plus"], res["minus"]
    return out


def references(model, dm, seqs, idx):
    """Oracle decibans and the extended-precision log z of both models (over the device's own P and pi)."""
    cod = window_codons(seqs, idx)
    ref = orc.run_tracks(orc.OracleModel(model.tree, model.S_c, model.f_c), orc.OracleModel(model.tree, model.S_nc, model.f_nc), cod)
    lz = []
    for which in (0, 1):
        _, pi, P = dm.get(which)
        lz.append(prune_longdouble(model.tree, P, pi, cod))
    return ref, lz


def check_against_references(model, dm, seqs, res, idx):
    """Within TOL64 of the oracle on every window whose oracle likelihoods are both normal doubles; within REL_LOGZ (relative, on
    log z of each model, expressed in decibans) of the extended-precision pruning on every window; finite everywhere."""
    got = interleave(res)[idx]
    assert np.isfinite(got).all()
    ref, lz = references(model, dm, seqs, idx)
    exact = (DB * (lz[0] - lz[1])).astype(np.float64)
    bound = (REL_LOGZ * DB * (np.abs(lz[0]) + np.abs(lz[1]))).astype(np.float64) + 1e-13
    assert (np.abs(got - exact) <= bound).all(), np.abs(got - exact).max()
    normal = (np.minimum(lz[0], lz[1]) > LOG_DBL_MIN + 1.0).astype(bool) & np.isfinite(ref)
    d = np.abs(got[normal] - ref[normal]).max() if normal.any() else 0.0
    assert d <= TOL64, d
    return d, int((~normal).sum())


def test_every_large_tree_gives_a_model(tree_dir):
    """pcsf_model_create succeeds on every tree of 129 to 512 leaves and refuses 513 with PCSF_ERR_UNSUPPORTED; PCSF_TRACKS_TC5 is
    refused with PCSF_ERR_UNSUPPORTED and the FP64 path runs on the same handle (within TOL64 of the oracle on a short input)."""
    for t in lt.ALL:
        model = model_of(tree_dir, t.name)
        dm = capi.DeviceModel(model)
        seqs = random_alignment(model.nl, 12, seed=t.nl, gap=0.5, conserve=0.9)
        with pytest.raises(capi.PcsfError) as ei:
            dm.tracks(seqs, tc5=True)
        assert ei.value.status == capi.PCSF_ERR_UNSUPPORTED and "tcgen05" in str(ei.value)
        f64 = dm.tracks(seqs)
        ref = orc.run_tracks(orc.OracleModel(model.tree, model.S_c, model.f_c), orc.OracleModel(model.tree, model.S_nc, model.f_nc),
                             orc.window_codons(seqs)[0])
        ok = np.isfinite(ref)
        assert np.isfinite(f64["plus"]).all() and (np.abs(f64["plus"][ok] - ref[ok]) <= TOL64).all(), t.name
        assert np.array_equal(f64["bls"], orc.bls(model.tree, seqs)[1]), t.name
        dm.close()
    with pytest.raises(capi.PcsfError) as ei:
        capi.DeviceModel(model_of(tree_dir, lt.TOO_LARGE.name))
    assert ei.value.status == capi.PCSF_ERR_UNSUPPORTED


@pytest.mark.parametrize("name", ["balanced129", "yule192", "caterpillar257", "balanced470", "yule470", "balanced512"])
def test_tracks_on_large_trees(tree_dir, name):
    """pcsf_tracks (FP64) on 120 random columns: every window against both references, BLS and pattern indices bit for bit."""
    t = lt.BY_NAME[name]
    model = model_of(tree_dir, name)
    seqs = random_alignment(model.nl, 120, seed=9000 + t.nl, gap=0.3, conserve=0.7)
    dm = capi.DeviceModel(model)
    res = dm.tracks(seqs, want_patterns=True)
    idx = np.arange(2 * (seqs.shape[1] - 2))
    d, n_under = check_against_references(model, dm, seqs, res, idx)
    assert np.array_equal(res["bls"], orc.bls(model.tree, seqs)[1])
    plus, minus = orc.window_codons(seqs)
    assert np.array_equal(res["pattern_index"], pattern_index_reference(plus, minus, 1 << 22))
    print(f"{name}: max |d| vs oracle {d:.3e} decibans, {n_under} of {len(idx)} windows outside the double range in the oracle")
    dm.close()


def test_underflow_on_the_long_caterpillar(tree_dir):
    """All-certain codons on the 512-leaf caterpillar whose branches are all long: the reference's unscaled likelihood is far below
    the double range and the oracle's score is not finite.  The device's is finite and agrees with the extended-precision pruning.
    Mostly-gap windows on the same tree stay in range: there the device agrees with the oracle."""
    model = model_of(tree_dir, lt.LONG_CATERPILLAR_512.name)
    rng = np.random.default_rng(5)
    seqs = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, size=(model.nl, 60))].copy()
    seqs[:, 40:] = ord("N")
    seqs[:24, 40:] = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, size=(24, 20))]    # 24 certain leaves: no underflow
    dm = capi.DeviceModel(model)
    res = dm.tracks(seqs)
    idx = np.arange(2 * (seqs.shape[1] - 2))
    ref, lz = references(model, dm, seqs, idx)
    got = interleave(res)[idx]
    under = idx < 2 * 38                                   # windows entirely in the all-certain columns
    assert not np.isfinite(ref[under]).any(), "the oracle is meant to underflow here"
    assert (np.minimum(lz[0], lz[1])[under] < LOG_DBL_MIN - 100).all()
    assert np.isfinite(got).all()
    exact = (DB * (lz[0] - lz[1])).astype(np.float64)
    rel = np.abs(got - exact) / (DB * (np.abs(lz[0]) + np.abs(lz[1]))).astype(np.float64)
    assert rel.max() <= REL_LOGZ, rel.max()
    calm = idx >= 2 * 40
    assert np.isfinite(ref[calm]).all() and np.abs(got[calm] - ref[calm]).max() <= TOL64
    print(f"long caterpillar512: log z down to {float(np.min(lz[0])):.1f}; max relative error of log z {rel.max():.2e}")
    dm.close()


def _with_env(monkeypatch, model, **env):
    for k, v in env.items():
        monkeypatch.setenv(k, str(v))
    try:
        return capi.DeviceModel(model)
    finally:
        for k in env:
            monkeypatch.delenv(k)


def _rc(seqs):
    return orc.reverse_complement(seqs)


@pytest.mark.parametrize("name", ["yule129", "caterpillar470", "balanced512"])
def test_large_tree_results_are_invariant(tree_dir, monkeypatch, name):
    """Bit-identical tracks with dedup on and off, with small chunks, with every warp count that fits (12, 8, 4), and '+' / '-'
    windows of the reverse-complemented alignment equal to '-' / '+' windows of the original."""
    model = model_of(tree_dir, name)
    seqs = random_alignment(model.nl, 3000, seed=model.nl, gap=0.3, conserve=0.8)
    dm = capi.DeviceModel(model)
    base = dm.tracks(seqs)
    nod = dm.tracks(seqs, dedup=False)
    dm.set_chunk_columns(700)
    chunked = dm.tracks(seqs)
    rc = dm.tracks(_rc(seqs))
    dm.close()
    for r in (nod, chunked):
        assert np.array_equal(r["plus"], base["plus"]) and np.array_equal(r["minus"], base["minus"])
        assert np.array_equal(r["bls"], base["bls"])
    assert np.array_equal(rc["plus"], base["minus"][::-1]) and np.array_equal(rc["minus"], base["plus"][::-1])
    assert np.array_equal(rc["bls"], base["bls"][::-1])
    # the host steps 12 -> 8 -> 4 warps until shared memory fits: every count that fits this tree runs once
    for nw in (12, 8, 4):
        dmw = _with_env(monkeypatch, model, PCSF_PRUNE_NWARP=nw)
        r = dmw.tracks(seqs, bls=False)
        dmw.close()
        assert np.array_equal(r["plus"], base["plus"]) and np.array_equal(r["minus"], base["minus"]), nw


def _alns(model, n, lo, hi, seed, conserve=(0.6, 0.95), gap=0.25):
    rng = np.random.default_rng(seed)
    return [random_alignment(model.nl, 3 * int(k), seed=seed + i, gap=gap, conserve=float(c))
            for i, (k, c) in enumerate(zip(rng.integers(lo, hi + 1, n), rng.uniform(*conserve, n)))]


def test_score_msa_fixed_on_a_470_leaf_model(tree_dir):
    """FIXED on 30 alignments: a batch equals its two halves bit for bit; BLS equals the oracle's bit for bit; phylo is within 1e-3
    decibans (plus float32 rounding) of the extended-precision pruning over the device's own P and pi on every alignment; phylo and
    anc are within 1e-3 of the oracle (the reference's CI tolerance) on every alignment whose codon likelihoods are all normal
    doubles in the oracle.  Where one is not, the oracle's unscaled product is -inf / NaN or, in the subnormal range, has lost most
    of its significant digits (measured: 0.009 decibans off on a codon at e^-737.7), so only the extended-precision pruning is
    a reference there."""
    model = model_of(tree_dir, "yule470")
    alns = _alns(model, 30, 10, 80, 470)
    mc = orc.OracleModel(model.tree, model.S_c, model.f_c)
    mnc = orc.OracleModel(model.tree, model.S_nc, model.f_nc)
    dm = capi.DeviceModel(model)
    phylo, anc, bls = dm.score_msa(alns, capi.STRATEGY_FIXED)
    h1, h2 = dm.score_msa(alns[:13], capi.STRATEGY_FIXED), dm.score_msa(alns[13:], capi.STRATEGY_FIXED)
    P_pi = [(dm.get(which)[2], dm.get(which)[1]) for which in (0, 1)]      # (P, pi) of each ECM as the device uses them
    dm.close()
    for k, full in enumerate((phylo, anc, bls)):
        assert np.array_equal(np.concatenate([h1[k], h2[k]]).view(np.uint32), np.asarray(full).view(np.uint32))
    peps = [orc.translate(a) for a in alns]
    cod = np.concatenate(peps, axis=1)
    lz = [prune_longdouble(model.tree, P, pi, cod) for P, pi in P_pi]
    ends = np.cumsum([0] + [p.shape[1] for p in peps])
    n_oracle = 0
    for i, (a, pep, p, an, b) in enumerate(zip(alns, peps, phylo, anc, bls)):
        exact = np.float64(DB * (lz[0][ends[i]:ends[i + 1]] - lz[1][ends[i]:ends[i + 1]]).sum())
        assert np.isfinite(p) and abs(float(p) - exact) <= 1e-3 + float(np.spacing(np.float32(exact))), (i, float(p), exact)
        assert np.float32(orc.bls(model.tree, a, per_base=False)[0]) == b
        if min(mc.lpr_leaves(pep)[2].min(), mnc.lpr_leaves(pep)[2].min()) > LOG_DBL_MIN:
            rp, ra = orc.run_fixed(mc, mnc, pep, True)
            assert abs(float(p) - float(rp)) <= 1e-3 and abs(float(an) - float(ra)) <= 1e-3, (i, float(p), rp, float(an), ra)
            n_oracle += 1
    assert 0 < n_oracle < len(alns), n_oracle      # both kinds of alignment are in the batch


def test_score_msa_mle_and_omega_on_a_470_leaf_model(tree_dir):
    """MLE within the reference's CI tolerance ((d phylo)^2 <= 1e-3) of the oracle on short alignments, OMEGA within its tolerance
    ((d)^2 <= 0.1) on a few; the slot budget gives the batch more than one slot.  The alignments are chosen so that the oracle's
    codon likelihoods stay normal doubles over the whole rho range of the fit (checked at its ends and in between), so the oracle
    is a valid reference for every evaluation of its Brent search."""
    model = model_of(tree_dir, "balanced470")
    alns = _alns(model, 4, 8, 20, 4700, conserve=(0.85, 0.95), gap=0.4)
    mc = orc.OracleModel(model.tree, model.S_c, model.f_c)
    mnc = orc.OracleModel(model.tree, model.S_nc, model.f_nc)
    for om in (mc, mnc):
        for rho in (1e-2, 1e-1, 1.0, 10.0):
            om.set_rho(rho)
            assert all(om.lpr_leaves(orc.translate(a))[2].min() > LOG_DBL_MIN for a in alns), (rho, "pick alignments without subnormal codons")
        om.set_rho(1.0)
    dm = capi.DeviceModel(model)
    phylo, anc, _ = dm.score_msa(alns, capi.STRATEGY_MLE)
    st = dm.score_msa_stats()
    om = dm.score_msa(alns[:2], capi.STRATEGY_OMEGA, comp_anc=False)[0]
    dm.close()
    assert st["slots"] >= min(len(alns), 2), st
    for a, p, an in zip(alns, phylo, anc):
        rp, ra, _ = orc.run_mle(mc, mnc, orc.translate(a), True)
        assert np.isfinite(rp) and (float(p) - float(rp)) ** 2 <= 1e-3 and (float(an) - float(ra)) ** 2 <= 1e-3, (p, rp, an, ra)
    for a, p in zip(alns[:2], om):
        rp = float(orc.run_omega(model.tree, orc.translate(a))[0])
        assert (float(p) - rp) ** 2 <= 0.1, (p, rp)


def test_reading_frames_on_a_470_leaf_model(tree_dir):
    """One --frames 6 --orf atgstop call returns, bit for bit, what pcsf_score_msa returns for the extracted regions."""
    model = model_of(tree_dir, "yule470")
    from tests.test_gpu_score_regions import planted
    alns = [planted(model.nl, L, 300 + L, (13 * L) % model.nl) for L in (90, 150, 301)]
    refs = [(13 * L) % model.nl for L in (90, 150, 301)]
    dm = capi.DeviceModel(model)
    rec = dm.score_regions(alns, refs, capi.STRATEGY_FIXED, 6, orf.ATGSTOP, 2)
    subs = []
    for x in rec:
        r = orf.Region(int(x["strand"]), int(x["frame"]), 0, int(x["codons"]), int(x["col_begin"]), int(x["col_end"]))
        subs.append(orf.sub_alignment(alns[int(x["aln"])], r))
    phylo, anc, bls = dm.score_msa(subs, capi.STRATEGY_FIXED)
    dm.close()
    assert len(rec) >= 3
    for got, exp in ((rec["phylo"], phylo), (rec["anc"], anc), (rec["bls"], bls)):
        assert np.array_equal(np.asarray(got, np.float32).view(np.uint32), np.asarray(exp, np.float32).view(np.uint32))


def test_mle_on_an_underflowing_input_is_finite(tree_dir):
    """MLE on all-certain alignments of the long-branch 512-leaf caterpillar, where the oracle's likelihoods underflow: finite scores."""
    model = model_of(tree_dir, lt.LONG_CATERPILLAR_512.name)
    rng = np.random.default_rng(11)
    alns = [np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, size=(model.nl, 3 * k))].copy() for k in (5, 9, 14)]
    mc = orc.OracleModel(model.tree, model.S_c, model.f_c)
    mnc = orc.OracleModel(model.tree, model.S_nc, model.f_nc)
    assert not np.isfinite(orc.run_fixed(mc, mnc, orc.translate(alns[0]), False)[0])
    dm = capi.DeviceModel(model)
    phylo, anc, _ = dm.score_msa(alns, capi.STRATEGY_MLE)
    fixed = dm.score_msa(alns, capi.STRATEGY_FIXED)[0]
    dm.close()
    assert np.isfinite(phylo).all() and np.isfinite(anc).all() and np.isfinite(fixed).all()


def _maf(path, model, seqs, start0):
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from make_synth_maf import write_synth_maf
    write_synth_maf(path, model, seqs.shape[1], seed=3, start0=start0, mean_block=10 ** 9, hole_p=0.0, ref_gap=0.0, alien_p=0.0,
                    mat=seqs)


def test_build_tracks_cli_on_a_300_leaf_model(tree_dir, tmp_path):
    """build-tracks (FP64) on a one-block MAF for a 300-leaf model writes the seven wig files the oracle's scores give, byte for
    byte; --species reduces the tree to 200 leaves and again matches the oracle on the reduced model; --precision tc5 stops with a
    message that names the tcgen05 path."""
    from tests.tree_shapes import Shape
    prefix = lt.write_model(str(tmp_path), Shape("yule", 300))
    model = load_model(prefix)
    seqs = random_alignment(model.nl, 400, seed=300, gap=0.3, conserve=0.8)
    seqs[0] = np.frombuffer(b"ACGT", np.uint8)[np.random.default_rng(1).integers(0, 4, seqs.shape[1])]   # no reference gaps
    maf = str(tmp_path / "large.maf")
    _maf(maf, model, seqs, 12345)

    def expected(m):
        alns = list(MafReader(maf, m.seqid_to_phyloid, m.nl, True, warn=False))
        mc, mnc = orc.OracleModel(m.tree, m.S_c, m.f_c), orc.OracleModel(m.tree, m.S_nc, m.f_nc)
        out = {k: [] for k in tracks.FRAMES}
        power = []
        for a in alns:
            plus, minus = orc.window_codons(a.seqs)
            p, mi = orc.run_tracks(mc, mnc, plus), orc.run_tracks(mc, mnc, minus)
            assert np.isfinite(p).all() and np.isfinite(mi).all(), "this input is meant to stay inside the double range"
            b = orc.bls(m.tree, a.seqs)[1]
            power += tracks.power_wig(a.chrom, a.start_pos, b)
            r = tracks.raw_wigs(a.chrom, a.start_pos, a.chrom_len, p, mi, b)
            for k in out:
                out[k] += r[k]
        return power, out

    def check(outdir, m):
        power, out = expected(m)
        with open(os.path.join(outdir, "PhyloCSFpower.wig")) as fh:
            assert fh.read().splitlines() == power
        for (s, f), lines in out.items():
            with open(os.path.join(outdir, tracks.wig_filename(s, f))) as fh:
                assert fh.read().splitlines() == lines, (s, f)

    out = str(tmp_path / "f64")
    subprocess.run([BIN, "build-tracks", "--threads", "2", "--output", out, prefix, maf], check=True, capture_output=True)
    check(out, model)
    species = ",".join(model.tree.labels[i] for i in range(0, 300) if i % 3 != 2)
    out = str(tmp_path / "species")
    subprocess.run([BIN, "build-tracks", "--threads", "2", "--species", species, "--output", out, prefix, maf], check=True,
                   capture_output=True)
    reduced = load_model(prefix, species)
    assert reduced.nl == 200
    check(out, reduced)
    r = subprocess.run([BIN, "build-tracks", "--precision", "tc5", "--output", str(tmp_path / "tc5"), prefix, maf], capture_output=True,
                       text=True)
    assert r.returncode != 0 and "tcgen05" in (r.stdout + r.stderr) and "CUDA" not in (r.stdout + r.stderr), r.stdout + r.stderr
