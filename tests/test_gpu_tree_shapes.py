"""Both pruning kernels on generated trees of 2 to 128 leaves (tests/tree_shapes.py), against the C oracle and an extended-precision
pruning of the device's own P and pi.

The built-in models only reach a few program shapes: every one gets 12 FP64 warps, and their tcgen05 programs have stack depths up
to 3 and about 100 steps.  The generated trees add 8- and 4-warp FP64 runs (32-window tiles), tcgen05 programs without any GEMM
step, starts made of cherries, stack depths 4 and 5 (spilled to global scratch), 117 steps, and trees on both sides of the 64-leaf
word boundary of k_bls's presence mask, up to PCSF_MAX_LEAVES.
"""
import functools
import os

import numpy as np
import pytest

from oracle import oracle as orc
from phylocsfpp_b200 import capi
from phylocsfpp_b200.models import load_model
from tests import tree_shapes as ts
from tests.util import pattern_index_reference, prune_longdouble, random_alignment

pytestmark = pytest.mark.gpu

TOL64 = 1e-6      # decibans, FP64 path against the oracle (the contract is 1e-3)
TOL5 = 2e-4       # decibans, tcgen05 path against the extended-precision reference (the contract is 1e-3)
MAX_REF_WINDOWS = 1100


@pytest.fixture(scope="module")
def tree_dir(tmp_path_factory):
    d = str(tmp_path_factory.mktemp("trees"))
    for spec in ts.BY_NAME.values():
        ts.write_model(d, spec)
    return d


@functools.lru_cache(maxsize=None)
def _load(prefix):
    return load_model(prefix)


def model_of(tree_dir, name):
    return _load(os.path.join(tree_dir, name))


def window_codons(seqs, idx):
    """Codon ids [nl, len(idx)] of windows idx (window 2 o + s: offset o, strand s, the pattern_index order)."""
    plus, minus = orc.window_codons(seqs)
    o, s = idx // 2, idx % 2
    return np.where(s[None, :] == 0, plus[:, o], minus[:, o])


def references(model, dm, seqs, idx):
    """(oracle, extended precision) decibans of windows idx.  The extended-precision pruning runs over the device's own P and pi."""
    cod = window_codons(seqs, idx)
    mc = orc.OracleModel(model.tree, model.S_c, model.f_c)
    mnc = orc.OracleModel(model.tree, model.S_nc, model.f_nc)
    ref = orc.run_tracks(mc, mnc, cod)
    lz = []
    for which in (0, 1):
        _, pi, P = dm.get(which)
        lz.append(prune_longdouble(model.tree, P, pi, cod))
    exact = (10.0 * (lz[0] - lz[1]) / np.log(np.longdouble(10.0))).astype(np.float64)
    return ref, exact


def sample_windows(nwin, rng, extra=()):
    if nwin <= MAX_REF_WINDOWS:
        return np.arange(nwin)
    idx = np.unique(np.concatenate([np.arange(128), np.arange(nwin - 128, nwin), rng.integers(0, nwin, 600),
                                    np.asarray(extra, np.int64)]))
    return idx[(idx >= 0) & (idx < nwin)]


def interleave(res):
    out = np.empty(2 * len(res["plus"]))
    out[0::2], out[1::2] = res["plus"], res["minus"]
    return out


def check_fp64(model, seqs, res, idx, ref, exact):
    """FP64 path: within TOL64 of the oracle wherever the oracle is finite and agrees with the extended-precision pruning to
    TOL64; finite exactly where the oracle is; BLS bit for bit."""
    got = interleave(res)[idx]
    assert np.array_equal(np.isfinite(got), np.isfinite(ref))
    ok = np.isfinite(ref) & (np.abs(ref - exact) < TOL64)
    assert ok.mean() >= 0.9, f"the oracle resolves only {ok.mean():.3f} of the windows"
    d = np.abs(got[ok] - ref[ok]).max()
    assert d <= TOL64, d
    assert np.array_equal(res["bls"], orc.bls(model.tree, seqs)[1]), "BLS must be bit-exact"
    return d


def check_tc5(t5, f64, idx, exact):
    """tcgen05 path: within TOL5 of the extended-precision pruning, finite, same BLS and pattern indices as the FP64 path."""
    got = interleave(t5)[idx]
    assert np.isfinite(interleave(t5)).all()
    d = np.abs(got - exact).max()
    assert d <= TOL5, d
    assert np.array_equal(t5["bls"], f64["bls"])
    if f64["pattern_index"] is not None:
        assert np.array_equal(t5["pattern_index"], f64["pattern_index"])
    return d


@pytest.mark.parametrize("name", list(ts.BY_NAME))
def test_every_tree_gives_a_model(tree_dir, name):
    """pcsf_model_create succeeds for every tree of 2 to 128 leaves.  The tcgen05 path is accepted on every tree that fits its
    shared memory (all trees of at most 123 leaves, balanced 125); on the others it is refused with PCSF_ERR_UNSUPPORTED and the
    FP64 path still runs on the same handle."""
    spec = ts.BY_NAME[name]
    assert spec.tc5_fits or spec.nl > 123
    model = model_of(tree_dir, name)
    dm = capi.DeviceModel(model)
    seqs = random_alignment(model.nl, 40, seed=spec.nl)
    f64 = dm.tracks(seqs)
    if spec.tc5_fits:
        t5 = dm.tracks(seqs, tc5=True)
        assert max(np.abs(t5["plus"] - f64["plus"]).max(), np.abs(t5["minus"] - f64["minus"]).max()) <= TOL5
    else:
        with pytest.raises(capi.PcsfError) as ei:
            dm.tracks(seqs, tc5=True)
        assert ei.value.status == capi.PCSF_ERR_UNSUPPORTED
        again = dm.tracks(seqs)
        assert np.array_equal(again["plus"], f64["plus"]) and np.array_equal(again["minus"], f64["minus"])
    ref_p = orc.run_tracks(orc.OracleModel(model.tree, model.S_c, model.f_c), orc.OracleModel(model.tree, model.S_nc, model.f_nc),
                           orc.window_codons(seqs)[0])
    assert np.abs(f64["plus"] - ref_p).max() <= TOL64
    dm.close()


@pytest.mark.parametrize("name", [s.name for s in ts.SHAPES])
def test_tracks_on_generated_trees(tree_dir, name):
    """Both paths on 500 random columns (996 windows, every one checked against both references).

    Measured on one B200 (1000 W power limit), max |tcgen05 - extended precision| in decibans: balanced2 6.0e-7, leafcherry3
    7.2e-7, balanced4 7.9e-7, caterpillar63 4.5e-5, caterpillar64 5.1e-5, caterpillar65 6.1e-5, balanced63 3.2e-5, balanced64
    3.0e-5, balanced65 4.1e-5, yule65 6.2e-5, yule100 8.6e-5, caterpillar120 6.7e-5, balanced125 4.5e-5 (the 128-leaf trees do
    not fit the tcgen05 path).  The FP64 path agreed with the oracle to 2.5e-13 decibans or better on every tree."""
    spec = ts.BY_NAME[name]
    model = model_of(tree_dir, name)
    seqs = random_alignment(model.nl, 500, seed=7000 + spec.nl + 100 * len(spec.shape), gap=0.3, conserve=0.7)
    dm = capi.DeviceModel(model)
    f64 = dm.tracks(seqs, want_patterns=True)
    idx = np.arange(2 * (seqs.shape[1] - 2))
    ref, exact = references(model, dm, seqs, idx)
    d64 = check_fp64(model, seqs, f64, idx, ref, exact)
    plus, minus = orc.window_codons(seqs)
    assert np.array_equal(f64["pattern_index"], pattern_index_reference(plus, minus, 1 << 22))
    msg = f"{name}: FP64 path max |d| vs oracle {d64:.3e}"
    if spec.tc5_fits:
        t5 = dm.tracks(seqs, want_patterns=True, tc5=True)
        msg += f", tcgen05 path max |d| vs extended precision {check_tc5(t5, f64, idx, exact):.3e} decibans"
    print(msg)
    dm.close()


def test_long_branches_all_certain_columns(tree_dir):
    """All-certain random codons on the 128-leaf caterpillar whose branches are all long (nearly stationary P): the reference's
    unscaled FP64 likelihood falls to about 1e-264, close to the bottom of the double range.  The FP64 path must still agree with
    the oracle wherever the oracle agrees with the extended-precision pruning (and be finite exactly where the oracle is)."""
    model = model_of(tree_dir, ts.LONG_CATERPILLAR.name)
    rng = np.random.default_rng(5)
    seqs = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, size=(model.nl, 300))]
    dm = capi.DeviceModel(model)
    f64 = dm.tracks(seqs)
    idx = np.arange(2 * (seqs.shape[1] - 2))
    ref, exact = references(model, dm, seqs, idx)
    cod = window_codons(seqs, idx)
    _, pi, P = dm.get(0)
    assert prune_longdouble(model.tree, P, pi, cod).min() < np.log(1e-250), "this input is meant to come close to underflow"
    print(f"long caterpillar: FP64 path max |d| vs oracle {check_fp64(model, seqs, f64, idx, ref, exact):.3e} decibans")
    dm.close()


def _tile_inputs(nl, n_sm):
    """(label, seqs, dedup, unique-pattern count) on nl leaves.  Even counts: dedup off, 2 (L - 2) windows.  Odd counts: dedup on
    and the last column all N, so that the '+' and '-' window of the last offset are one pattern (every leaf's codon is missing)."""
    out = [("1", np.full((nl, 3), ord("N"), np.uint8), True, 1)]
    for k in (255, 257, 2 * n_sm * 256 + 1):
        L = (k - 1) // 2 + 3
        seqs = random_alignment(nl, L, seed=k, gap=0.3, conserve=0.7)
        seqs[:, -1] = ord("N")
        out.append((str(k), seqs, True, k))
    out.append(("256", random_alignment(nl, 130, seed=256), False, 256))
    return out


def test_tile_boundaries_on_a_deep_tree(tree_dir):
    """The balanced 125-leaf tree (FP64: 4 warps, 32-window tiles, stack depth 5; tcgen05: stack depth 5, the deepest that fits)
    with 1, 255, 256, 257 and 2 x SMs x 256 + 1 unique patterns: one window, one short of a pair of 128-window tiles, exactly
    one pair, one over, and one pair more than two passes of the persistent grid."""
    import torch
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    model = model_of(tree_dir, "balanced125")
    dm = capi.DeviceModel(model)
    rng = np.random.default_rng(125)
    for label, seqs, dedup, k in _tile_inputs(model.nl, n_sm):
        f64 = dm.tracks(seqs, dedup=dedup, want_patterns=True)
        t5 = dm.tracks(seqs, dedup=dedup, want_patterns=True, tc5=True)
        assert f64["stats"]["n_unique"] == k and t5["stats"]["n_unique"] == k, (label, f64["stats"], t5["stats"])
        nwin = 2 * (seqs.shape[1] - 2)
        if dedup:
            plus, minus = orc.window_codons(seqs)
            assert np.array_equal(f64["pattern_index"], pattern_index_reference(plus, minus, 1 << 22))
        else:
            assert np.array_equal(f64["pattern_index"], np.arange(nwin, dtype=np.uint32))
        # every pattern rank here is its window index up to the last offset, so these are the tiles' edges
        edges = [r + e for r in range(0, nwin, 256 * n_sm) for e in (-1, 0, 1)] + [r + e for r in range(0, nwin, 256) for e in (-1, 0)][:400]
        idx = sample_windows(nwin, rng, edges)
        ref, exact = references(model, dm, seqs, idx)
        d64 = check_fp64(model, seqs, f64, idx, ref, exact)
        d5 = check_tc5(t5, f64, idx, exact)
        full = max(np.abs(t5["plus"] - f64["plus"]).max(), np.abs(t5["minus"] - f64["minus"]).max())
        assert full <= TOL5, full
        print(f"balanced125, {k} patterns: FP64 {d64:.3e}, tcgen05 {d5:.3e} (vs FP64 on all {nwin} windows: {full:.3e})")
    dm.close()


def _with_env(monkeypatch, model, **env):
    """A DeviceModel created with the given PCSF_* knobs (pcsf_model_create reads them once)."""
    for k, v in env.items():
        monkeypatch.setenv(k, str(v))
    try:
        return capi.DeviceModel(model)
    finally:
        for k in env:
            monkeypatch.delenv(k)


@pytest.mark.parametrize("name", ["yule128", "58mammals"])
def test_fp64_warp_count_does_not_change_results(tree_dir, monkeypatch, name):
    """k_prune with 12, 8 and 4 compute warps per CTA (8-window slices of 96-, 64- and 32-window tiles; the host itself steps 12 ->
    8 -> 4 until shared memory fits): every window is pruned by one warp on its own, so the tracks are bit-identical."""
    model = model_of(tree_dir, name) if name in ts.BY_NAME else load_model(name)
    seqs = random_alignment(model.nl, 20000, seed=128, gap=0.3, conserve=0.8)
    runs = []
    for nwarp in (12, 8, 4):
        dm = _with_env(monkeypatch, model, PCSF_PRUNE_NWARP=nwarp)
        runs.append(dm.tracks(seqs, bls=False))
        dm.close()
    for r in runs[1:]:
        assert np.array_equal(r["plus"], runs[0]["plus"]) and np.array_equal(r["minus"], runs[0]["minus"])


@pytest.mark.parametrize("name", ["balanced4", "caterpillar63", "balanced63"])
def test_tc5_ring_depths_do_not_change_results(tree_dir, monkeypatch, name):
    """k_prune_tc5 with its default rings and with PCSF_TC5_NSTAGE=2, PCSF_TC5_NIDS=1 (a single codon-id buffer), on more pairs
    of tiles than SMs: bit-identical.  These trees double-buffer the codon ids by default; from 64 leaves up the ids of a pair of
    tiles are too large for two buffers and every tree already runs with nstage 2, nids 1."""
    import torch
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    model = model_of(tree_dir, name)
    seqs = random_alignment(model.nl, 40000, seed=63, gap=0.3, conserve=0.7)
    dm = capi.DeviceModel(model)
    a = dm.tracks(seqs, bls=False, dedup=False, tc5=True)
    dm.close()
    dm = _with_env(monkeypatch, model, PCSF_TC5_NSTAGE=2, PCSF_TC5_NIDS=1)
    b = dm.tracks(seqs, bls=False, dedup=False, tc5=True)
    dm.close()
    assert a["stats"]["n_unique"] > 2 * 256 * n_sm
    assert np.array_equal(a["plus"], b["plus"]) and np.array_equal(a["minus"], b["minus"])


MSA_ORACLE_MLE = 10       # alignments per tree checked against the oracle's MLE fit (each costs seconds of CPU on 128 leaves)
MSA_ORACLE_OMEGA = 6      # and against its OMEGA fit (several seconds each)


def reachable_fit(om, pep):
    """What the reference's MLE fit of one model can return (fixed_lik.hpp:469-544): its Brent search over the tree scale rho in
    [1e-2, 10] stops once the bracket around the best point is 1 % of it wide, and reports the LAST evaluation, which lies in that
    bracket.  So the reported rho is within 1.02 % of the true maximiser rho*, whichever way tiny differences in P(t) steer the
    trajectory.  Returns (min, max) of lpr and of the ancestral term over that range; rho* is found far more tightly than the
    reference does (a log grid, then a bracketed Brent search to 1e-12)."""
    from scipy.optimize import minimize_scalar

    def f(r):
        om.set_rho(r)
        return -om.lpr_leaves(pep)[0]
    grid = np.geomspace(1e-2, 10.0, 60)
    i = int(np.argmin([f(r) for r in grid]))
    x = minimize_scalar(f, bracket=(grid[i - 1], grid[i], grid[i + 1]), tol=1e-12).x if 0 < i < len(grid) - 1 else grid[i]
    vals = []
    for r in np.linspace(max(1e-2, x * (1 - 0.0102)), min(10.0, x * (1 + 0.0102)), 41):
        om.set_rho(r)
        vals.append(om.lpr_leaves(pep, True)[:2])
    om.set_rho(1.0)
    v = np.array(vals)
    return v[:, 0].min(), v[:, 0].max(), v[:, 1].min(), v[:, 1].max()


@pytest.mark.parametrize("name", ["balanced64", "yule128"])
def test_score_msa_on_generated_trees(tree_dir, monkeypatch, name):
    """pcsf_score_msa (FIXED, MLE, OMEGA) on 40 random alignments of 30 to 200 codons, against the oracle at the tolerances of
    test_gpu_score_msa.py; MLE rows whose Brent search forked are held to what the reference's own search can return.  balanced64 always runs k_prune<true> with 4 warps (32-window tiles in the MLE / OMEGA tile plans);
    on yule128 the three warp counts 12, 8 and 4 must give bit-identical scores for each strategy."""
    model = model_of(tree_dir, name)
    rng = np.random.default_rng(64)
    alns = [random_alignment(model.nl, 3 * int(k), seed=500 + i, gap=0.25, conserve=float(c))
            for i, (k, c) in enumerate(zip(rng.integers(30, 201, 40), rng.uniform(0.5, 0.95, 40)))]
    mc = orc.OracleModel(model.tree, model.S_c, model.f_c)
    mnc = orc.OracleModel(model.tree, model.S_nc, model.f_nc)
    warps = (12, 8, 4) if name == "yule128" else (None,)
    res = {}
    for nw in warps:
        dm = capi.DeviceModel(model) if nw is None else _with_env(monkeypatch, model, PCSF_PRUNE_NWARP=nw)
        res[nw] = {s: dm.score_msa(alns, s) for s in (capi.STRATEGY_FIXED, capi.STRATEGY_MLE)}
        res[nw][capi.STRATEGY_OMEGA] = dm.score_msa(alns, capi.STRATEGY_OMEGA, comp_anc=False)
        dm.close()
    base = res[warps[0]]
    for nw in warps[1:]:
        for s, out in res[nw].items():
            for x, y in zip(base[s], out):
                assert x is None or np.array_equal(x, y, equal_nan=True), (nw, s)
    phylo, anc, bls = base[capi.STRATEGY_FIXED]
    for a, p, an, b in zip(alns, phylo, anc, bls):
        rp, ra = orc.run_fixed(mc, mnc, orc.translate(a), True)
        assert abs(float(p) - float(rp)) <= 1e-3 and abs(float(an) - float(ra)) <= 1e-3
        assert np.float32(orc.bls(model.tree, a, per_base=False)[0]) == b
    phylo, anc, bls = base[capi.STRATEGY_MLE]
    assert np.array_equal(bls, base[capi.STRATEGY_FIXED][2])
    tight, forks = 0, []
    db = 10.0 / np.log(10.0)
    for a, p, an in list(zip(alns, phylo, anc))[:MSA_ORACLE_MLE]:
        pep = orc.translate(a)
        rp, ra, info = orc.run_mle(mc, mnc, pep, True)
        if (float(p) - float(rp)) ** 2 <= 0.001 and (float(an) - float(ra)) ** 2 <= 0.001:
            tight += abs(float(p) - float(rp)) <= 1e-3 and abs(float(an) - float(ra)) <= 1e-3
            continue
        # A Brent trajectory that forks on ~1e-13 differences in P(t) (DESIGN.md section 7) ends at another point of the final 1 %
        # bracket.  With 128 leaves and hundreds of codons the likelihood is so sharply peaked in rho that two such endpoints can
        # differ by more than the reference's CI tolerance (either the oracle or the device may land nearer the maximum); the device
        # must then give scores the reference's own search can return.
        c_lo, c_hi, ca_lo, ca_hi = reachable_fit(mc, pep)
        n_lo, n_hi, na_lo, na_hi = reachable_fit(mnc, pep)
        p_rng, a_rng = (db * (c_lo - n_hi), db * (c_hi - n_lo)), (db * (ca_lo - na_hi), db * (ca_hi - na_lo))
        forks.append((a.shape[1], float(p), float(rp), p_rng, float(an), float(ra), a_rng))
        assert p_rng[0] - 1e-3 <= float(p) <= p_rng[1] + 1e-3 and a_rng[0] - 1e-3 <= float(an) <= a_rng[1] + 1e-3, (forks[-1], info)
    print(f"{name}: MLE {tight}/{MSA_ORACLE_MLE} rows within 1e-3 of the oracle; forked rows (columns, device, oracle, reachable "
          f"range; the same for anc): {forks}")
    assert tight >= MSA_ORACLE_MLE // 2
    phylo, _, bls = base[capi.STRATEGY_OMEGA]
    assert np.array_equal(bls, base[capi.STRATEGY_FIXED][2])
    order = np.argsort([a.shape[1] for a in alns])[:MSA_ORACLE_OMEGA]
    d = [abs(float(phylo[i]) - float(orc.run_omega(model.tree, orc.translate(alns[i]))[0])) for i in order]
    print(f"{name}: OMEGA |d| vs oracle on the {MSA_ORACLE_OMEGA} shortest alignments: {d}")
    assert max(d) ** 2 <= 0.1
    # OMEGA reports the last evaluation of six Brent fits that stop at 1 % brackets.  On balanced64 some rows still agree to 1e-3;
    # on yule128 the likelihood is so sharply peaked that no row does (measured on one B200: 0.0037 to 0.12 decibans over the six
    # rows), as the MLE forks above show for the simpler fit
    if name == "balanced64":
        assert min(d) <= 1e-3
