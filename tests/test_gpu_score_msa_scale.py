"""pcsf_score_msa at batch scale: more alignments than fitting slots, so that slots are recycled (a slot that finishes one
alignment pulls the next from the queue), the tile plan runs with more than 1024 slots, and FIXED sees a config-5-sized batch.

Every alignment's tiles start at its own window 0 and its sums run sequentially in codon order; no reduction crosses
alignments.  So an alignment's outputs must not depend on the batch around it: batches are compared bit for bit (NaN-aware)
with the same alignments in sub-batches, in reverse order, and in a second call on the same handle.  Samples are compared with
the oracle.  Measured times are printed (-s).
"""
import time

import numpy as np
import pytest

from oracle import oracle as orc
from phylocsfpp_b200 import capi, orf
from phylocsfpp_b200.models import load_model
from tests.util import random_alignment

pytestmark = pytest.mark.gpu

SPECIES12 = "Human,Chimp,Mouse,Dog,Cow,Horse,Elephant,Armadillo,Rat,Rabbit,Cat,Megabat"
BUDGET = 6 << 30          # the scratch budget of mle_run / omega_run
HIGH = (0.6, 0.75, 0.85, 0.9, 0.95, 0.7, 0.8)          # no random restarts: keeps the 100-species oracle fits short


def _lengths(n, lo, hi, seed, tiny=()):
    rng = np.random.default_rng(seed)
    lens = np.exp(rng.uniform(np.log(lo), np.log(hi), n)).astype(np.int64)
    lens[:len(tiny)] = tiny
    return lens


def _batch(nl, lens, seed, conserve=(0.3, 0.6, 0.75, 0.85, 0.9, 0.95, 0.7, 0.8, 0.92, 0.65, 0.88, 0.97, 0.8, 0.9, 0.6, 0.85, 0.95,
                                     0.75, 0.9, 0.82)):
    """Alignment i is cut from block i % len(conserve), a random alignment of that conservation and a gap rate of 0 .. 0.4."""
    nb = len(conserve)
    owner = np.arange(len(lens)) % nb
    blocks = [random_alignment(nl, int(lens[owner == b].sum()), seed=seed + b, gap=0.4 * b / nb, conserve=c) for b, c in enumerate(conserve)]
    pos = np.zeros(nb, np.int64)
    out = []
    for i, L in enumerate(lens):
        b = owner[i]
        out.append(np.ascontiguousarray(blocks[b][:, pos[b]:pos[b] + L]))
        pos[b] += L
    return out


def _same(x, y):
    """Bit identity, NaN-aware (the device writes one NaN pattern)."""
    if x is None or y is None:
        return x is None and y is None
    return np.array_equal(np.asarray(x, np.float32).view(np.uint32), np.asarray(y, np.float32).view(np.uint32))


def _score(dm, alns, strategy, comp_anc=True):
    out = dm.score_msa(alns, strategy, comp_anc=comp_anc)
    st = dm.score_msa_stats() if strategy == capi.STRATEGY_MLE else None
    return out, st


def _in_parts(dm, alns, strategy, part, comp_anc=True):
    res, evals = [[], [], []], 0
    for i in range(0, len(alns), part):
        (p, a, b), st = _score(dm, alns[i:i + part], strategy, comp_anc)
        for r, x in zip(res, (p, a, b)):
            r.append(x)
        evals += st["evaluations"] if st else 0
    return tuple(np.concatenate(r) for r in res), evals


def _assert_same(x, y, what):
    for k, (u, v) in enumerate(zip(x, y)):
        if not _same(u, v):
            bad = np.flatnonzero(np.asarray(u, np.float32).view(np.uint32) != np.asarray(v, np.float32).view(np.uint32))
            raise AssertionError(f"{what}: output {('phylo', 'anc', 'bls')[k]} differs at {bad[:10].tolist()} ({len(bad)} rows)")


def _recycling_checks(dm, alns, strategy, part, label, comp_anc=True):
    """(a) = sub-batches of <= part (MLE: with the same total evaluations), (b) = reversed batch, (c) = a second call."""
    t0 = time.perf_counter()
    full, st = _score(dm, alns, strategy, comp_anc)
    t1 = time.perf_counter()
    parts, ev = _in_parts(dm, alns, strategy, part, comp_anc)
    _assert_same(full, parts, f"{label}: batch vs sub-batches of {part}")
    if st:
        assert ev == st["evaluations"], (ev, st["evaluations"])
    rev, _ = _score(dm, alns[::-1], strategy, comp_anc)
    _assert_same(full, tuple(None if r is None else r[::-1] for r in rev), f"{label}: reversed batch")
    again, st2 = _score(dm, alns, strategy, comp_anc)
    _assert_same(full, again, f"{label}: second call")
    if st:
        assert st2["evaluations"] == st["evaluations"]
    print(f"{label}: {len(alns)} alignments, one call {t1 - t0:.2f} s, all checks {time.perf_counter() - t0:.2f} s"
          + (f", {st['slots']} slots, {st['evaluations']} evaluations, {st['rounds']} rounds" if st else ""))
    return full, st


def _restarts(mc, mnc, pep):
    """fit_find_init draws random restarts when the likelihood at rho = 1 does not beat both ends of [0.01, 10]."""
    out = False
    for om in (mc, mnc):
        f = {}
        for r in (0.01, 10.0, 1.0):
            om.set_rho(r)
            f[r] = om.lpr_leaves(pep)[0]
        om.set_rho(1.0)
        out |= f[1.0] <= f[0.01] or f[1.0] <= f[10.0]
    return out


def _fit_evals(om, pep, gen, noise=None, amp=0.0, lo=1e-2, hi=10.0, init=1.0):
    """Likelihood evaluations of one max_lik_lpr_leaves (fit_find_init + GSL Brent, as oracle/phylocsf_oracle.c max_lik_core),
    with every lpr optionally perturbed by amp * |lpr| * N(0, 1): the evaluation counts the reference's own algorithm reaches
    when lpr carries rounding differences of that size (another summation order, another eigensolver)."""
    n = [0]

    def F(x):          # minimizer_lpr_leaves: -lpr
        n[0] += 1
        om.set_rho(x)
        lpr = om.lpr_leaves(pep)[0]
        return -(lpr + (amp * abs(lpr) * noise.standard_normal() if amp else 0.0))

    flo, fhi, x = -F(lo), -F(hi), init
    fx, tries = -F(init), 0
    while tries < 250 and (fx <= flo or fx <= fhi):
        x = float(np.exp(np.log(lo) + gen.uniform(np.log(hi) - np.log(lo))))
        fx, tries = -F(x), tries + 1
    if tries == 250:
        x = lo if flo > fhi else hi
    F(x)
    if lo < x < hi:
        z, xl, xu = x, lo, hi
        F(xl), F(xu)
        fz = F(z)
        g = 0.3819660
        v = w = xl + g * (xu - xl)
        d = e = 0.0
        fv = fw = F(v)
        for _ in range(250):
            dd, ee = e, d
            tol = 1.4901161193847656e-08 * abs(z)
            mid, wl, wu = 0.5 * (xl + xu), z - xl, xu - z
            p = q = r = 0.0
            if abs(ee) > tol:
                r, q = (z - w) * (fz - fv), (z - v) * (fz - fw)
                p, q = (z - v) * q - (z - w) * r, 2 * (q - r)
                p, q = (-p, q) if q > 0 else (p, -q)
                r, ee = ee, dd
            if abs(p) < abs(0.5 * q * r) and p < q * wl and p < q * wu:
                dd = p / q
                u = z + dd
                if (u - xl) < 2 * tol or (xu - u) < 2 * tol:
                    dd = tol if z < mid else -tol
            else:
                ee = xu - z if z < mid else -(z - xl)
                dd = g * ee
            u = z + dd if abs(dd) >= tol else z + (tol if dd > 0 else -tol)
            e, d = ee, dd
            fu = F(u)
            if fu <= fz:
                xl, xu = (xl, z) if u < z else (z, xu)
                v, fv, w, fw, z, fz = w, fw, z, fz, u, fu
            else:
                xl, xu = (u, xu) if u < z else (xl, u)
                if fu <= fw or w == z:
                    v, fv, w, fw = w, fw, u, fu
                elif fu <= fv or v == z or v == w:
                    v, fv = u, fu
            if (xu - xl) / z <= 0.01:
                break
    om.set_rho(1.0)
    return n[0]


def _forked_counts(mc, mnc, pep, info, amp=1e-14, trials=24):
    """Total evaluation counts (coding + non-coding, one mt19937(42) stream) of the reference's fit under lpr perturbations of
    relative size amp.  The restatement is first held to the oracle's own counts without perturbation."""
    gen = orc.MT19937(42)
    assert (_fit_evals(mc, pep, gen), _fit_evals(mnc, pep, gen)) == (info["evals_c"], info["evals_nc"])
    out = set()
    for s in range(trials):
        noise, gen = np.random.default_rng(s), orc.MT19937(42)
        out.add(_fit_evals(mc, pep, gen, noise, amp) + _fit_evals(mnc, pep, gen, noise, amp))
    return out


def _mle_vs_oracle(model, dm, alns, full, idx, min_tight, label, max_forks=2):
    """Every sampled row within the reference's CI tolerance (squared error <= 1e-3) of the oracle, at least min_tight within
    1e-3; for each tight row, the alignment scored alone gives the same bits, and the same number of likelihood evaluations as
    the oracle's Brent trajectory (evals_c + evals_nc).  A tight row may differ in that number only where the trajectory is a
    knife edge: the reference's own algorithm must reach the device's count when lpr is perturbed at the 1e-14 level (e.g. a
    Brent parabola on a nearly flat likelihood); at most max_forks such rows."""
    mc = orc.OracleModel(model.tree, model.S_c, model.f_c)
    mnc = orc.OracleModel(model.tree, model.S_nc, model.f_nc)
    phylo, anc, _ = full
    tight, restarts, forks = 0, 0, []
    t0 = time.perf_counter()
    for i in idx:
        pep = orc.translate(alns[i])
        rp, ra, info = orc.run_mle(mc, mnc, pep, True)
        restarts += _restarts(mc, mnc, pep)
        if np.isnan(rp):
            assert np.isnan(phylo[i]) and np.isnan(anc[i]), (i, info)
            continue
        assert (float(phylo[i]) - float(rp)) ** 2 <= 1e-3 and (float(anc[i]) - float(ra)) ** 2 <= 1e-3, (i, phylo[i], rp, anc[i], ra, info)
        if abs(float(phylo[i]) - float(rp)) <= 1e-3 and abs(float(anc[i]) - float(ra)) <= 1e-3:
            tight += 1
            one = dm.score_msa([alns[i]], capi.STRATEGY_MLE)
            assert _same(one[0], phylo[i:i + 1]) and _same(one[1], anc[i:i + 1]), (i, one, phylo[i], anc[i])
            ev = dm.score_msa_stats()["evaluations"]
            if ev != info["evals_c"] + info["evals_nc"]:
                reach = _forked_counts(mc, mnc, pep, info)
                assert ev in reach, (i, ev, info, sorted(reach))
                forks.append((i, ev, info["evals_c"] + info["evals_nc"]))
    print(f"{label}: {tight}/{len(idx)} sampled rows within 1e-3 of the oracle, {restarts} of them with random restarts, "
          f"Brent forks (row, device evaluations, oracle evaluations): {forks} ({time.perf_counter() - t0:.1f} s)")
    assert tight >= min_tight and len(forks) <= max_forks
    return restarts


def test_mle_config5_shape_recycles_slots():
    """MLE with the 12-species reduction of 29mammals, 12 000 alignments of 30..600 columns (plus lengths 0, 1, 2, 3, 5) over
    8192 slots."""
    model = load_model("29mammals", SPECIES12)
    n = 12000
    alns = _batch(model.nl, _lengths(n, 30, 600, 1, tiny=(0, 1, 2, 3, 5)), 100)
    dm = capi.DeviceModel(model)
    full, st = _recycling_checks(dm, alns, capi.STRATEGY_MLE, 1000, "MLE 29mammals/12")
    assert st["slots"] == 8192 < n
    # the tiny ones, the last one dequeued, a few of low conservation (block 0) and a random rest
    rng = np.random.default_rng(3)
    idx = sorted(set([0, 1, 2, 3, 4, n - 1] + list(range(20, 20 * 6, 20)) + rng.choice(n, 40, replace=False).tolist()))
    restarts = _mle_vs_oracle(model, dm, alns, full, idx, len(idx) - 2, "MLE 29mammals/12")
    assert restarts >= 3          # state a slot's previous occupant left behind only matters for such fits
    dm.close()


def test_mle_budget_bound_recycles_slots():
    """MLE with 100vertebrates: the 6 GiB scratch budget caps the slots well below the 2000 alignments."""
    model = load_model("100vertebrates")
    n = 2000
    alns = _batch(model.nl, _lengths(n, 30, 90, 2), 200, conserve=HIGH)
    dm = capi.DeviceModel(model)
    full, st = _recycling_checks(dm, alns, capi.STRATEGY_MLE, 700, "MLE 100vertebrates")
    stride = (model.nl - 2) * 4096 + model.nl * 65 * 64
    assert st["slots"] == BUDGET // (stride * 8) < n
    idx = sorted(set([0, n - 1] + np.random.default_rng(4).choice(n, 6, replace=False).tolist()))
    _mle_vs_oracle(model, dm, alns, full, idx, len(idx) - 1, "MLE 100vertebrates")
    dm.close()


def test_omega_recycles_slots():
    """OMEGA with 100vertebrates, 2000 alignments of 30..60 columns (more than the budget's slots): batch = sub-batches of 500,
    reversed, second call; anc is all NaN; BLS equals FIXED's; two short alignments against the oracle."""
    model = load_model("100vertebrates")
    n = 2000
    stride = (model.nl - 2) * 4096 + model.nl * 65 * 64 + 64 + 2 * 4096
    assert BUDGET // (stride * 8) < n
    alns = _batch(model.nl, _lengths(n, 30, 60, 5), 500, conserve=HIGH)
    dm = capi.DeviceModel(model)
    full, _ = _recycling_checks(dm, alns, capi.STRATEGY_OMEGA, 500, "OMEGA 100vertebrates")
    phylo, anc, bls = full
    assert np.isnan(anc).all()
    assert np.isfinite(phylo).sum() > n // 2
    _, _, bls_fixed = dm.score_msa(alns, capi.STRATEGY_FIXED)
    assert _same(bls, bls_fixed)
    d = []
    for i in (0, n - 1):
        s, info = orc.run_omega(model.tree, orc.translate(alns[i]))
        d.append(abs(float(phylo[i]) - float(s)))
        print(f"OMEGA row {i}: device {float(phylo[i])}, oracle {float(s)}")
    assert max(d) ** 2 <= 0.1 and min(d) <= 1e-3
    dm.close()


def test_fixed_config5_size():
    """FIXED on 65 536 alignments in one call (one dedup domain) = sub-batches of 4096 (sixteen domains) bit for bit; 500 samples
    against the oracle."""
    model = load_model("29mammals", SPECIES12)
    n = 65536
    alns = _batch(model.nl, _lengths(n, 30, 600, 6, tiny=(0, 1, 2, 3, 5)), 600)
    dm = capi.DeviceModel(model)
    t0 = time.perf_counter()
    full = dm.score_msa(alns, capi.STRATEGY_FIXED)
    t1 = time.perf_counter()
    parts, _ = _in_parts(dm, alns, capi.STRATEGY_FIXED, 4096)
    _assert_same(full, parts, "FIXED: batch vs sub-batches of 4096")
    print(f"FIXED 29mammals/12: {n} alignments, one call {t1 - t0:.2f} s, with sub-batches {time.perf_counter() - t0:.2f} s")
    phylo, anc, bls = full
    mc = orc.OracleModel(model.tree, model.S_c, model.f_c)
    mnc = orc.OracleModel(model.tree, model.S_nc, model.f_nc)
    idx = sorted(set([0, 1, 2, 3, 4, n - 1] + np.random.default_rng(7).choice(n, 494, replace=False).tolist()))
    for i in idx:
        a = alns[i]
        rp, ra = orc.run_fixed(mc, mnc, orc.translate(a), True)
        assert abs(float(phylo[i]) - float(rp)) <= 1e-3 and abs(float(anc[i]) - float(ra)) <= 1e-3, (i, phylo[i], rp, anc[i], ra)
        if a.shape[1] > 0:
            assert np.float32(orc.bls(model.tree, a, per_base=False)[0]) == bls[i], i
    dm.close()


def _regions(dm, alns):
    return dm.score_regions(alns, np.arange(len(alns)) % dm.nl, capi.STRATEGY_MLE, 6, orf.ATGSTOP, 25)


def _same_records(x, y):
    return (len(x) == len(y) and all(np.array_equal(x[k], y[k]) for k in ("aln", "strand", "frame", "col_begin", "col_end", "codons"))
            and all(_same(x[k], y[k]) for k in ("phylo", "anc", "bls")))


def _last_records(dm, n):
    out = np.zeros(n, capi.REGION_DTYPE)
    capi._check(capi.load().pcsf_score_regions_get(dm.h, out.ctypes.data if n else None, n))
    return out


def test_handle_reuse_small_large_small():
    """One handle alternates score_msa and six-frame ATG-to-stop score_regions calls (which share the staging and the scratch) on
    a small batch, a large one (the page-locked staging and the scratch reservations grow), then the small one again; each equals
    what a fresh handle computes, and a score_msa call leaves the records of the last score_regions call in place."""
    model = load_model("29mammals", SPECIES12)
    small = _batch(model.nl, _lengths(40, 30, 300, 8, tiny=(0, 4)), 800)
    large = _batch(model.nl, _lengths(9000, 30, 600, 9), 900)
    calls = [("msa", small), ("regions", large), ("msa", small), ("msa", large), ("regions", small), ("msa", small)]
    dm = capi.DeviceModel(model)
    seq, last = [], None
    for kind, b in calls:
        if kind == "msa":
            seq.append(dm.score_msa(b, capi.STRATEGY_MLE))
            if last is not None:
                assert _same_records(_last_records(dm, len(last)), last)
        else:
            last = _regions(dm, b)
            seq.append(last)
    dm.close()
    for (kind, b), got in zip(calls, seq):
        fresh = capi.DeviceModel(model)
        if kind == "msa":
            _assert_same(got, fresh.score_msa(b, capi.STRATEGY_MLE), f"reused handle, score_msa, batch of {len(b)}")
        else:
            assert len(got) > 0 and _same_records(got, _regions(fresh, b)), f"reused handle, score_regions, batch of {len(b)}"
        fresh.close()
