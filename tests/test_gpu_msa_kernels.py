"""The batched kernels of score-msa (k_omega_eig, k_mle_expm, k_mle_plan, k_omega_counts) one at a time, against
high-precision references.

tests/kernel_harness.cu wraps each kernel in a C entry point (compiled here with __graft_entry__.NVCC_FLAGS, loaded with
ctypes).  The references are mpmath restatements of the same operations (tests/golden/make_msa_kernel_refs.py, stored in
tests/golden/msa-kernels/refs.npz), exact Python restatements (tile plan), or numpy (F3x4 counts).

Tolerances.  A reversible Q is diagonalised through its symmetric form A = D^1/2 Q D^-1/2, so S = D^-1/2 U and
(S f(lam) S^-1)_ij = sqrt(w_j / w_i) (U f(lam) U^T)_ij: an error of eps in U reaches Q and P(t) amplified by sqrt(w_j / w_i),
up to 1e7 for the skewed F3x4 cases (w spans 1e-14 .. 1).  Entry (i, j) of Q (relative to max|lam|) and of P(t) is
therefore held to TOL * max(1, sqrt(w_j / w_i)), TOL = 1e-12; eigenvalues to TOL * max|lam|, S^-1 S to TOL, the prior to TOL.
The measured maxima are printed (-s).  On one B200 (1000 W power limit): k_omega_eig over the 24 cases lam 7.4e-14, Q 8.5e-14,
S^-1 S 8.7e-14, prior 8.9e-16, P(t) 5.6e-14; k_mle_expm 1.7e-14 (ECM route) and 4.1e-14 (OMEGA route) against the float32-rounded
t, 1.6e-8 and 1.7e-8 against the unrounded t.
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import __graft_entry__ as G

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HARNESS = os.path.join(ROOT, "tests", "kernel_harness.cu")
REFS = os.path.join(ROOT, "tests", "golden", "msa-kernels", "refs.npz")
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import make_msa_kernel_refs as mkr  # noqa: E402

TOL = 1e-12
EIG_STRIDE = 64 + 2 * 4096
TIMES = (1e-4, 0.01, 0.3, 3.0, 30.0)
EXPORTS = ("h_omega_eig", "h_mle_expm", "h_mle_plan", "h_omega_counts")


@pytest.fixture(scope="module")
def harness_so(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("harness") / "kernel_harness.so")
    subprocess.check_call([G.NVCC] + G.NVCC_FLAGS + ["-o", out, HARNESS])
    return out


@pytest.fixture(scope="module")
def H(harness_so):
    L = C.CDLL(harness_so)
    p = C.c_void_p
    L.h_omega_eig.argtypes = [C.c_int, p, p, p, C.c_int, p, p]
    L.h_mle_expm.argtypes = [C.c_int, p, p, p, p, C.c_int, C.c_int, p, p, p, p, C.c_int, p, p, p, p]
    L.h_mle_plan.argtypes = [C.c_int, p, p, p, p, p, C.c_int, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_int, p, p]
    L.h_omega_counts.argtypes = [C.c_int, p, C.c_int64, p, C.c_int64, C.c_int, p, p, p]
    assert L.h_eig_stride() == EIG_STRIDE
    return L


@pytest.fixture(scope="module")
def refs():
    return dict(np.load(REFS))


def _p(a):
    return None if a is None else a.ctypes.data


def test_harness_compiles(harness_so):
    """Runs without a GPU: a change of a kernel's signature or of the structs it reads breaks here first."""
    L = C.CDLL(harness_so)
    for name in EXPORTS:
        assert hasattr(L, name), name


def test_reference_regenerates():
    """One OMEGA case (random F3x4, kappa 2.5) recomputed from scratch in mpmath equals what refs.npz stores, and its eigen-route
    P(t) equals mpmath's independent expm(Q t)."""
    r = np.load(REFS)
    cases = mkr.case_list()
    i = next(k for k, c in enumerate(cases) if c[2] == "random" and c[1][0] == 2.5 and c[1][1] == 1.0)
    kind, params, _ = cases[i]
    assert np.array_equal(r["omega_params"][i], params[:3]) and np.array_equal(r["omega_f3x4"][i], params[3])
    got = mkr.compute_case(kind, params)
    for k in ("Q", "sq", "pistat"):
        assert np.array_equal(got[k], r[k][i]), k
    assert np.abs(got["lam"] - r["lam"][i]).max() <= 1e-15
    assert np.abs(got["U"] - r["U"][i]).max() <= 1e-15
    d = mkr.validate_with_expm(got, kind, params, 3.0)
    assert d <= 1e-15, d


# ---------------------------------------------------------------------------------------------------------------------------
def _weights(ref_sq):
    w = ref_sq.astype(np.float64) ** 2
    return np.maximum(1.0, np.sqrt(w[None, :] / w[:, None]))


def _run_eig(H, alns, kso, f3x4):
    n = len(alns)
    eig = np.full((n, EIG_STRIDE), np.nan)
    pi = np.full((n, 64), np.nan)
    alns = np.ascontiguousarray(alns, np.int32)          # held by a name until the call returns
    kso = np.ascontiguousarray(kso, np.float64)
    f3x4 = np.ascontiguousarray(f3x4, np.float64)
    rc = H.h_omega_eig(n, _p(alns), _p(kso), _p(f3x4), len(f3x4), _p(eig), _p(pi))
    assert rc == 0, rc
    return eig, pi


def _split(e):
    return e[:64], e[64:64 + 4096].reshape(64, 64), e[64 + 4096:].reshape(64, 64)


@pytest.mark.gpu
def test_omega_eig_vs_mpmath(H, refs):
    """k_omega_eig over kappa {1, 1 + 1e-9, 2.5, 10} x (omega, sigma) {(1, 1), (0.2, 0.01)} x F3x4 {uniform (the 12-fold
    degenerate spectrum), random, one base dominating}: eigenvalues, S diag(lam) S^-1 = Q, S^-1 S = I, a single zero eigenvalue,
    the prior = the stationary distribution, and S diag(exp(lam t)) S^-1 = P(t) for t in 1e-4 .. 30."""
    kso, f3 = refs["omega_params"], refs["omega_f3x4"]
    n = len(kso)
    eig, pi = _run_eig(H, np.arange(n), kso, f3)
    LD = np.longdouble
    worst = dict(lam=0.0, Q=0.0, inv=0.0, pi=0.0, P=0.0)
    for i in range(n):
        lam, S, Si = _split(eig[i])
        ref = {k: refs[k][i] for k in ("Q", "lam", "U", "sq", "pistat")}
        scale = np.abs(ref["lam"]).max()
        wt = _weights(ref["sq"])
        dl = np.abs(np.sort(lam) - np.sort(ref["lam"])).max() / scale
        Qd = ((S.astype(LD) * lam.astype(LD)[None, :]) @ Si.astype(LD)).astype(np.float64)
        dq = (np.abs(Qd - ref["Q"]) / wt).max() / scale
        dinv = np.abs((Si.astype(LD) @ S.astype(LD)).astype(np.float64) - np.eye(64)).max()
        nzero = int((np.abs(lam) < 1e-12 * scale).sum())
        dpi = np.abs(pi[i] - ref["pistat"]).max()
        dp = 0.0
        for t in TIMES:
            Pd = ((S.astype(LD) * np.exp(lam.astype(LD) * LD(t))[None, :]) @ Si.astype(LD)).astype(np.float64)
            dp = max(dp, (np.abs(Pd - mkr.p_of_t(ref, t).astype(np.float64)) / wt).max())
        label = f"case {i} ({refs['omega_kind'][i]}, kappa {kso[i][0]!r}, omega {kso[i][1]}, sigma {kso[i][2]})"
        assert np.abs(np.sort(np.abs(ref["lam"]))[1]) > 1e-10 * scale, label          # the reference has one zero, no near-zero
        assert nzero == 1, (label, nzero)
        assert dl <= TOL and dq <= TOL and dinv <= TOL and dpi <= TOL and dp <= TOL, (label, dl, dq, dinv, dpi, dp)
        for k, v in zip(worst, (dl, dq, dinv, dpi, dp)):
            worst[k] = max(worst[k], v)
    print("k_omega_eig max errors over %d cases: " % n + ", ".join(f"{k} {v:.2e}" for k, v in worst.items()))


@pytest.mark.gpu
def test_omega_eig_batch_position_invariant(H, refs):
    """A slot's eigensystem is the same bits whether it is launched alone or anywhere in a batch with idle slots."""
    kso, f3 = refs["omega_params"], refs["omega_f3x4"]
    n = len(kso)
    alone = [_run_eig(H, [i], kso[i:i + 1], f3) for i in range(n)]
    perm = np.random.default_rng(5).permutation(n)
    alns = []
    for i in perm:
        alns += [i, -1]
    kso_b = np.concatenate([[kso[i], kso[i]] for i in perm])
    eig, pi = _run_eig(H, alns, kso_b, f3)
    for pos, a in enumerate(alns):
        if a < 0:
            assert np.isnan(eig[pos]).all() and np.isnan(pi[pos]).all(), "an idle slot was written"
            continue
        assert np.array_equal(eig[pos], alone[a][0][0]) and np.array_equal(pi[pos], alone[a][1][0]), (pos, a)


# ---------------------------------------------------------------------------------------------------------------------------
_FRAG = np.zeros((4096, 2), np.int64)          # flat fragment index -> (a, b) of P, mle.cuh:367-369
for _ks in range(16):
    for _ntp in range(4):
        for _lane in range(32):
            for _e in range(2):
                _FRAG[((_ks * 4 + _ntp) * 32 + _lane) * 2 + _e] = (8 * (2 * _ntp + _e) + _lane // 4,
                                                                   8 * (_ks // 2) + 2 * (_lane % 4) + _ks % 2)


def test_fragment_order_is_a_permutation():
    """The GEMM tile layout of k_mle_expm (mle.cuh:367-369) names every P entry exactly once."""
    flat = _FRAG[:, 0] * 64 + _FRAG[:, 1]
    assert np.array_equal(np.sort(flat), np.arange(4096))


def _decode_gemm(tile):
    P = np.full((64, 64), np.nan)
    P[_FRAG[:, 0], _FRAG[:, 1]] = tile
    return P


def _fixups(P):
    """PhyloModel_make's row fix-ups (instance.hpp:602-640): negative entries to 0, diagonal = 1 - off-diagonal sum."""
    P = np.where(P < 0, 0.0, P)
    off = P.sum(1) - np.diag(P)
    P[np.diag_indices(64)] = 1.0 - off
    return P


def _edge_to_gemm(tree, seed):
    """Leaf edges -1, inner edges a random bijection onto 0 .. n_gemm-1 (the kernel must follow whatever mapping it is given)."""
    n_br = tree.n - 1
    e2g = np.full(n_br, -1, np.int32)
    inner = np.arange(tree.nl, n_br)
    e2g[inner] = np.random.default_rng(seed).permutation(len(inner))
    return e2g


def _run_expm(H, tree, slots, e2g, eig0=None, eig1=None, eig_slots=None, rho_slots=None):
    n = len(slots)
    n_br, nl, n_gemm = tree.n - 1, tree.nl, int((e2g >= 0).sum())
    stride = n_gemm * 4096 + nl * 65 * 64
    p = np.full((n, stride), np.nan)
    err = np.zeros(n, np.int32)
    # every array handed to the harness is held by a name until the call returns (a temporary's buffer would be freed first)
    aln, pending, model = (np.array([s[k] for s in slots], np.int32) for k in ("aln", "pending", "model"))
    x = np.array([s["x"] for s in slots], np.float64)
    bl = np.ascontiguousarray(tree.branch_len[:n_br], np.float32)
    e2g = np.ascontiguousarray(e2g, np.int32)
    rc = H.h_mle_expm(n, _p(aln), _p(pending), _p(model), _p(x), n_br, nl, _p(bl), _p(eig0), _p(eig1), _p(e2g), n_gemm,
                      _p(eig_slots), _p(rho_slots), _p(p), _p(err))
    assert rc == 0, rc
    return p, err, n_gemm


def _unpack(p_slot, e2g, nl, n_gemm, b):
    """P of branch b as the kernel left it: decoded from its GEMM tile, or from its leaf table (checking the row-sum row)."""
    g = e2g[b]
    if g >= 0:
        return _decode_gemm(p_slot[g * 4096:(g + 1) * 4096]), None
    pt = p_slot[n_gemm * 4096 + b * 65 * 64:n_gemm * 4096 + (b + 1) * 65 * 64].reshape(65, 64)
    return pt[:64].T.copy(), pt[64]


def _eig_blob(lam, SR, SRi):
    return np.concatenate([lam, np.ascontiguousarray(SR).ravel(), np.ascontiguousarray(SRi).ravel()])


def _check_expm_slots(tree, slots, p, e2g, n_gemm, refs_of_slot, wts, label):
    """Every branch of every active slot against the rounded-t reference; returns (max weighted error, max error against the
    unrounded-t reference)."""
    n_br, nl = tree.n - 1, tree.nl
    worst = worst_unrounded = 0.0
    for si, s in enumerate(slots):
        if s["aln"] < 0 or not s["pending"]:
            assert np.isnan(p[si]).all(), f"{label}: slot {si} (idle or not pending) was written"
            continue
        assert not np.isnan(p[si]).any(), f"{label}: slot {si} has NaN entries (unwritten or NaN computed)"
        ref, wt, rho = refs_of_slot(si)
        for b in range(n_br):
            P, rowsum = _unpack(p[si], e2g, nl, n_gemm, b)
            if rowsum is not None:
                assert np.abs(rowsum - P.sum(1)).max() <= 1e-15 and np.abs(rowsum - 1.0).max() <= TOL, (label, si, b)
            t = float(np.float32(float(tree.branch_len[b]) * rho))          # instantiate_tree (instance.hpp:299-307)
            R = _fixups(mkr.p_of_t(ref, t).astype(np.float64))
            d = (np.abs(P - R) / wt).max()
            assert d <= TOL, (label, si, b, t, d)
            worst = max(worst, d)
            tu = float(tree.branch_len[b]) * rho
            if tu != t:
                worst_unrounded = max(worst_unrounded, (np.abs(P - _fixups(mkr.p_of_t(ref, tu).astype(np.float64))) / wt).max())
    return worst, worst_unrounded


@pytest.mark.gpu
def test_mle_expm_ecm_route(H, refs):
    """k_mle_expm with the 58mammals coding / non-coding eigensystems (OracleModel.eigen()) at rho {0.01, 1, 10}: every P(t_b)
    entry of every branch in both layouts against mpmath at t_b = float32(double(bl_b) rho), idle and non-pending slots untouched,
    and the device provably resolves the float32 rounding of t."""
    from oracle import oracle as orc
    from phylocsfpp_b200.models import load_model
    m = load_model("58mammals")
    tree = m.tree
    eig = []
    for S, f in ((m.S_c, m.f_c), (m.S_nc, m.f_nc)):
        lam, SR, SRi, _ = orc.OracleModel(tree, S, f).eigen()
        eig.append(_eig_blob(lam, SR, SRi))
    slots = [dict(aln=i, pending=1, model=model, x=rho) for i, (model, rho) in enumerate((m_, r_) for m_ in (0, 1) for r_ in (0.01, 1.0, 10.0))]
    slots.insert(2, dict(aln=-1, pending=1, model=0, x=1.0))          # idle
    slots.insert(5, dict(aln=7, pending=0, model=1, x=1.0))           # fitting, but no evaluation requested
    e2g = _edge_to_gemm(tree, 3)
    p, err, n_gemm = _run_expm(H, tree, slots, e2g, eig0=eig[0], eig1=eig[1])
    assert not err.any()
    ecm = [{k: refs[k][24 + w] for k in ("Q", "lam", "U", "sq")} for w in (0, 1)]
    wts = [_weights(r["sq"]) for r in ecm]
    worst, worst_u = _check_expm_slots(tree, slots, p, e2g, n_gemm,
                                       lambda si: (ecm[slots[si]["model"]], wts[slots[si]["model"]], slots[si]["x"]), wts, "ECM")
    print(f"k_mle_expm (ECM route): max weighted |P - P_ref(t_f32)| = {worst:.2e}; against the unrounded t: {worst_u:.2e}")
    assert worst_u > 100 * worst


@pytest.mark.gpu
def test_mle_expm_omega_route(H, refs):
    """k_mle_expm with per-slot eigensystems from k_omega_eig and per-slot tree scales (the OMEGA route)."""
    from phylocsfpp_b200.models import load_model
    tree = load_model("58mammals").tree
    kso, f3 = refs["omega_params"], refs["omega_f3x4"]
    cases = [int(np.flatnonzero((refs["omega_kind"] == "random") & (kso[:, 0] == 2.5) & (kso[:, 1] == 1.0))[0]),
             int(np.flatnonzero((refs["omega_kind"] == "skew") & (kso[:, 0] == 2.5) & (kso[:, 1] == 0.2))[0])]
    eig, _ = _run_eig(H, cases, kso[cases], f3)
    slots, es, rhos, case_of = [], [], [], []
    for ci, c in enumerate(cases):
        for rho in (0.01, 1.0, 10.0):
            slots.append(dict(aln=len(slots), pending=1, model=0, x=0.0))
            es.append(eig[ci]); rhos.append(rho); case_of.append(c)
    for extra in (dict(aln=-1, pending=1), dict(aln=9, pending=0)):
        slots.insert(2, dict(extra, model=0, x=0.0)); es.insert(2, eig[0]); rhos.insert(2, 1.0); case_of.insert(2, cases[0])
    e2g = _edge_to_gemm(tree, 4)
    p, err, n_gemm = _run_expm(H, tree, slots, e2g, eig_slots=np.ascontiguousarray(es), rho_slots=np.array(rhos))
    assert not err.any()
    R = {c: {k: refs[k][c] for k in ("Q", "lam", "U", "sq")} for c in cases}
    W = {c: _weights(R[c]["sq"]) for c in cases}
    worst, worst_u = _check_expm_slots(tree, slots, p, e2g, n_gemm, lambda si: (R[case_of[si]], W[case_of[si]], rhos[si]), W, "OMEGA")
    print(f"k_mle_expm (OMEGA route): max weighted |P - P_ref(t_f32)| = {worst:.2e}; against the unrounded t: {worst_u:.2e}")
    assert worst_u > 100 * worst


@pytest.mark.gpu
def test_mle_expm_flags_exactly_the_failing_slots(H):
    """expm_err is set for exactly the slots whose P(t) has an entry below -1e-6 (PhyloModel_make's check): 12flies with
    branches shortened 1000-fold and one negative exchangeability, whose most negative entry (scipy expm, float64) is about
    -3.4e-7 at rho = 1 and -3.0e-6 at rho = 10."""
    import copy

    import scipy.linalg as sl

    from oracle import oracle as orc
    from phylocsfpp_b200.models import load_model
    m = copy.deepcopy(load_model("12flies"))
    tree = m.tree
    tree.branch_len = (np.asarray(tree.branch_len, np.float64) * 1e-3).astype(np.float32)
    S = m.S_c.copy()
    S[5, 9] = S[9, 5] = -0.02
    f = m.f_c
    Q = S * f[None, :]
    np.fill_diagonal(Q, 0.0)
    Q[np.diag_indices(64)] = -Q.sum(1)
    Q /= -(np.diag(Q) * f).sum()
    bad = {}
    for rho in (1.0, 10.0):
        worst = min(sl.expm(Q * float(np.float32(float(tree.branch_len[b]) * rho))).min() for b in range(tree.n - 1))
        assert not (-2e-6 < worst < -0.5e-6), worst          # clear of the threshold either way
        bad[rho] = worst < -1e-6
    assert bad == {1.0: False, 10.0: True}
    lam, SR, SRi, _ = orc.OracleModel(tree, S, f).eigen()
    e = _eig_blob(lam, SR, SRi)
    rhos = [1.0, 10.0, 10.0, 1.0, 10.0]
    slots = [dict(aln=i, pending=1, model=0, x=r) for i, r in enumerate(rhos)]
    slots[4]["pending"] = 0
    p, err, _ = _run_expm(H, tree, slots, _edge_to_gemm(tree, 5), eig0=e, eig1=e)
    assert err.tolist() == [0, 1, 1, 0, 0], err


# ---------------------------------------------------------------------------------------------------------------------------
def _plan_reference(aln, pending, model, K, win0, tw, stride, leaf_off, with_pi):
    out = []
    for si in range(len(aln)):
        if aln[si] < 0 or not pending[si]:
            continue
        nt = (int(K[si]) + tw - 1) // tw
        for t in range(nt):
            out.append((si * stride, si * stride + leaf_off, int(model[si]), min(int(K[si]) - tw * t, tw),
                        (int(win0[si]) + tw * t) & 0xFFFFFFFF, 0, si * 64 if with_pi else -1))
    return np.array(out, np.int64).reshape(-1, 7)


@pytest.mark.gpu
@pytest.mark.parametrize("tw", [64, 96])
def test_mle_plan_vs_python(H, tw):
    """k_mle_plan's tile descriptors (one block of 1024 threads, runs of ceil(n_slots / 1024) slots per thread) equal a
    sequential restatement exactly, with idle and non-pending slots and K in {0, 1, tw-1, tw, tw+1, 10 tw + 3}."""
    rng = np.random.default_rng(tw)
    stride, leaf_off = 470656, 229376
    pbase, pi_base = 1 << 40, 1 << 41
    for n in (1, 5, 1023, 1024, 1025, 1500, 4097, 8191, 8192):
        aln = np.where(rng.random(n) < 0.15, -1, rng.integers(0, 1 << 20, n)).astype(np.int32)
        pending = (rng.random(n) < 0.85).astype(np.int32)
        model = rng.integers(0, 2, n).astype(np.int32)
        K = rng.choice([0, 1, tw - 1, tw, tw + 1, 10 * tw + 3], n).astype(np.int64)
        if n > 1:
            aln[-1], pending[-1], K[-1] = 3, 1, 10 * tw + 3          # the last slot, and the last of a thread's run, is active
        win0 = np.cumsum(K) - K + rng.integers(0, 1000, n)
        for with_pi in (0, 1):
            ref = _plan_reference(aln, pending, model, K, win0, tw, stride, leaf_off, with_pi)
            max_tiles = len(ref) + 8
            desc = np.full((max_tiles, 7), -7, np.int64)
            nt = np.zeros(1, np.uint32)
            rc = H.h_mle_plan(n, _p(aln), _p(pending), _p(model), _p(K), _p(win0), tw, stride, leaf_off, pbase,
                              pi_base if with_pi else 0, max_tiles, _p(desc), _p(nt))
            assert rc == 0, rc
            assert int(nt[0]) == len(ref), (n, tw, int(nt[0]), len(ref))
            assert np.array_equal(desc[:len(ref)], ref), (n, tw, with_pi)


# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_omega_counts_bit_exact(H):
    """k_omega_counts: F3x4 ratios (1 + c) / (1 + c_T) of the certain codons of all species equal numpy bit for bit, for lengths
    0, 1, 2, not multiples of 3, and K * nl below and above the block's 256 threads."""
    rng = np.random.default_rng(11)
    nl = 13
    lens = np.array([0, 1, 2, 3, 4, 5, 8, 30, 31, 59, 61, 200, 301, 1000, 3001], np.int64)
    K = lens // 3
    starts = np.cumsum(lens + 2) - (lens + 2)
    Ltot = int((lens + 2).sum())
    ld = (Ltot + 15) // 16 * 16
    codes = rng.choice(5, size=(nl, ld), p=[0.3, 0.2, 0.2, 0.15, 0.15]).astype(np.uint8)
    win_start = np.cumsum(K) - K
    win_off = np.concatenate([starts[i] + 3 * np.arange(K[i]) for i in range(len(lens))]).astype(np.uint32)
    f = np.full((len(lens), 9), np.nan)
    rc = H.h_omega_counts(nl, _p(codes), ld, _p(win_off), len(win_off), len(lens), _p(win_start), _p(lens), _p(f))
    assert rc == 0, rc
    assert (K * nl < 256).any() and (K * nl > 256).any()
    for i in range(len(lens)):
        cnt = np.zeros((3, 4), np.int64)
        for k in range(K[i]):
            c = codes[:, starts[i] + 3 * k:starts[i] + 3 * k + 3]
            ok = (c < 4).all(1)
            for pos in range(3):
                cnt[pos] += np.bincount(c[ok, pos], minlength=4)
        ref = np.array([(1.0 + cnt[p, j]) / (1.0 + cnt[p, 3]) for p in range(3) for j in range(3)])
        assert np.array_equal(f[i], ref), (int(lens[i]), f[i], ref)
