"""Writes tests/golden/msa-kernels/refs.npz: high-precision references for the score-msa kernels (tests/test_gpu_msa_kernels.py).

Every case is a rate matrix Q, restated in mpmath (mp.dps = 40) from the semantics the kernels implement, and its exact
spectral data, rounded to float64 only at the end:
  * OMEGA cases: Q(kappa, omega, sigma, F3x4) of pi_expr + comp_q_p14n + comp_q_scale (omega.hpp:8-103, quoted in
    phylocsfpp_b200/csrc/omega.cuh; the oracle's omega_pi_sc / omega_set_q state the same), over a grid of kappa,
    (omega, sigma) and three kinds of F3x4 ratios (uniform, random, one base dominating);
  * ECM cases: Q of build_q (instance.hpp:648-685, phylocsfpp_b200/csrc/model_prep.hpp) for the 58mammals coding and
    non-coding models.
Per case: Q, lam and U of mp.eigsy(D^1/2 Q D^-1/2) (D = diag of the equilibrium weights w), sqrt(w), and the stationary
distribution from solving pi Q = 0, sum(pi) = 1 directly.  P(t) = D^-1/2 U diag(exp(lam t)) U^T D^1/2.

mpmath takes seconds per 64 x 64 eigensystem, so the tests read this file instead of recomputing; one test regenerates a
single case and compares.  Run from the repository root:  python tests/golden/make_msa_kernel_refs.py
"""
from __future__ import annotations

import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
OUT = os.path.join(HERE, "msa-kernels", "refs.npz")
DPS = 40

KAPPAS = (1.0, 1.0 + 1e-9, 2.5, 10.0)
OMEGA_SIGMA = ((1.0, 1.0), (0.2, 0.01))
TCAG = "FFLLSSSSYY**CC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG"


def f3x4_kinds():
    """F3x4 ratios (count + 1) / (count_T + 1) per codon position, as k_omega_counts writes them: [A, C, G] x 3."""
    rng = np.random.default_rng(2024)
    uniform = np.ones(9)
    rand = (1.0 + rng.integers(0, 400, 9)) / (1.0 + rng.integers(0, 400, 3)).repeat(3)
    # one base dominating at every position: T (ratios 1/3001), A (3001 / 1), G (3000 / 1 with C absent)
    skew = np.array([1 / 3001, 1 / 3001, 1 / 3001, 3001.0, 1.0, 1.0, 1.0, 1 / 3001, 3000.0])
    return {"uniform": uniform, "random": rand, "skew": skew}


def case_list():
    """[(kind, params)]: kind 'omega' with (kappa, omega, sigma, f3x4[9]) or 'ecm' with (model name, 0 coding / 1 non-coding)."""
    out = []
    for fname, f in f3x4_kinds().items():
        for om, sg in OMEGA_SIGMA:
            for k in KAPPAS:
                out.append(("omega", (k, om, sg, f), fname))
    out.append(("ecm", ("58mammals", 0), "58mammals coding"))
    out.append(("ecm", ("58mammals", 1), "58mammals non-coding"))
    return out


def _aa(c):
    to_tcag = (2, 1, 3, 0)
    return TCAG[16 * to_tcag[c >> 4] + 4 * to_tcag[(c >> 2) & 3] + to_tcag[c & 3]]


def omega_q(kappa, omega, sigma, f):
    """pi_expr (omega.hpp:8-36), comp_q_p14n (:38-95), comp_q_scale (:97-103) in mpmath.  Returns (Q, w)."""
    import mpmath as mp
    kappa, omega, sigma = mp.mpf(kappa), mp.mpf(omega), mp.mpf(sigma)
    f = [mp.mpf(x) for x in f]

    def pi_sc(c):
        i = (c >> 4, (c >> 2) & 3, c & 3)
        r = mp.mpf(1)
        for p in range(3):
            r *= (mp.mpf(1) if i[p] == 3 else f[3 * p + i[p]]) / (1 + f[3 * p] + f[3 * p + 1] + f[3 * p + 2])
        return r

    denom = 1 - (1 - sigma) * (pi_sc(48) + pi_sc(50) + pi_sc(56))          # TAA, TAG, TGA
    w = [pi_sc(c) / denom for c in range(64)]
    Q = mp.zeros(64, 64)
    for i in range(64):
        for j in range(64):
            a = (i >> 4, (i >> 2) & 3, i & 3)
            b = (j >> 4, (j >> 2) & 3, j & 3)
            diff = [p for p in range(3) if a[p] != b[p]]
            if len(diff) != 1:
                continue
            p = diff[0]
            val = kappa if a[p] + b[p] in (2, 4) else mp.mpf(1)          # A<->G, C<->T
            ia, ja = _aa(i), _aa(j)
            if ia != "*" and ja != "*" and ia != ja:
                val *= omega
            Q[i, j] = val * w[j]
    for i in range(64):
        Q[i, i] = -mp.fsum(Q[i, j] for j in range(64) if j != i)
    scale = -mp.fsum(w[i] * Q[i, i] for i in range(64))
    return Q / scale, w


def ecm_q(S, f):
    """build_q (instance.hpp:648-685): Q_ij = S_ij f_j, rows summing to zero, scaled to one expected substitution."""
    import mpmath as mp
    w = [mp.mpf(float(x)) for x in f]
    Q = mp.zeros(64, 64)
    for i in range(64):
        for j in range(64):
            if j != i:
                Q[i, j] = mp.mpf(float(S[i, j])) * w[j]
        Q[i, i] = -mp.fsum(Q[i, j] for j in range(64) if j != i)
    scale = -mp.fsum(w[i] * Q[i, i] for i in range(64))
    return Q / scale, w


def stationary(Q):
    """pi Q = 0 with sum(pi) = 1, solved directly (the last balance equation replaced by the normalisation)."""
    import mpmath as mp
    A = Q.T.copy()
    for j in range(64):
        A[63, j] = mp.mpf(1)
    rhs = mp.zeros(64, 1)
    rhs[63] = mp.mpf(1)
    return mp.lu_solve(A, rhs)


def compute_case(kind, params):
    """The float64-rounded reference of one case: dict(Q, lam, U, sq, pistat)."""
    import mpmath as mp
    mp.mp.dps = DPS
    if kind == "omega":
        Q, w = omega_q(*params)
    else:
        sys.path.insert(0, ROOT)
        from phylocsfpp_b200.models import load_model
        m = load_model(params[0])
        S, f = (m.S_c, m.f_c) if params[1] == 0 else (m.S_nc, m.f_nc)
        Q, w = ecm_q(S, f)
    sq = [mp.sqrt(x) for x in w]
    A = mp.zeros(64, 64)
    for i in range(64):
        for j in range(64):
            A[i, j] = sq[i] * Q[i, j] / sq[j]
    for i in range(64):
        for j in range(i + 1, 64):
            A[i, j] = A[j, i] = (A[i, j] + A[j, i]) / 2
    lam, U = mp.eigsy(A)
    ps = stationary(Q)
    f64 = lambda M, r, c: np.array([[float(M[i, j]) for j in range(c)] for i in range(r)])
    return dict(Q=f64(Q, 64, 64), lam=np.array([float(lam[i]) for i in range(64)]), U=f64(U, 64, 64),
                sq=np.array([float(x) for x in sq]), pistat=np.array([float(ps[i]) for i in range(64)]))


def p_of_t(ref, t):
    """P(t) = D^-1/2 U diag(exp(lam t)) U^T D^1/2 in x87 extended precision (about 1e-18 per entry from float64-rounded factors)."""
    LD = np.longdouble
    U, lam, sq = ref["U"].astype(LD), ref["lam"].astype(LD), ref["sq"].astype(LD)
    M = (U * np.exp(lam * LD(t))[None, :]) @ U.T
    return M / sq[:, None] * sq[None, :]


def validate_with_expm(ref, kind, params, t):
    """The eigen route against mpmath's own expm(Q t) (an independent algorithm) at one t: returns max |difference|."""
    import mpmath as mp
    mp.mp.dps = DPS
    Q = omega_q(*params)[0] if kind == "omega" else None
    if Q is None:
        sys.path.insert(0, ROOT)
        from phylocsfpp_b200.models import load_model
        m = load_model(params[0])
        Q = ecm_q(*((m.S_c, m.f_c) if params[1] == 0 else (m.S_nc, m.f_nc)))[0]
    E = mp.expm(Q * mp.mpf(t))
    Pe = np.array([[float(E[i, j]) for j in range(64)] for i in range(64)])
    return float(np.abs(p_of_t(ref, t).astype(np.float64) - Pe).max())


def _work(i):
    kind, params, _ = case_list()[i]
    return compute_case(kind, params)


def main():
    from multiprocessing import Pool
    cases = case_list()
    with Pool(min(8, os.cpu_count() or 1)) as pool:
        refs = pool.map(_work, range(len(cases)))
    # the eigen route against an independent expm, on a random-F3x4 OMEGA case and on an ECM
    for i in (next(i for i, c in enumerate(cases) if c[2] == "random"), len(cases) - 1):
        d = validate_with_expm(refs[i], cases[i][0], cases[i][1], 0.3)
        print(f"case {i} ({cases[i][2]}): eigen route vs mp.expm at t = 0.3: max |d| = {d:.2e}")
        assert d < 1e-15, d
    omega = [c for c in cases if c[0] == "omega"]
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    np.savez_compressed(
        OUT,
        omega_params=np.array([[p[0], p[1], p[2]] for _, p, _ in omega]),
        omega_f3x4=np.array([p[3] for _, p, _ in omega]),
        omega_kind=np.array([n for _, _, n in omega]),
        **{k: np.stack([r[k] for r in refs]) for k in ("Q", "lam", "U", "sq", "pistat")})
    print(f"wrote {OUT}: {len(cases)} cases ({len(omega)} OMEGA, {len(cases) - len(omega)} ECM)")


if __name__ == "__main__":
    main()
