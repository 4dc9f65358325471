"""Shared helpers for GPU-vs-oracle parity runs (used by tests/ and tools/explore_parity.py).
Test infrastructure: imports the oracle."""
import importlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle.slod_oracle import CoefficientTable, GlibcRand, SlodOracle, SlodProblem, reference_random_table  # noqa: E402

pkg = importlib.import_module("dealii-slod_b200")
EPS = 2.220446049250313e-16


def make_tables(dim, s, r, kind, seed):
    rs = np.random.default_rng(seed)
    n = (2 ** r) ** dim
    out = []
    for f in range(1 if s == 1 else 2):
        if kind == "uniform100":
            out.append(1.0 + 99.0 * rs.random(n))
        elif kind == "uniform1e4":
            out.append(1.0 + (1e4 - 1.0) * rs.random(n))
        elif kind == "binary1e4":
            out.append(np.where(rs.random(n) < 0.5, 1.0, 1e4))
        elif kind == "const":
            out.append(np.ones(n))
        else:
            raise ValueError(kind)
    return out


def case_id(case):
    """Test id of a case dict; the expected plan is not part of it."""
    return "-".join(f"{k}{v}" for k, v in case.items() if k != "plan")


def check_plan(ctx, want):
    """The kernels slod_create chose (slod_get_plan) include ``want`` ({PLAN_KEYS entry: value})."""
    got = ctx.plan()
    assert {k: got[k] for k in want} == want, got


def build_pair(dim=2, s=1, ref=3, n=2, ell=1, stabilize=True, r=None, kind="uniform100", seed=1234, quirk=False,
               tables=None, plan=None):
    """GPU handle and oracle of one configuration.  ``plan``: the kernel variants the configuration exists to run,
    asserted through slod_get_plan once the coefficients are set."""
    r = min(ref + int(np.log2(n)), 8 if dim == 2 else 6) if r is None else r
    tables = make_tables(dim, s, r, kind, seed) if tables is None else tables
    problem = "diffusion" if s == 1 else "elasticity"
    ctx = pkg.SlodContext(dim=dim, spacedim=s, n_global_refinements=ref, n_subdivisions=n, oversampling=ell,
                          stabilize=stabilize, problem=0 if s == 1 else 1, quirk_presaved=quirk)
    for f, t in enumerate(tables):
        ctx.set_coefficient(f, r, t)
    if plan is not None:
        check_plan(ctx, plan)
    prob = SlodProblem(dim=dim, spacedim=s, n_global_refinements=ref, n_subdivisions=n, oversampling=ell,
                       stabilize=stabilize, problem=problem, quirk_presaved=quirk,
                       coefficients=[CoefficientTable(dim, r, t) for t in tables])
    return ctx, SlodOracle(prob)


def cond_eff(info, d):
    """sigma_0 / smallest singular value still used after thresholding + truncation."""
    sig = info["sigma"][d]
    steps = info["trunc_steps"][d]
    kept = sig[: len(sig) - steps]
    kept = kept[kept > 1e-15 * sig[0]]
    return float(sig[0] / kept[-1]) if len(kept) else 1.0


def patch_tolerance(info, d, c=200.0):
    """1e-10 for well-conditioned selections, c * eps * cond_eff otherwise (SURVEY Appendix E)."""
    if not info.get("slod", False):
        return 1e-10
    return max(1e-10, c * EPS * cond_eff(info, d))


def margin_safe(info, d):
    """False when a discontinuous decision of the reference rule is within rounding of flipping: the computed d carries
    an error of about eps * cond(G) * ||d||, so ||d||_inf within max(1e-8, 1e3 eps cond(G)) of the 0.5 threshold
    (source/LOD.cc:703) can fall on either side in any fp64 implementation, LAPACK's included."""
    if not info.get("slod", False):
        return True
    sig = np.asarray(info["sigma"][d])
    kept = sig[sig > 1e-15 * sig[0]]
    cond_full = float(sig[0] / kept[-1]) if len(kept) else 1.0
    if abs(info["dinf"][d] - 0.5) <= max(1e-8, 1e3 * EPS * cond_full):
        return False
    # the singular-value threshold 1e-15 * sigma_0 (source/LOD.cc:667): a singular value of size ~eps * sigma_0 is
    # only known to O(1) relative accuracy, so a ratio within two decades of the threshold can fall on either side
    # (LAPACK's dgesdd included) and the selected d changes completely
    ratio = sig / sig[0]
    return not np.any((ratio > 1e-17) & (ratio < 1e-13))


def selection_from_G(G, Minv, X, d, s_dim=None):
    """The reference's selection (source/LOD.cc:637-752) restated on given stage matrices; returns the
    interior part of the normalised basis function."""
    ncd = G.shape[0]
    other = [k for k in range(ncd) if k != d]
    Go = G[np.ix_(other, other)]
    g = G[other, d]
    U, sig, Vt = np.linalg.svd(Go)
    winv = np.where(sig > 1e-15 * sig[0], 1.0 / np.where(sig > 0, sig, 1.0), 0.0)
    d_i = -(Vt.T @ (winv * (U.T @ g)))
    for i in range(len(other) - 1, -1, -1):
        if np.abs(d_i).max() < 0.5:
            break
        d_i = d_i + Vt[i, :] * (U[:, i] @ g) * winv[i]
    c = Minv[:, d].copy()
    for idx, k in enumerate(other):
        c += d_i[idx] * Minv[:, k]
    phi = X @ c
    return phi / np.linalg.norm(phi)


def selection_sensitivity(info, d, trials=4, rel=4 * EPS, seed=0):
    """Change of the selected basis under a few-ulp symmetric perturbation of the Gram matrix: the accuracy
    floor of ANY fp64 implementation of the reference's Gram/SVD selection on this patch."""
    G, Minv, X = info["G"], info["Minv"], info["X"]
    base = selection_from_G(G, Minv, X, d)
    rs = np.random.default_rng(seed)
    worst = 0.0
    for _ in range(trials):
        E = rs.standard_normal(G.shape)
        E = (E + E.T) * 0.5 * rel * np.abs(G).max()
        worst = max(worst, np.linalg.norm(selection_from_G(G + E, Minv, X, d) - base))
    return worst
