"""CPU checks of the selection test infrastructure: the extended-precision restatement of the reference's selection
rule (tools/select_reference.py) against mpmath, against the fp64 restatement the parity tests use and against the
oracle; the synthetic families (tools/select_families.py) against their designs; and the host-side refusals of
slod_debug_select on a handle without a device."""
import importlib
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tools"))
import select_families as sf  # noqa: E402
import select_reference as sr  # noqa: E402

pkg = importlib.import_module("dealii-slod_b200")
precise = pytest.mark.skipif(not sr.PRECISE, reason=f"numpy longdouble has eps {sr.EPS_LD:.1e} here (> 1e-18): "
                             "the reference needs x87 extended precision")


def _random_problem(n, seed, spread=8):
    rs = np.random.default_rng(seed)
    lam = 10.0 ** (-spread * rs.random(n))
    lam[0] = 1.0
    Q = sf.orthogonal(n, rs)
    return sf.embed(((Q * lam) @ Q.T + ((Q * lam) @ Q.T).T) / 2, rs.standard_normal(n), 0)


@precise
@pytest.mark.parametrize("n", [5, 17, 40])
def test_reference_matches_mpmath(n):
    """Eigenvalues to 1e-17 sigma_0 and every candidate d(r) to 1e-12 relative against mpmath.eigsy at 32 digits on
    the same fp64 matrix (spectrum spread over 8 decades: d(0) has cond 1e8, so 1e-12 needs more than fp64)."""
    mpmath = pytest.importorskip("mpmath")
    mpmath.mp.dps = 32
    G = _random_problem(n, n)
    ref = sr.select(G, np.eye(n + 1), 0)
    Go, g, _ = sr.split(G, 0)
    E, Qm = mpmath.eigsy(mpmath.matrix(Go.tolist()))
    lam = np.array([np.longdouble(mpmath.nstr(x, 30)) for x in E])
    order = np.argsort(-np.abs(lam), kind="stable")
    assert np.abs(np.sort(lam) - np.sort(ref["lam_ld"])).max() <= 1e-17 * ref["sigma0"]
    gm = mpmath.matrix(g.tolist())
    terms = []
    for k in order:
        v = Qm[:, int(k)]
        terms.append([float(x) for x in v * ((v.T * gm)[0] / E[int(k)])])
    terms = np.array(terms)                       # row j: the j-th largest term
    for r in range(n + 1):
        want = -terms[: n - r].sum(axis=0) if r < n else np.zeros(n)
        assert np.linalg.norm(ref["cand"][r] - want) <= 1e-12 * max(np.linalg.norm(want), 1e-300), r


@precise
@pytest.mark.parametrize("label", ["fast", "truncation", "clusters"])
def test_reference_matches_fp64_restatement(label):
    """On well-conditioned designs (cond <= 1e6) the parity tests' fp64 restatement (parity_common.selection_from_G,
    LAPACK SVD) and this one agree: same normalised c to 1e-9 (1e3 eps cond)."""
    pc = pytest.importorskip("parity_common")
    rs = np.random.default_rng(5)
    for n, d in ((8, 0), (31, 1), (65, 0)):
        G, expect = sf.family(label, n, d, 0, R=3 if label == "truncation" else None)
        Minv = sf.random_minv(n + 1, rs)
        ref = sr.select(G, Minv, d)
        assert ref["steps"] == expect["steps"]
        want = pc.selection_from_G(G, Minv, np.eye(n + 1), d)
        assert np.linalg.norm(ref["c"] / np.linalg.norm(ref["c"]) - want) <= 1e-9


@precise
def test_reference_matches_oracle():
    """The oracle's own selection (its SVD on its own G) on the margin-safe patches of a small SLOD case: the same step
    counts and the same basis function at the parity tests' 1e-10 / conditioning tolerance."""
    pc = pytest.importorskip("parity_common")
    from oracle.slod_oracle import morton_decode
    orc = pc.SlodOracle(pc.SlodProblem(dim=2, spacedim=2, n_global_refinements=3, n_subdivisions=2, oversampling=1,
                                       stabilize=True, problem="elasticity",
                                       coefficients=[pc.CoefficientTable(2, 4, t)
                                                     for t in pc.make_tables(2, 2, 4, "uniform100", 3)]))
    pids = [0, 9, 27, 36, 63]
    orc.compute_basis(pids)
    checked = 0
    for res in orc.patches:
        shape, _ = orc.shape_for(morton_decode(res.pid, 2, 3))
        for d in range(2):
            ref = sr.select(res.info["G"], res.info["Minv"], d)
            if not (pc.margin_safe(res.info, d) and sr.margins_safe(ref)):
                continue
            checked += 1
            assert ref["steps"] == res.info["trunc_steps"][d]
            phi = res.info["X"] @ ref["c"]
            phi /= np.linalg.norm(phi)
            assert np.linalg.norm(phi - res.basis[d][shape.internal]) <= pc.patch_tolerance(res.info, d), res.pid
    assert checked >= 4


@precise
@pytest.mark.parametrize("n", [3, 7, 8, 15, 17, 31, 65])
def test_family_designs(n):
    """Every synthetic family reproduces its design (step count, fast-path eligibility) on the fp64 matrix, with every
    decision margin above its bound.  The large sizes are checked where they are used (tests/test_select_gpu.py)."""
    for d in (0, 1):
        for label, G, expect in sf.cases(n, d):
            ref = sf.check_design(G, d, expect)
            if label == "zero_load":
                assert not ref["d"].any()


def test_debug_select_refusals():
    """slod_debug_select checks its input on the host before anything runs: out-of-range and repeated patch ids and
    non-finite entries are SLOD_ERR_INVALID (1) even without a device; valid input on a maps-only handle is
    SLOD_ERR_CUDA (3), as every computing entry point."""
    pkg.build_library()
    ctx = pkg.SlodContext(dim=2, n_global_refinements=3, oversampling=1, stabilize=True, device=-2)
    import ctypes as C
    ncd = ctx.patch_info(0)["n_coarse"]
    eye = np.eye(ncd)
    for pids, G in (([0, 0], [eye, eye]), ([0], [np.full((ncd, ncd), np.nan)]), ([0], [np.where(eye > 0, np.inf, 0.0)])):
        with pytest.raises(pkg.SlodError) as e:
            ctx.debug_select(pids, G, [eye] * len(pids))
        assert e.value.code == 1 and ("repeated" in str(e.value) or "non-finite" in str(e.value)), pids
    ids = np.array([ctx.n_patches], dtype=np.int64)
    c, diag = np.empty(ncd), np.empty(8)
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))   # noqa: E731
    assert ctx.lib.slod_debug_select(ctx.h, 1, ids.ctypes.data_as(C.POINTER(C.c_int64)), dp(eye), dp(eye), dp(c),
                                     dp(diag)) == 1
    with pytest.raises(pkg.SlodError) as e:
        ctx.debug_select([0], [eye], [eye])
    assert e.value.code == 3
    with pytest.raises(ValueError):
        ctx.debug_select([0], [np.eye(ncd + 1)], [np.eye(ncd + 1)])
