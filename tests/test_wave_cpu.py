"""CPU checks of Newmark time stepping for the wave equation on the SLOD space (slod_wave_solve / _batch,
slod_fem_wave_solve) that need no GPU: the reference in tools/wave_oracle.py against the Chebyshev closed form on
generalized eigenvectors, its energy conservation and order in time, the stable explicit step on the SLOD space against
the fine grid, the pinned SLOD-vs-fine trajectory errors the GPU tests use, and every argument refusal on a maps-only
handle."""
import ctypes as C
import importlib
import os
import sys

import numpy as np
import pytest
import scipy.linalg as sl
import scipy.sparse.linalg as spla

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tools"))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from heat_oracle import fine_operators  # noqa: E402
from test_heat_theta_cpu import T_END, _problem, pulse, ramp  # noqa: E402
from wave_oracle import energy, newmark_coarse, newmark_fine  # noqa: E402

pkg = importlib.import_module("dealii-slod_b200")

NEW = ["slod_wave_solve", "slod_wave_solve_batch", "slod_fem_wave_solve"]


def test_new_symbols_are_exported():
    pkg.build_library()
    lib = pkg.load_library()
    for name in NEW:
        assert name in pkg.EXPORTS
        getattr(lib, name)


def chebyshev(k, c):
    """T_0 .. T_k at c (three-term recurrence; |c| > 1 included)."""
    t = [1.0, c]
    for _ in range(k - 1):
        t.append(2.0 * c * t[-1] - t[-2])
    return np.array(t[:k + 1])


def amplification(beta, z2):
    """c of the mode u_k = T_k(c) x for dt^2 lambda = z2; the scheme is stable for the mode iff |c| <= 1."""
    return (1.0 - (0.5 - beta) * z2) / (1.0 + beta * z2)


def stable_z2(beta):
    """The largest stable dt^2 lambda for beta < 1/4."""
    return 4.0 / (1.0 - 4.0 * beta)


@pytest.mark.parametrize("ell", [1, 2])
@pytest.mark.parametrize("beta", [0.0, 1.0 / 12, 0.25, 0.5])
def test_chebyshev_closed_form(beta, ell):
    """u_0 = x with K x = lambda M_H x, v_0 = 0, no forcing: u_k = T_k(c) x.  At a stable dt for three eigenpairs (the
    top one, a middle one, the lowest); for beta < 1/4 at dt^2 lambda_max 5 % above the limit, where the top mode grows
    like T_k(c) with c < -1."""
    _, K, _, M, _ = _problem(1, ell)
    lam, X = sl.eigh(K.toarray(), M.toarray())
    n_steps = 40
    dts = [0.9 * np.sqrt(stable_z2(beta) / lam[-1]) if beta < 0.25 else 3.0 / np.sqrt(lam[-1])]
    if beta < 0.25:
        dts.append(np.sqrt(1.05 * stable_z2(beta) / lam[-1]))
    for i, dt in enumerate(dts):
        for m in ((len(lam) - 1,) if i else (len(lam) - 1, len(lam) // 2, 0)):
            x = X[:, m]
            c = amplification(beta, dt * dt * lam[m])
            U, _ = newmark_coarse(K, M, None, None, x, None, beta, dt, n_steps)
            T = chebyshev(n_steps, c)
            err = np.abs(U - T[:, None] * x[None]).max(axis=1) / (np.maximum(np.abs(T), 1.0) * np.abs(x).max())
            assert err.max() <= 1e-9, (beta, dt, m, c, err.max())
            if i:
                assert c < -1.0 and abs(T[-1]) > 1e3, (beta, c, T[-1])
            else:
                assert abs(c) <= 1.0


def test_energy_conserved_average_acceleration():
    """beta = 1/4, no forcing, seeded u_0 and v_0: E = 1/2 v^T M_H v + 1/2 u^T K u is the same to 1e-12 over 500 steps,
    at a step 10x above the explicit limit."""
    _, K, _, M, _ = _problem(1, 2)
    lam_max = spla.eigsh(K.tocsc(), k=1, M=M.tocsc(), which="LA", return_eigenvectors=False)[0]
    rng = np.random.default_rng(1)
    n = K.shape[0]
    dt = 20.0 / np.sqrt(lam_max)
    U, V = newmark_coarse(K, M, None, None, rng.standard_normal(n), rng.standard_normal(n), 0.25, dt, 500)
    E = energy(K, M, U, V)
    assert np.abs(E / E[0] - 1.0).max() <= 1e-12, np.abs(E / E[0] - 1.0).max()


def _m_norm(M, v):
    return float(np.sqrt(v @ (M @ v)))


@pytest.mark.parametrize("beta", [0.0, 0.25])
def test_second_order_in_time(beta):
    """2-D diffusion, 8^2 cells, l = 2, u0 = v0 = 0, g = sin(pi t / T), T = 0.2: the error of u at T against a dt / 64
    run falls by about 4x per halving of dt.  From dt = T / 64, inside the explicit limit (dt^2 lambda_max = 0.71)."""
    _, K, Cm, M, F = _problem(1, 2)
    b = (Cm.T @ F)[None]
    n0 = 64
    dt0 = T_END / n0
    ref = newmark_coarse(K, M, b, pulse(64 * n0, dt0 / 64), None, None, beta, dt0 / 64, 64 * n0)[0][-1]
    errs = [_m_norm(M, newmark_coarse(K, M, b, pulse(n0 * 2 ** j, dt0 / 2 ** j), None, None, beta, dt0 / 2 ** j,
                                      n0 * 2 ** j)[0][-1] - ref) for j in range(3)]
    ratios = [errs[j] / errs[j + 1] for j in range(2)]
    print(f"beta {beta}: errors {errs}, ratios {ratios}")
    assert all(3.5 <= r <= 4.5 for r in ratios), (beta, errs, ratios)


# sqrt(lambda_max(M_h^-1 A_h) / lambda_max(M_H^-1 K)) on the problem above (8^2 cells, n = 2, coefficients in [1, 100]):
# the explicit step the SLOD space allows over the one the fine grid allows, for every oversampling l = 1, 2, 3
STEP_RATIO = 2.10


def lambda_max(A, M):
    return float(spla.eigsh(A.tocsc(), k=1, M=M.tocsc(), which="LA", return_eigenvectors=False)[0])


@pytest.mark.parametrize("ell", [1, 2, 3])
def test_stable_explicit_step_ratio(ell):
    o, K, _, M, _ = _problem(1, ell)
    A, Mh, ii = fine_operators(o)
    lam_H, lam_h = lambda_max(K, M), lambda_max(A[ii][:, ii], Mh[ii][:, ii])
    ratio = np.sqrt(lam_h / lam_H)
    print(f"l = {ell}: lambda_max SLOD {lam_H:.6g}, fine {lam_h:.6g}, explicit step ratio {ratio:.4f}")
    assert abs(ratio - STEP_RATIO) <= 0.01, ratio


# SLOD-vs-fine relative energy error of u at T = 0.2 of the beta = 1/4 trajectory (dt = 1e-2, g = the ramp, u0 = v0 =
# 0) on the problem above; the GPU test bounds its own run by the same values.  The error decreases with l but levels
# off: the load excites fine-scale modes that oscillate undamped in the fine trajectory and are absent from the SLOD space.
WAVE_ERRORS = {1: 1.15e-1, 2: 2.05e-3, 3: 1.85e-3}


def wave_trajectory_error(o, K, Cm, M_H, F):
    n, dt = 20, T_END / 20
    U, _ = newmark_coarse(K, M_H, (Cm.T @ F)[None], ramp(n, dt), None, None, 0.25, dt, n)
    Uf, _ = newmark_fine(o, F[None], ramp(n, dt), None, None, 0.25, dt, n)
    A, _, _ = fine_operators(o)
    e = Cm @ U[-1] - Uf[-1]
    return float(np.sqrt(e @ (A @ e)) / np.sqrt(Uf[-1] @ (A @ Uf[-1])))


def test_wave_trajectory_error_decreases():
    prev = None
    for ell in (1, 2, 3):
        err = wave_trajectory_error(*_problem(1, ell))
        print(f"l = {ell}: {err:.3e}")
        assert 0.95 * WAVE_ERRORS[ell] <= err <= 1.05 * WAVE_ERRORS[ell], (ell, err)
        if prev is not None:
            assert err < prev
        prev = err


def test_fine_reference_ignores_boundary_rows():
    """newmark_fine keeps u, v zero on the boundary whatever the boundary rows of F, u0 and v0 hold."""
    o, _, _, _, F = _problem(1, 1)
    _, _, ii = fine_operators(o)
    rng = np.random.default_rng(3)
    n = F.size
    bnd = np.setdiff1d(np.arange(n), ii)
    u0, v0 = rng.standard_normal(n), rng.standard_normal(n)
    U, V = newmark_fine(o, F[None], None, u0, v0, 0.25, 1e-2, 3)
    u0b, v0b, Fb = u0.copy(), v0.copy(), F.copy()
    u0b[bnd] = v0b[bnd] = Fb[bnd] = 7.0
    U2, V2 = newmark_fine(o, Fb[None], None, u0b, v0b, 0.25, 1e-2, 3)
    assert np.array_equal(U, U2) and np.array_equal(V, V2) and not U[:, bnd].any() and not V[:, bnd].any()


# ---- argument refusals on a maps-only handle ------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx():
    pkg.build_library()
    c = pkg.SlodContext(dim=2, n_global_refinements=3, device=-2)
    yield c
    c.close()


def test_maps_only_handle_refusals(ctx):
    """Every argument is checked before the device (SLOD_ERR_INVALID = 1); a valid call then reports the missing device
    (SLOD_ERR_CUDA = 3)."""
    nf, nc = ctx.n_fine, ctx.n_patches * ctx.s
    buf = np.zeros(max(nf, nc) * 16)
    dp = buf.ctypes.data_as(C.POINTER(C.c_double))
    lib, h = ctx.lib, ctx.h
    n_steps = 4
    g_ok = np.ones((3, n_steps + 1, 2))
    g_nan = g_ok.copy()
    g_nan[0, 2, 1] = np.nan
    g_inf = g_ok.copy()
    g_inf[0, 0, 0] = np.inf

    def gp(a):
        return np.ascontiguousarray(a).ctypes.data_as(C.POINTER(C.c_double))

    def calls(beta=0.25, dt=1e-2, n=n_steps, every=1, nq=2, f=dp, g="ok", out=dp, ms=100, tol=0.0, red=1e-10):
        g = gp(g_ok) if isinstance(g, str) else g
        yield lib.slod_wave_solve(h, beta, dt, n, every, nq, f, g, None, None, out, None, None, ms, tol, red, None)
        yield lib.slod_wave_solve_batch(h, 3, beta, dt, n, every, nq, f, g, None, None, out, None, None, ms, tol, red,
                                        None)
        yield lib.slod_fem_wave_solve(h, beta, dt, n, every, nq, f, g, None, None, out, None, None, ms, tol, red, None)

    refusals = [dict(beta=-1e-3), dict(beta=0.51), dict(beta=float("nan")), dict(beta=float("inf")),
                dict(nq=0), dict(nq=-3), dict(g=gp(g_nan)), dict(g=gp(g_inf)),
                dict(dt=0.0), dict(dt=-1e-2), dict(dt=float("inf")), dict(n=0), dict(every=0),
                dict(every=n_steps + 1), dict(out=None), dict(ms=-1), dict(tol=-1.0), dict(red=float("nan"))]
    for kw in refusals:
        assert list(calls(**kw)) == [1, 1, 1], kw
    assert lib.slod_wave_solve_batch(h, 0, 0.25, 1e-2, 2, 1, 1, dp, None, None, None, dp, None, None, 100, 0.0, 1e-10,
                                     None) == 1
    # the batch reads g of every column: a NaN in the last column's last row is found
    g_last = g_ok.copy()
    g_last[2, n_steps, 1] = np.nan
    assert lib.slod_wave_solve_batch(h, 3, 0.25, 1e-2, n_steps, 1, 2, dp, gp(g_last), None, None, dp, None, None, 100,
                                     0.0, 1e-10, None) == 1
    # accepted: the bounds themselves, g = NULL, no fields (n_fields and g are then not read), every output given
    for kw in (dict(beta=0.0), dict(beta=0.5), dict(every=n_steps), dict(g=None), dict(f=None, nq=0, g=gp(g_nan))):
        assert list(calls(**kw)) == [3, 3, 3], kw
    assert lib.slod_wave_solve(h, 0.25, 1e-2, n_steps, 1, 2, dp, gp(g_ok), dp, dp, dp, dp, dp, 100, 0.0, 1e-10,
                               None) == 3
    with pytest.raises(pkg.SlodError) as e:
        ctx.wave_solve(np.ones((2, nf)), None, None, None, 0.25, 1e-2, 3)
    assert e.value.code == 3 and "without a device" in str(e.value)
    with pytest.raises(pkg.SlodError) as e:
        ctx.wave_solve(np.ones((2, nf)), None, None, None, 0.6, 1e-2, 3)
    assert e.value.code == 1 and "beta" in str(e.value)
    with pytest.raises(pkg.SlodError) as e:
        ctx.fem_wave_solve(None, None, None, None, -0.1, 1e-2, 3)
    assert e.value.code == 1 and "beta" in str(e.value)
    with pytest.raises(ValueError):
        ctx.wave_solve(np.ones((2, nf)), np.ones((3, 2)), None, None, 0.25, 1e-2, 3)   # g needs n_steps + 1 rows
    with pytest.raises(ValueError):
        ctx.wave_solve_batch(None, None, None, None, 0.25, 1e-2, 3)
