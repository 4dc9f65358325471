"""CPU checks of the theta scheme on the SLOD space (slod_heat_theta_solve / _batch, slod_fem_heat_theta_solve) that need
no GPU: the reference in tools/heat_oracle.py against closed forms and the backward-Euler loop it replaces, its order in
time, the pinned SLOD-vs-fine trajectory errors the GPU tests use, and every argument refusal on a maps-only handle."""
import ctypes as C
import importlib
import os
import sys

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from oracle.slod_oracle import CoefficientTable, SlodOracle, SlodProblem

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tools"))
from heat_oracle import (coarse_mass, fine_operators, heat_solve_coarse, heat_solve_fine,  # noqa: E402
                         theta_solve_coarse, theta_solve_fine)

pkg = importlib.import_module("dealii-slod_b200")

NEW = ["slod_heat_theta_solve", "slod_heat_theta_solve_batch", "slod_fem_heat_theta_solve"]
T_END = 0.2


def _problem(s, ell, seed=11):
    """The problem of tests/test_heat_cpu.py: 8^2 cells, n = 2, coefficients in [1, 100] (seed 11)."""
    dim, ref = 2, 3
    r = ref + 1
    rs = np.random.default_rng(seed)
    tabs = [1.0 + 99.0 * rs.random((2 ** r) ** dim) for _ in range(1 if s == 1 else 2)]
    prob = SlodProblem(dim=dim, spacedim=s, n_global_refinements=ref, n_subdivisions=2, oversampling=ell,
                       stabilize=True, problem="diffusion" if s == 1 else "elasticity",
                       coefficients=[CoefficientTable(dim, r, t) for t in tabs])
    o = SlodOracle(prob)
    o.compute_basis()
    K, Cm, _ = o.assemble_global_matrix()
    F = o.fem_rhs(lambda p: np.tile([1.0] if s == 1 else [1.0, -0.5], (len(p), 1)))
    return o, K, Cm, coarse_mass(o, Cm), F


def ramp(n_steps, dt):
    """g(t) = sin(pi t / (2 T)) at t_k = k dt, one field: 0 at t = 0, 1 at T = 0.2."""
    return np.sin(np.pi * np.arange(n_steps + 1) * dt / (2 * T_END))[:, None]


def pulse(n_steps, dt):
    """g(t) = sin(pi t / T) at t_k = k dt, one field: 0 at t = 0 and at T."""
    return np.sin(np.pi * np.arange(n_steps + 1) * dt / T_END)[:, None]


# ---- the reference itself ----------------------------------------------------------------------------------------------
def _be_coarse(K, M_H, b, u0, dt, n_steps):
    """The backward-Euler loop the theta reference replaced, restated."""
    solve = spla.factorized(sp.csc_matrix(M_H + dt * K))
    u = np.zeros(K.shape[0]) if u0 is None else np.array(u0, dtype=float)
    b = np.zeros(K.shape[0]) if b is None else np.asarray(b, dtype=float)
    out = []
    for _ in range(n_steps):
        u = u + solve(dt * (b - K @ u))
        out.append(u.copy())
    return np.array(out)


def test_new_symbols_are_exported():
    pkg.build_library()
    lib = pkg.load_library()
    for name in NEW:
        assert name in pkg.EXPORTS
        getattr(lib, name)


def test_theta_one_is_backward_euler_bit_for_bit():
    o, K, Cm, M_H, F = _problem(1, 1)
    rng = np.random.default_rng(1)
    u0 = rng.standard_normal(K.shape[0])
    b = Cm.T @ F
    ref = _be_coarse(K, M_H, b, u0, 1e-2, 5)
    assert np.array_equal(theta_solve_coarse(K, M_H, b[None], None, u0, 1.0, 1e-2, 5), ref)
    assert np.array_equal(heat_solve_coarse(K, M_H, b, u0, 1e-2, 5), ref)
    assert np.array_equal(theta_solve_coarse(K, M_H, None, None, u0, 1.0, 1e-2, 5),
                          _be_coarse(K, M_H, None, u0, 1e-2, 5))
    # the fine reference: the same loop on the interior dofs
    A, M, ii = fine_operators(o)
    Aii, Mii = A[ii][:, ii], M[ii][:, ii]
    solve = spla.factorized(sp.csc_matrix(Mii + 1e-2 * Aii))
    u0f = rng.standard_normal(A.shape[0])
    u = u0f.copy()
    mask = np.zeros(A.shape[0], dtype=bool)
    mask[ii] = True
    u[~mask] = 0.0
    ref_f = []
    for _ in range(4):
        u[ii] += solve(1e-2 * (F[ii] - Aii @ u[ii]))
        ref_f.append(u.copy())
    assert np.array_equal(theta_solve_fine(o, F[None], None, u0f, 1.0, 1e-2, 4), np.array(ref_f))
    assert np.array_equal(heat_solve_fine(o, F, u0f, 1e-2, 4), np.array(ref_f))


def _amp(theta, z):
    return (1.0 - (1.0 - theta) * z) / (1.0 + theta * z)


@pytest.mark.parametrize("theta", [0.5, 0.75, 1.0])
def test_scalar_closed_form(theta):
    """m u' + k u = b(t) with one dof: u^k = R u^{k-1} + dt (theta b_k + (1 - theta) b_{k-1}) / (m + theta dt k),
    R = (1 - (1 - theta) z) / (1 + theta z), z = dt k / m."""
    m, kk, dt, n = 2.0, 3.0, 0.1, 12
    K, M = sp.csr_matrix([[kk]]), sp.csr_matrix([[m]])
    g = np.cos(np.arange(n + 1) * dt)[:, None]
    U = theta_solve_coarse(K, M, np.array([[1.5]]), g, [0.7], theta, dt, n)
    u, z = 0.7, dt * kk / m
    for k in range(1, n + 1):
        u = _amp(theta, z) * u + dt * 1.5 * (theta * g[k, 0] + (1 - theta) * g[k - 1, 0]) / (m + theta * dt * kk)
        assert abs(U[k - 1, 0] - u) <= 1e-13 * max(abs(u), 1.0), (k, U[k - 1, 0], u)


def test_stiff_mode_crank_nicolson_and_rannacher():
    """dt k / m = 1e3: Crank-Nicolson flips the sign of the mode and nearly keeps its size (R = -0.996); two Rannacher start-up
    steps (four backward-Euler half steps, 1 / (1 + z / 2) each) damp it to the closed-form value."""
    m, kk, dt, n = 1.0, 1e3, 1.0, 10
    K, M = sp.csr_matrix([[kk]]), sp.csr_matrix([[m]])
    z = dt * kk / m
    U = theta_solve_coarse(K, M, None, None, [1.0], 0.5, dt, n)[:, 0]
    assert np.allclose(U, _amp(0.5, z) ** np.arange(1, n + 1), rtol=1e-12, atol=0)
    assert abs(U[0]) > 0.99 and abs(U[-1]) > 0.95 and (np.sign(U) == (-1.0) ** np.arange(1, n + 1)).all()
    for ns in (1, 2):
        Ur = theta_solve_coarse(K, M, None, None, [1.0], 0.5, dt, n, n_startup=ns)[:, 0]
        closed = [(1.0 / (1.0 + z / 2)) ** (2 * min(k, ns)) * _amp(0.5, z) ** max(k - ns, 0) for k in range(1, n + 1)]
        assert np.allclose(Ur, closed, rtol=1e-12, atol=0)
        assert abs(Ur[-1]) < 1e-5
    # the half-step load is g at the midpoint (g_{k-1} + g_k) / 2, then g_k
    g = np.array([[0.0], [2.0], [2.0]])
    Ur = theta_solve_coarse(K, M, np.array([[1.0]]), g, [0.0], 0.5, dt, 2, n_startup=1)[:, 0]
    h = 0.5 * dt
    u1 = h * 1.0 / (m + h * kk)
    u2 = (u1 * m + h * 2.0) / (m + h * kk)
    assert abs(Ur[0] - u2) <= 1e-15 * abs(u2)


def _m_norm(M, v):
    return float(np.sqrt(v @ (M @ v)))


def test_self_convergence_in_time():
    """2-D diffusion, 8^2 cells, l = 2, u0 = 0, g = sin(pi t / T): the error at T against a dt / 64 run falls by at
    least 3.5x per halving of dt for Crank-Nicolson and by about 2x for backward Euler.  From dt = T / 32 (measured
    ratios 4.30, 4.02 and 2.62, 2.42; backward Euler still carries a second-order part at these steps)."""
    _, K, Cm, M_H, F = _problem(1, 2)
    b = (Cm.T @ F)[None]
    n0 = 32
    dt0 = T_END / n0
    for theta, lo, hi in ((0.5, 3.5, 4.5), (1.0, 1.8, 2.7)):
        ref = theta_solve_coarse(K, M_H, b, pulse(64 * n0, dt0 / 64), None, theta, dt0 / 64, 64 * n0)[-1]
        errs = [_m_norm(M_H, theta_solve_coarse(K, M_H, b, pulse(n0 * 2 ** j, dt0 / 2 ** j), None, theta,
                                                dt0 / 2 ** j, n0 * 2 ** j)[-1] - ref) for j in range(3)]
        ratios = [errs[j] / errs[j + 1] for j in range(2)]
        print(f"theta {theta}: errors {errs}, ratios {ratios}")
        assert all(lo <= r <= hi for r in ratios), (theta, errs, ratios)


# SLOD-vs-fine relative energy error at T = 0.2 of the Crank-Nicolson trajectory (dt = 1e-2, two start-up steps, g = the
# ramp, u0 = 0) on the problem above; the GPU test bounds its own run by the same values.
CN_ERRORS = {1: 1.2e-1, 2: 9.4e-4, 3: 1.3e-6}


def cn_trajectory_error(o, K, Cm, M_H, F):
    n, dt = 20, T_END / 20
    U = theta_solve_coarse(K, M_H, (Cm.T @ F)[None], ramp(n, dt), None, 0.5, dt, n, n_startup=2)
    Uf = theta_solve_fine(o, F[None], ramp(n, dt), None, 0.5, dt, n, n_startup=2)
    A, _, _ = fine_operators(o)
    e = Cm @ U[-1] - Uf[-1]
    return float(np.sqrt(e @ (A @ e)) / np.sqrt(Uf[-1] @ (A @ Uf[-1])))


def test_cn_trajectory_error_decays():
    prev = None
    for ell in (1, 2, 3):
        err = cn_trajectory_error(*_problem(1, ell))
        print(f"l = {ell}: {err:.3e}")
        assert 0.8 * CN_ERRORS[ell] <= err <= 1.25 * CN_ERRORS[ell], (ell, err)
        if prev is not None:
            assert err < prev / 20.0
        prev = err


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

    def calls(theta=0.5, dt=1e-2, n=n_steps, every=1, ns=0, nq=2, f=dp, g="ok", out=dp, ms=100, tol=0.0, red=1e-10):
        g = gp(g_ok) if isinstance(g, str) else g
        yield lib.slod_heat_theta_solve(h, theta, dt, n, every, ns, nq, f, g, None, out, ms, tol, red, None)
        yield lib.slod_heat_theta_solve_batch(h, 3, theta, dt, n, every, ns, nq, f, g, None, out, ms, tol, red, None)
        yield lib.slod_fem_heat_theta_solve(h, theta, dt, n, every, ns, nq, f, g, None, out, ms, tol, red, None)

    refusals = [dict(theta=0.49), dict(theta=1.01), dict(theta=float("nan")), dict(theta=-1.0),
                dict(ns=-1), dict(ns=n_steps + 1), dict(nq=0), dict(nq=-3), dict(g=gp(g_nan)), dict(g=gp(g_inf)),
                dict(dt=0.0), dict(dt=float("inf")), dict(n=0), dict(every=0), dict(every=n_steps + 1),
                dict(out=None), dict(ms=-1), dict(tol=-1.0), dict(red=float("nan"))]
    for kw in refusals:
        assert list(calls(**kw)) == [1, 1, 1], kw
    assert lib.slod_heat_theta_solve_batch(h, 0, 0.5, 1e-2, 2, 1, 0, 1, dp, None, None, dp, 100, 0.0, 1e-10, None) == 1
    # the batch reads g of every column: a NaN in the last column's last row is found
    g_last = g_ok.copy()
    g_last[2, n_steps, 1] = np.nan
    assert lib.slod_heat_theta_solve_batch(h, 3, 0.5, 1e-2, n_steps, 1, 0, 2, dp, gp(g_last), None, dp, 100, 0.0,
                                           1e-10, None) == 1
    # accepted: the bounds themselves, g = NULL, no fields (n_fields and g are then not read)
    for kw in (dict(theta=0.5), dict(theta=1.0), dict(ns=n_steps), dict(g=None), dict(f=None, nq=0, g=gp(g_nan))):
        assert list(calls(**kw)) == [3, 3, 3], kw
    with pytest.raises(pkg.SlodError) as e:
        ctx.heat_theta_solve(np.ones((2, nf)), None, None, 0.5, 1e-2, 3)
    assert e.value.code == 3 and "without a device" in str(e.value)
    with pytest.raises(pkg.SlodError) as e:
        ctx.heat_theta_solve(np.ones((2, nf)), None, None, 0.4, 1e-2, 3)
    assert e.value.code == 1 and "theta" in str(e.value)
    with pytest.raises(ValueError):
        ctx.heat_theta_solve(np.ones((2, nf)), np.ones((3, 2)), None, 0.5, 1e-2, 3)   # g needs n_steps + 1 rows
