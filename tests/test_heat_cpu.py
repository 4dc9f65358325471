"""CPU checks of the coarse mass matrix and the heat-equation entry points: a handle without a device refuses them, the
symbols are exported, and an anchor of backward Euler on the SLOD space that depends on no GPU run: the oracle's SLOD
trajectory against its fine trajectory shows the super-exponential decay of the localization error in the oversampling."""
import ctypes as C
import importlib
import os
import sys

import numpy as np
import pytest

from oracle.slod_oracle import CoefficientTable, SlodOracle, SlodProblem

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tools"))
from heat_oracle import coarse_mass, fine_operators, heat_solve_coarse, heat_solve_fine  # noqa: E402

pkg = importlib.import_module("dealii-slod_b200")

NEW = ["slod_assemble_coarse_mass", "slod_get_coarse_mass_csr", "slod_l2_project_batch", "slod_heat_solve",
       "slod_heat_solve_batch", "slod_fem_heat_solve"]


@pytest.fixture(scope="module")
def ctx():
    pkg.build_library()
    c = pkg.SlodContext(dim=2, n_global_refinements=3, device=-2)
    yield c
    c.close()


def test_new_symbols_are_exported(ctx):
    for name in NEW:
        assert name in pkg.EXPORTS
        getattr(ctx.lib, name)


def test_maps_only_handle_refuses_heat_calls(ctx):
    nf, nc = ctx.n_fine, ctx.n_patches * ctx.s
    for call in (ctx.assemble_coarse_mass, ctx.coarse_mass_csr,
                 lambda: ctx.l2_project_batch(np.ones((2, nf))),
                 lambda: ctx.heat_solve(np.ones(nf), None, 1e-2, 3),
                 lambda: ctx.heat_solve_batch(np.ones((2, nf)), None, 1e-2, 3),
                 lambda: ctx.fem_heat_solve(np.ones(nf), None, 1e-2, 3)):
        with pytest.raises(pkg.SlodError) as e:
            call()
        assert e.value.code == 3 and "without a device" in str(e.value)
    # through the C ABI directly, invalid arguments included: the missing device is reported first
    buf = np.zeros(max(nf, nc) * 4)
    dp = buf.ctypes.data_as(C.POINTER(C.c_double))
    lib, h = ctx.lib, ctx.h
    assert lib.slod_assemble_coarse_mass(h) == 3
    i64 = np.zeros(nc + 1, dtype=np.int64).ctypes.data_as(C.POINTER(C.c_int64))
    assert lib.slod_get_coarse_mass_csr(h, i64, i64, dp, None, None) == 3
    assert lib.slod_l2_project_batch(h, 0, dp, dp, 10, 0.0, 1e-10, None, None) == 3
    assert lib.slod_heat_solve(h, dp, dp, -1.0, 0, 0, dp, 10, 0.0, 1e-10, None) == 3
    assert lib.slod_heat_solve_batch(h, 1, dp, dp, 1e-2, 2, 1, dp, 10, 0.0, 1e-10, None) == 3
    assert lib.slod_fem_heat_solve(h, dp, dp, 1e-2, 2, 1, dp, 10, 0.0, 1e-10, None) == 3


def _energy(A, e):
    return float(np.sqrt(e @ (A @ e)))


def _trajectory_errors(s, ell, steps=20, dt=1e-2, seed=11):
    """Relative energy error of the prolongated SLOD trajectory against the fine one, per step.  The problem of
    tests/test_oracle_convergence.py: 8^2 cells, n = 2, coefficients in [1, 100] (seed 11), constant forcing, u0 = 0."""
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
    M_H = coarse_mass(o, Cm)
    rhs = [1.0] if s == 1 else [1.0, -0.5]
    F = o.fem_rhs(lambda p: np.tile(rhs, (len(p), 1)))
    U = heat_solve_coarse(K, M_H, Cm.T @ F, None, dt, steps)
    Uf = heat_solve_fine(o, F, None, dt, steps)
    A, _, _ = fine_operators(o)
    return np.array([_energy(A, Cm @ U[k] - Uf[k]) / _energy(A, Uf[k]) for k in range(steps)]), M_H, K


def test_oracle_mass_matrix_is_spd_on_the_pattern_of_K():
    _, M_H, K = _trajectory_errors(1, 1, steps=1)
    assert np.array_equal(M_H.indptr, K.indptr) and np.array_equal(M_H.indices, K.indices)
    D = (M_H - M_H.T).toarray()
    assert np.abs(D).max() <= 1e-14 * np.abs(M_H.data).max()
    assert np.linalg.eigvalsh(M_H.toarray()).min() > 0


@pytest.mark.parametrize("s,ells,bounds,first", [
    # measured at t = 0.2: 1.16e-1 / 8.9e-4 / 1.17e-6; first step 1.16e-1 / 1.08e-3 / 5.5e-4
    (1, (1, 2, 3), (0.2, 2e-3, 5e-6), (None, 2e-3, 2e-3)),
    # measured: 1.48e-1 / 4.3e-3
    (2, (1, 2), (0.3, 1e-2), (None, None)),
])
def test_slod_trajectory_error_decays(s, ells, bounds, first):
    """Final-time energy error: each layer gains more than a factor 20.  The first step does not keep decaying: for
    dt << H^2 the mass term dominates the step, and the basis was built for the elliptic operator (the floor DESIGN.md
    records), so it is only bounded."""
    prev = None
    for ell, bound, b1 in zip(ells, bounds, first):
        err, _, _ = _trajectory_errors(s, ell)
        assert err[-1] < bound, (ell, err[-1])
        if b1 is not None:
            assert err[0] < b1, (ell, err[0])
        if prev is not None:
            assert err[-1] < prev / 20.0, (ell, err[-1], prev)
        prev = err[-1]
