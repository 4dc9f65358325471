"""Tensor diffusion (SLOD_PROBLEM_DIFFUSION_TENSOR) on the CPU: the reference restatement against the scalar oracle, a
mirror symmetry that pins the orientation of the off-diagonal term, the method's super-exponential decay with an
anisotropic coefficient, and the C ABI's argument checks on a maps-only handle."""
import importlib
import math
import os
import sys

import numpy as np
import pytest

from oracle.slod_oracle import CoefficientTable, SlodOracle, SlodProblem

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from aniso_oracle import VOIGT, grid_points, laminate, make_oracle, manufactured  # noqa: E402
from parity_common import margin_safe, patch_tolerance  # noqa: E402

pkg = importlib.import_module("dealii-slod_b200")


def _isotropic(dim, alpha):
    t = np.zeros((alpha.size, len(VOIGT[dim])))
    t[:, :dim] = alpha[:, None]
    return t


@pytest.mark.parametrize("dim,ref,ell,stabilize", [(2, 2, 1, True), (2, 2, 1, False), (2, 3, 2, True),
                                                   (3, 1, 1, True), (3, 2, 1, True), (3, 2, 1, False)])
def test_isotropic_tensor_reproduces_scalar_oracle(dim, ref, ell, stabilize):
    r = ref + 1
    alpha = 1.0 + 99.0 * np.random.default_rng(3).random((2 ** r) ** dim)
    sc = SlodOracle(SlodProblem(dim=dim, spacedim=1, n_global_refinements=ref, n_subdivisions=2, oversampling=ell,
                                stabilize=stabilize, coefficients=[CoefficientTable(dim, r, alpha)]))
    te = make_oracle(dim, ref, 2, ell, stabilize, r, _isotropic(dim, alpha))
    sc.compute_basis()
    te.compute_basis()
    Ks, _, _ = sc.assemble_global_matrix()
    Kt, _, _ = te.assemble_global_matrix()
    # 1e-12 on LOD-branch patches.  The SLOD selection (Gram matrix, thresholded SVD, truncation) amplifies the rounding
    # difference of the two sums (sum_f a_f K_f against alpha K): 7e-11 on a well-conditioned patch, and 3.3 times the
    # GPU parity tests' bound of 200 eps cond_eff on an ill-conditioned one (tools/parity_common.patch_tolerance).  Two
    # fp64 evaluations of the rule in numpy are held to 1e-10, or 2000 eps cond_eff.
    tol = [patch_tolerance(a.info, 0, c=2000.0) if a.info.get("slod", False) else 1e-12 for a in sc.patches]
    assert np.abs(Ks.data - Kt.data).max() <= max(tol) * np.abs(Ks.data).max()
    for a, b, t in zip(sc.patches, te.patches, tol):
        if not margin_safe(a.info, 0):
            continue   # a truncation decision within rounding of flipping: either answer is the oracle's
        assert np.linalg.norm(a.basis - b.basis) <= t * np.linalg.norm(a.basis)


def _fem_solution(o, load):
    F = o.fem_rhs(load)
    u, _ = o.fem_solve(F)
    o.compute_basis()
    K, C, _ = o.assemble_global_matrix()
    uc, _ = o.solve_coarse(K, C.T @ F, direct=True)
    return u, C @ uc


def test_mirror_symmetry_pins_off_diagonal_orientation():
    dim, ref, r = 2, 2, 3
    nl = 2 ** r
    t = laminate(dim, r, contrast=20.0, angle=0.4)
    # transpose the coefficient grid and swap a_xx, a_yy (a_xy stays: the mirror x <-> y keeps it)
    tm = t.reshape(nl, nl, 3).transpose(1, 0, 2).reshape(-1, 3)[:, [1, 0, 2]]
    load = lambda p: (1.0 + p[:, 0] + 3.0 * p[:, 1] ** 2)[:, None]
    load_m = lambda p: (1.0 + p[:, 1] + 3.0 * p[:, 0] ** 2)[:, None]
    u, us = _fem_solution(make_oracle(dim, ref, 2, 1, True, r, t), load)
    um, usm = _fem_solution(make_oracle(dim, ref, 2, 1, True, r, tm), load_m)
    G = 2 ** ref * 2 + 1
    tr = lambda v: v.reshape(G, G).T.ravel()
    assert np.abs(tr(u) - um).max() <= 1e-12 * np.abs(u).max()
    assert np.abs(tr(us) - usm).max() <= 1e-10 * np.abs(us).max()
    # with a_xy negated instead the solution is a different one: the test sees the off-diagonal term's sign
    tn = tm.copy()
    tn[:, 2] *= -1.0
    un, _ = _fem_solution(make_oracle(dim, ref, 2, 1, True, r, tn), load_m)
    assert np.abs(tr(u) - un).max() > 1e-3 * np.abs(u).max()


# constant tensors with non-zero off-diagonal entries, and the refinements of the manufactured-solution test
MANUFACTURED = {2: ([[2.0, 0.7], [0.7, 1.0]], (1, 2, 3)),
                3: ([[2.0, 0.3, 0.5], [0.3, 1.5, -0.6], [0.5, -0.6, 1.0]], (1, 2))}


def manufactured_errors(dim, solve, scale_off_diagonal=1.0):
    """Max nodal error of the fine FEM against u = prod sin(pi x_a) for each refinement; solve(ref, tensors, F) -> u_h.
    The off-diagonal components can be scaled to show that the test sees their factor."""
    A, refs = MANUFACTURED[dim]
    A = np.array(A)
    u, f = manufactured(dim, A)
    t = np.array([[A[a, b] for a, b in VOIGT[dim]]])
    t[:, dim:] *= scale_off_diagonal
    errs = []
    for ref in refs:
        F = make_oracle(dim, ref, 2, 1, True, 0, t).fem_rhs(lambda p: f(p)[:, None])
        uh = solve(ref, t, F)
        errs.append(np.abs(uh - u(grid_points(dim, 2 ** ref * 2 + 1))).max())
    return errs


def oracle_fem(dim):
    return lambda ref, t, F: make_oracle(dim, ref, 2, 1, True, 0, t).fem_solve(F)[0]


@pytest.mark.parametrize("dim", [2, 3])
def test_manufactured_solution_pins_component_factors(dim):
    """Second order in h (Q1 nodal error) only if every component, a_xy included, enters with the right factor: with
    the off-diagonal part halved the error stalls (measured: rates 1.7 then 1.0 in 2-D)."""
    errs = manufactured_errors(dim, oracle_fem(dim))
    for e0, e1 in zip(errs, errs[1:]):
        assert 3.8 < e0 / e1 < 4.3, errs
    wrong = manufactured_errors(dim, oracle_fem(dim), scale_off_diagonal=0.5)
    assert wrong[-1] / wrong[-2] < 2.0 and wrong[-1] > 2.0 * errs[-1], wrong


def laminate_errors(ell, dim=2, ref=3):
    o = make_oracle(dim, ref, 2, ell, True, ref + 1, laminate(dim, ref + 1))
    o.compute_basis()
    K, C, _ = o.assemble_global_matrix()
    F = o.fem_rhs(lambda p: np.ones((len(p), 1)))
    u_fem, A = o.fem_solve(F)
    u, _ = o.solve_coarse(K, C.T @ F, direct=True)
    e = C @ u - u_fem
    return math.sqrt(e @ (A @ e)) / math.sqrt(u_fem @ (A @ u_fem))


# relative energy errors of SLOD against the fine FEM, rotated laminate of contrast 100, 8^2 cells, n = 2
LAMINATE_ERRORS_2D = {1: 7.804e-1, 2: 7.000e-2, 3: 6.709e-5}


def test_laminate_error_decays_superexponentially():
    errs = {ell: laminate_errors(ell) for ell in (1, 2, 3)}
    for ell, want in LAMINATE_ERRORS_2D.items():
        assert errs[ell] == pytest.approx(want, rel=1e-3), (ell, errs[ell])
    assert errs[2] < errs[1] / 10.0 and errs[3] < errs[2] / 100.0   # the gain per layer grows


# ---- C ABI on a maps-only handle ----

def _maps_only(dim, problem=pkg.PROBLEM_DIFFUSION_TENSOR, spacedim=1):
    return pkg.SlodContext(dim=dim, spacedim=spacedim, n_global_refinements=2, n_subdivisions=2, oversampling=1,
                           problem=problem, device=-2)


@pytest.mark.parametrize("dim", [2, 3])
def test_tensor_problem_accepted(dim):
    ctx = _maps_only(dim)
    assert ctx.n_patches == 4 ** dim
    for s in (2, 3):
        with pytest.raises(pkg.SlodError) as e:
            _maps_only(dim, spacedim=s)
        assert e.value.code == 1


@pytest.mark.parametrize("dim", [2, 3])
def test_set_coefficient_tensor_refusals(dim):
    ctx = _maps_only(dim)
    nc = len(VOIGT[dim])
    r = 3
    good = _isotropic(dim, np.ones((2 ** r) ** dim))

    def code(call):
        with pytest.raises(pkg.SlodError) as e:
            call()
        return e.value.code, str(e.value)

    assert code(lambda: ctx.set_coefficient_tensor(r, good[:-1]))[0] == 1
    bad = good.copy()
    bad[5, nc - 1] = np.nan
    c, msg = code(lambda: ctx.set_coefficient_tensor(r, bad))
    assert c == 1 and "cell 5" in msg
    bad = good.copy()
    bad[7, nc - 1] = 1.5          # |a_xy| > 1 with a_xx = a_yy = 1: indefinite
    c, msg = code(lambda: ctx.set_coefficient_tensor(r, bad))
    assert c == 1 and "cell 7" in msg and "positive definite" in msg
    bad = good.copy()
    bad[2, 0] = 0.0               # a zero pivot
    c, msg = code(lambda: ctx.set_coefficient_tensor(r, bad))
    assert c == 1 and "cell 2" in msg
    # finer than the sub-cells (2^4 > 4 * 2): the Gauss-point mode is scalar only
    fine = _isotropic(dim, np.ones((2 ** 4) ** dim))
    assert code(lambda: ctx.set_coefficient_tensor(4, fine))[0] == 2
    # a valid table passes every check and stops at the device
    assert code(lambda: ctx.set_coefficient_tensor(r, good))[0] == 3
    # the per-field call on a tensor handle names the right call
    c, msg = code(lambda: ctx.set_coefficient(0, r, np.ones((2 ** r) ** dim)))
    assert c == 1 and "slod_set_coefficient_tensor" in msg
    # and the tensor call on a scalar handle
    sc = _maps_only(dim, problem=pkg.PROBLEM_DIFFUSION)
    c, msg = code(lambda: sc.set_coefficient_tensor(r, good))
    assert c == 1 and "slod_set_coefficient" in msg


def test_plan_of_tensor_handles():
    # cfg-4 geometry (3-D, 32^3 cells, n = 2, l = 2): the split solver stages one field at a time and stays available
    p3 = pkg.SlodContext(dim=3, n_global_refinements=5, n_subdivisions=2, oversampling=2, stabilize=True,
                         problem=pkg.PROBLEM_DIFFUSION_TENSOR, device=-2).plan()
    s3 = pkg.SlodContext(dim=3, n_global_refinements=5, n_subdivisions=2, oversampling=2, stabilize=True,
                         device=-2).plan()
    assert p3 == s3 and p3["split_solver"] == 1


@pytest.mark.parametrize("ell", [1, 2])
def test_large_3d_tensor_patches_are_planned(ell):
    # 3-D, 4 subdivisions: six fields of the coefficient window fit no shared-memory plan at l = 2 (384 KB); the SIMT
    # solver, the SIMT dense stage and k_patch_finish then read it from global memory, and the handle is accepted with
    # the scalar handle's plan
    kw = dict(dim=3, n_global_refinements=3, n_subdivisions=4, oversampling=ell, stabilize=True, device=-2)
    pt = pkg.SlodContext(problem=pkg.PROBLEM_DIFFUSION_TENSOR, **kw).plan()
    assert pt["mma_variant"] == -1 and pt["gmem_window"] == 1
    if ell == 2:
        assert pt == pkg.SlodContext(**kw).plan()
