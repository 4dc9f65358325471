"""Tensor diffusion (SLOD_PROBLEM_DIFFUSION_TENSOR) on the GPU against the reference restatement (tools/aniso_oracle.py):
basis and K in every kernel plan a tensor handle can take, an isotropic tensor against the scalar problem, the fine
reference problem and the method's decay with a laminate, the incremental update, and two GPUs."""
import math
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from aniso_oracle import VOIGT, laminate, make_oracle  # noqa: E402
from parity_common import check_plan, margin_safe, patch_tolerance, pkg, selection_sensitivity  # noqa: E402
from oracle.slod_oracle import CoefficientTable, SlodOracle, SlodProblem  # noqa: E402

pytestmark = pytest.mark.gpu

T = pkg.PROBLEM_DIFFUSION_TENSOR


def _ctx(dim, ref, n, ell, stabilize, quirk=False, problem=T, n_gpus=0):
    return pkg.SlodContext(dim=dim, spacedim=1, n_global_refinements=ref, n_subdivisions=n, oversampling=ell,
                           stabilize=stabilize, problem=problem, quirk_presaved=quirk, n_gpus=n_gpus)


def _isotropic(dim, alpha):
    t = np.zeros((alpha.size, len(VOIGT[dim])))
    t[:, :dim] = alpha[:, None]
    return t


def _compare(ctx, orc):
    """The criterion of tests/test_parity_gpu.py: 1e-10 where the selection is well conditioned, else 50 x the change a
    few-ulp perturbation of G causes in the oracle's answer; patches whose truncation decision is within rounding of
    flipping are not comparable; K entries against the tolerances of the two rows' bases."""
    ctx.compute_basis()
    ctx.assemble_coarse()
    orc.compute_basis()
    tol_of = {}
    for res in orc.patches:
        phi, aphi = ctx.basis(res.pid)
        assert ctx.diagnostics(res.pid)[7] == 0
        if not margin_safe(res.info, 0):
            tol_of[res.pid] = None
            continue
        err = np.linalg.norm(phi - res.basis[0])
        tol = 1e-10
        if err > tol and res.info["slod"]:
            tol = max(tol, 50.0 * selection_sensitivity(res.info, 0))
        tol_of[res.pid] = tol
        assert err <= tol, (res.pid, err, tol)
        ref = res.basis_premultiplied[0]
        assert np.linalg.norm(aphi - ref) <= 10 * tol * np.linalg.norm(ref), res.pid
    K, _, _ = orc.assemble_global_matrix()
    rowptr, col, val = ctx.coarse_csr()
    assert np.array_equal(rowptr, K.indptr) and np.array_equal(col, K.indices)
    rows = np.repeat(np.arange(K.shape[0]), np.diff(K.indptr))
    tol_row = np.array([tol_of.get(r) or np.inf for r in range(K.shape[0])])
    assert (np.abs(val - K.data) <= 20 * (tol_row[rows] + tol_row[col]) * np.abs(K.data).max()).all()


# (dim, ref, n, ell, stabilize, quirk, environment, plan entries the case exists to run)
CASES = [
    (2, 3, 2, 1, True, False, {}, {"mma_variant": 1}),
    (2, 3, 2, 3, True, False, {}, {"mma_variant": 2}),
    (2, 3, 2, 1, False, False, {}, {}),
    (2, 3, 2, 1, True, True, {}, {}),
    (2, 3, 2, 1, True, False, {"SLOD_FORCE_SIMT_SOLVER": "1"}, {"mma_variant": -1}),
    (2, 3, 2, 1, True, False, {"SLOD_FORCE_SIMT_DENSE": "1"}, {"dense_ntile": 0}),
    (3, 2, 2, 1, True, False, {}, {"mma_variant": 0, "split_solver": 0}),     # fused solver: l = 1 has no split plan
    (3, 3, 2, 2, True, False, {}, {"split_solver": 1}),
    # at l = 2 six fields do not fit the fused solver's shared memory: the plan drops to the global-memory SIMT solver
    (3, 3, 2, 2, True, False, {"SLOD_FUSED_SOLVER": "1"}, {"split_solver": 0, "mma_variant": -1, "gmem_window": 1}),
    (3, 2, 2, 1, True, False, {"SLOD_FORCE_GMEM_SOLVER": "1"}, {"mma_variant": -1, "gmem_window": 1}),
    (3, 2, 2, 1, False, False, {"SLOD_FORCE_SIMT_DENSE": "1"}, {"dense_ntile": 0}),
]


@pytest.mark.parametrize("dim,ref,n,ell,stabilize,quirk,env,plan", CASES)
def test_parity_with_oracle(monkeypatch, dim, ref, n, ell, stabilize, quirk, env, plan):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    r = ref + int(math.log2(n))
    t = laminate(dim, r, contrast=50.0, seed=ref + ell)
    ctx = _ctx(dim, ref, n, ell, stabilize, quirk)
    ctx.set_coefficient_tensor(r, t)
    check_plan(ctx, plan)
    _compare(ctx, make_oracle(dim, ref, n, ell, stabilize, r, t, quirk_presaved=quirk))


@pytest.mark.parametrize("stabilize", [False, True])
@pytest.mark.parametrize("dim,ref,ell", [(2, 3, 2), (3, 3, 2)])
def test_isotropic_tensor_matches_scalar_handle(dim, ref, ell, stabilize):
    r = ref + 1
    alpha = 1.0 + 99.0 * np.random.default_rng(5).random((2 ** r) ** dim)
    sc = _ctx(dim, ref, 2, ell, stabilize, problem=pkg.PROBLEM_DIFFUSION)
    sc.set_coefficient(0, r, alpha)
    te = _ctx(dim, ref, 2, ell, stabilize)
    te.set_coefficient_tensor(r, _isotropic(dim, alpha))
    assert sc.plan() == te.plan()
    out = []
    for c in (sc, te):
        c.compute_basis()
        c.assemble_coarse()
        phi, aphi = c.all_basis()
        out.append((phi.copy(), aphi.copy(), c.coarse_csr()[2].copy()))
    if not stabilize:
        # LOD branch everywhere: phi, A phi and K to 1e-12
        for a, b in zip(out[0], out[1]):
            assert np.abs(a - b).max() <= 1e-12 * np.abs(a).max()
        return
    # The SLOD selection amplifies the rounding difference of the two sums (sum_f a_f K_f against alpha K) with its
    # conditioning: phi and A phi per patch and K per row to the bound of tests/test_aniso_cpu.py, from the scalar
    # oracle's selection data (1e-12 on LOD-branch patches, else 1e-10 or 2000 eps cond_eff); patches whose truncation
    # decision is within rounding of flipping are not comparable.  The stages up to the Gram matrix agree to 1e-12.
    orc = SlodOracle(SlodProblem(dim=dim, spacedim=1, n_global_refinements=ref, n_subdivisions=2, oversampling=ell,
                                 stabilize=True, coefficients=[CoefficientTable(dim, r, alpha)]))
    orc.compute_basis()
    tol = np.full(sc.n_patches, np.inf)
    for res in orc.patches:
        if margin_safe(res.info, 0):
            tol[res.pid] = patch_tolerance(res.info, 0, c=2000.0) if res.info["slod"] else 1e-12
    ok = np.isfinite(tol)
    assert ok.sum() >= sc.n_patches // 2
    for a, b in zip(out[0][:2], out[1][:2]):
        err = np.linalg.norm((a - b)[:, 0], axis=1)
        assert (err[ok] <= tol[ok] * np.linalg.norm(a[:, 0], axis=1)[ok]).all()
    rowptr, _, _ = sc.coarse_csr()
    rows = np.repeat(np.arange(sc.n_patches), np.diff(rowptr))
    col = sc.coarse_csr()[1]
    both = ok[rows] & ok[col]
    assert (np.abs(out[0][2] - out[1][2])[both] <= (20 * (tol[rows] + tol[col]))[both] * np.abs(out[0][2]).max()).all()
    for pid in np.arange(0, sc.n_patches, 37):
        for x, y in zip(sc.debug_stages(pid), te.debug_stages(pid)):
            assert np.abs(x - y).max() <= 1e-12 * np.abs(x).max(), pid


def _laminate_errors_gpu(dim, ref, ell):
    r = ref + 1
    t = laminate(dim, r)
    ctx = _ctx(dim, ref, 2, ell, True)
    ctx.set_coefficient_tensor(r, t)
    ctx.compute_basis()
    ctx.assemble_coarse()
    orc = make_oracle(dim, ref, 2, ell, True, r, t)
    F = orc.fem_rhs(lambda p: np.ones((len(p), 1)))
    u_fem, _, _ = ctx.fem_solve(F)
    u = ctx.prolongate(ctx.coarse_solve(ctx.coarse_rhs(F))[0])
    return ctx, orc, F, u_fem, u


def test_fem_and_laminate_errors_2d():
    from test_aniso_cpu import LAMINATE_ERRORS_2D
    for ell in (1, 2, 3):
        ctx, orc, F, u_fem, u = _laminate_errors_gpu(2, 3, ell)
        if ell == 1:
            u_ref, A = orc.fem_solve(F)
            assert np.abs(u_fem - u_ref).max() <= 1e-8 * np.abs(u_ref).max()
            en = ctx.fine_norms(u_ref)[2]
            assert en == pytest.approx(math.sqrt(u_ref @ (A @ u_ref)), rel=1e-10)
        err = ctx.fine_norms(u - u_fem)[2] / ctx.fine_norms(u_fem)[2]
        # the pins carry four digits (rounding <= 6.5e-4 relative); the CG solves stop at 1e-10 / 1e-12
        assert err == pytest.approx(LAMINATE_ERRORS_2D[ell], rel=1e-3), (ell, err)


def test_laminate_errors_decrease_3d():
    errs = []
    for ell in (1, 2):
        ctx, _, _, u_fem, u = _laminate_errors_gpu(3, 3, ell)
        errs.append(ctx.fine_norms(u - u_fem)[2] / ctx.fine_norms(u_fem)[2])
    assert errs[1] < errs[0] / 5.0, errs


@pytest.mark.parametrize("dim,ref,ell", [(2, 4, 2), (3, 3, 2)])
def test_update_after_one_cell_matches_fresh(dim, ref, ell):
    r = ref
    t = laminate(dim, r, contrast=30.0)
    ctx = _ctx(dim, ref, 2, ell, True)
    ctx.set_coefficient_tensor(r, t)
    ctx.compute_basis()
    ctx.assemble_coarse()
    t2 = t.copy()
    c = (2 ** r) ** dim // 2 + 3
    t2[c, -1] += 0.05          # only the off-diagonal entry of one coarse cell changes
    ctx.set_coefficient_tensor(r, t2)
    got = ctx.update_basis()
    from update_expect import expected_patches
    comps = lambda tt: [tt[:, f] for f in range(tt.shape[1])]
    assert got["patches"] == len(expected_patches(ctx, dim, ref, 2, ell, (comps(t), r), (comps(t2), r)))
    phi_u, aphi_u = [a.copy() for a in ctx.all_basis()]
    K_u = ctx.coarse_csr()[2].copy()
    fresh = _ctx(dim, ref, 2, ell, True)
    fresh.set_coefficient_tensor(r, t2)
    fresh.compute_basis()
    fresh.assemble_coarse()
    phi_f, aphi_f = fresh.all_basis()
    assert np.array_equal(phi_u, phi_f) and np.array_equal(aphi_u, aphi_f)
    assert np.array_equal(K_u, fresh.coarse_csr()[2])


def test_two_gpus_bit_identical():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    r, dim, ref, ell = 3, 3, 3, 1
    t = laminate(dim, r)
    out = []
    for g in (0, 2):
        ctx = _ctx(dim, ref, 2, ell, True, n_gpus=g)
        ctx.set_coefficient_tensor(r, t)
        ctx.compute_basis()
        ctx.assemble_coarse()
        phi, aphi = ctx.all_basis()
        out.append((phi.copy(), aphi.copy(), ctx.coarse_csr()[2].copy()))
    for a, b in zip(*out):
        assert np.array_equal(a, b)


def test_large_3d_patches_coefficient_window_in_global_memory():
    """3-D, 4 subdivisions, oversampling 2: six fields of a 20^3 sub-cell window (384 KB) fit no shared-memory plan.
    The SIMT solver (global-memory windows), the SIMT dense stage and k_patch_finish read the window from a per-CTA
    global scratch; the scalar handle of the same geometry has the same plan."""
    dim, ref, n, ell = 3, 3, 4, 2
    r = ref + 2
    t = laminate(dim, r, contrast=20.0)
    ctx = _ctx(dim, ref, n, ell, True)
    ctx.set_coefficient_tensor(r, t)
    check_plan(ctx, {"mma_variant": -1, "gmem_window": 1, "dense_coef_gmem": 1})
    ctx.compute_basis()
    ctx.assemble_coarse()
    full = next(p for p in range(ctx.n_patches) if ctx.patch_info(p)["n_cells"] == 125)
    orc = make_oracle(dim, ref, n, ell, True, r, t)
    orc.compute_basis([0, full, ctx.n_patches - 1])
    for res in orc.patches:
        phi, aphi = ctx.basis(res.pid)
        assert ctx.diagnostics(res.pid)[7] == 0
        if not margin_safe(res.info, 0):
            continue
        tol = max(1e-10, 50.0 * selection_sensitivity(res.info, 0))
        assert np.linalg.norm(phi - res.basis[0]) <= tol, (res.pid, tol)
        ref_a = res.basis_premultiplied[0]
        assert np.linalg.norm(aphi - ref_a) <= 10 * tol * np.linalg.norm(ref_a)


@pytest.mark.parametrize("dim", [2, 3])
def test_fem_solve_manufactured_solution(dim):
    """slod_fem_solve on a tensor handle converges at second order to the manufactured solution, like the oracle's fine
    FEM: the factor of every component, a_xy included, is right in k_fine_apply."""
    from test_aniso_cpu import manufactured_errors, oracle_fem

    def gpu(ref, t, F):
        ctx = _ctx(dim, ref, 2, 1, True)
        ctx.set_coefficient_tensor(0, t)
        return ctx.fem_solve(F)[0]
    errs = manufactured_errors(dim, gpu)
    want = manufactured_errors(dim, oracle_fem(dim))
    assert np.allclose(errs, want, rtol=1e-6), (errs, want)
    for e0, e1 in zip(errs, errs[1:]):
        assert 3.8 < e0 / e1 < 4.3, errs
