"""GPU tests of the coarse mass matrix, the L2 projection and backward Euler on the SLOD space
(slod_assemble_coarse_mass, slod_l2_project_batch, slod_heat_solve / _batch, slod_fem_heat_solve).

Operator-level checks use the GPU's own basis and matrices in the reference formulas of tools/heat_oracle.py, so that the
new kernels are tested at rounding level whatever the conditioning of the basis selection; the oracle's own basis is
compared at basis accuracy (the discrepancy K itself shows)."""
import ctypes as C
import os
import sys

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from heat_oracle import coarse_mass, heat_solve_coarse, heat_solve_fine  # noqa: E402
from parity_common import build_pair, case_id, pkg  # noqa: E402
from test_online_gpu import _forcing, _host_C  # noqa: E402

pytestmark = pytest.mark.gpu

CASES = [
    dict(dim=2, s=1, ref=3, n=2, ell=1),
    dict(dim=2, s=1, ref=3, n=2, ell=2),
    dict(dim=2, s=2, ref=3, n=2, ell=1),
    dict(dim=2, s=2, ref=3, n=2, ell=2),
    dict(dim=3, s=1, ref=2, n=2, ell=1),
    dict(dim=3, s=1, ref=2, n=2, ell=2),
    # wide ELL rows (361 and 450 slots: k_ell_residual and the CG kernels over several 128-entry passes plus a tail) and
    # one coefficient per Gauss point
    dict(dim=2, s=1, ref=4, n=2, ell=4, plan=dict(mma_variant=0, dense_ntile=16)),
    dict(dim=2, s=2, ref=3, n=2, ell=3, plan=dict(mma_variant=0, dense_ntile=16)),
    dict(dim=2, s=1, ref=3, n=2, ell=1, r=5, plan=dict(gauss_coef=1)),
]
IDS = [case_id(c) for c in CASES]
CG = dict(max_steps=5000, tolerance=0.0, reduction=1e-13)
DP = C.POINTER(C.c_double)


def _dp(a):
    return None if a is None else a.ctypes.data_as(DP)


def _rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def _csr(t, n):
    rowptr, col, val = t
    return sp.csr_matrix((val.copy(), col.copy(), rowptr.copy()), shape=(n, n))


def _ready(case):
    ctx, orc = build_pair(**case)
    ctx.compute_basis()
    ctx.assemble_coarse()
    ctx.assemble_coarse_mass()
    nc = ctx.n_patches * ctx.s
    return ctx, orc, _csr(ctx.coarse_csr(), nc), _csr(ctx.coarse_mass_csr(), nc)


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_coarse_mass_matrix(case):
    """M_H against the oracle's formula on the GPU's own phi (rounding level), its pattern, symmetry and definiteness, and
    against the oracle's own M_H at the accuracy K shows."""
    ctx, orc, K, M = _ready(case)
    Cm = _host_C(ctx, case["n"], case["s"], case["ref"])
    M_ref = coarse_mass(orc, Cm)
    assert np.array_equal(M.indptr, K.indptr) and np.array_equal(M.indices, K.indices)
    assert np.array_equal(M_ref.indptr, M.indptr) and np.array_equal(M_ref.indices, M.indices)
    scale = np.abs(M.data).max()
    assert np.abs(M.data - M_ref.data).max() <= 1e-14 * scale
    assert np.abs((M - M.T).toarray()).max() <= 1e-14 * scale
    assert np.linalg.eigvalsh(M.toarray()).min() > 0.0
    orc.compute_basis()
    K_o, C_o, _ = orc.assemble_global_matrix()
    err_K = np.abs(K.data - K_o.data).max() / np.abs(K_o.data).max()
    err_M = np.abs(M.data - coarse_mass(orc, C_o).data).max() / scale
    assert err_M <= max(1e-10, 10.0 * err_K), (err_M, err_K)
    ctx.close()


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_l2_projection(case):
    """A function of the space projects onto itself; a general field gives M_H^-1 C^T M_h v (scipy, GPU's own M_H)."""
    ctx, orc, _, M = _ready(case)
    nc = ctx.n_patches * ctx.s
    rng = np.random.default_rng(2)
    U = rng.standard_normal((3, nc))
    P, steps, res = ctx.l2_project_batch(ctx.prolongate_batch(U), **CG)
    assert np.linalg.norm(P - U) <= 1e-9 * np.linalg.norm(U)
    assert (steps > 0).all()
    V = rng.standard_normal((2, ctx.n_fine))
    P, _, _ = ctx.l2_project_batch(V, **CG)
    Cm = _host_C(ctx, case["n"], case["s"], case["ref"])
    Mh = orc.fine_norm_matrices()[0]
    solve = spla.factorized(M.tocsc())
    for j in range(2):
        ref = solve(Cm.T @ (Mh @ V[j]))
        assert np.linalg.norm(P[j] - ref) <= 1e-9 * np.linalg.norm(ref)
    ctx.close()


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_heat_trajectories(case):
    """heat_solve and heat_solve_batch against the direct increment scheme on the GPU's own K and M_H at every output,
    fem_heat_solve against the oracle's fine trajectory (it needs only the coefficient)."""
    ctx, orc, K, M = _ready(case)
    rng = np.random.default_rng(7)
    F = orc.fem_rhs(_forcing(case["s"]))
    u0 = rng.standard_normal(ctx.n_patches * ctx.s)
    dt, n_steps, every = 1e-2, 6, 2
    U, st = ctx.heat_solve(F, u0, dt, n_steps, every, **CG)
    Ub, stb = ctx.heat_solve_batch(F[None], u0[None], dt, n_steps, every, **CG)
    ref = heat_solve_coarse(K, M, ctx.coarse_rhs(F), u0, dt, n_steps)[every - 1::every]
    assert U.shape == (3, u0.size) and Ub.shape == (3, 1, u0.size) and st.shape == (6,) and stb.shape == (6, 1)
    for o in range(3):
        assert np.linalg.norm(U[o] - ref[o]) <= 1e-9 * np.linalg.norm(ref[o])
        assert np.linalg.norm(Ub[o, 0] - ref[o]) <= 1e-9 * np.linalg.norm(ref[o])
    assert (st > 0).all() and (np.abs(st - stb[:, 0]) <= 1).all()
    u0f = ctx.prolongate(u0)
    Uf, stf = ctx.fem_heat_solve(F, u0f, dt, n_steps, every, max_steps=200000, tolerance=0.0, reduction=1e-13)
    ref_f = heat_solve_fine(orc, F, u0f, dt, n_steps)[every - 1::every]
    for o in range(3):
        assert np.linalg.norm(Uf[o] - ref_f[o]) <= 1e-9 * np.linalg.norm(ref_f[o])
    assert (stf > 0).all()
    ctx.close()


def _heat_batch_case():
    ctx, orc = build_pair(dim=2, s=1, ref=4, n=2, ell=2)
    ctx.compute_basis()
    ctx.assemble_coarse()
    ctx.assemble_coarse_mass()
    return ctx, orc


def test_heat_batch_independence():
    """n_rhs = 37 (three groups): a column is bit-identical across runs, permutations and n_rhs = 1; the single-vector
    form agrees with it to the solver tolerance."""
    ctx, _ = _heat_batch_case()
    rng = np.random.default_rng(5)
    k, nc = 37, ctx.n_patches
    F = rng.standard_normal((k, ctx.n_fine)) * np.logspace(-3, 3, k)[:, None]
    U0 = rng.standard_normal((k, nc))
    F[7] = 0.0
    U0[7] = 0.0
    args = (2e-3, 5, 1)
    U, st = ctx.heat_solve_batch(F, U0, *args, **CG)
    U2, st2 = ctx.heat_solve_batch(F, U0, *args, **CG)
    assert np.array_equal(U, U2) and np.array_equal(st, st2)
    assert not U[:, 7].any() and not st[:, 7].any()
    perm = rng.permutation(k)
    Up, stp = ctx.heat_solve_batch(F[perm], U0[perm], *args, **CG)
    assert np.array_equal(Up, U[:, perm]) and np.array_equal(stp, st[:, perm])
    for j in (0, 15, 16, 17, 36):
        u1, s1 = ctx.heat_solve_batch(F[j:j + 1], U0[j:j + 1], *args, **CG)
        assert np.array_equal(u1[:, 0], U[:, j]) and np.array_equal(s1[:, 0], st[:, j])
        us, ss = ctx.heat_solve(F[j], U0[j], *args, **CG)
        assert np.linalg.norm(us - U[:, j]) <= 1e-9 * np.linalg.norm(U[:, j])
        assert (np.abs(ss - st[:, j]) <= 1).all()
    ctx.close()


def test_heat_reaches_steady_state():
    """With dt >> the slowest time scale a few steps reach the elliptic solution K^-1 C^T f."""
    ctx, orc = _heat_batch_case()
    F = orc.fem_rhs(_forcing(1))
    U, _ = ctx.heat_solve(F, None, 1e4, 8, 8, **CG)
    u_inf, _, _ = ctx.coarse_solve(ctx.coarse_rhs(F), **CG)
    assert np.linalg.norm(U[0] - u_inf) <= 1e-9 * np.linalg.norm(u_inf)
    ctx.close()


def test_slod_trajectory_error_decays():
    """The prolongated SLOD trajectory against fem_heat_solve: the oracle's decay in the oversampling (tests/
    test_heat_cpu.py: energy error 1.16e-1 / 8.9e-4 at t = 0.2 for l = 1 / 2)."""
    errs = []
    for ell in (1, 2):
        rs = np.random.default_rng(11)
        tab = 1.0 + 99.0 * rs.random(16 ** 2)
        ctx = pkg.SlodContext(dim=2, spacedim=1, n_global_refinements=3, n_subdivisions=2, oversampling=ell,
                              stabilize=True)
        ctx.set_coefficient(0, 4, tab)
        ctx.compute_basis()
        ctx.assemble_coarse()
        ctx.assemble_coarse_mass()
        G = 8 * 2 + 1
        F = np.full((G, G), (1.0 / 16) ** 2)
        U, _ = ctx.heat_solve(F.ravel(), None, 1e-2, 20, 20, **CG)
        Uf, _ = ctx.fem_heat_solve(F.ravel(), None, 1e-2, 20, 20, reduction=1e-13)
        e = ctx.fine_norms(ctx.prolongate(U[0]) - Uf[0])[2] / ctx.fine_norms(Uf[0])[2]
        errs.append(e)
        ctx.close()
    print("SLOD trajectory energy error at t = 0.2, l = 1, 2:", errs)
    assert 0.05 < errs[0] < 0.2 and 4e-4 < errs[1] < 2e-3 and errs[1] < errs[0] / 20.0


def test_heat_errors():
    """Call order (stale M_H / S after a new basis or K), argument checks."""
    ctx, _ = build_pair(dim=2, s=1, ref=3, n=2, ell=1)
    nf, nc = ctx.n_fine, ctx.n_patches
    F, u0 = np.ones(nf), np.zeros(nc)

    def code(call):
        with pytest.raises(pkg.SlodError) as ei:
            call()
        return ei.value.code

    assert code(ctx.assemble_coarse_mass) == 4
    assert code(lambda: ctx.heat_solve(F, u0, 1e-2, 2)) == 4
    ctx.compute_basis()
    assert code(lambda: ctx.l2_project_batch(np.ones((1, nf)))) == 4
    assert code(ctx.coarse_mass_csr) == 4
    ctx.assemble_coarse_mass()
    assert code(lambda: ctx.heat_solve(F, u0, 1e-2, 2)) == 4          # no K yet
    ctx.assemble_coarse()                                             # a new K makes M_H (and S) stale
    for call in (lambda: ctx.heat_solve(F, u0, 1e-2, 2), lambda: ctx.heat_solve_batch(F[None], None, 1e-2, 2),
                 lambda: ctx.l2_project_batch(np.ones((1, nf))), ctx.coarse_mass_csr):
        assert code(call) == 4
    ctx.assemble_coarse_mass()
    ref, _ = ctx.heat_solve(F, u0, 1e-2, 2, **CG)
    ctx.compute_basis()                                               # so does a new basis
    assert code(lambda: ctx.heat_solve(F, u0, 1e-2, 2)) == 4
    ctx.assemble_coarse()
    ctx.assemble_coarse_mass()
    again, _ = ctx.heat_solve(F, u0, 1e-2, 2, **CG)
    assert np.array_equal(ref, again)
    out = np.zeros(4 * nc)
    lib, h = ctx.lib, ctx.h
    for dt, n_steps, every in ((0.0, 2, 1), (-1e-2, 2, 1), (float("nan"), 2, 1), (1e-2, 0, 1), (1e-2, 2, 0),
                               (1e-2, 2, 3)):
        assert lib.slod_heat_solve(h, _dp(F), _dp(u0), dt, n_steps, every, _dp(out), 100, 0.0, 1e-10, None) == 1
        assert lib.slod_heat_solve_batch(h, 1, _dp(F), _dp(u0), dt, n_steps, every, _dp(out), 100, 0.0, 1e-10,
                                         None) == 1
        assert lib.slod_fem_heat_solve(h, _dp(F), None, dt, n_steps, every, _dp(np.zeros(4 * nf)), 100, 0.0, 1e-10,
                                       None) == 1
    assert lib.slod_heat_solve_batch(h, 0, _dp(F), _dp(u0), 1e-2, 2, 1, _dp(out), 100, 0.0, 1e-10, None) == 1
    assert lib.slod_heat_solve(h, _dp(F), _dp(u0), 1e-2, 2, 1, None, 100, 0.0, 1e-10, None) == 1
    assert lib.slod_l2_project_batch(h, 0, _dp(F), _dp(out), 100, 0.0, 1e-10, None, None) == 1
    ctx.close()


def test_heat_cg_failure_names_step_and_column():
    """Column 1 starts where the increment of step 1 is an eigenvector of the Jacobi-preconditioned M_H + dt K: CG needs
    one step there and many at step 2.  With max_steps set to step 1's count, step 2 fails: the error names step 2 and
    column 1, and the outputs of step 1 are written."""
    ctx, _ = build_pair(dim=2, s=1, ref=3, n=2, ell=1)
    ctx.compute_basis()
    ctx.assemble_coarse()
    ctx.assemble_coarse_mass()
    nc, dt = ctx.n_patches, 1e-2
    K = _csr(ctx.coarse_csr(), nc).toarray()
    S = _csr(ctx.coarse_mass_csr(), nc).toarray() + dt * K
    d = np.sqrt(np.diag(S))
    _, vec = np.linalg.eigh(S / d[:, None] / d[None, :])
    U0 = np.zeros((3, nc))
    for j, m in ((1, nc // 2), (2, nc // 3)):
        r = d * vec[:, m]                                  # S D^-1 r = lambda r
        U0[j] = -np.linalg.solve(K, r) / dt                # so that dt (0 - K u0) = r
    ctl = dict(tolerance=0.0, reduction=1e-6)
    _, st = ctx.heat_solve_batch(None, U0, dt, 3, 1, max_steps=1000, **ctl)
    m = int(st[0].max())
    assert m <= 2 and st[1, 1] > m, st
    out = np.full((3, 3, nc), np.nan)
    cg = np.full((3, 3), -1, dtype=np.int32)
    rc = ctx.lib.slod_heat_solve_batch(ctx.h, 3, None, _dp(U0), dt, 3, 1, _dp(out), m, 0.0, 1e-6,
                                       cg.ctypes.data_as(C.POINTER(C.c_int32)))
    msg = ctx.lib.slod_last_error(ctx.h).decode()
    assert rc == 5 and "time step 2 column 1" in msg and "did not converge" in msg, msg
    ref, _ = ctx.heat_solve_batch(None, U0, dt, 1, 1, max_steps=1000, **ctl)
    assert np.array_equal(out[0], ref[0]) and np.isnan(out[1:]).all()
    assert (cg[0] == st[0]).all() and cg[1, 1] == m and (cg[2] == -1).all()
    # the single-vector form: step 2 named, step 1 written
    out1 = np.full((3, nc), np.nan)
    u0 = np.ascontiguousarray(U0[1])
    rc = ctx.lib.slod_heat_solve(ctx.h, None, _dp(u0), dt, 3, 1, _dp(out1), m, 0.0, 1e-6, None)
    msg = ctx.lib.slod_last_error(ctx.h).decode()
    assert rc == 5 and "time step 2:" in msg, msg
    assert np.isfinite(out1[0]).all() and np.isnan(out1[1:]).all()
    ctx.close()


def test_heat_after_checkpoint(tmp_path):
    """A restored handle needs M_H assembled again and then gives the same bits."""
    ctx, orc = _heat_batch_case()
    rng = np.random.default_rng(3)
    F = rng.standard_normal((4, ctx.n_fine))
    U0 = rng.standard_normal((4, ctx.n_patches))
    M1 = [a.copy() for a in ctx.coarse_mass_csr()]
    T1, s1 = ctx.heat_solve_batch(F, U0, 1e-2, 4, 2, **CG)
    path = str(tmp_path / "offline.slod")
    ctx.save_state(path)
    ctx.close()
    ctx2 = pkg.SlodContext(dim=2, spacedim=1, n_global_refinements=4, n_subdivisions=2, oversampling=2, stabilize=True)
    ctx2.load_state(path)
    with pytest.raises(pkg.SlodError) as ei:
        ctx2.heat_solve_batch(F, U0, 1e-2, 4, 2, **CG)
    assert ei.value.code == 4
    ctx2.assemble_coarse_mass()
    for a, b in zip(M1, ctx2.coarse_mass_csr()):
        assert np.array_equal(a, b)
    T2, s2 = ctx2.heat_solve_batch(F, U0, 1e-2, 4, 2, **CG)
    assert np.array_equal(T1, T2) and np.array_equal(s1, s2)
    ctx2.close()


def test_heat_two_gpus():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    from parity_common import make_tables
    tab = make_tables(2, 1, 6, "uniform100", 1234)[0]
    out = []
    for n_gpus in (1, 2):
        ctx = pkg.SlodContext(dim=2, spacedim=1, n_global_refinements=4, n_subdivisions=2, oversampling=2,
                              stabilize=True, n_gpus=n_gpus, device=0)
        ctx.set_coefficient(0, 6, tab)
        ctx.compute_basis()
        ctx.assemble_coarse()
        ctx.assemble_coarse_mass()
        rng = np.random.default_rng(4)
        F = rng.standard_normal((5, ctx.n_fine))
        out.append([a.copy() for a in ctx.coarse_mass_csr()] + list(ctx.heat_solve_batch(F, None, 1e-2, 3, 1, **CG))
                   + [ctx.l2_project_batch(F, **CG)[0].copy()])
        ctx.close()
    for a, b in zip(*out):
        assert np.array_equal(a, b)


def test_heat_full_size():
    """The headline workload (3-D, 32^3 cells, oversampling 2): M_H assembles, 10 backward-Euler steps run, and the
    energy error of the prolongated trajectory against the fine one is printed and bounded."""
    import bench
    w = bench.WORKLOADS[bench.DEFAULT_WORKLOAD]
    ctx = pkg.SlodContext(dim=w["dim"], spacedim=w["s"], n_global_refinements=w["ref"], n_subdivisions=w["n"],
                          oversampling=w["ell"], stabilize=True, problem=0 if w["s"] == 1 else 1)
    for f, t in enumerate(bench.make_tables(w)):
        ctx.set_coefficient(f, w["r"], t)
    ctx.compute_basis()
    ctx.assemble_coarse()
    ctx.assemble_coarse_mass()
    ms = ctx.timings()
    assert ms[6] > 0 and ms[7] > 0
    _, _, val = ctx.coarse_mass_csr()
    assert np.isfinite(val).all()
    G = 2 ** w["ref"] * w["n"] + 1
    h = 1.0 / (G - 1)
    F = np.full(ctx.n_fine, h ** 3)
    dt, n_steps = 1e-3, 10
    U, st = ctx.heat_solve(F, None, dt, n_steps, n_steps, **CG)
    Uf, stf = ctx.fem_heat_solve(F, None, dt, n_steps, n_steps, max_steps=200000, reduction=1e-12)
    e = ctx.fine_norms(ctx.prolongate(U[0]) - Uf[0])[2] / ctx.fine_norms(Uf[0])[2]
    print(f"full size: M_h phi {ms[6]:.2f} ms, M_H {ms[7]:.2f} ms; CG steps SLOD {st.tolist()} fine {stf.tolist()}; "
          f"energy error at t = {dt * n_steps:g}: {e:.3e}")
    assert e < 0.1
    ctx.close()
