"""GPU tests of the batched online phase (slod_coarse_rhs_batch / slod_coarse_solve_batch / slod_prolongate_batch):
rounding-level operator checks against C built on the host from the GPU's own basis, agreement with the single-vector
calls, bit-identity of a column however it is batched, per-column stopping, errors, checkpoint, end to end against the
oracle, and the full-size workload."""
import ctypes as C
import os
import sys

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from parity_common import build_pair, case_id, pkg  # noqa: E402
from test_online_gpu import END_TO_END, OPERATOR_CASES, _forcing, _host_C  # noqa: E402

pytestmark = pytest.mark.gpu

CG = dict(max_steps=5000, tolerance=0.0, reduction=1e-13)


def _rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def _ready(case):
    ctx, orc = build_pair(**case)
    ctx.compute_basis()
    ctx.assemble_coarse()
    return ctx, orc


def _K(ctx):
    rowptr, col, val = ctx.coarse_csr()
    n = ctx.n_patches * ctx.s
    return sp.csr_matrix((val.copy(), col.copy(), rowptr.copy()), shape=(n, n))


def _block(rng, k, n, zero=1, repeat=(3, 0)):
    """k random rows, row `zero` zero, row repeat[0] a copy of row repeat[1]."""
    F = rng.standard_normal((k, n))
    F[zero] = 0.0
    F[repeat[0]] = F[repeat[1]]
    return F


@pytest.mark.parametrize("case", OPERATOR_CASES, ids=case_id)
def test_batch_operators(case):
    """k = 5 with a zero and a repeated column (k = 17, two groups with the last one partial, on the cases added for a
    kernel plan): C^T F and C U at rounding level, the solve against scipy's direct solve on the GPU's own K, the true
    residual, and each column against the single-vector calls."""
    ctx, _ = _ready(case)
    Cm = _host_C(ctx, case["n"], case["s"], case["ref"])
    K = _K(ctx)
    rng = np.random.default_rng(11)
    k = 17 if "plan" in case else 5
    F = _block(rng, k, ctx.n_fine)
    B = ctx.coarse_rhs_batch(F)
    assert B.shape == (k, Cm.shape[1])
    U, steps, res = ctx.coarse_solve_batch(B, **CG)
    Ur = _block(rng, k, Cm.shape[1])
    Uf = ctx.prolongate_batch(Ur)
    solve = spla.factorized(K.tocsc())
    for j in range(k):
        b_ref = Cm.T @ F[j]
        uf_ref = Cm @ Ur[j]
        if j == 1:   # the zero column
            assert not B[j].any() and not Uf[j].any() and not U[j].any() and steps[j] == 0 and res[j] == 0.0
            continue
        assert _rel(B[j], b_ref) <= 1e-12
        assert _rel(Uf[j], uf_ref) <= 1e-12
        x_ref = solve(B[j])
        assert np.linalg.norm(U[j] - x_ref) <= 1e-9 * np.linalg.norm(x_ref)
        assert np.linalg.norm(K @ U[j] - B[j]) <= 1e-11 * np.linalg.norm(B[j])
        # against the single-vector entry points
        assert _rel(B[j], ctx.coarse_rhs(F[j])) <= 1e-12
        assert _rel(Uf[j], ctx.prolongate(Ur[j])) <= 1e-12
        u1, s1, _ = ctx.coarse_solve(B[j], **CG)
        assert np.linalg.norm(U[j] - u1) <= 1e-9 * np.linalg.norm(u1)
        assert abs(int(steps[j]) - s1) <= 1
    for X in (B, U, Uf):                       # the repeated column
        assert np.array_equal(X[3], X[0])
    assert steps[3] == steps[0] and res[3] == res[0]
    ctx.close()


def _chain(ctx, F, U_in, **cg):
    B = ctx.coarse_rhs_batch(F)
    U, steps, res = ctx.coarse_solve_batch(B, **cg)
    return B.copy(), U.copy(), steps.copy(), res.copy(), ctx.prolongate_batch(U_in).copy()


def test_batch_independence():
    """n_rhs = 37 (three groups, the last one partial): every column is bit-identical to the n_rhs = 1 call on it and to
    the same column in a permuted batch; two runs are bit-identical."""
    ctx, _ = _ready(dict(dim=2, s=1, ref=4, n=2, ell=2))
    rng = np.random.default_rng(5)
    k = 37
    F = rng.standard_normal((k, ctx.n_fine)) * np.logspace(-3, 3, k)[:, None]
    F[7] = 0.0
    Ui = rng.standard_normal((k, ctx.n_patches))
    B, U, steps, res, Uf = _chain(ctx, F, Ui, **CG)
    B2, U2, steps2, res2, Uf2 = _chain(ctx, F, Ui, **CG)
    for a, b in ((B, B2), (U, U2), (steps, steps2), (res, res2), (Uf, Uf2)):
        assert np.array_equal(a, b)
    perm = rng.permutation(k)
    Bp, Up, sp_, rp, Ufp = _chain(ctx, F[perm], Ui[perm], **CG)
    assert np.array_equal(Bp, B[perm]) and np.array_equal(Up, U[perm]) and np.array_equal(Ufp, Uf[perm])
    assert np.array_equal(sp_, steps[perm]) and np.array_equal(rp, res[perm])
    for j in (0, 7, 15, 16, 17, 31, 32, 36):
        b1, u1, s1, r1, uf1 = _chain(ctx, F[j:j + 1], Ui[j:j + 1], **CG)
        assert np.array_equal(b1[0], B[j]) and np.array_equal(u1[0], U[j]) and np.array_equal(uf1[0], Uf[j])
        assert s1[0] == steps[j] and r1[0] == res[j]
    ctx.close()


def test_per_column_stopping():
    """Columns scaled by 1e-8 .. 1e8 under an absolute tolerance stop at different steps; each equals its own n_rhs = 1
    call.  A failing column is reported by index with steps and residual filled for every column."""
    ctx, _ = _ready(dict(dim=2, s=1, ref=4, n=2, ell=2))
    rng = np.random.default_rng(9)
    k = 9
    b0 = ctx.coarse_rhs(rng.standard_normal(ctx.n_fine))
    B = np.logspace(-8, 8, k)[:, None] * b0[None, :]
    ctl = dict(max_steps=5000, tolerance=1e-4 * np.linalg.norm(b0), reduction=0.0)   # 1e-12 relative at the top
    U, steps, res = ctx.coarse_solve_batch(B, **ctl)
    assert len(set(steps.tolist())) >= 3, steps
    for j in range(k):
        u1, s1, r1 = ctx.coarse_solve_batch(B[j:j + 1], **ctl)
        assert s1[0] == steps[j] and r1[0] == res[j] and np.array_equal(u1[0], U[j])
        assert res[j] <= ctl["tolerance"]
    # max_steps = 1 with a tight reduction: SLOD_ERR_NUMERIC naming column 0, outputs filled
    Bn = np.ascontiguousarray(np.stack([b0, 2.0 * b0, -b0]))
    u = np.full_like(Bn, np.nan)
    st = np.full(3, -1, dtype=np.int32)
    r = np.full(3, np.nan)
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))  # noqa: E731
    rc = ctx.lib.slod_coarse_solve_batch(ctx.h, 3, dp(Bn), dp(u), 1, 0.0, 1e-14,
                                         st.ctypes.data_as(C.POINTER(C.c_int32)), dp(r))
    assert rc == 5
    msg = ctx.lib.slod_last_error(ctx.h).decode()
    assert "column 0" in msg and "did not converge" in msg
    assert (st == 1).all() and np.isfinite(r).all() and (r > 0).all() and np.isfinite(u).all()
    with pytest.raises(pkg.SlodError) as ei:
        ctx.coarse_solve_batch(Bn, max_steps=1, tolerance=0.0, reduction=1e-14)
    assert ei.value.code == 5
    ctx.close()


def test_batch_errors():
    ctx, _ = build_pair(dim=2, s=1, ref=3, n=2, ell=1)
    nf, nc = ctx.n_fine, ctx.n_patches
    for call in (lambda: ctx.coarse_rhs_batch(np.ones((2, nf))), lambda: ctx.prolongate_batch(np.ones((2, nc))),
                 lambda: ctx.coarse_solve_batch(np.ones((2, nc)))):
        with pytest.raises(pkg.SlodError) as ei:          # basis not computed
            call()
        assert ei.value.code == 4
    ctx.compute_basis()
    with pytest.raises(pkg.SlodError) as ei:              # coarse matrix not assembled
        ctx.coarse_solve_batch(np.ones((2, nc)))
    assert ei.value.code == 4
    ctx.assemble_coarse()
    buf = np.ones(nf * 2)
    dp = buf.ctypes.data_as(C.POINTER(C.c_double))
    assert ctx.lib.slod_coarse_rhs_batch(ctx.h, 0, dp, dp) == 1
    assert ctx.lib.slod_coarse_solve_batch(ctx.h, 0, dp, dp, 10, 0.0, 1e-10, None, None) == 1
    assert ctx.lib.slod_prolongate_batch(ctx.h, -1, dp, dp) == 1
    assert ctx.lib.slod_coarse_rhs_batch(ctx.h, 1, None, dp) == 1
    ctx.close()


def test_batch_after_checkpoint(tmp_path):
    ctx, _ = _ready(dict(dim=2, s=1, ref=4, n=2, ell=2))
    rng = np.random.default_rng(3)
    F = rng.standard_normal((6, ctx.n_fine))
    Ui = rng.standard_normal((6, ctx.n_patches))
    ref = _chain(ctx, F, Ui, max_steps=5000, tolerance=0.0, reduction=1e-12)
    path = str(tmp_path / "offline.slod")
    ctx.save_state(path)
    ctx.close()
    ctx2 = pkg.SlodContext(dim=2, spacedim=1, n_global_refinements=4, n_subdivisions=2, oversampling=2, stabilize=True)
    ctx2.load_state(path)
    got = _chain(ctx2, F, Ui, max_steps=5000, tolerance=0.0, reduction=1e-12)
    for a, b in zip(ref, got):
        assert np.array_equal(a, b)
    ctx2.close()


@pytest.mark.parametrize("case", [END_TO_END[0], END_TO_END[6]],
                         ids=lambda c: "-".join(f"{k}{v}" for k, v in c.items()))
def test_batch_end_to_end(case):
    """Three forcings through the batched chain against the oracle's direct chain: 1e-9 relative on the fine solution."""
    assert case["ell"] == 1
    ctx, orc = _ready(case)
    orc.compute_basis()
    K, Cm, _ = orc.assemble_global_matrix()
    forcings = [_forcing(case["s"]), lambda p: np.ones((len(p), 1)),
                lambda p: np.exp(p[:, [0]]) * (1.0 + p[:, [1]] ** 2)]
    F = np.stack([orc.fem_rhs(fn) for fn in forcings])
    B = ctx.coarse_rhs_batch(F)
    U, _, _ = ctx.coarse_solve_batch(B, **CG)
    Uf = ctx.prolongate_batch(U)
    for j in range(len(forcings)):
        u_dir, _ = orc.solve_coarse(K, Cm.T @ F[j], direct=True)
        uh_ref = Cm @ u_dir
        assert np.linalg.norm(Uf[j] - uh_ref) <= 1e-9 * np.linalg.norm(uh_ref)
    ctx.close()


def test_batch_full_size():
    """The headline workload (3-D, 32^3 cells, oversampling 2), k = 8: every column within 1e-9 of its single solve."""
    import bench
    w = bench.WORKLOADS[bench.DEFAULT_WORKLOAD]
    ctx = pkg.SlodContext(dim=w["dim"], spacedim=w["s"], n_global_refinements=w["ref"], n_subdivisions=w["n"],
                          oversampling=w["ell"], stabilize=True, problem=0 if w["s"] == 1 else 1)
    for f, t in enumerate(bench.make_tables(w)):
        ctx.set_coefficient(f, w["r"], t)
    ctx.compute_basis()
    ctx.assemble_coarse()
    rng = np.random.default_rng(21)
    F = rng.standard_normal((8, ctx.n_fine))
    ctl = dict(max_steps=20000, tolerance=0.0, reduction=1e-13)
    B = ctx.coarse_rhs_batch(F)
    U, steps, _ = ctx.coarse_solve_batch(B, **ctl)
    Uf = ctx.prolongate_batch(U)
    for j in range(8):
        b1 = ctx.coarse_rhs(F[j])
        assert _rel(B[j], b1) <= 1e-12
        u1, s1, _ = ctx.coarse_solve(B[j], **ctl)
        assert np.linalg.norm(U[j] - u1) <= 1e-9 * np.linalg.norm(u1)
        assert abs(int(steps[j]) - s1) <= 1
        uf1 = ctx.prolongate(u1)
        assert np.linalg.norm(Uf[j] - uf1) <= 1e-9 * np.linalg.norm(uf1)
    ctx.close()


def test_batch_two_gpus():
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
        rng = np.random.default_rng(4)
        out.append(_chain(ctx, rng.standard_normal((20, ctx.n_fine)), rng.standard_normal((20, ctx.n_patches)), **CG))
        ctx.close()
    for a, b in zip(*out):
        assert np.array_equal(a, b)
