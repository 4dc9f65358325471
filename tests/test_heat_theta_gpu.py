"""GPU tests of the theta scheme on the SLOD space (slod_heat_theta_solve / _batch, slod_fem_heat_theta_solve).

Trajectories are compared with tools/heat_oracle.py on the GPU's own K and M_H (direct solves), so the new kernels are
tested at the solver tolerance whatever the conditioning of the basis selection."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from heat_oracle import theta_solve_coarse, theta_solve_fine  # noqa: E402
from parity_common import build_pair, pkg  # noqa: E402
from test_heat_gpu import CASES, CG, IDS, _csr, _dp, _ready  # noqa: E402
from test_heat_theta_cpu import CN_ERRORS, T_END, pulse, ramp  # noqa: E402
from test_online_gpu import _forcing  # noqa: E402

pytestmark = pytest.mark.gpu

# (theta, n_fields, n_startup); n_fields = 0: per-step loads, n_fields = n_steps + 1 with g the identity
SCHEMES = [(0.5, 1, 0), (0.5, 3, 2), (0.75, 3, 0), (0.75, 1, 1), (1.0, 3, 1), (1.0, 1, 0), (0.5, 0, 1)]


def _fields(ctx, orc, case, nq, n_steps, seed):
    """nq fine fields (the first the smooth forcing of the heat tests, then seeded ones) and g [2][n_steps + 1][nq]."""
    rng = np.random.default_rng(seed)
    n = n_steps + 1 if nq == 0 else nq
    F = np.empty((n, ctx.n_fine))
    F[0] = orc.fem_rhs(_forcing(case["s"]))
    F[1:] = rng.standard_normal((n - 1, ctx.n_fine)) * np.abs(F[0]).max()
    if nq == 0:
        return F, np.broadcast_to(np.eye(n), (2, n, n)).copy()
    t = np.arange(n_steps + 1)[:, None] * 1e-2
    G = np.stack([np.cos(3 * t + np.arange(nq)) + 0.2 * rng.standard_normal((n_steps + 1, nq)) for _ in range(2)])
    return F, G


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_theta_trajectories(case):
    """heat_theta_solve and heat_theta_solve_batch (two columns with different g and u0) against theta_solve_coarse at
    every output; fem_heat_theta_solve against theta_solve_fine for two of the schemes."""
    ctx, orc, K, M = _ready(case)
    nc = ctx.n_patches * ctx.s
    dt, n_steps, every = 1e-2, 6, 2
    rng = np.random.default_rng(7)
    U0 = rng.standard_normal((2, nc))
    for theta, nq, ns in SCHEMES:
        F, G = _fields(ctx, orc, case, nq, n_steps, 11)
        B = ctx.coarse_rhs_batch(F)
        U, st = ctx.heat_theta_solve(F, G[0], U0[0], theta, dt, n_steps, every, n_startup=ns, **CG)
        Ub, stb = ctx.heat_theta_solve_batch(np.stack([F, F]), G, U0, theta, dt, n_steps, every, n_startup=ns, **CG)
        assert U.shape == (3, nc) and Ub.shape == (3, 2, nc) and st.shape == (6,) and stb.shape == (6, 2)
        for j in range(2):
            ref = theta_solve_coarse(K, M, B, G[j], U0[j], theta, dt, n_steps, ns)[every - 1::every]
            for o in range(3):
                assert np.linalg.norm(Ub[o, j] - ref[o]) <= 1e-9 * np.linalg.norm(ref[o]), (theta, nq, ns, j, o)
                if j == 0:
                    assert np.linalg.norm(U[o] - ref[o]) <= 1e-9 * np.linalg.norm(ref[o]), (theta, nq, ns, o)
        assert (st > 0).all() and (stb > 0).all()
        if (theta, nq, ns) in ((0.5, 3, 2), (0.75, 3, 0)):
            u0f = ctx.prolongate(U0[0])
            Uf, stf = ctx.fem_heat_theta_solve(F, G[0], u0f, theta, dt, n_steps, every, n_startup=ns,
                                               max_steps=200000, tolerance=0.0, reduction=1e-13)
            ref_f = theta_solve_fine(orc, F, G[0], u0f, theta, dt, n_steps, ns)[every - 1::every]
            for o in range(3):
                assert np.linalg.norm(Uf[o] - ref_f[o]) <= 1e-9 * np.linalg.norm(ref_f[o]), (theta, nq, ns, o)
            assert (stf > 0).all()
    ctx.close()


def test_startup_step_is_two_half_steps():
    """A start-up step is two backward-Euler solves of dt / 2: the state after it and its cg_steps (the sum of the two
    solves) equal, bit for bit, those of a theta = 1 run of two steps of dt / 2 whose g holds the midpoint value
    (g_0 + g_1) / 2 and then g_1.  Single, batch and fine calls."""
    ctx, orc, _, _ = _ready(dict(dim=2, s=1, ref=3, n=2, ell=2))
    rng = np.random.default_rng(21)
    F, _ = _fields(ctx, orc, dict(s=1), 2, 2, 21)
    g = 1.0 + rng.random((3, 2))
    gh = np.stack([g[0], 0.5 * (g[0] + g[1]), g[1]])
    u0 = rng.standard_normal(ctx.n_patches)
    dt = 1e-2
    U, st = ctx.heat_theta_solve(F, g, u0, 0.5, dt, 2, 1, n_startup=1, **CG)
    Uh, sth = ctx.heat_theta_solve(F, gh, u0, 1.0, dt / 2, 2, 1, **CG)
    assert np.array_equal(U[0], Uh[1]) and st[0] == sth.sum() and sth.min() > 0, (st, sth)
    Ub, stb = ctx.heat_theta_solve_batch(F[None], g[None], u0[None], 0.5, dt, 2, 1, n_startup=1, **CG)
    Ubh, stbh = ctx.heat_theta_solve_batch(F[None], gh[None], u0[None], 1.0, dt / 2, 2, 1, **CG)
    assert np.array_equal(Ub[0, 0], Ubh[1, 0]) and stb[0, 0] == stbh[:, 0].sum(), (stb, stbh)
    u0f = ctx.prolongate(u0)
    Uf, stf = ctx.fem_heat_theta_solve(F, g, u0f, 0.5, dt, 2, 1, n_startup=1, reduction=1e-12)
    Ufh, stfh = ctx.fem_heat_theta_solve(F, gh, u0f, 1.0, dt / 2, 2, 1, reduction=1e-12)
    assert np.array_equal(Uf[0], Ufh[1]) and stf[0] == stfh.sum(), (stf, stfh)
    ctx.close()


def test_backward_euler_calls_are_theta_one():
    """slod_heat_solve / _batch / slod_fem_heat_solve equal the theta calls at theta = 1, g = NULL, no start-up, bit for
    bit, with and without forcing."""
    ctx, orc = build_pair(dim=2, s=1, ref=4, n=2, ell=2)
    ctx.compute_basis()
    ctx.assemble_coarse()
    ctx.assemble_coarse_mass()
    rng = np.random.default_rng(9)
    k, nc = 19, ctx.n_patches
    F = rng.standard_normal((k, ctx.n_fine))
    U0 = rng.standard_normal((k, nc))
    for f in (F, None):
        U, st = ctx.heat_solve(None if f is None else f[0], U0[0], 2e-3, 5, 1, **CG)
        Ut, stt = ctx.heat_theta_solve(None if f is None else f[:1], None, U0[0], 1.0, 2e-3, 5, 1, **CG)
        assert np.array_equal(U, Ut) and np.array_equal(st, stt)
        Ub, stb = ctx.heat_solve_batch(f, U0, 2e-3, 5, 1, **CG)
        Ubt, stbt = ctx.heat_theta_solve_batch(None if f is None else f[:, None], None, U0, 1.0, 2e-3, 5, 1, **CG)
        assert np.array_equal(Ub, Ubt) and np.array_equal(stb, stbt)
    u0f = ctx.prolongate(U0[0])
    Uf, stf = ctx.fem_heat_solve(F[0], u0f, 2e-3, 3, 1, max_steps=200000, reduction=1e-12)
    Uft, stft = ctx.fem_heat_theta_solve(F[:1], None, u0f, 1.0, 2e-3, 3, 1, max_steps=200000, reduction=1e-12)
    assert np.array_equal(Uf, Uft) and np.array_equal(stf, stft)
    ctx.close()


def test_batch_fields_beyond_the_largest_copy_pitch():
    """In the host array [n_rhs][n_fields][n_fine], field q of consecutive columns lies n_fields n_fine doubles apart;
    here that is more than 2 GiB, beyond the largest pitch of a 2-D copy.  g is zero on all but the first and the last
    field, whose fields are the only nonzero ones: the result equals, bit for bit, the run with those two fields alone."""
    ctx, _ = build_pair(dim=2, s=1, ref=7, n=2, ell=1)
    ctx.compute_basis()
    ctx.assemble_coarse()
    ctx.assemble_coarse_mass()
    nf = ctx.n_fine
    nq = 2 ** 31 // (8 * nf) + 2
    rng = np.random.default_rng(8)
    F = np.zeros((2, nq, nf))   # zero pages: only the four nonzero fields take memory
    F[:, 0] = rng.standard_normal((2, nf))
    F[:, -1] = rng.standard_normal((2, nf))
    G = np.zeros((2, 3, nq))
    G[:, :, 0] = 1.0 + rng.random((2, 3))
    G[:, :, -1] = rng.standard_normal((2, 3))
    assert nq * nf * 8 > 2 ** 31
    U, st = ctx.heat_theta_solve_batch(F, G, None, 0.5, 1e-2, 2, 1, n_startup=1, **CG)
    U2, st2 = ctx.heat_theta_solve_batch(np.ascontiguousarray(F[:, [0, -1]]), np.ascontiguousarray(G[:, :, [0, -1]]),
                                         None, 0.5, 1e-2, 2, 1, n_startup=1, **CG)
    assert np.array_equal(U, U2) and np.array_equal(st, st2) and np.abs(U).max() > 0
    ctx.close()


def test_theta_batch_independence():
    """n_rhs = 37 (three groups), three fields, Crank-Nicolson with one start-up step: a column is bit-identical across
    runs, permutations and n_rhs = 1."""
    ctx, _ = build_pair(dim=2, s=1, ref=4, n=2, ell=2)
    ctx.compute_basis()
    ctx.assemble_coarse()
    ctx.assemble_coarse_mass()
    rng = np.random.default_rng(5)
    k, nc, nq, n_steps = 37, ctx.n_patches, 3, 5
    F = rng.standard_normal((k, nq, ctx.n_fine)) * np.logspace(-3, 3, k)[:, None, None]
    G = rng.standard_normal((k, n_steps + 1, nq))
    U0 = rng.standard_normal((k, nc))
    F[7] = 0.0
    U0[7] = 0.0
    args = (0.5, 2e-3, n_steps, 1)
    U, st = ctx.heat_theta_solve_batch(F, G, U0, *args, n_startup=1, **CG)
    U2, st2 = ctx.heat_theta_solve_batch(F, G, U0, *args, n_startup=1, **CG)
    assert np.array_equal(U, U2) and np.array_equal(st, st2)
    assert not U[:, 7].any() and not st[:, 7].any()
    perm = rng.permutation(k)
    Up, stp = ctx.heat_theta_solve_batch(F[perm], G[perm], U0[perm], *args, n_startup=1, **CG)
    assert np.array_equal(Up, U[:, perm]) and np.array_equal(stp, st[:, perm])
    rep = np.array([3, 3, 20, 3, 36, 20])   # repeated columns
    Ur, str_ = ctx.heat_theta_solve_batch(F[rep], G[rep], U0[rep], *args, n_startup=1, **CG)
    assert np.array_equal(Ur, U[:, rep]) and np.array_equal(str_, st[:, rep])
    for j in (0, 15, 16, 17, 36):
        u1, s1 = ctx.heat_theta_solve_batch(F[j:j + 1], G[j:j + 1], U0[j:j + 1], *args, n_startup=1, **CG)
        assert np.array_equal(u1[:, 0], U[:, j]) and np.array_equal(s1[:, 0], st[:, j])
        us, ss = ctx.heat_theta_solve(F[j], G[j], U0[j], *args, n_startup=1, **CG)
        assert np.linalg.norm(us - U[:, j]) <= 1e-9 * np.linalg.norm(U[:, j])
    ctx.close()


def test_crank_nicolson_second_order():
    """The GPU's own 2-D l = 2 system, u0 = 0, g = sin(pi t / T): the error at T against a direct dt / 64 run on the same
    K and M_H falls by at least 3.5x per halving of dt (tests/test_heat_theta_cpu.py on the oracle's system)."""
    ctx, _, K, M = _ready(dict(dim=2, s=1, ref=3, n=2, ell=2))
    G0 = 2 ** 3 * 2 + 1
    F = np.full((1, G0 * G0), (1.0 / 16) ** 2)
    B = ctx.coarse_rhs_batch(F)
    n0 = 32
    dt0 = T_END / n0
    ref = theta_solve_coarse(K, M, B, pulse(64 * n0, dt0 / 64), None, 0.5, dt0 / 64, 64 * n0)[-1]
    errs = []
    for j in range(3):
        n = n0 * 2 ** j
        U, _ = ctx.heat_theta_solve(F, pulse(n, T_END / n), None, 0.5, T_END / n, n, n, max_steps=5000, tolerance=0.0,
                                    reduction=1e-14)
        e = U[0] - ref
        errs.append(float(np.sqrt(e @ (M @ e))))
    print("Crank-Nicolson errors at T:", errs)
    assert all(errs[j] / errs[j + 1] >= 3.5 for j in range(2)), errs
    ctx.close()


def test_cn_trajectory_error_decays():
    """The prolongated Crank-Nicolson trajectory (two start-up steps, g the ramp) against fem_heat_theta_solve on the
    problem of tests/test_heat_theta_cpu.py: within the oracle's pinned errors, more than 20x per layer."""
    errs = []
    n, dt = 20, T_END / 20
    for ell in (1, 2, 3):
        rs = np.random.default_rng(11)
        tab = 1.0 + 99.0 * rs.random(16 ** 2)
        ctx = pkg.SlodContext(dim=2, spacedim=1, n_global_refinements=3, n_subdivisions=2, oversampling=ell,
                              stabilize=True)
        ctx.set_coefficient(0, 4, tab)
        ctx.compute_basis()
        ctx.assemble_coarse()
        ctx.assemble_coarse_mass()
        G0 = 8 * 2 + 1
        F = np.full((1, G0 * G0), (1.0 / 16) ** 2)
        U, _ = ctx.heat_theta_solve(F, ramp(n, dt), None, 0.5, dt, n, n, n_startup=2, **CG)
        Uf, _ = ctx.fem_heat_theta_solve(F, ramp(n, dt), None, 0.5, dt, n, n, n_startup=2, reduction=1e-13)
        errs.append(ctx.fine_norms(ctx.prolongate(U[0]) - Uf[0])[2] / ctx.fine_norms(Uf[0])[2])
        ctx.close()
    print("CN trajectory energy error at t = 0.2, l = 1, 2, 3:", errs, "oracle:", CN_ERRORS)
    for ell, e in zip((1, 2, 3), errs):
        assert e <= 1.25 * CN_ERRORS[ell], (ell, e)
    assert errs[0] >= 0.8 * CN_ERRORS[1] and errs[1] >= 0.8 * CN_ERRORS[2]
    assert errs[1] < errs[0] / 20 and errs[2] < errs[1] / 20


def test_mass_norm_does_not_grow_full_size():
    """The headline workload (3-D, 32^3 cells, oversampling 2), f = 0, 16 seeded initial values: ||u^k||_{M_H} does not
    increase for theta = 1/2, 3/4, 1 (with and without start-up), up to the CG tolerance."""
    import bench
    w = bench.WORKLOADS[bench.DEFAULT_WORKLOAD]
    ctx = pkg.SlodContext(dim=w["dim"], spacedim=w["s"], n_global_refinements=w["ref"], n_subdivisions=w["n"],
                          oversampling=w["ell"], stabilize=True, problem=0 if w["s"] == 1 else 1)
    for f, t in enumerate(bench.make_tables(w)):
        ctx.set_coefficient(f, w["r"], t)
    ctx.compute_basis()
    ctx.assemble_coarse()
    ctx.assemble_coarse_mass()
    nc = ctx.n_patches * ctx.s
    M = _csr(ctx.coarse_mass_csr(), nc)
    U0 = np.random.default_rng(16).standard_normal((16, nc))
    n0 = np.sqrt(np.einsum("ij,ij->i", U0, (M @ U0.T).T))
    for theta, ns in ((0.5, 0), (0.5, 1), (0.75, 0), (1.0, 0)):
        U, st = ctx.heat_theta_solve_batch(None, None, U0, theta, 1e-3, 6, 1, n_startup=ns, max_steps=20000,
                                           tolerance=0.0, reduction=1e-12)
        norms = np.array([np.sqrt(np.einsum("ij,ij->i", U[k], (M @ U[k].T).T)) for k in range(6)])
        prev = np.vstack([n0, norms[:-1]])
        print(f"theta {theta} start-up {ns}: max ratio {np.max(norms / prev):.6f}, CG steps {st.max(axis=1).tolist()}")
        assert (norms <= prev * (1.0 + 1e-9)).all(), (theta, ns)
    ctx.close()


def test_theta_cg_failure_names_step_and_column():
    """The construction of tests/test_heat_gpu.py for M_H + theta dt K at theta = 1/2: column 1's step-1 increment is an
    eigenvector of the Jacobi-preconditioned matrix; with max_steps at step 1's count, step 2 of column 1 fails."""
    ctx, _ = build_pair(dim=2, s=1, ref=3, n=2, ell=1)
    ctx.compute_basis()
    ctx.assemble_coarse()
    ctx.assemble_coarse_mass()
    nc, dt, theta = ctx.n_patches, 1e-2, 0.5
    K = _csr(ctx.coarse_csr(), nc).toarray()
    S = _csr(ctx.coarse_mass_csr(), nc).toarray() + theta * dt * K
    d = np.sqrt(np.diag(S))
    _, vec = np.linalg.eigh(S / d[:, None] / d[None, :])
    U0 = np.zeros((3, nc))
    for j, m in ((1, nc // 2), (2, nc // 3)):
        U0[j] = -np.linalg.solve(K, d * vec[:, m]) / dt   # dt (0 - K u0) = D^1/2 v
    ctl = dict(tolerance=0.0, reduction=1e-6)
    _, st = ctx.heat_theta_solve_batch(None, None, U0, theta, dt, 3, 1, max_steps=1000, **ctl)
    m = int(st[0].max())
    assert m <= 2 and st[1, 1] > m, st
    out = np.full((3, 3, nc), np.nan)
    cg = np.full((3, 3), -1, dtype=np.int32)
    rc = ctx.lib.slod_heat_theta_solve_batch(ctx.h, 3, theta, dt, 3, 1, 0, 1, None, None, _dp(U0), _dp(out), m, 0.0,
                                             1e-6, cg.ctypes.data_as(C.POINTER(C.c_int32)))
    msg = ctx.lib.slod_last_error(ctx.h).decode()
    assert rc == 5 and "time step 2 column 1" in msg and "did not converge" in msg, msg
    assert "M_H + c K (c = 0.005)" in msg, msg   # the matrix that failed: c = theta dt
    assert np.isfinite(out[0]).all() and np.isnan(out[1:]).all() and (cg[2] == -1).all()
    out1 = np.full((3, nc), np.nan)
    rc = ctx.lib.slod_heat_theta_solve(ctx.h, theta, dt, 3, 1, 0, 1, None, None, _dp(np.ascontiguousarray(U0[1])),
                                       _dp(out1), m, 0.0, 1e-6, None)
    msg = ctx.lib.slod_last_error(ctx.h).decode()
    assert rc == 5 and "time step 2:" in msg, msg
    assert np.isfinite(out1[0]).all() and np.isnan(out1[1:]).all()
    ctx.close()


def test_theta_call_order_and_checkpoint(tmp_path):
    """SLOD_ERR_STATE before K / M_H; a restored handle needs M_H assembled again and then gives the same bits."""
    ctx, _ = build_pair(dim=2, s=1, ref=4, n=2, ell=2)
    nf = ctx.n_fine
    F = np.random.default_rng(3).standard_normal((2, 2, nf))
    G = np.random.default_rng(4).standard_normal((2, 5, 2))

    def code(call):
        with pytest.raises(pkg.SlodError) as ei:
            call()
        return ei.value.code

    run = (lambda c: c.heat_theta_solve_batch(F, G, None, 0.5, 1e-2, 4, 2, n_startup=1, **CG))
    assert code(lambda: run(ctx)) == 4
    ctx.compute_basis()
    ctx.assemble_coarse()
    assert code(lambda: run(ctx)) == 4
    ctx.assemble_coarse_mass()
    T1, s1 = run(ctx)
    path = str(tmp_path / "offline.slod")
    ctx.save_state(path)
    ctx.close()
    ctx2 = pkg.SlodContext(dim=2, spacedim=1, n_global_refinements=4, n_subdivisions=2, oversampling=2, stabilize=True)
    ctx2.load_state(path)
    assert code(lambda: run(ctx2)) == 4
    ctx2.assemble_coarse_mass()
    T2, s2 = run(ctx2)
    assert np.array_equal(T1, T2) and np.array_equal(s1, s2)
    ctx2.close()


def test_theta_two_gpus():
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
        F = rng.standard_normal((5, 2, ctx.n_fine))
        G = rng.standard_normal((5, 4, 2))
        out.append(list(ctx.heat_theta_solve_batch(F, G, None, 0.5, 1e-2, 3, 1, n_startup=1, **CG))
                   + list(ctx.heat_theta_solve(F[0], G[0], None, 0.75, 1e-2, 3, 1, **CG)))
        ctx.close()
    for a, b in zip(*out):
        assert np.array_equal(a, b)
