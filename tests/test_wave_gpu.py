"""GPU tests of Newmark time stepping for the wave equation on the SLOD space (slod_wave_solve / _batch,
slod_fem_wave_solve).

Trajectories are compared with tools/wave_oracle.py on the GPU's own K and M_H (direct solves), so the new kernels are
tested at the solver tolerance whatever the conditioning of the basis selection."""
import ctypes as C
import os
import sys

import numpy as np
import pytest
import scipy.linalg as sl

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from heat_oracle import fine_operators  # noqa: E402
from parity_common import build_pair, pkg  # noqa: E402
from test_heat_gpu import CASES, CG, IDS, _dp, _ready  # noqa: E402
from test_heat_theta_cpu import T_END, ramp  # noqa: E402
from test_heat_theta_gpu import _fields  # noqa: E402
from test_wave_cpu import WAVE_ERRORS, amplification, chebyshev  # noqa: E402
from wave_oracle import energy, newmark_coarse, newmark_fine  # noqa: E402

pytestmark = pytest.mark.gpu


def _rel(a, b):
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


def _lambda_max(K, M):
    return float(sl.eigh(K.toarray(), M.toarray(), eigvals_only=True)[-1])


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_wave_trajectories(case):
    """wave_solve and a two-column wave_solve_batch (different g, u0, v0) against newmark_coarse for u and v at every
    output, beta in {0, 1/4, 1/2}, with and without three forcing fields; energy_out against 1/2 v^T M v + 1/2 u^T K u
    from the CSR copies.  fem_wave_solve against newmark_fine (beta = 0 at a quarter of the step, inside the fine
    grid's explicit limit)."""
    ctx, orc, K, M = _ready(case)
    nc = ctx.n_patches * ctx.s
    dt = 0.5 * 2.0 / np.sqrt(_lambda_max(K, M))   # half the explicit limit of the SLOD space
    n_steps, every = 6, 2
    rng = np.random.default_rng(7)
    U0, V0 = rng.standard_normal((2, nc)), rng.standard_normal((2, nc))
    F, G = _fields(ctx, orc, case, 3, n_steps, 11)
    B = ctx.coarse_rhs_batch(F)
    for beta in (0.0, 0.25, 0.5):
        for forced in (True, False):
            Fx, Gx = (F, G) if forced else (None, None)
            U, V, E, st = ctx.wave_solve(Fx, None if Gx is None else Gx[0], U0[0], V0[0], beta, dt, n_steps, every, **CG)
            Ub, Vb, Eb, stb = ctx.wave_solve_batch(None if Fx is None else np.stack([F, F]), Gx, U0, V0, beta, dt,
                                                   n_steps, every, **CG)
            assert U.shape == V.shape == (3, nc) and Ub.shape == Vb.shape == (3, 2, nc)
            assert E.shape == (4,) and Eb.shape == (4, 2) and st.shape == (7,) and stb.shape == (7, 2)
            for j in range(2):
                Ur, Vr = newmark_coarse(K, M, B if forced else None, G[j] if forced else None, U0[j], V0[j], beta, dt,
                                        n_steps)
                Ur, Vr = Ur[every::every], Vr[every::every]
                for o in range(3):
                    assert _rel(Ub[o, j], Ur[o]) <= 1e-9 and _rel(Vb[o, j], Vr[o]) <= 1e-9, (beta, forced, j, o)
                    if j == 0:
                        assert _rel(U[o], Ur[o]) <= 1e-9 and _rel(V[o], Vr[o]) <= 1e-9, (beta, forced, o)
                Eref = energy(K, M, np.vstack([U0[j], Ub[:, j]]), np.vstack([V0[j], Vb[:, j]]))
                assert np.abs(Eb[:, j] - Eref).max() <= 1e-12 * Eref.max(), (beta, forced, j, Eb[:, j], Eref)
            Eref = energy(K, M, np.vstack([U0[0], U]), np.vstack([V0[0], V]))
            assert np.abs(E - Eref).max() <= 1e-12 * Eref.max(), (beta, forced)
            assert (st > 0).all() and (stb > 0).all()
    u0f, v0f = ctx.prolongate(U0[0]), ctx.prolongate(V0[0])
    A, Mh, _ = fine_operators(orc)
    for beta, dtf in ((0.0, dt / 4), (0.25, dt)):
        Uf, Vf, Ef, stf = ctx.fem_wave_solve(F, G[0], u0f, v0f, beta, dtf, n_steps, every, max_steps=200000,
                                             tolerance=0.0, reduction=1e-13)
        Ur, Vr = newmark_fine(orc, F, G[0], u0f, v0f, beta, dtf, n_steps)
        for o in range(3):
            assert _rel(Uf[o], Ur[every * (o + 1)]) <= 1e-9 and _rel(Vf[o], Vr[every * (o + 1)]) <= 1e-9, (beta, o)
        Eref = energy(A, Mh, np.vstack([Ur[:1], Uf]), np.vstack([Vr[:1], Vf]))
        assert np.abs(Ef - Eref).max() <= 1e-12 * Eref.max(), (beta, Ef, Eref)
        assert (stf > 0).all()
    ctx.close()


def test_wave_batch_bit_identity():
    """n_rhs = 17 (crosses a group of 16), three fields, beta = 1/4 and 0: a column is bit-identical across runs,
    permutations, repeated columns, n_rhs = 1 and 5; the single-vector call agrees to the tolerance."""
    ctx, _ = build_pair(dim=2, s=1, ref=4, n=2, ell=2)
    ctx.compute_basis()
    ctx.assemble_coarse()
    ctx.assemble_coarse_mass()
    rng = np.random.default_rng(5)
    k, nc, nq, n_steps = 17, ctx.n_patches, 3, 5
    F = rng.standard_normal((k, nq, ctx.n_fine)) * np.logspace(-3, 3, k)[:, None, None]
    G = rng.standard_normal((k, n_steps + 1, nq))
    U0, V0 = rng.standard_normal((k, nc)), rng.standard_normal((k, nc))
    for beta in (0.25, 0.0):
        args = (beta, 1e-3, n_steps, 1)
        R = ctx.wave_solve_batch(F, G, U0, V0, *args, **CG)
        R2 = ctx.wave_solve_batch(F, G, U0, V0, *args, **CG)
        assert all(np.array_equal(a, b) for a, b in zip(R, R2))
        perm = rng.permutation(k)
        Rp = ctx.wave_solve_batch(F[perm], G[perm], U0[perm], V0[perm], *args, **CG)
        assert all(np.array_equal(a, b[..., perm, :] if b.ndim == 3 else b[:, perm]) for a, b in zip(Rp, R))
        for sel in ([3, 3, 16, 0, 9], [16], [0], [15, 16, 2, 7, 11]):
            Rs = ctx.wave_solve_batch(F[sel], G[sel], U0[sel], V0[sel], *args, **CG)
            assert all(np.array_equal(a, b[..., sel, :] if b.ndim == 3 else b[:, sel]) for a, b in zip(Rs, R)), sel
        for j in (0, 16):
            U, V, E, _ = ctx.wave_solve(F[j], G[j], U0[j], V0[j], *args, **CG)
            assert _rel(U, R[0][:, j]) <= 1e-9 and _rel(V, R[1][:, j]) <= 1e-9 and _rel(E, R[2][:, j]) <= 1e-9
    ctx.close()


def test_explicit_step_on_the_top_mode():
    """The top generalized eigenpair of the GPU's own (K, M_H), u_0 = x, beta = 0: at z = dt sqrt(lambda) = 1.9 the
    trajectory is cos(k phi) x, cos phi = 1 - z^2 / 2; at z = 2.1 it grows like T_k(c), c < -1.  At 0.9 x the SLOD
    stable step, the fine reference with beta = 0 blows up (its largest eigenvalue is about 2.1^2 x larger) while the
    SLOD energy stays bounded."""
    ctx, _, K, M = _ready(dict(dim=2, s=1, ref=3, n=2, ell=2))
    lam, X = sl.eigh(K.toarray(), M.toarray())
    x = X[:, -1]
    n_steps = 40
    for z in (1.9, 2.1):
        dt = z / np.sqrt(lam[-1])
        c = amplification(0.0, z * z)
        U, _, _, _ = ctx.wave_solve(None, None, x, None, 0.0, dt, n_steps, 1, **CG)
        T = chebyshev(n_steps, c)[1:]
        if z < 2:
            assert np.allclose(T, np.cos(np.arange(1, n_steps + 1) * np.arccos(c)), rtol=0, atol=1e-12)
        err = np.abs(U - T[:, None] * x[None]).max(axis=1) / (np.maximum(np.abs(T), 1.0) * np.abs(x).max())
        print(f"z = {z}: c = {c:.4f}, |T_40| = {abs(T[-1]):.3e}, max rel. error {err.max():.2e}")
        assert err.max() <= 1e-8, (z, err.max())
        if z > 2:
            assert abs(T[-1]) > 1e9
    dt = 0.9 * 2.0 / np.sqrt(lam[-1])
    rng = np.random.default_rng(2)
    n = 30
    _, _, E, _ = ctx.wave_solve(None, None, rng.standard_normal(ctx.n_patches), None, 0.0, dt, n, 1, **CG)
    _, _, Ef, _ = ctx.fem_wave_solve(None, None, rng.standard_normal(ctx.n_fine), None, 0.0, dt, n, 1,
                                     reduction=1e-12)
    print(f"explicit step 0.9 x the SLOD limit: SLOD energy max ratio {np.max(E / E[0]):.3f}, fine energy ratio after "
          f"{n} steps {Ef[-1] / Ef[0]:.3e}")
    assert np.max(E / E[0]) <= 10.0 and Ef[-1] / Ef[0] >= 1e6
    ctx.close()


def test_wave_trajectory_error_decreases():
    """The prolongated beta = 1/4 trajectory (g the ramp, u0 = v0 = 0) against fem_wave_solve on the problem of
    tests/test_wave_cpu.py: within the oracle's pinned errors, decreasing with the oversampling."""
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
        U, _, _, _ = ctx.wave_solve(F, ramp(n, dt), None, None, 0.25, dt, n, n, **CG)
        Uf, _, _, _ = ctx.fem_wave_solve(F, ramp(n, dt), None, None, 0.25, dt, n, n, reduction=1e-13)
        errs.append(ctx.fine_norms(ctx.prolongate(U[0]) - Uf[0])[2] / ctx.fine_norms(Uf[0])[2])
        ctx.close()
    print("wave trajectory energy error at t = 0.2, l = 1, 2, 3:", errs, "oracle:", WAVE_ERRORS)
    for ell, e in zip((1, 2, 3), errs):
        assert 0.8 * WAVE_ERRORS[ell] <= e <= 1.25 * WAVE_ERRORS[ell], (ell, e)
    assert errs[0] > errs[1] > errs[2]


# relative energy drift of 50 average-acceleration steps at the headline workload with the CG reduction 1e-10 (measured
# on a B200: 3.7e-11 for one trajectory, 5.7e-11 over a batch of 16)
FULL_SIZE_DRIFT = 5e-10


def test_energy_drift_full_size():
    """The headline workload (3-D, 32^3 cells, oversampling 2), no forcing, beta = 1/4, 50 steps from seeded u0 and v0
    (one trajectory and a batch of 16): E changes by no more than FULL_SIZE_DRIFT relative; the scheme conserves it
    exactly and the acceleration solves stop at a reduction of 1e-10."""
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
    rng = np.random.default_rng(16)
    U0, V0 = rng.standard_normal((16, nc)), rng.standard_normal((16, nc))
    ctl = dict(max_steps=20000, tolerance=0.0, reduction=1e-10)
    _, _, E, st = ctx.wave_solve(None, None, U0[0], V0[0], 0.25, 1e-3, 50, 5, **ctl)
    _, _, Eb, stb = ctx.wave_solve_batch(None, None, U0, V0, 0.25, 1e-3, 50, 5, **ctl)
    d, db = np.abs(E / E[0] - 1).max(), np.abs(Eb / Eb[0] - 1).max()
    print(f"energy drift over 50 steps: single {d:.3e}, batch of 16 {db:.3e}; CG steps {st.max()}, {stb.max()}")
    assert d <= FULL_SIZE_DRIFT and db <= FULL_SIZE_DRIFT
    ctx.close()


def test_wave_cg_failure_names_step_and_column():
    """u0 = v0 = 0 and a forcing that column 1 alone switches on at t_2: steps 0 and 1 need no CG step, and with
    max_steps = 5 step 2 of column 1 fails, naming the step and the column; the outputs of step 1 are written, the later
    ones are not.  max_steps = 0 with u0 != 0 fails the start solve (step 0)."""
    ctx, _ = build_pair(dim=2, s=1, ref=3, n=2, ell=1)
    ctx.compute_basis()
    ctx.assemble_coarse()
    ctx.assemble_coarse_mass()
    nc, n_steps, k = ctx.n_patches, 4, 3
    rng = np.random.default_rng(12)
    F = np.ascontiguousarray(np.broadcast_to(rng.standard_normal(ctx.n_fine), (k, 1, ctx.n_fine)))
    G = np.zeros((k, n_steps + 1, 1))
    G[1, 2:, 0] = 1.0
    ctl = dict(tolerance=0.0, reduction=1e-10)
    U, _, _, st = ctx.wave_solve_batch(F, G, None, None, 0.25, 1e-2, n_steps, 1, max_steps=1000, **ctl)
    assert not st[:2].any() and st[2, 1] > 5 and not st[:, [0, 2]].any(), st
    out = np.full((n_steps, k, nc), np.nan)
    cg = np.full((n_steps + 1, k), -1, dtype=np.int32)
    rc = ctx.lib.slod_wave_solve_batch(ctx.h, k, 0.25, 1e-2, n_steps, 1, 1, _dp(F), _dp(G), None, None, _dp(out), None,
                                       None, 5, 0.0, 1e-10, cg.ctypes.data_as(C.POINTER(C.c_int32)))
    msg = ctx.lib.slod_last_error(ctx.h).decode()
    assert rc == 5 and "time step 2 column 1" in msg and "CG on M_H + c K (c = 2.5e-05)" in msg, msg
    assert "did not converge" in msg, msg
    assert np.array_equal(out[0], U[0]) and np.isnan(out[1:]).all()
    assert np.array_equal(cg[:2], st[:2]) and cg[2, 1] == 5 and (cg[3:] == -1).all(), cg
    out1 = np.full((n_steps, nc), np.nan)
    rc = ctx.lib.slod_wave_solve(ctx.h, 0.25, 1e-2, n_steps, 1, 1, _dp(np.ascontiguousarray(F[1])),
                                 _dp(np.ascontiguousarray(G[1])), None, None, _dp(out1), None, None, 5, 0.0, 1e-10, None)
    msg = ctx.lib.slod_last_error(ctx.h).decode()
    assert rc == 5 and "time step 2:" in msg and "column" not in msg, msg
    assert np.array_equal(out1[0], U[0, 1]) and np.isnan(out1[1:]).all()
    u0 = np.ascontiguousarray(rng.standard_normal(nc))
    rc = ctx.lib.slod_wave_solve(ctx.h, 0.25, 1e-2, n_steps, 1, 1, None, None, _dp(u0), None, _dp(out1), None, None, 0,
                                 0.0, 1e-10, None)
    msg = ctx.lib.slod_last_error(ctx.h).decode()
    assert rc == 5 and "start solve (step 0)" in msg and "CG on M_H" in msg, msg
    ctx.close()


def test_wave_call_order_checkpoint_and_heat_unchanged(tmp_path):
    """SLOD_ERR_STATE before K / M_H; a restored handle needs M_H assembled again and then gives the same bits; a heat
    trajectory is bit-identical before and after a wave call on the same handle (they share the cache of M_H + c K),
    and a wave trajectory before and after a heat call."""
    ctx, _ = build_pair(dim=2, s=1, ref=4, n=2, ell=2)
    nf, nc = ctx.n_fine, ctx.n_patches
    rng = np.random.default_rng(3)
    F, G = rng.standard_normal((2, 2, nf)), rng.standard_normal((2, 5, 2))
    U0, V0 = rng.standard_normal((2, nc)), rng.standard_normal((2, nc))

    def code(call):
        with pytest.raises(pkg.SlodError) as ei:
            call()
        return ei.value.code

    def run(c):
        return c.wave_solve_batch(F, G, U0, V0, 0.25, 1e-2, 4, 2, **CG)

    def heat(c):
        return c.heat_theta_solve(F[0], G[0], U0[0], 0.5, 3e-3, 4, 1, **CG)

    assert code(lambda: run(ctx)) == 4
    ctx.compute_basis()
    ctx.assemble_coarse()
    assert code(lambda: run(ctx)) == 4
    Uz, _, Ez, _ = ctx.fem_wave_solve(None, None, None, None, 0.25, 1e-2, 2)   # needs only the coefficient
    assert not Uz.any() and not Ez.any()
    ctx.assemble_coarse_mass()
    H1 = heat(ctx)
    W1 = run(ctx)
    H2 = heat(ctx)
    W2 = run(ctx)
    assert all(np.array_equal(a, b) for a, b in zip(H1, H2)) and all(np.array_equal(a, b) for a, b in zip(W1, W2))
    path = str(tmp_path / "offline.slod")
    ctx.save_state(path)
    ctx.close()
    ctx2 = pkg.SlodContext(dim=2, spacedim=1, n_global_refinements=4, n_subdivisions=2, oversampling=2, stabilize=True)
    ctx2.load_state(path)
    assert code(lambda: run(ctx2)) == 4
    ctx2.assemble_coarse_mass()
    W3 = run(ctx2)
    assert all(np.array_equal(a, b) for a, b in zip(W1, W3))
    ctx2.close()
