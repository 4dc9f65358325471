"""Reference computations for Newmark time stepping of the wave equation on the SLOD space, built from the numpy
oracle's own matrices (oracle/slod_oracle.py) with direct solves.

    newmark_coarse(K, M_H, B, g, u0, v0, beta, dt, n_steps)   M_H u'' + K u = b(t), b(t) = sum_q g_q(t) B_q
    newmark_fine(orc, F, g, u0, v0, beta, dt, n_steps)         the same with M_h, A_h on the interior dofs of the global
                                                                grid (homogeneous Dirichlet rows)
    energy(K, M, U, V)                                          1/2 v^T M v + 1/2 u^T K u row by row

The scheme is the one the library uses (gamma = 1/2): M a_0 = b(t_0) - K u_0, then per step
ut = u + dt v + (1/2 - beta) dt^2 a, (M + beta dt^2 K) a_new = b(t_{k+1}) - K ut, u = ut + beta dt^2 a_new,
v += dt/2 (a + a_new).  The load is summed from its first term in field order, as the library does.  Trajectories are
returned with the initial state: U[k] is u at t_k = k dt, k = 0 .. n_steps."""
import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from heat_oracle import _load, fine_operators


def _newmark_loop(apply_K, solve_M, solve_S, B, g, u, v, beta, dt, n_steps):
    B = np.zeros((1, u.size)) if B is None else np.asarray(B, dtype=float)
    g = np.ones((n_steps + 1, B.shape[0])) if g is None else np.asarray(g, dtype=float)
    a = solve_M(_load(g[0], B) - apply_K(u))
    U, V = [u.copy()], [v.copy()]
    for k in range(1, n_steps + 1):
        ut = u + dt * v + (0.5 - beta) * dt * dt * a
        a_new = solve_S(_load(g[k], B) - apply_K(ut))
        u = ut + beta * dt * dt * a_new
        v = v + 0.5 * dt * (a + a_new)
        a = a_new
        U.append(u.copy())
        V.append(v.copy())
    return np.array(U), np.array(V)


def _solvers(K, M, beta, dt):
    solve_M = spla.factorized(sp.csc_matrix(M))
    return solve_M, (solve_M if beta == 0.0 else spla.factorized(sp.csc_matrix(M + beta * dt * dt * K)))


def newmark_coarse(K, M_H, B, g, u0, v0, beta, dt, n_steps):
    """(U, V), each [n_steps + 1][n_coarse], on the coarse space.  B: (n_fields, n_coarse) loads C^T f_q or None (zero);
    g: (n_steps + 1, n_fields) or None (g = 1); u0, v0 or None (zero)."""
    n = K.shape[0]
    u = np.zeros(n) if u0 is None else np.array(u0, dtype=float)
    v = np.zeros(n) if v0 is None else np.array(v0, dtype=float)
    solve_M, solve_S = _solvers(K, M_H, beta, dt)
    return _newmark_loop(lambda x: K @ x, solve_M, solve_S, B, g, u, v, beta, dt, n_steps)


def newmark_fine(orc, F, g, u0, v0, beta, dt, n_steps):
    """(U, V), each [n_steps + 1][n_fine], on the fine grid with homogeneous Dirichlet rows (the boundary rows of F, u0
    and v0 are ignored).  F: (n_fields, n_fine) or None; g as in newmark_coarse."""
    A, M, ii = fine_operators(orc)
    Aii, Mii = A[ii][:, ii], M[ii][:, ii]
    n = A.shape[0]
    u = np.zeros(len(ii)) if u0 is None else np.asarray(u0, dtype=float)[ii]
    v = np.zeros(len(ii)) if v0 is None else np.asarray(v0, dtype=float)[ii]
    B = None if F is None else np.asarray(F, dtype=float)[:, ii]
    solve_M, solve_S = _solvers(Aii, Mii, beta, dt)
    Ui, Vi = _newmark_loop(lambda x: Aii @ x, solve_M, solve_S, B, g, u, v, beta, dt, n_steps)
    U, V = np.zeros((n_steps + 1, n)), np.zeros((n_steps + 1, n))
    U[:, ii] = Ui
    V[:, ii] = Vi
    return U, V


def energy(K, M, U, V):
    """1/2 v^T M v + 1/2 u^T K u for every row of U, V (or for one pair of vectors)."""
    U, V = np.atleast_2d(U), np.atleast_2d(V)
    return 0.5 * np.einsum("ij,ij->i", V, (M @ V.T).T) + 0.5 * np.einsum("ij,ij->i", U, (K @ U.T).T)
