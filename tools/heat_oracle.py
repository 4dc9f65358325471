"""Reference computations for the coarse mass matrix and backward Euler on the SLOD space, built from the numpy oracle's
own matrices (oracle/slod_oracle.py) with direct solves.

    coarse_mass(orc, C)                  M_H = C^T M_h C on the structural pattern of K (the oracle's galerkin_product)
    theta_solve_coarse(K, M_H, B, g, ...)  the theta scheme (M_H + theta dt K) delta = dt (theta b(t_k) + (1 - theta)
                                           b(t_{k-1}) - K u^{k-1}), b(t) = sum_q g_q(t) B_q, Rannacher start-up included
    theta_solve_fine(orc, F, g, ...)       the same with M_h + theta dt A_h on the interior dofs of the global grid
    heat_solve_coarse / heat_solve_fine    backward Euler with a forcing constant in time: their theta = 1 case
    theta_stages(theta, dt, g, ...)        the solves of the time loop: (step, tau, coefficient of K, weights w_q)

The increment form is the one the library uses: r = tau (sum_q w_q b_q - K u^{k-1}), S delta = r, u^k = u^{k-1} + delta,
the load summed from its first term in field order as the library does."""
import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from oracle.slod_oracle import PatchShape, SlodOracle


def coarse_mass(orc, C):
    """M_H[(p,d),(q,e)] = phi_{p,d} . (M_h phi_{q,e}), M_h = the oracle's exact Q1 mass matrix (fine_norm_matrices)."""
    M = orc.fine_norm_matrices()[0]
    C = sp.csc_matrix(C)
    ones = C.copy()
    ones.data = np.ones_like(ones.data)
    return SlodOracle.galerkin_product(C, (M @ C).tocsc(), ones)


def theta_stages(theta, dt, g, n_steps, n_startup=0):
    """[(k, tau, coef, w)]: one solve of M + coef K with the load tau (sum_q w_q b_q - K u); u^k after the last solve of
    step k.  g: (n_steps + 1, n_fields) values at t_k = k dt.  A start-up step is two backward-Euler solves of dt / 2
    with the loads (g_{k-1} + g_k) / 2 and g_k."""
    g = np.asarray(g, dtype=float)
    out = []
    for k in range(1, n_steps + 1):
        if k <= n_startup:
            out.append((k, 0.5 * dt, 0.5 * dt, 0.5 * (g[k - 1] + g[k])))
            out.append((k, 0.5 * dt, 0.5 * dt, g[k].copy()))
        else:
            out.append((k, dt, theta * dt, theta * g[k] + (1.0 - theta) * g[k - 1]))
    return out


def _load(w, B):
    acc = w[0] * B[0]
    for q in range(1, len(w)):
        acc = acc + w[q] * B[q]
    return acc


def _theta_loop(apply_K, factor, B, g, u, theta, dt, n_steps, n_startup):
    """Trajectory [n_steps][n] of the theta scheme; factor(coef) -> a solver of M + coef K (cached per coefficient)."""
    B = np.zeros((1, u.size)) if B is None else np.asarray(B, dtype=float)
    g = np.ones((n_steps + 1, B.shape[0])) if g is None else np.asarray(g, dtype=float)
    solvers, out = {}, []
    for k, tau, coef, w in theta_stages(theta, dt, g, n_steps, n_startup):
        if coef not in solvers:
            solvers[coef] = factor(coef)
        u = u + solvers[coef](tau * (_load(w, B) - apply_K(u)))
        if len(out) < k:
            out.append(None)
        out[k - 1] = u.copy()
    return np.array(out)


def theta_solve_coarse(K, M_H, B, g, u0, theta, dt, n_steps, n_startup=0):
    """Trajectory [n_steps][n_coarse] of the theta scheme on the coarse space (direct solves).  B: (n_fields, n_coarse)
    loads C^T f_q or None (zero); g: (n_steps + 1, n_fields) or None (g = 1)."""
    u = np.zeros(K.shape[0]) if u0 is None else np.array(u0, dtype=float)
    return _theta_loop(lambda v: K @ v, lambda c: spla.factorized(sp.csc_matrix(M_H + c * K)), B, g, u, theta, dt,
                       n_steps, n_startup)


def heat_solve_coarse(K, M_H, b, u0, dt, n_steps):
    """Trajectory [n_steps][n_coarse] of backward Euler on the coarse space (direct solves)."""
    return theta_solve_coarse(K, M_H, None if b is None else np.asarray(b, dtype=float)[None], None, u0, 1.0, dt,
                              n_steps)


def fine_operators(orc):
    """(A_h, M_h, interior dofs) of the global grid, lexicographic numbering node * spacedim + comp."""
    pr = orc.prob
    whole = PatchShape(pr.dim, pr.spacedim, pr.n_subdivisions, (pr.N,) * pr.dim, (True,) * pr.dim, (True,) * pr.dim,
                       (0,) * pr.dim)
    A = orc.assemble_patch_stiffness(whole, (0,) * pr.dim).tocsr()
    return A, orc.fine_norm_matrices()[0], whole.internal


def theta_solve_fine(orc, F, g, u0, theta, dt, n_steps, n_startup=0):
    """Trajectory [n_steps][n_fine] of the theta scheme on the fine grid, homogeneous Dirichlet rows.  F: (n_fields,
    n_fine) or None; g as in theta_solve_coarse."""
    A, M, ii = fine_operators(orc)
    Aii, Mii = A[ii][:, ii], M[ii][:, ii]
    n = A.shape[0]
    u = np.zeros(n) if u0 is None else np.array(u0, dtype=float)
    mask = np.zeros(n, dtype=bool)
    mask[ii] = True
    u[~mask] = 0.0
    B = None if F is None else np.asarray(F, dtype=float)[:, ii]
    U = _theta_loop(lambda v: Aii @ v, lambda c: spla.factorized(sp.csc_matrix(Mii + c * Aii)), B, g, u[ii], theta, dt,
                    n_steps, n_startup)
    out = np.zeros((n_steps, n))
    out[:, ii] = U
    return out


def heat_solve_fine(orc, F, u0, dt, n_steps):
    """Trajectory [n_steps][n_fine] of backward Euler on the fine grid, homogeneous Dirichlet rows."""
    return theta_solve_fine(orc, None if F is None else np.asarray(F, dtype=float)[None], None, u0, 1.0, dt, n_steps)
