"""Reference computations for the coarse mass matrix and backward Euler on the SLOD space, built from the numpy oracle's
own matrices (oracle/slod_oracle.py) with direct solves.

    coarse_mass(orc, C)                  M_H = C^T M_h C on the structural pattern of K (the oracle's galerkin_product)
    heat_solve_coarse(K, M_H, b, ...)    (M_H + dt K) u^k = M_H u^{k-1} + dt b, in increment form
    heat_solve_fine(orc, F, ...)         (M_h + dt A_h) u^k = M_h u^{k-1} + dt F on the interior dofs of the global grid

The increment form is the one the library uses: r = dt (b - K u^{k-1}), S delta = r, u^k = u^{k-1} + delta."""
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


def heat_solve_coarse(K, M_H, b, u0, dt, n_steps):
    """Trajectory [n_steps][n_coarse] of backward Euler on the coarse space (direct solves)."""
    solve = spla.factorized(sp.csc_matrix(M_H + dt * K))
    u = np.zeros(K.shape[0]) if u0 is None else np.array(u0, dtype=float)
    b = np.zeros(K.shape[0]) if b is None else np.asarray(b, dtype=float)
    out = []
    for _ in range(n_steps):
        u = u + solve(dt * (b - K @ u))
        out.append(u.copy())
    return np.array(out)


def fine_operators(orc):
    """(A_h, M_h, interior dofs) of the global grid, lexicographic numbering node * spacedim + comp."""
    pr = orc.prob
    whole = PatchShape(pr.dim, pr.spacedim, pr.n_subdivisions, (pr.N,) * pr.dim, (True,) * pr.dim, (True,) * pr.dim,
                       (0,) * pr.dim)
    A = orc.assemble_patch_stiffness(whole, (0,) * pr.dim).tocsr()
    return A, orc.fine_norm_matrices()[0], whole.internal


def heat_solve_fine(orc, F, u0, dt, n_steps):
    """Trajectory [n_steps][n_fine] of the same scheme on the fine grid, homogeneous Dirichlet rows."""
    A, M, ii = fine_operators(orc)
    Aii, Mii = A[ii][:, ii], M[ii][:, ii]
    solve = spla.factorized(sp.csc_matrix(Mii + dt * Aii))
    n = A.shape[0]
    u = np.zeros(n) if u0 is None else np.array(u0, dtype=float)
    mask = np.zeros(n, dtype=bool)
    mask[ii] = True
    u[~mask] = 0.0
    f = np.zeros(n) if F is None else np.asarray(F, dtype=float)
    out = []
    for _ in range(n_steps):
        u[ii] += solve(dt * (f[ii] - Aii @ u[ii]))
        out.append(u.copy())
    return np.array(out)
