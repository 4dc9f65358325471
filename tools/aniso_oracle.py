"""Reference restatement of the tensor-diffusion problem (SLOD_PROBLEM_DIFFUSION_TENSOR) on top of the numpy oracle.

-div(A grad u) with a symmetric positive definite tensor A per coefficient cell.  The coefficient is d (d + 1) / 2
CoefficientTables in Voigt order (2-D a_xx, a_yy, a_xy; 3-D a_xx, a_yy, a_zz, a_yz, a_xz, a_xy).  The sub-cell matrix
is sum_f a_f K_f with K_f = d_a N_i d_b N_j (+ d_b N_i d_a N_j for a != b) for component f = (a, b), integrated with
the 2-point Gauss rule per axis like the scalar problem.  Everything else (projection, Gram matrix, selection, coarse
product) is the scalar oracle's: the coefficient enters only through the patch stiffness.
"""
from __future__ import annotations

import itertools
import math
import os
import sys

import numpy as np
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle.slod_oracle import CoefficientTable, PatchShape, SlodOracle, SlodProblem  # noqa: E402

VOIGT = {2: [(0, 0), (1, 1), (0, 1)], 3: [(0, 0), (1, 1), (2, 2), (1, 2), (0, 2), (0, 1)]}


def tensor_component_matrices(dim: int, h: float):
    """(gauss_unit_points, K[q][f][i][j]): the component matrices at each Gauss point, local nodes lexicographic."""
    g = 0.5 / math.sqrt(3.0)
    pts1 = (0.5 - g, 0.5 + g)
    qpts = [tuple(reversed(q)) for q in itertools.product(*([pts1] * dim))]
    nodes = [tuple(reversed(v)) for v in itertools.product(*([(0, 1)] * dim))]
    jxw = (h / 2.0) ** dim
    K = np.zeros((len(qpts), len(VOIGT[dim]), len(nodes), len(nodes)))
    for qi, x in enumerate(qpts):
        G = np.empty((len(nodes), dim))
        for i, nd in enumerate(nodes):
            for a in range(dim):
                val = 1.0
                for b in range(dim):
                    val *= ((1.0 if nd[b] else -1.0) / h) if b == a else (x[b] if nd[b] else 1.0 - x[b])
                G[i, a] = val
        for f, (a, b) in enumerate(VOIGT[dim]):
            K[qi, f] = (np.outer(G[:, a], G[:, a]) if a == b
                        else np.outer(G[:, a], G[:, b]) + np.outer(G[:, b], G[:, a])) * jxw
    return qpts, K


class TensorSlodOracle(SlodOracle):
    """SlodOracle for problem "diffusion_tensor": prob.coefficients holds the Voigt components' tables."""

    def __init__(self, prob: SlodProblem):
        assert prob.problem == "diffusion_tensor" and prob.spacedim == 1
        assert len(prob.coefficients) == len(VOIGT[prob.dim])
        self.prob = prob
        self._shapes = {}
        self._presaved = None
        self.qpts, self.Kt = tensor_component_matrices(prob.dim, prob.h)
        self.patches = []

    def assemble_patch_stiffness(self, shape: PatchShape, lo):
        pr = self.prob
        h = pr.h
        origin = (np.array(lo) * pr.n_subdivisions + shape.sub_coords) * h
        pts = origin[:, None, :] + np.array(self.qpts)[None, :, :] * h              # (n_sub, nq, dim)
        loc = 0.0
        for f, tab in enumerate(pr.coefficients):
            loc = loc + np.einsum("sq,qij->sij", tab.at(pts), self.Kt[:, f])
        nd = shape.sub_dofs.shape[1]
        rows = np.repeat(shape.sub_dofs, nd, axis=1).ravel()
        cols = np.tile(shape.sub_dofs, (1, nd)).ravel()
        A = sp.coo_matrix((loc.ravel(), (rows, cols)), shape=(shape.Nf, shape.Nf)).tocsr()
        A.sum_duplicates()
        return A


def make_oracle(dim, ref, n, ell, stabilize, r, tensors, quirk_presaved=False):
    """Oracle of a tensor problem from a (n_cells, ncomp) table on the 2^r grid (the C ABI's layout)."""
    tensors = np.asarray(tensors, dtype=float)
    prob = SlodProblem(dim=dim, spacedim=1, n_global_refinements=ref, n_subdivisions=n, oversampling=ell,
                       stabilize=stabilize, problem="diffusion_tensor", quirk_presaved=quirk_presaved,
                       coefficients=[CoefficientTable(dim, r, tensors[:, f].copy()) for f in range(tensors.shape[1])])
    return TensorSlodOracle(prob)


def laminate(dim, r, contrast=100.0, angle=math.pi / 6, seed=0):
    """A rotated laminate of the given contrast on the 2^r grid: layers normal to the unit vector nu (angle in the x-y
    plane; in 3-D tilted by angle / 2 towards z) alternate between conductivities 1 and `contrast` across the layers,
    with conductivity 1 along them, plus a small random isotropic part so that no two cells repeat exactly.  Returns
    (n_cells, ncomp) in Voigt order."""
    nl = 2 ** r
    rng = np.random.default_rng(seed)
    if dim == 2:
        nu = np.array([math.cos(angle), math.sin(angle)])
    else:
        nu = np.array([math.cos(angle) * math.cos(angle / 2), math.sin(angle) * math.cos(angle / 2), math.sin(angle / 2)])
    centres = np.stack(np.meshgrid(*[(np.arange(nl) + 0.5) / nl] * dim, indexing="ij"), axis=-1)
    centres = np.transpose(centres, tuple(reversed(range(dim))) + (dim,)).reshape(-1, dim)   # x fastest
    layer = np.floor(centres @ nu * 8.0).astype(int) % 2
    across = np.where(layer == 1, contrast, 1.0)
    out = np.empty((nl ** dim, len(VOIGT[dim])))
    for c in range(nl ** dim):
        A = np.eye(dim) + (across[c] - 1.0) * np.outer(nu, nu) + 0.1 * rng.random() * np.eye(dim)
        out[c] = [A[a, b] for a, b in VOIGT[dim]]
    return out


def manufactured(dim, A):
    """u = prod_a sin(pi x_a) (zero on the boundary) and f = -div(A grad u) for a constant symmetric tensor A: the pair
    a convergence test of the fine FEM uses to pin the factor of every tensor component, the off-diagonal ones included.
    Returns (u(points), f(points)) as functions of points [npts, dim]."""
    A = np.asarray(A, dtype=float)

    def u(p):
        return np.prod(np.sin(np.pi * p), axis=1)

    def f(p):
        s, c = np.sin(np.pi * p), np.cos(np.pi * p)
        out = np.zeros(len(p))
        for a in range(dim):
            for b in range(dim):
                # d_a d_b u = -pi^2 u (a == b), pi^2 c_a c_b prod_{other} s (a != b)
                if a == b:
                    d2 = -np.pi ** 2 * np.prod(s, axis=1)
                else:
                    d2 = np.pi ** 2 * c[:, a] * c[:, b] * np.prod(np.delete(s, [a, b], axis=1), axis=1)
                out -= A[a, b] * d2
        return out
    return u, f


def grid_points(dim, G):
    """Fine nodes of the (G - 1)^dim sub-cell grid on the unit cube, lexicographic x fastest: [G^dim, dim]."""
    g = np.linspace(0.0, 1.0, G)
    mesh = np.meshgrid(*[g] * dim, indexing="ij")
    return np.stack([m.transpose(tuple(reversed(range(dim)))).ravel() for m in mesh], axis=-1)
