"""Rounding-error checks of the patch stages and the coarse assembly, each on the inputs that stage was given.

Every check restates one stage in extended precision (numpy longdouble, x87 80-bit here: eps 1.1e-19, four thousand
times below fp64's) from the stage's own inputs, takes the patch operators from the oracle (assemble_patch_stiffness,
projection_PT, shape.b / db / internal), and compares the stage's output entry by entry with a componentwise a priori
rounding-error bound.  Each check returns (err, bound) arrays of the same shape; err <= bound everywhere is the test.
Because the inputs are the implementation's own, the checks do not depend on how well conditioned the later stages
(the Gram selection) are, and a bound of a few hundred u still resolves a wrong summand in the smallest entry.

    stage  restatement from the stage's inputs                  bound (u = 2^-53)
    X      R = P_i - A_ii X                                     per column, normwise backward error (check_X)
    Minv   R = Minv M - I,  M = P_i^T X / H^dim                 |R| <= u |Minv| (8 Ncd |L||U||Minv||M| + Ni |P_i|^T|X| / H^dim)
    G      BD = (S_b X - P_b) Minv,  G = BD^T BD                first-order propagation through W, BD, G (check_G)
    A phi  semi phi (domain-boundary rows of semi: identity)    c_apply u |semi|~ |phi|
    K      sum over the overlap of phi_i (A phi)_j              (n_ov + 1) u sum |phi_i| |(A phi)_j|
    M_H    sum over the overlap of phi_i (M_h phi_j)            (n_ov + 3^dim + 2 dim) u sum |phi_i| (|M_h| |phi_j|)

Counting the roundings.  A computed sum of products in which every term passes through at most k roundings (its
product, the additions on its path to the result, and the rounding of its factors from exact values) is within
k u sum |terms| of the exact sum, to first order, whatever the order of the additions (Higham, Accuracy and Stability
of Numerical Algorithms, 2nd ed., section 3.1); an addition of an exact zero does not round.  The constants below are
such counts; each carries one extra u for the second-order terms and for the longdouble restatement itself.

Operator entries.  Neither the library nor the oracle forms the exact stiffness entries.  Both build them from the
sub-cell matrices at the Gauss points (a product of dim shape-function factors per gradient component, a dim-term
gradient dot product or strain contraction: at most C_K = dim^2 + 4 dim - 4 roundings from the exact rational value,
counted for elasticity, the longer of the two), sum 2^dim Gauss points, multiply by the coefficient, add the lambda
part (elasticity) and sum the 2^dim sub-cells that share the entry: at most C_ENTRY = C_K + 2 * 2^dim - 1 + [s > 1]
roundings per contribution, relative to |A|~, the assembly of the absolute values of the contributions (|A|~ >= |A|;
it is the right majorant when Gauss-point matrices of mixed sign cancel).  The check compares the library's operator
with the oracle's, so both counts enter: 2 C_ENTRY.

A applied to a vector: one product per term and at most max(3^dim s, 2^dim s + 2^dim) - 1 additions on a term's path
(a stencil row of 3^dim s entries, or the library's sub-cell-wise order: 2^dim s local terms, then 2^dim sub-cells):
C_APPLY = 2 C_ENTRY + 3^dim s + 2 (3^dim s >= 2^dim s + 2^dim - 1 for dim >= 2).

X.  The patch solvers are banded Cholesky factorisations followed by two banded triangular solves (the tensor-core
variants multiply by explicit inverses of the 8 x 8 diagonal blocks).  Each of the three steps is a sum of at most
w + 1 products per entry (w = half band width), hence a backward error of gamma_{w+1} each: the normwise backward
error of a column is at most 3 (w + 1) u (Higham, sections 10.1 and 8.1; Cholesky of a symmetric positive definite
band matrix needs no pivoting).  The library's matrix differs from the oracle's by the entry roundings above, which
adds 2 C_ENTRY u |A_ii|~ |x| to the residual.  Per column j:
    max_i |R_ij| <= 3 (w + 1) u (||A_ii||_inf ||x_j||_inf + ||p_j||_inf) + 2 C_ENTRY u || |A_ii|~ ||_inf ||x_j||_inf.
w is taken over every axis order of the interior nodes (the solvers order them x-fastest or z-fastest).

Minv.  M = P_i^T X / H^dim: P entries are exact (powers of two times 1, 2, 4, 8), H^dim is a power of two, so the
library's M is within Ni u |P_i|^T |X| / H^dim of M (a dot product of length Ni).  The inverse is a blocked Gauss-
Jordan elimination without pivoting.  Gauss-Jordan elimination is forward stable, not backward stable: its error is
|Minv - M^-1| <= 8 Ncd u |Minv| |L||U| |Minv| (Higham, section 14.4), L U = M the unpivoted LU factorisation, taken
here in longdouble, so the residual (Minv - M^-1) M carries one more factor |M|.  A residual bound without it (the
backward-stable |Minv| |L||U|) does not hold: on the high-contrast case of the parity list (cond(M) ~ 1e4) both the
library and the C++ port (partial pivoting) exceed it several times.  Together:
    |Minv M_ld - I| <= u |Minv| (8 Ncd |L||U| |Minv| |M| + Ni |P_i|^T |X| / H^dim).

G.  W = S_b X - P_b is an operator application plus one subtraction: E_W = (C_APPLY + 1) u (|S_b|~ |X| + |P_b|).
BD = W Minv is a dot product of length Ncd on a perturbed W: E_BD = E_W |Minv| + Ncd u |W| |Minv|.  G = BD^T BD is a
dot product of length Nb on a perturbed BD: E_G = |BD|^T E_BD + E_BD^T |BD| + Nb u |BD|^T |BD|.

K and M_H.  k_coarse_blocked (and k_coarse) form K[(p, d), (q, e)] as the sum over the nodes both patches hold and the
components of phi_{p,d} times (A phi)_{q,e}: the row's patch gives phi, the column's patch gives A phi, both the arrays
slod_get_all_basis returns.  With A phi given that is a dot product of n_ov terms: (n_ov + 1) u.  M_H is the same
product with M_h phi in place of A phi, and k_mass_apply forms M_h phi inside the library from the 1-D weights h/6 and
2h/3 (one rounding each), a product of dim weights (dim - 1 roundings), the product with phi and 3^dim - 1 additions:
3^dim + 2 dim - 1 roundings relative to |M_h| |phi| -- (n_ov + 3^dim + 2 dim) u in all.  An empty overlap contributes
no term: the entry must be exactly 0.0."""
import itertools
import math
import os
import sys

import numpy as np
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
from oracle.slod_oracle import _patch_extent, morton_decode  # noqa: E402

LD = np.longdouble
U = 2.0 ** -53


def c_entry(dim, s):
    c_k = dim * dim + 4 * dim - 4
    return c_k + 2 * 2 ** dim - 1 + (1 if s > 1 else 0)


def c_apply(dim, s):
    return 2 * c_entry(dim, s) + 3 ** dim * s + 2


def _abs_stiffness(orc, shape, lo):
    """assemble_patch_stiffness with the absolute value of every Gauss-point contribution: |A|~ >= |A|."""
    pr = orc.prob
    h = pr.h
    origin = (np.array(lo) * pr.n_subdivisions + shape.sub_coords) * h
    pts = origin[:, None, :] + np.array(orc.qpts)[None, :, :] * h
    if pr.problem == "diffusion":
        loc = np.einsum("sq,qij->sij", np.abs(pr.coefficients[0].at(pts)), np.abs(orc.Kq))
    else:
        loc = (np.einsum("sq,qij->sij", np.abs(pr.coefficients[1].at(pts)), np.abs(orc.Kmu)) +
               np.einsum("sq,qij->sij", np.abs(pr.coefficients[0].at(pts)), np.abs(orc.Klam)))
    nd = shape.sub_dofs.shape[1]
    rows = np.repeat(shape.sub_dofs, nd, axis=1).ravel()
    cols = np.tile(shape.sub_dofs, (1, nd)).ravel()
    A = sp.coo_matrix((loc.ravel(), (rows, cols)), shape=(shape.Nf, shape.Nf)).tocsr()
    A.sum_duplicates()
    return A


def _identity_rows(A, rows):
    A = A.tolil(copy=True)
    for j in rows:
        A.rows[j] = [int(j)]
        A.data[j] = [1.0]
    return A.tocsr()


class PatchOps:
    """The oracle's operators of one patch: A_ii, P_i, S_b, P_b, semi (and their |.|~ majorants), in longdouble."""

    def __init__(self, orc, pid):
        pr = orc.prob
        dim, ell = pr.dim, pr.oversampling
        self.pid, self.dim, self.s = pid, dim, pr.spacedim
        shape, lo = orc.shape_for(morton_decode(pid, dim, pr.n_global_refinements))
        self.shape = shape
        full = shape.Nc == (2 * ell + 1) ** dim
        lo_a = _quirk_donor_lo(orc) if pr.quirk_presaved and full else lo   # quirk B: the first full-size patch's A
        A = orc.assemble_patch_stiffness(shape, lo_a)
        Aabs = _abs_stiffness(orc, shape, lo_a)
        PT = shape.projection_PT(pr.h)
        it, b, db = shape.internal, shape.b, shape.db
        self.slod = not (not pr.stabilize or ell == 0 or pr.N ** dim == shape.Nc)
        self.Hd = LD(pr.H) ** dim
        self.Aii, self.Aii_abs = (M[it, :][:, it].tocsr() for M in (A, Aabs))
        self.Pi = PT[it, :]
        self.Sb, self.Sb_abs = (M[b, :][:, it].tocsr() for M in (A, Aabs))
        self.Pb = PT[b, :]
        self.semi = _identity_rows(A, db)
        self.semi_abs = _identity_rows(Aabs, db)
        # half band width of A_ii over every axis order of the interior node grid
        nint = [pp - 2 for pp in shape.p]
        w = 0
        for perm in itertools.permutations(range(dim)):
            stride, tot = self.s, self.s - 1
            for a in perm:
                tot += stride
                stride *= nint[a]
            w = max(w, tot)
        self.w = w


def _quirk_donor_lo(orc):
    if not hasattr(orc, "_stage_donor_lo"):
        pr = orc.prob
        for p in range(pr.N ** pr.dim):
            shape, lo = orc.shape_for(morton_decode(p, pr.dim, pr.n_global_refinements))
            if shape.Nc == (2 * pr.oversampling + 1) ** pr.dim:
                orc._stage_donor_lo = lo
                break
    return orc._stage_donor_lo


def _ld(a):
    return np.asarray(a).astype(LD)


def _spld(A):
    return sp.csr_matrix(A).astype(LD)


def check_X(ops, X, sparse_lu=False):
    """Per column: (max |P_i - A_ii X|, bound); see the module docstring.  sparse_lu: X is the oracle's, solved with a
    sparse LU factorisation of the whole constrained patch matrix (order Nf, partial pivoting on a fill-reducing order),
    not a band Cholesky: the band count 3 (w + 1) is replaced by Wilkinson's 3 Nf for LU with partial pivoting (Higham,
    Theorem 9.5), with growth factor 1 (the matrix is symmetric positive definite and diagonally dominant in its
    interior rows: the pivots are its diagonal)."""
    X = np.asarray(X)
    R = _ld(ops.Pi) - _spld(ops.Aii) @ _ld(X)
    err = np.abs(R).max(axis=0).astype(float)
    nA = np.abs(ops.Aii).sum(axis=1).max()
    nAabs = np.abs(ops.Aii_abs).sum(axis=1).max()
    xn, pn = np.abs(X).max(axis=0), np.abs(ops.Pi).max(axis=0)
    band = 3 * ops.shape.Nf if sparse_lu else 3 * (ops.w + 1)
    bound = band * U * (nA * xn + pn) + 2 * c_entry(ops.dim, ops.s) * U * nAabs * xn
    return err, bound


def _lu_abs(M):
    """|L| |U| of the unpivoted LU factorisation of M (longdouble)."""
    A = M.copy()
    n = A.shape[0]
    L = np.eye(n, dtype=LD)
    for k in range(n - 1):
        L[k + 1:, k] = A[k + 1:, k] / A[k, k]
        A[k + 1:, k:] -= np.outer(L[k + 1:, k], A[k, k:])
        A[k + 1:, k] = 0
    return np.abs(L) @ np.abs(A)


def check_Minv(ops, X, Minv):
    """(|Minv M - I|, bound) entrywise, M = P_i^T X / H^dim from the stage's X, in longdouble."""
    Xl, Ml = _ld(X), _ld(Minv)
    M = _ld(ops.Pi).T @ Xl / ops.Hd
    err = np.abs(Ml @ M - np.eye(M.shape[0], dtype=LD)).astype(float)
    ncd, ni = M.shape[0], X.shape[0]
    PX = (np.abs(ops.Pi).T @ np.abs(np.asarray(X))) / float(ops.Hd)
    aMi = np.abs(Minv)
    bound = U * (8 * ncd * aMi @ _lu_abs(M).astype(float) @ aMi @ np.abs(M).astype(float) + ni * aMi @ PX)
    return err, bound


def check_G(ops, X, Minv, G):
    """(|G - BD^T BD|, E_G), BD = (S_b X - P_b) Minv from the stage's X and Minv, in longdouble."""
    X, Minv = np.asarray(X), np.asarray(Minv)
    W = _spld(ops.Sb) @ _ld(X) - _ld(ops.Pb)
    BD = W @ _ld(Minv)
    err = np.abs(_ld(G) - BD.T @ BD).astype(float)
    ncd, nb = Minv.shape[0], ops.Pb.shape[0]
    Wf, BDa = np.abs(W).astype(float), np.abs(BD).astype(float)
    EW = (c_apply(ops.dim, ops.s) + 1) * U * (np.abs(ops.Sb_abs) @ np.abs(X) + np.abs(ops.Pb))
    EBD = EW @ np.abs(Minv) + ncd * U * Wf @ np.abs(Minv)
    bound = BDa.T @ EBD + EBD.T @ BDa + nb * U * BDa.T @ BDa
    return err, bound


def check_aphi(ops, phi, aphi):
    """(|A phi - semi phi|, c_apply u |semi|~ |phi|) on every patch dof; phi, aphi: (s, >= Nf) rows of one patch."""
    nf = ops.shape.Nf
    P = np.asarray(phi)[:, :nf]
    Y = np.asarray(aphi)[:, :nf]
    err = np.abs(_ld(Y) - (_spld(ops.semi) @ _ld(P).T).T).astype(float)
    bound = c_apply(ops.dim, ops.s) * U * (ops.semi_abs @ np.abs(P).T).T
    return err, bound


def _box_views(prob, phi, grow=0):
    """Per patch: (lo node, hi node) per axis and phi reshaped to [s][z][y][x][comp] on its node box; grow: the box
    widened by that many zero node layers, within the domain."""
    dim, s, n, N, ell = prob.dim, prob.spacedim, prob.n_subdivisions, prob.N, prob.oversampling
    out = []
    for p in range(N ** dim):
        lo, hi, m = _patch_extent(morton_decode(p, dim, prob.n_global_refinements), ell, N)
        pp = [mm * n + 1 for mm in m]
        nf = s * int(np.prod(pp))
        arr = np.asarray(phi[p])[:, :nf].reshape((s,) + tuple(pp[::-1]) + (s,))
        b0, b1 = np.array(lo) * n, (np.array(hi) + 1) * n
        g0, g1 = np.maximum(b0 - grow, 0), np.minimum(b1 + grow, N * n)
        pad = [(0, 0)] + [(int(b0[a] - g0[a]), int(g1[a] - b1[a])) for a in reversed(range(dim))] + [(0, 0)]
        out.append((g0, g1, np.pad(arr, pad)))
    return out


def mass_apply(prob, box, lo):
    """M_h on a node box with lowest global node `lo` (zero outside it), axis by axis with the 1-D weights
    (h/6, 2h/3, h/6) -- h/3 on the diagonal at the domain boundary -- in the dtype of box."""
    h = box.dtype.type(prob.h)
    wo = h / 6
    last = prob.N * prob.n_subdivisions
    out = box
    for a in range(prob.dim):
        ax = prob.dim - a                      # [s][z][y][x][comp]: axis a of the grid
        L = out.shape[ax]
        g = lo[a] + np.arange(L)
        wd = np.where((g == 0) | (g == last), h / 3, 2 * h / 3).astype(box.dtype)
        wd = wd.reshape([L if k == ax else 1 for k in range(out.ndim)])
        pad = [(0, 0)] * out.ndim
        pad[ax] = (1, 1)
        q = np.pad(out, pad)
        sl = lambda a0, a1: tuple(slice(a0, a1) if k == ax else slice(None) for k in range(out.ndim))
        out = wo * q[sl(0, L)] + wd * q[sl(1, L + 1)] + wo * q[sl(2, L + 2)]
    return out


def check_coarse(prob, phi, csr, aphi=None, rows=None):
    """Every stored entry of the coarse rows `rows` (all when None) of K (aphi given: the column patch's A phi) or of
    M_H (aphi None: M_h phi formed here in longdouble).  phi, aphi: [n_patches][s][>= Nf].  csr: (rowptr, col, val).
    Returns (err, bound) over the checked entries in CSR order."""
    dim, s = prob.dim, prob.spacedim
    rowptr, col, val = csr
    P = _box_views(prob, phi)
    if aphi is None:
        # M_h phi on the box widened by one node layer, with the domain-boundary weights: C^T M_h C whatever phi holds on
        # the box and domain boundaries (the library's phi is exactly zero there, and k_mass_apply stays on the box with
        # the interior weights; a chain with rounding residue there does not)
        Yp = _box_views(prob, phi, grow=1)
        Y = [(lo, hi, mass_apply(prob, a.astype(LD), lo)) for lo, hi, a in Yp]
        Yabs = [mass_apply(prob, np.abs(a), lo) for lo, _, a in Yp]
        extra = 3 ** dim + 2 * dim
    else:
        Y = _box_views(prob, aphi)
        Yabs = [np.abs(a) for _, _, a in Y]
        extra = 1
    n_patch = len(P)
    rows = range(n_patch * s) if rows is None else rows
    errs, bounds = [], []
    for r in rows:
        p, d = divmod(int(r), s)
        lo_p, hi_p, ap = P[p]
        for k in range(rowptr[r], rowptr[r + 1]):
            q, e = divmod(int(col[k]), s)
            lo_q, hi_q, aq = Y[q]
            b0, b1 = np.maximum(lo_p, lo_q), np.minimum(hi_p, hi_q)
            if (b1 < b0).any():
                errs.append(abs(val[k]))
                bounds.append(0.0)
                continue
            cut = lambda lo: (slice(None),) + tuple(slice(b0[a] - lo[a], b1[a] - lo[a] + 1) for a in reversed(range(dim)))
            x = ap[cut(lo_p)][d]
            y = aq[cut(lo_q)][e]
            ya = Yabs[q][cut(lo_q)][e]
            ref = (x.astype(LD) * y.astype(LD)).sum()
            n_ov = x.size
            errs.append(float(abs(LD(val[k]) - ref)))
            bounds.append((n_ov + extra) * U * float((np.abs(x) * ya).sum()))
    return np.array(errs), np.array(bounds)


def patch_class(prob, pid):
    """Number of axes on which the patch is cut by the domain boundary: 0 interior, 1 face, 2 edge, 3 corner."""
    lo, hi, _ = _patch_extent(morton_decode(pid, prob.dim, prob.n_global_refinements), prob.oversampling, prob.N)
    return sum(1 for a in range(prob.dim) if lo[a] == 0 or hi[a] == prob.N - 1)


def sample_patches(prob, at_least=32):
    """Every patch up to 256 patches; otherwise at least `at_least` spread evenly over the patch classes."""
    n = prob.N ** prob.dim
    if n <= 256:
        return list(range(n))
    by_class = {}
    for p in range(n):
        by_class.setdefault(patch_class(prob, p), []).append(p)
    per = math.ceil(at_least / len(by_class))
    out = []
    for ids in by_class.values():
        k = min(per, len(ids))
        out += [ids[int(i)] for i in np.linspace(0, len(ids) - 1, k).round()]
    return sorted(set(out))


def ratio(err, bound):
    """max err / bound (0 / 0 = 0: an exact zero where nothing may round)."""
    err, bound = np.asarray(err, dtype=float), np.asarray(bound, dtype=float)
    if err.size == 0:
        return 0.0
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(err == 0.0, 0.0, err / bound)
    return float(r.max())
