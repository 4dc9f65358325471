"""Restatement of which patches slod_update_basis recomputes (include/slod.h), for the tests.

Tables -> device coefficient array (the expansion of prepare_coefficients in csrc/capi.cu: one value per sub-cell, or
one per Gauss point of the 2-point rule once a table is finer than the sub-cells, looked up at floor(gp * ratio)) ->
coarse cells holding a bitwise-changed value -> patches whose coefficient window (the coarse cells of the patch box;
under quirk_presaved the box of the first full-size patch for every full-size patch) contains such a cell."""
import numpy as np

GP = (0.5 - 0.5 / np.sqrt(3.0), 0.5 + 0.5 / np.sqrt(3.0))


def device_coefficients(dim, ref, n, tables, r):
    """[fields][z][y][x][q] array of what the kernels read; tables: one flat table per field on (2^r)^dim cells."""
    nsub = (2 ** ref) * n
    nl = 2 ** r
    gauss = nl > nsub
    nq = 2 ** dim if gauss else 1
    out = []
    for tab in tables:
        t = np.asarray(tab, dtype=np.float64).reshape((nl,) * dim)   # [z][y][x] / [y][x]
        sub = np.arange(nsub)
        per_q = []
        for q in range(nq):
            idx = []
            for a in range(dim):   # axis a: bit a of q
                if nl <= nsub:
                    idx.append(sub // (nsub // nl))
                else:
                    ratio = nl // nsub
                    idx.append(sub * ratio + int(np.floor(GP[(q >> a) & 1] * ratio)))
            # t is indexed [z][y][x]: axis a of the table is dimension dim - 1 - a
            grid = np.ix_(*reversed(idx))
            per_q.append(t[grid])
        f = np.stack(per_q, axis=-1)
        if dim == 2:
            f = f[None]
        out.append(f)
    return np.stack(out)


def changed_cells(dim, ref, n, old, new):
    """Boolean [N]*3 array (z, y, x; z of size 1 in 2-D) of coarse cells with a bitwise change, or None when the
    layout of the device array differs (every patch is recomputed).  old / new: (tables, r)."""
    a = device_coefficients(dim, ref, n, *old)
    b = device_coefficients(dim, ref, n, *new)
    if a.shape != b.shape:
        return None
    diff = (a.view(np.uint64) != b.view(np.uint64)).any(axis=(0, 4))   # [z][y][x] sub-cells
    N = 2 ** ref
    if dim == 3:
        return diff.reshape(N, n, N, n, N, n).any(axis=(1, 3, 5))
    return diff.reshape(1, N, n, N, n).any(axis=(2, 4))


def coefficient_windows(ctx, ell, quirk):
    """Per patch: (lo, m), padded to 3 axes, of the coefficient window it reads."""
    full = 2 * ell + 1
    wins, is_full = [], []
    for pid in range(ctx.n_patches):
        info = ctx.patch_info(pid)
        pad = 3 - len(info["lo"])
        wins.append((list(info["lo"]) + [0] * pad, list(info["m"]) + [1] * pad))
        is_full.append(all(x == full for x in info["m"]))
    if quirk:   # the first full-size patch in patch-id order donates its window to every full-size patch
        donor = next((lo for (lo, m), f in zip(wins, is_full) if f), None)
        if donor is not None:
            wins = [(donor if f else lo, m) for (lo, m), f in zip(wins, is_full)]
    return wins


def expected_patches(ctx, dim, ref, n, ell, old, new, quirk=False):
    """Sorted patch ids slod_update_basis recomputes for a change of the tables from old to new ((tables, r) each)."""
    cells = changed_cells(dim, ref, n, old, new)
    if cells is None:
        return list(range(ctx.n_patches))
    return [pid for pid, (lo, m) in enumerate(coefficient_windows(ctx, ell, quirk))
            if cells[lo[2]:lo[2] + m[2], lo[1]:lo[1] + m[1], lo[0]:lo[0] + m[0]].any()]
