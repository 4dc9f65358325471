"""slod_update_basis without a GPU: the symbol, the maps-only refusal, and the restatement of which patches an update
recomputes (tools/update_expect.py), pinned on hand-worked cases so that tests/test_update_gpu.py can rely on it."""
import importlib
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from update_expect import changed_cells, device_coefficients, expected_patches  # noqa: E402

pkg = importlib.import_module("dealii-slod_b200")


def morton2(x, y, ref):
    code = 0
    for b in range(ref):
        code |= ((x >> b) & 1) << (2 * b) | ((y >> b) & 1) << (2 * b + 1)
    return code


def maps(dim=2, s=1, ref=3, n=2, ell=1, quirk=False):
    return pkg.SlodContext(dim=dim, spacedim=s, n_global_refinements=ref, n_subdivisions=n, oversampling=ell,
                           stabilize=True, problem=0 if s == 1 else 1, quirk_presaved=quirk, device=-2)


def centres(xs, ys, ref=3):
    return sorted(morton2(x, y, ref) for x in xs for y in ys)


def test_symbol_exported():
    pkg.build_library()
    lib = pkg.load_library()
    assert "slod_update_basis" in pkg.EXPORTS
    assert lib.slod_update_basis is not None


def test_maps_only_handle_refuses():
    pkg.build_library()
    ctx = maps()
    with pytest.raises(pkg.SlodError) as e:
        ctx.update_basis()
    assert e.value.code == 3


def table(r, dim=2, seed=0):
    return np.random.default_rng(seed).uniform(1.0, 100.0, (2 ** r) ** dim)


def test_one_cell_interior():
    """N = 8, n = 2, table on the 16 x 16 sub-cells: coarse cell (3, 4) = sub-cells x 6..7, y 8..9; the patches that
    read it are the 3 x 3 centres around it."""
    ctx = maps()
    t0 = table(4)
    t1 = t0.copy()
    t1[8 * 16 + 7] *= 2.0     # sub-cell (7, 8)
    got = expected_patches(ctx, 2, 3, 2, 1, ([t0], 4), ([t1], 4))
    assert got == centres(range(2, 5), range(3, 6))


def test_corner_and_coarse_table():
    ctx = maps()
    t0 = table(3)
    t1 = t0.copy()
    t1[0] = 5.0               # coarse cell (0, 0): centres (0..1, 0..1)
    assert expected_patches(ctx, 2, 3, 2, 1, ([t0], 3), ([t1], 3)) == centres(range(2), range(2))
    # a table coarser than the sub-cells: table cell (1, 0) of 2 x 2 covers coarse cells x 4..7, y 0..3
    c0 = table(1)
    c1 = c0.copy()
    c1[1] += 1.0
    assert expected_patches(ctx, 2, 3, 2, 1, ([c0], 1), ([c1], 1)) == centres(range(3, 8), range(0, 5))


def test_bitwise_rule():
    ctx = maps()
    t0 = table(4)
    t0[5] = 0.0
    t1 = t0.copy()
    t1[5] = -0.0              # sub-cell (5, 0) = coarse cell (2, 0): counts
    assert expected_patches(ctx, 2, 3, 2, 1, ([t0], 4), ([t1], 4)) == centres(range(1, 4), range(0, 2))
    assert expected_patches(ctx, 2, 3, 2, 1, ([t0], 4), ([t0.copy()], 4)) == []


def test_gauss_lookup():
    """N = 4, n = 2 (8 sub-cells per axis) and a 32 x 32 table: ratio 4, the Gauss points sample table cells
    4 x + floor(0.211 * 4) = 4 x and 4 x + floor(0.789 * 4) = 4 x + 3; cells 4 x + 1 and 4 x + 2 are never read."""
    ctx = maps(ref=2)
    t0 = table(5)
    a = device_coefficients(2, 2, 2, [t0], 5)
    assert a.shape == (1, 1, 8, 8, 4)
    assert a[0, 0, 0, 1, 0] == t0[4] and a[0, 0, 0, 1, 1] == t0[7] and a[0, 0, 1, 0, 2] == t0[7 * 32 + 0]
    t1 = t0.copy()
    t1[1] = t1[2] = t1[32 + 1] = 7.0          # unsampled
    assert expected_patches(ctx, 2, 2, 2, 1, ([t0], 5), ([t1], 5)) == []
    t2 = t0.copy()
    t2[3 * 32 + 11] = 7.0                     # x 11 = 4 * 2 + 3: sub-cell (2, 0), coarse cell (1, 0)
    assert expected_patches(ctx, 2, 2, 2, 1, ([t0], 5), ([t2], 5)) == centres(range(0, 3), range(0, 2), ref=2)


def test_layout_change_recomputes_everything():
    ctx = maps(ref=2)
    t = table(3)
    assert changed_cells(2, 2, 2, ([t], 3), ([table(5)], 5)) is None      # per sub-cell -> per Gauss point
    assert expected_patches(ctx, 2, 2, 2, 1, ([t], 3), ([table(5)], 5)) == list(range(16))
    # same layout at another eta: the values decide
    t2 = np.repeat(np.repeat(table(2).reshape(4, 4), 2, axis=0), 2, axis=1).ravel()
    assert expected_patches(ctx, 2, 2, 2, 1, ([table(2)], 2), ([t2], 3)) == []


def test_quirk_donor_window():
    """quirk B, N = 8, ell = 1: the first full-size patch in id order is centre (1, 1), window cells 0..2; every
    full-size patch (centres 1..6) reads that window instead of its own."""
    ctx = maps(quirk=True)
    t0 = table(3)
    t1 = t0.copy()
    t1[0] = 3.0               # cell (0, 0): inside the donor window
    got = expected_patches(ctx, 2, 3, 2, 1, ([t0], 3), ([t1], 3), quirk=True)
    assert got == sorted(set(centres(range(1, 7), range(1, 7)) + centres(range(2), range(2))))
    t2 = t0.copy()
    t2[6 * 8 + 6] = 3.0       # cell (6, 6): only the non-full patches around it
    got = expected_patches(ctx, 2, 3, 2, 1, ([t0], 3), ([t2], 3), quirk=True)
    assert got == sorted(set(centres(range(5, 8), range(5, 8))) - set(centres(range(1, 7), range(1, 7))))
    assert len(got) == 5


def test_elasticity_fields_and_3d():
    ctx = maps(s=2)
    lam, mu = table(3, seed=1), table(3, seed=2)
    mu2 = mu.copy()
    mu2[3 * 8 + 4] = 1.0      # only mu, cell (4, 3)
    assert expected_patches(ctx, 2, 3, 2, 1, ([lam, mu], 3), ([lam, mu2], 3)) == centres(range(3, 6), range(2, 5))
    ctx3 = maps(dim=3, ref=2, ell=1)
    t0 = table(2, dim=3)
    t1 = t0.copy()
    t1[(3 * 4 + 0) * 4 + 1] = 1.0   # cell (1, 0, 3)
    got = expected_patches(ctx3, 3, 2, 2, 1, ([t0], 2), ([t1], 2))
    want = []
    for pid in range(64):
        c = [sum(((pid >> (3 * b + a)) & 1) << b for b in range(2)) for a in range(3)]
        if abs(c[0] - 1) <= 1 and abs(c[1] - 0) <= 1 and abs(c[2] - 3) <= 1:
            want.append(pid)
    assert got == want and len(want) == 12
