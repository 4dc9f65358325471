"""slod_update_basis on the GPU: after a change of the coefficient tables, an update must leave the basis, the
diagnostics and the coarse matrix bit-identical to a fresh handle that computes everything from the same tables, and it
must recompute exactly the patches the restatement in tools/update_expect.py names."""
import importlib
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from parity_common import check_plan, make_tables  # noqa: E402
from update_expect import expected_patches  # noqa: E402

pkg = importlib.import_module("dealii-slod_b200")
pytestmark = pytest.mark.gpu

V0_SIMT = dict(mma_variant=0, dense_ntile=0)
V1_T4 = dict(mma_variant=1, dense_ntile=4)
V2_T8 = dict(mma_variant=2, dense_ntile=8)
SPLIT = dict(mma_variant=0, split_solver=1, dense_ntile=16)
GMEM = dict(mma_variant=-1, gmem_window=1, dense_ntile=0, dense_coef_gmem=1)

CASES = [
    dict(id="2d_l1", dim=2, s=1, ref=4, n=2, ell=1, plan=dict(V1_T4, coarse_blocked=1)),
    dict(id="2d_l2", dim=2, s=1, ref=4, n=2, ell=2, plan=V1_T4),
    dict(id="elasticity_l2", dim=2, s=2, ref=4, n=2, ell=2, plan=V2_T8),
    dict(id="3d_l1", dim=3, s=1, ref=3, n=2, ell=1, plan=V0_SIMT),
    dict(id="3d_l2_split", dim=3, s=1, ref=3, n=2, ell=2, kind="uniform1e4", seed=3001, plan=SPLIT),
    dict(id="gauss", dim=2, s=1, ref=3, n=2, ell=1, r=6, plan=dict(V1_T4, gauss_coef=1)),
    dict(id="coarse_table", dim=2, s=2, ref=3, n=2, ell=1, r=2, plan=dict(V1_T4, gauss_coef=0)),
    dict(id="quirk", dim=2, s=1, ref=4, n=2, ell=2, quirk=True, plan=V1_T4),
    dict(id="lod", dim=2, s=1, ref=3, n=2, ell=1, stabilize=False, plan=V1_T4),
    dict(id="gmem", dim=2, s=1, ref=3, n=2, ell=1, env=("SLOD_FORCE_GMEM_SOLVER", "1"), plan=GMEM),
    dict(id="simple_coarse", dim=2, s=2, ref=3, n=2, ell=1, env=("SLOD_SIMPLE_COARSE", "1"),
         plan=dict(coarse_blocked=0)),
    dict(id="chunk7", dim=3, s=1, ref=2, n=2, ell=1, env=("SLOD_CHUNK", "7"), plan=V0_SIMT),
]


def table_r(case):
    return case.get("r", case["ref"] + int(np.log2(case["n"])))


def make_ctx(case, tables, r):
    ctx = pkg.SlodContext(dim=case["dim"], spacedim=case["s"], n_global_refinements=case["ref"],
                          n_subdivisions=case["n"], oversampling=case["ell"], stabilize=case.get("stabilize", True),
                          problem=0 if case["s"] == 1 else 1, quirk_presaved=case.get("quirk", False))
    for f, t in enumerate(tables):
        ctx.set_coefficient(f, r, t)
    return ctx


def fresh(case, tables, r, coarse=True):
    ctx = make_ctx(case, tables, r)
    ctx.compute_basis()
    if coarse:
        ctx.assemble_coarse()
    return ctx


def state(ctx, path, coarse=True):
    """phi, A phi, the diagnostics of every patch, CSR of K, and the checkpoint bytes (phi, A phi and the block-ELL rows
    of K with their zero slots)."""
    phi, aphi = ctx.all_basis()
    out = {"phi": phi.copy(), "aphi": aphi.copy(),
           "diag": np.array([[ctx.diagnostics(p, d) for d in range(ctx.s)] for p in range(ctx.n_patches)])}
    if coarse:
        out.update(zip(("rowptr", "col", "val"), (a.copy() for a in ctx.coarse_csr())))
    ctx.save_state(str(path))
    out["checkpoint"] = np.fromfile(str(path), dtype=np.uint8)
    return out


def assert_same(a, b):
    assert a.keys() == b.keys()
    for k in a:
        assert np.array_equal(a[k], b[k]), k


def needed_rows(ctx, ids):
    rowptr, col, _ = ctx.coarse_csr()
    s = ctx.s
    return {int(c) // s for q in ids for c in col[rowptr[q * s]:rowptr[q * s + 1]]}


def update_and_check(ctx, case, old, new, tmp_path, coarse=True):
    """Apply the tables `new` ((tables, r)), update, check counts against the restatement and results against a fresh
    handle; returns the recomputed patches."""
    for f, t in enumerate(new[0]):
        ctx.set_coefficient(f, new[1], t)
    l0 = ctx.launch_count
    got = ctx.update_basis()
    exp = expected_patches(ctx, case["dim"], case["ref"], case["n"], case["ell"], old, new, case.get("quirk", False))
    assert got["patches"] == len(exp)
    tm = ctx.timings()
    if not exp:
        assert got["row_blocks"] == 0 and ctx.launch_count == l0 + 1     # the comparison kernel only
        assert not tm[:5].any()
    else:
        assert (tm[:4] >= 0).all() and tm[:4].sum() > 0
        if coarse:
            need = needed_rows(ctx, exp)
            group = 2 ** case["dim"]
            rounded = {p // group * group + k for p in need for k in range(group)}
            assert len(need) <= got["row_blocks"] <= len(rounded)
            assert tm[4] > 0
        else:
            assert got["row_blocks"] == 0
    ref = fresh(case, *new, coarse=coarse)
    assert_same(state(ctx, tmp_path / "a.bin", coarse), state(ref, tmp_path / "b.bin", coarse))
    return exp


def coarse_cell_slices(case, r, cell):
    """Table index ranges (z, y, x) of coarse cell `cell` (x, y, z): a table coarser than the coarse cells gives the one
    table cell that covers it."""
    N, nl = 2 ** case["ref"], 2 ** r
    sl = []
    for a in range(case["dim"]):
        if nl >= N:
            k = nl // N
            sl.append(slice(cell[a] * k, (cell[a] + 1) * k))
        else:
            c = cell[a] * nl // N
            sl.append(slice(c, c + 1))
    return tuple(reversed(sl))


def with_cell(case, tables, r, cell, fn, fields=None):
    out = []
    for f, t in enumerate(tables):
        t = t.copy()
        if fields is None or f in fields:
            v = t.reshape((2 ** r,) * case["dim"])
            sl = coarse_cell_slices(case, r, cell)
            v[sl] = fn(v[sl])
        out.append(t)
    return out


@pytest.mark.parametrize("case", CASES, ids=[c["id"] for c in CASES])
def test_update_matches_fresh(case, tmp_path, monkeypatch):
    if "env" in case:
        monkeypatch.setenv(*case["env"])
    dim, r = case["dim"], table_r(case)
    N = 2 ** case["ref"]
    tables = make_tables(dim, case["s"], r, case.get("kind", "uniform100"), case.get("seed", 1234))
    ctx = fresh(case, tables, r)
    check_plan(ctx, case["plan"])
    cur = (tables, r)

    def step(new_tables, new_r=None):
        nonlocal cur
        new = (new_tables, cur[1] if new_r is None else new_r)
        exp = update_and_check(ctx, case, cur, new, tmp_path)
        cur = new
        return exp

    assert step(cur[0]) == []                                                   # nothing changed
    # one table entry in the middle (one sub-cell where the table resolves the sub-cells)
    nl = 2 ** r
    one = [t.copy() for t in cur[0]]
    one[0][np.ravel_multi_index((nl // 2,) * dim, (nl,) * dim)] *= 1.7
    exp = step(one)
    # under quirk B every full-size patch reads the donor window, which this cell lies outside of
    assert len(exp) > 0 or case.get("quirk")
    assert len(step(with_cell(case, cur[0], r, (N - 1,) * 3, lambda v: v * 0 + 50.0))) > 0   # domain corner
    # a cell just outside the box of the patch centred at (ell, ..., ell): that patch is not recomputed
    ell = case["ell"]
    if 2 * ell + 1 < N:
        centre = [ell] * dim
        pid = sum(((centre[a] >> b) & 1) << (dim * b + a) for b in range(case["ref"]) for a in range(dim))
        exp = step(with_cell(case, cur[0], r, (2 * ell + 1,) + (ell,) * 2, lambda v: v * 1.5, fields={0}))
        assert len(exp) > 0
        if nl >= N:      # else the table cell covers cells inside the box too
            assert pid not in exp
    if case.get("quirk"):
        exp = step(with_cell(case, cur[0], r, (1,) * 3, lambda v: v + 1.0))        # inside the donor window
        assert len(exp) > 0
    if case["s"] == 2:
        assert len(step(with_cell(case, cur[0], r, (N // 2,) * 3, lambda v: v * 0.5, fields={1}))) > 0   # mu only
    if r >= case["ref"] + int(np.log2(case["n"])):
        # 0.0 -> -0.0 on one table cell at sub-cell resolution or finer (a zero coarse cell would make A_ii singular);
        # under quirk B in coarse cell (1, ..., 1), inside the donor window, elsewhere in the middle
        at = np.ravel_multi_index((nl // N if case.get("quirk") else nl // 2,) * dim, (nl,) * dim)
        z = [t.copy() for t in cur[0]]
        z[0][at] = 0.0
        step(z)
        nz = [t.copy() for t in z]
        nz[0][at] = -0.0
        assert len(step(nz)) > 0
    if r - (case["ref"] + int(np.log2(case["n"]))) >= 2:
        un = [t.copy() for t in cur[0]]
        un[0][1] = 12345.0           # x = 1 of a table with 4+ cells per sub-cell: no Gauss point samples it
        assert step(un) == []
    assert len(step([t * 1.25 for t in cur[0]])) == ctx.n_patches             # every cell
    eta = make_tables(dim, case["s"], r - 1, case.get("kind", "uniform100"), 99)
    assert len(step(eta, r - 1)) == ctx.n_patches                              # another eta_refinement


def test_sequence_with_online_and_heat(tmp_path):
    """Five updates of a moving high-contrast inclusion; coarse and heat solves in between; M_H is stale after each."""
    case = dict(dim=2, s=1, ref=4, n=2, ell=2)
    r = 5
    base = np.ones((2 ** r) ** 2)
    ctx = fresh(case, [base], r)
    cur = ([base], r)
    f = np.ones(ctx.n_fine)
    for k in range(5):
        t = base.reshape(32, 32).copy()
        t[6:10, 4 + 2 * k:8 + 2 * k] = 1e4
        new = ([t.ravel()], r)
        update_and_check(ctx, case, cur, new, tmp_path)
        cur = new
        with pytest.raises(pkg.SlodError) as e:
            ctx.heat_solve(None, np.zeros(ctx.n_patches), 0.01, 2)
        assert e.value.code == 4
        u, _, _ = ctx.coarse_solve(ctx.coarse_rhs(f))
        ctx.assemble_coarse_mass()
        U, _ = ctx.heat_solve(f, u, 0.01, 2)
        assert np.isfinite(U).all()


def test_baseline_survives_fem_solve(tmp_path):
    case = dict(dim=2, s=1, ref=3, n=2, ell=1)
    t0 = make_tables(2, 1, 4, "uniform100", 5)
    ctx = fresh(case, t0, 4)
    t1 = [t0[0].copy()]
    t1[0][40] = 3.0
    ctx.set_coefficient(0, 4, t1[0])
    ctx.fem_solve(np.ones(ctx.n_fine))          # expands the new tables onto the device array
    ctx.fine_norms(np.ones(ctx.n_fine))
    got = ctx.update_basis()
    exp = expected_patches(ctx, 2, 3, 2, 1, (t0, 4), (t1, 4))
    assert got["patches"] == len(exp) > 0
    assert_same(state(ctx, tmp_path / "a.bin"), state(fresh(case, t1, 4), tmp_path / "b.bin"))


def test_full_compute_and_debug_after_update(tmp_path):
    case = dict(dim=3, s=1, ref=3, n=2, ell=2, kind="uniform1e4", seed=3001)
    t0 = make_tables(3, 1, 4, "uniform1e4", 3001)
    ctx = fresh(case, t0, 4)
    t1 = [t0[0].copy()]
    t1[0][:7] = 2.0
    update_and_check(ctx, case, (t0, 4), (t1, 4), tmp_path)
    ref = fresh(case, t1, 4)
    for p in (0, 77, 300):
        X, M, G = ctx.debug_stages(p)
        X2, M2, G2 = ref.debug_stages(p)
        assert np.array_equal(X, X2) and np.array_equal(M, M2) and np.array_equal(G, G2)
        c, d = ctx.debug_select([p], [G], [M])
        c2, d2 = ref.debug_select([p], [G2], [M2])
        assert np.array_equal(c[0], c2[0]) and np.array_equal(d, d2)
    ctx.compute_basis()                         # the device work list of the update must not be taken for the range
    ctx.assemble_coarse()
    assert_same(state(ctx, tmp_path / "a.bin"), state(ref, tmp_path / "b.bin"))


def test_two_handles_interleaved(tmp_path):
    a_case, b_case = dict(dim=2, s=1, ref=4, n=2, ell=1), dict(dim=2, s=1, ref=4, n=2, ell=2)
    t0 = make_tables(2, 1, 5, "uniform100", 8)
    t1 = [t0[0].copy()]
    t1[0][100:104] = 77.0
    a = fresh(a_case, t0, 5)
    b = fresh(b_case, t0, 5)
    a.set_coefficient(0, 5, t1[0])
    b.set_coefficient(0, 5, t1[0])
    b.compute_basis()                           # the other handle's parameter block is resident in between
    a.update_basis()
    b.assemble_coarse()
    assert_same(state(a, tmp_path / "a.bin"), state(fresh(a_case, t1, 5), tmp_path / "a2.bin"))
    assert_same(state(b, tmp_path / "b.bin"), state(fresh(b_case, t1, 5), tmp_path / "b2.bin"))


def test_basis_without_coarse_matrix(tmp_path):
    case = dict(dim=2, s=2, ref=3, n=2, ell=1)
    t0 = make_tables(2, 2, 4, "uniform100", 4)
    ctx = fresh(case, t0, 4, coarse=False)
    t1 = [t.copy() for t in t0]
    t1[1][17] = 1.0
    update_and_check(ctx, case, (t0, 4), (t1, 4), tmp_path, coarse=False)
    with pytest.raises(pkg.SlodError) as e:
        ctx.coarse_csr()
    assert e.value.code == 4


def test_state_errors(tmp_path):
    case = dict(dim=2, s=1, ref=3, n=2, ell=1)
    r = 3
    t0 = make_tables(2, 1, r, "uniform100", 6)
    ctx = make_ctx(case, t0, r)
    with pytest.raises(pkg.SlodError) as e:
        ctx.update_basis()                      # no basis yet
    assert e.value.code == 4
    ctx.compute_basis()
    ctx.assemble_coarse()
    ctx.save_state(str(tmp_path / "s.bin"))
    restored = make_ctx(case, t0, r)
    restored.load_state(str(tmp_path / "s.bin"))
    with pytest.raises(pkg.SlodError) as e:
        restored.update_basis()                 # the checkpoint holds no coefficient
    assert e.value.code == 4
    bad = t0[0].copy()
    bad[3 * 8 + 5] = -1.0                       # one coarse cell: A_ii indefinite
    ctx.set_coefficient(0, r, bad)
    with pytest.raises(pkg.SlodError) as e:
        ctx.compute_basis()
    assert e.value.code == 5
    ctx.set_coefficient(0, r, t0[0])
    with pytest.raises(pkg.SlodError) as e:
        ctx.update_basis()                      # the last compute failed
    assert e.value.code == 4


def test_numerical_failure_matches_compute(tmp_path):
    case = dict(dim=2, s=1, ref=3, n=2, ell=1)
    r = 3
    t0 = make_tables(2, 1, r, "uniform100", 9)
    ctx = fresh(case, t0, r)
    bad = t0[0].copy()
    bad[3 * 8 + 5] = -1.0                       # one coarse cell
    ref_ctx = make_ctx(case, [bad], r)
    with pytest.raises(pkg.SlodError) as e_ref:
        ref_ctx.compute_basis()
    ctx.set_coefficient(0, r, bad)
    with pytest.raises(pkg.SlodError) as e:
        ctx.update_basis()
    assert e.value.code == e_ref.value.code == 5
    assert str(e.value) == str(e_ref.value)
    with pytest.raises(pkg.SlodError) as e2:
        ctx.basis(0)
    assert e2.value.code == 4
    with pytest.raises(pkg.SlodError) as e3:
        ctx.update_basis()
    assert e3.value.code == 4
    ctx.set_coefficient(0, r, t0[0])
    ctx.compute_basis()
    ctx.assemble_coarse()
    assert_same(state(ctx, tmp_path / "a.bin"), state(fresh(case, t0, r), tmp_path / "b.bin"))


def test_multi_gpu_refused():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two devices")
    ctx = pkg.SlodContext(dim=2, spacedim=1, n_global_refinements=3, n_subdivisions=2, oversampling=1, stabilize=True,
                          device=0, n_gpus=2)
    ctx.set_coefficient(0, 4, make_tables(2, 1, 4, "uniform100", 1)[0])
    ctx.compute_basis()
    with pytest.raises(pkg.SlodError) as e:
        ctx.update_basis()
    assert e.value.code == 2 and "single-device" in str(e.value)
