"""The stage checks of tools/stage_bounds.py on the two CPU chains: the oracle's fp64 stages and the C++ port's
(slod_debug_patch_stages, basis, K).  Both must lie within the bounds.  Then defects planted in the oracle's stages,
each small enough that the tolerances the parity tests used before pass it, must fail the matching check."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tools"))
import stage_bounds as sb  # noqa: E402
from cpu_port import CpuSlod  # noqa: E402
from heat_oracle import coarse_mass  # noqa: E402
from parity_common import CoefficientTable, SlodOracle, SlodProblem, case_id, make_tables  # noqa: E402

CASES = [
    dict(dim=2, s=1, ref=3, n=2, ell=2),                                   # diffusion, SLOD
    dict(dim=2, s=2, ref=3, n=2, ell=1),                                   # elasticity
    dict(dim=3, s=1, ref=2, n=2, ell=1, kind="uniform1e4", seed=3001),     # 3-D, contrast 1e4
    dict(dim=2, s=1, ref=3, n=2, ell=1, stabilize=False),                  # LOD branch
    dict(dim=2, s=1, ref=3, n=2, ell=1, r=5),                              # one coefficient per Gauss point
]
# what the parity tests compared these stages with before: X, Minv, G at 1e-10 max|want| (tests/test_parity_gpu.py),
# K at 1e-12 max|K| (tests/test_online_gpu.py)
OLD_STAGE, OLD_K = 1e-10, 1e-12


def _oracle(dim=2, s=1, ref=3, n=2, ell=1, stabilize=True, r=None, kind="uniform100", seed=1234):
    """The oracle of a configuration, with the coefficient tables parity_common.build_pair gives the GPU handle."""
    r = min(ref + int(np.log2(n)), 8 if dim == 2 else 6) if r is None else r
    tabs = make_tables(dim, s, r, kind, seed)
    prob = SlodProblem(dim=dim, spacedim=s, n_global_refinements=ref, n_subdivisions=n, oversampling=ell,
                       stabilize=stabilize, problem="diffusion" if s == 1 else "elasticity",
                       coefficients=[CoefficientTable(dim, r, t) for t in tabs])
    return SlodOracle(prob), r, tabs


def _stacked(patches, s, key):
    nf = max(getattr(r, key).shape[1] for r in patches)
    out = np.zeros((len(patches), s, nf))
    for r in patches:
        v = getattr(r, key)
        out[r.pid, :, :v.shape[1]] = v
    return out


def _oracle_chain(case):
    orc = _oracle(**case)[0]
    orc.compute_basis()
    K, C, _ = orc.assemble_global_matrix()
    s = orc.prob.spacedim
    return orc, _stacked(orc.patches, s, "basis"), _stacked(orc.patches, s, "basis_premultiplied"), K, C


@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_oracle_chain_within_bounds(case):
    orc, phi, aphi, K, C = _oracle_chain(case)
    worst = {}
    for res in orc.patches:
        ops = sb.PatchOps(orc, res.pid)
        checks = {"Aphi": sb.check_aphi(ops, res.basis, res.basis_premultiplied)}
        if res.info["slod"]:
            checks["X"] = sb.check_X(ops, res.info["X"], sparse_lu=True)
            checks["Minv"] = sb.check_Minv(ops, res.info["X"], res.info["Minv"])
            checks["G"] = sb.check_G(ops, res.info["X"], res.info["Minv"], res.info["G"])
        for k, (e, b) in checks.items():
            worst[k] = max(worst.get(k, 0.0), sb.ratio(e, b))
    worst["K"] = sb.ratio(*sb.check_coarse(orc.prob, phi, (K.indptr, K.indices, K.data), aphi=aphi))
    M = coarse_mass(orc, C)
    worst["M_H"] = sb.ratio(*sb.check_coarse(orc.prob, phi, (M.indptr, M.indices, M.data)))
    print(f"STAGE-BOUNDS oracle {case_id(case)} " + " ".join(f"{k} {v:.3g}" for k, v in worst.items()))
    assert all(v <= 1.0 for v in worst.values()), worst


@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_cpu_port_within_bounds(case):
    dim, s = case["dim"], case["s"]
    orc, r, tabs = _oracle(**case)
    cpu = CpuSlod(dim=dim, spacedim=s, n_global_refinements=case["ref"], n_subdivisions=case["n"],
                  oversampling=case["ell"], stabilize=case.get("stabilize", True), problem=0 if s == 1 else 1)
    for f, t in enumerate(tabs):
        cpu.set_coefficient(f, r, t)
    cpu.compute_basis()
    cpu.assemble_coarse()
    phi, aphi = cpu.all_basis()
    worst = {}
    for pid in range(cpu.n_patches):
        ops = sb.PatchOps(orc, pid)
        X, Minv, G = cpu.debug_stages(pid, want_G=ops.slod)
        checks = {"X": sb.check_X(ops, X), "Minv": sb.check_Minv(ops, X, Minv),
                  "Aphi": sb.check_aphi(ops, phi[pid], aphi[pid])}
        if ops.slod:
            checks["G"] = sb.check_G(ops, X, Minv, G)
        for k, (e, b) in checks.items():
            worst[k] = max(worst.get(k, 0.0), sb.ratio(e, b))
    worst["K"] = sb.ratio(*sb.check_coarse(orc.prob, phi, cpu.coarse_csr(), aphi=aphi))
    print(f"STAGE-BOUNDS cpu_port {case_id(case)} " + " ".join(f"{k} {v:.3g}" for k, v in worst.items()))
    assert all(v <= 1.0 for v in worst.values()), worst


@pytest.fixture(scope="module")
def planted():
    """2-D diffusion, l = 3 on 8 x 8 cells (SLOD; K entries down to 1e-15 max|K|): the oracle's chain, the C++ port's
    stages of the same patch (band Cholesky, as in the library) and a patch cut on the fewest axes."""
    case = dict(dim=2, s=1, ref=3, n=2, ell=3)
    orc, phi, aphi, K, C = _oracle_chain(case)
    res = min((r for r in orc.patches if r.info["slod"]), key=lambda r: sb.patch_class(orc.prob, r.pid))
    orc_, r, tabs = _oracle(**case)
    cpu = CpuSlod(dim=2, spacedim=1, n_global_refinements=3, n_subdivisions=2, oversampling=3, stabilize=True)
    cpu.set_coefficient(0, r, tabs[0])
    return orc, phi, aphi, K, res, cpu.debug_stages(res.pid)[0]


def _old_passes(got, want, tol):
    return np.abs(got - want).max() <= tol * np.abs(want).max()


def test_planted_X_scaled(planted):
    """On the band-Cholesky X of the C++ port (the oracle's sparse LU has a looser a priori bound)."""
    orc, _, _, _, res, X = planted
    ops = sb.PatchOps(orc, res.pid)
    assert sb.ratio(*sb.check_X(ops, X)) <= 1.0
    bad = X * (1.0 + 1e-13)
    assert _old_passes(bad, res.info["X"], OLD_STAGE)
    assert sb.ratio(*sb.check_X(ops, bad)) > 1.0


def test_planted_Minv_entry(planted):
    orc, _, _, _, res, _ = planted
    ops = sb.PatchOps(orc, res.pid)
    X, Minv = res.info["X"], res.info["Minv"]
    assert sb.ratio(*sb.check_Minv(ops, X, Minv)) <= 1.0
    bad = Minv.copy()
    i, j = np.unravel_index(np.abs(Minv).argmax(), Minv.shape)
    bad[i, j] *= 1.0 + 1e-12
    assert _old_passes(bad, Minv, OLD_STAGE)
    assert sb.ratio(*sb.check_Minv(ops, X, bad)) > 1.0


def test_planted_G_entry(planted):
    orc, _, _, _, res, _ = planted
    ops = sb.PatchOps(orc, res.pid)
    X, Minv, G = res.info["X"], res.info["Minv"], res.info["G"]
    assert sb.ratio(*sb.check_G(ops, X, Minv, G)) <= 1.0
    bad = G.copy()
    i, j = np.unravel_index(np.abs(G).argmax(), G.shape)
    bad[i, j] += 1e-13 * np.abs(G).max()
    assert _old_passes(bad, G, OLD_STAGE)
    assert sb.ratio(*sb.check_G(ops, X, Minv, bad)) > 1.0


def test_planted_small_K_entry(planted):
    orc, phi, aphi, K, _, _ = planted
    kmax = np.abs(K.data).max()
    # below 1e-6 max|K|; the old tolerance (1e-12 max|K|) lets a 1e-3 relative error through below 1e-9 max|K|
    k = int(np.flatnonzero((np.abs(K.data) < 1e-9 * kmax) & (K.data != 0))[0])
    bad = K.data.copy()
    bad[k] *= 1.0 + 1e-3
    assert _old_passes(bad, K.data, OLD_K)
    assert sb.ratio(*sb.check_coarse(orc.prob, phi, (K.indptr, K.indices, K.data), aphi=aphi)) <= 1.0
    assert sb.ratio(*sb.check_coarse(orc.prob, phi, (K.indptr, K.indices, bad), aphi=aphi)) > 1.0


def test_planted_dropped_overlap_cell(planted):
    """A sweep box that misses one coarse cell of the overlap: the entry loses that cell's nodes.  Among the far
    entries (overlap of one cell layer), one whose change stays below the old K tolerance must still fail."""
    orc, phi, aphi, K, _, _ = planted
    pr = orc.prob
    n, s = pr.n_subdivisions, pr.spacedim
    kmax = np.abs(K.data).max()
    P = sb._box_views(pr, phi)
    Y = sb._box_views(pr, aphi)
    found = 0
    for r in range(K.shape[0]):
        p, d = divmod(r, s)
        for k in range(K.indptr[r], K.indptr[r + 1]):
            q, e = divmod(int(K.indices[k]), s)
            b0 = np.maximum(P[p][0], Y[q][0])
            b1 = np.minimum(P[p][1], Y[q][1])
            if ((b1 - b0) != n).any():        # far entries: the overlap is a single coarse cell per axis
                continue
            # the cell without its nodes shared with the rest of the overlap box is the whole box here: drop the
            # interior nodes of the cell (those no neighbouring cell of either patch would have covered)
            cut = lambda lo: (slice(None),) + tuple(slice(b0[a] - lo[a] + 1, b1[a] - lo[a]) for a in
                                                    reversed(range(pr.dim)))
            drop = float((P[p][2][cut(P[p][0])][d] * Y[q][2][cut(Y[q][0])][e]).sum())
            if drop == 0.0 or abs(drop) > OLD_K * kmax:
                continue
            bad = K.data.copy()
            bad[k] -= drop
            assert _old_passes(bad, K.data, OLD_K)
            err, bound = sb.check_coarse(pr, phi, (K.indptr, K.indices, bad), aphi=aphi, rows=[r])
            assert sb.ratio(err, bound) > 1.0, (r, k, drop)
            found += 1
            if found == 3:
                return
    assert found > 0, "no far entry whose dropped cell stays under the old tolerance"


def test_empty_overlap_must_be_exact_zero():
    """A stored entry whose patches share no node: exactly 0.0 passes, anything else fails."""
    pr = _oracle(dim=2, s=1, ref=2, n=2, ell=0)[0].prob
    phi = np.ones((pr.N ** 2, 1, 9))
    rowptr, col = np.array([0, 1]), np.array([15])      # patches 0 and 15 of a 4 x 4 mesh are two cells apart
    assert sb.ratio(*sb.check_coarse(pr, phi, (rowptr, col, np.array([0.0])), aphi=phi, rows=[0])) == 0.0
    assert sb.ratio(*sb.check_coarse(pr, phi, (rowptr, col, np.array([1e-300])), aphi=phi, rows=[0])) > 1.0
