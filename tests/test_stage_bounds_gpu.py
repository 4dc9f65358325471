"""The patch solver, the dense stage, A phi and the coarse assembly (K and M_H) entry by entry against rounding-error
bounds on their own inputs (tools/stage_bounds.py), on every plan of the parity cases: X, Minv and G from
slod_debug_patch_stages_list, phi and A phi from the basis, K and M_H from the assembled matrices.  Every patch is
checked up to 256 patches, otherwise at least 32 spread over the interior / face / edge / corner classes; LOD-branch
patches get every check but G.  Every stored entry of K and M_H in the rows of the checked patches is checked.

The list call runs the patches as one work list in cost order (the persistent kernels keep their shape tables from one
patch to the next): it must agree bit for bit with the one-patch call and leave the handle's state unchanged."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tools"))
import stage_bounds as sb  # noqa: E402
from parity_common import build_pair, case_id  # noqa: E402
from test_parity_gpu import CASES  # noqa: E402

pytestmark = pytest.mark.gpu


def _state(ctx, pids):
    phi, aphi = ctx.all_basis()
    diag = [ctx.diagnostics(p, d) for p in pids for d in range(ctx.s)]
    return [phi.copy(), aphi.copy(), *[a.copy() for a in ctx.coarse_csr()],
            *[a.copy() for a in ctx.coarse_mass_csr()], np.array(diag)]


@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_stage_bounds(case, monkeypatch):
    case = dict(case)
    case.pop("sample", None)
    env = case.pop("env", None)
    if env:
        monkeypatch.setenv(env, "1")   # read by slod_create
    ctx, orc = build_pair(**case)
    ctx.compute_basis()
    ctx.assemble_coarse()
    ctx.assemble_coarse_mass()
    prob, s = orc.prob, ctx.s
    pids = sb.sample_patches(prob)
    before = _state(ctx, pids)
    Xs, Ms, Gs = ctx.debug_stages_list(pids)
    after = _state(ctx, pids)
    assert all(np.array_equal(a, b) for a, b in zip(before, after)), "the list call changed the handle's state"
    phi, aphi = before[0], before[1]
    worst, n_lod = {}, 0
    for k, pid in enumerate(pids):
        ops = sb.PatchOps(orc, pid)
        X1, M1, G1 = ctx.debug_stages(pid, want_G=ops.slod)
        assert np.array_equal(X1, Xs[k]) and np.array_equal(M1, Ms[k]), pid
        assert (Gs[k] is None) == (not ops.slod) and (G1 is None or np.array_equal(G1, Gs[k])), pid
        checks = {"X": sb.check_X(ops, Xs[k]), "Minv": sb.check_Minv(ops, Xs[k], Ms[k]),
                  "Aphi": sb.check_aphi(ops, phi[pid], aphi[pid])}
        if ops.slod:
            checks["G"] = sb.check_G(ops, Xs[k], Ms[k], Gs[k])
        else:
            n_lod += 1
        for name, (e, b) in checks.items():
            worst[name] = max(worst.get(name, 0.0), sb.ratio(e, b))
    rows = None if len(pids) == ctx.n_patches else [p * s + d for p in pids for d in range(s)]
    worst["K"] = sb.ratio(*sb.check_coarse(prob, phi, before[2:5], aphi=aphi, rows=rows))
    worst["M_H"] = sb.ratio(*sb.check_coarse(prob, phi, before[5:8], rows=rows))
    for name, v in worst.items():
        print(f"STAGE-BOUNDS {case_id(case)} {name} {v:.3g}")
    print(f"STAGE-BOUNDS {case_id(case)} patches {len(pids)} of {ctx.n_patches}, LOD branch {n_lod}")
    assert all(v <= 1.0 for v in worst.values()), worst
    ctx.close()
