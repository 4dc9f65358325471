"""The selection kernels (csrc/select.cuh) on their own: slod_debug_select runs them, as slod_compute_basis does, on
given Gram matrices, and the answers are compared with the reference rule (source/LOD.cc:637-743) evaluated in extended
precision on the same fp64 input (tools/select_reference.py).  The comparison does not depend on cond(G):

  backward error   ||P (G_o d + g)|| <= 8 n eps (sigma_0 ||d|| + ||g||) + 8 n eps (sigma_0 / gap) ||ghat_dropped||.
                   n eps is the backward error of a Cholesky or Householder / QL solve; P projects onto the eigenvectors
                   the reference keeps (the identity without truncation), and the second term is the error of the kept
                   eigenspace (eps sigma_0 / gap) acting on the dropped components of g (zero without truncation).
  sigma_0          1e-13 relative: the largest eigenvalue is perfectly conditioned (Weyl: n eps sigma_0 at most).
  smallest kept    8 n eps sigma_0 absolute (Weyl's bound for a backward-stable eigen-solver).
  forward          ||d - d_ref|| <= 10 n eps sigma_0 / min(lambda_kept, gap) (||d_ref|| + ||ghat_dropped|| / lambda_kept)
                   (select_reference.forward_bound): first-order perturbation of the truncated pseudo-inverse.  The
                   Jacobi fallback (path 2) adds the dropped terms back to d(0) one at a time, as the reference's loop
                   does, and gets 10 n eps ||d(0)|| more for that loop's cancellation.
  step counts, path codes, status: exact.
  diagnostics [2], [3]: path 1 -> sigma_0 / n <= [2] <= sigma_0 and lambda_min <= [3] <= [2] (within the Weyl term);
                   paths 2, 3 -> sigma_0 and the smallest kept sigma as above (include/slod.h).

A decision of the rule that is within rounding on the given G (a singular value within 8 n eps sigma_0 of the 1e-15
threshold, or ||d(r)||_inf within the forward bound of 0.5) is not comparable in any fp64 implementation: synthetic
matrices are designed with safe margins (a margin below its bound is a generator error), real patches are counted as
margin-unsafe and only the checks that do not depend on those decisions are made there."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tools"))
import select_families as sf  # noqa: E402
import select_reference as sr  # noqa: E402
from parity_common import EPS, make_tables, pkg  # noqa: E402

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(not sr.PRECISE, reason="the reference needs x87 extended precision (longdouble)")]

# handles whose patch shapes give the sizes n = n_coarse - 1 below (no patch shape gives n = 9, 16, 32, 33, 64 or 96:
# n + 1 is not a product of reachable patch widths)
HANDLES = {
    "2d_l1": (dict(dim=2, spacedim=1, n_global_refinements=3, oversampling=1), [3, 8]),
    "2d_l2": (dict(dim=2, spacedim=1, n_global_refinements=3, oversampling=2), [15]),
    "3d_l1": (dict(dim=3, spacedim=1, n_global_refinements=2, oversampling=1), [7, 17]),
    "2d_l5": (dict(dim=2, spacedim=1, n_global_refinements=4, oversampling=5), [63, 65, 120]),
    "elast_l3": (dict(dim=2, spacedim=2, n_global_refinements=4, oversampling=3, problem=1), [31, 97]),
    "3d_l2_split": (dict(dim=3, spacedim=1, n_global_refinements=3, oversampling=2), [63, 124]),
}
ENVS = ["default", "SLOD_NO_FAST_SELECT", "SLOD_FORCE_JACOBI"]
STATS = {}


def _handle(kw, monkeypatch, env=None, **extra):
    for e in ENVS[1:] + ["SLOD_EIG_CAP", "SLOD_CHUNK"]:
        monkeypatch.delenv(e, raising=False)
    if env and env != "default":
        monkeypatch.setenv(env, "1")
    for k, v in extra.items():
        monkeypatch.setenv(k, str(v))
    return pkg.SlodContext(stabilize=True, **kw)


def _patches_by_size(ctx):
    out = {}
    for p in range(ctx.n_patches):
        out.setdefault(ctx.patch_info(p)["n_coarse"] - 1, []).append(p)
    return out


_REF = {}


def _cases(n, d):
    """Designed matrices of size n for component d with their checked references; scaled copies G 2^k reuse them."""
    key = (n, d)
    if key not in _REF:
        items = []
        for label, G, expect in sf.cases(n, d):
            ref = sf.check_design(G, d, expect)
            items.append((label, G, expect, ref, 0))
            if label in ("fast", f"truncation{min(33, n)}"):
                items += [(f"{label}*2^{k}", G * 2.0 ** k, expect, ref, k) for k in sf.SCALES]
        _REF[key] = items
    return _REF[key]


def _scaled_ref(ref, k):
    """The reference of 2^k G: d unchanged, eigenvalues and g scaled (exact in binary floating point)."""
    if k == 0:
        return ref
    f = 2.0 ** k
    return dict(ref, lam=ref["lam"] * f, sigma=ref["sigma"] * f, lam_ld=ref["lam_ld"] * f, ghat_ld=ref["ghat_ld"] * f,
                sigma0=ref["sigma0"] * f, kept_min=ref["kept_min"] * f, gap=ref["gap"] * f)


def _ghat_dropped(ref):
    drop = ~ref["used"]
    return float(np.sqrt(np.sum(np.asarray(ref["ghat_ld"][drop], dtype=np.float64) ** 2))) if drop.any() else 0.0


def _backward_ok(G, d, x, ref):
    err, bound = sr.backward_error(G, d, x, ref)
    if not ref["used"].all() and ref["used"].any():
        bound += 8 * ref["n"] * EPS * ref["sigma0"] / ref["gap"] * _ghat_dropped(ref)
    return err, bound


def _check_diag(dg, ref, path, n):
    """Diagnostics [2], [3] as include/slod.h documents them per path."""
    weyl = 8 * n * EPS * ref["sigma0"]
    if path == 1:
        assert ref["sigma0"] / n * (1 - 1e-13) <= dg[2] <= ref["sigma0"] * (1 + 1e-13), (dg, ref["sigma0"])
        assert ref["sigma"][-1] - weyl <= dg[3] <= dg[2] and dg[3] > 1e-12 * dg[2], (dg, ref["sigma"][-1])
        assert dg[0] < 0.49 and dg[6] == 0
    else:
        assert abs(dg[2] - ref["sigma0"]) <= 1e-13 * ref["sigma0"], (dg, ref["sigma0"])
        assert abs(dg[3] - ref["kept_min"]) <= weyl, (dg, ref["kept_min"])


def _run_items(ctx, pids, items, d, env, rng, stats):
    """One slod_debug_select call per batch of distinct patches with M^{-1} = I (c shows d) and one with a random
    M^{-1}; every item checked against its reference."""
    s = ctx.s
    for b0 in range(0, len(items), len(pids)):
        batch = items[b0:b0 + len(pids)]
        ids = pids[:len(batch)]
        ncd = batch[0][1].shape[0]
        n = ncd - 1
        other = [k for k in range(ncd) if k != d]
        eye = np.eye(ncd)
        minv = [sf.random_minv(ncd, rng) for _ in batch]
        c_id, dg_id = ctx.debug_select(ids, [it[1] for it in batch], [eye] * len(batch))
        c_rm, dg_rm = ctx.debug_select(ids, [it[1] for it in batch], minv)
        for i, (label, G, expect, ref0, k) in enumerate(batch):
            ref = _scaled_ref(ref0, k)
            dg = dg_id[i, d]
            what = (label, n, d, env, dg.tolist())
            assert np.array_equal(dg_rm[i, d], dg), what           # M^{-1} does not enter the selection
            path = 1 if expect["fast"] and env != "SLOD_NO_FAST_SELECT" else (2 if env == "SLOD_FORCE_JACOBI" else 3)
            assert dg[5] == path and dg[7] == 0, what
            assert int(dg[1]) == ref["steps"], what
            c = c_id[i][d]
            assert c[d] == 1.0, what
            x = c[other]
            fb = sr.forward_bound(ref)
            if path == 2:
                # the Jacobi fallback runs the reference's loop literally: the dropped terms are added back to d(0)
                # one by one (source/LOD.cc:703-725), so d(r) carries that loop's cancellation error n eps ||d(0)||
                # (and d(n) is rounding residue, not 0)
                fb += 10 * n * EPS * np.linalg.norm(ref["cand"][0])
            ferr = np.linalg.norm(x - ref["d"])
            assert ferr <= fb, (what, ferr, fb)
            berr, bb = _backward_ok(G, d, x, ref)
            assert berr <= bb, (what, berr, bb)
            assert abs(dg[0] - ref["norms"][0]) <= max(sr.forward_bound(ref, 0), 1e-15), what
            _check_diag(dg, ref, path, n)
            # c = M^{-1} (e_d + sum_k d_k e_other[k]): a dot product of length n_coarse per entry
            e = c.copy()
            want = minv[i] @ e
            assert (np.abs(c_rm[i][d] - want) <= 2 * ncd * EPS * (np.abs(minv[i]) @ np.abs(e))).all(), what
            if label == "zero_load":
                assert np.array_equal(c, eye[d]) and np.array_equal(c_rm[i][d], minv[i][:, d]), what
            st = stats.setdefault("scaling" if "*" in label else label.rstrip("0123456789"), {})
            st[n] = st.get(n, 0) + 1
            stats["_max_backward"] = max(stats.get("_max_backward", 0.0), berr / bb if bb > 0 else 0.0)
            stats["_max_forward"] = max(stats.get("_max_forward", 0.0), ferr / fb if fb > 0 else 0.0)


@pytest.mark.parametrize("env", ENVS)
@pytest.mark.parametrize("handle", list(HANDLES))
def test_synthetic_families(handle, env, monkeypatch):
    """Every family (tools/select_families.py) at every size the handle's patch shapes give, for each component,
    under the default plan, without the fast path and with the Jacobi eigen-solver only; M^{-1} = I and a random SPD
    M^{-1}.  Truncation counts 1, 2, 31-33, 63-65, 96, n - 1 and n cross the 32-candidate batches of k_eig_finish:
    the step count is asserted equal to the design."""
    kw, sizes = HANDLES[handle]
    ctx = _handle(kw, monkeypatch, env)
    by_size = _patches_by_size(ctx)
    rng = np.random.default_rng(17)
    stats = STATS.setdefault(f"{handle}-{env}", {})
    for n in sizes:
        pids = by_size[n]
        for d in range(ctx.s):
            _run_items(ctx, pids, _cases(n, d), d, env, rng, stats)
    print(f"\nSELECT-STATS {handle} {env} {stats}")
    assert all(n in stats.get("fast", {}) for n in sizes)
    assert stats["truncation"]


def test_lod_branch_and_chunks(monkeypatch):
    """LOD-branch patches: c = M^{-1} e_d bit-exactly and zero diagnostics whatever G holds.  A forced workspace of
    3 patches (SLOD_CHUNK) gives bit-identical results to one chunk."""
    kw = dict(dim=2, spacedim=2, n_global_refinements=3, oversampling=1, problem=1)
    rng = np.random.default_rng(3)
    ctx = _handle(kw, monkeypatch)
    ctx_lod = pkg.SlodContext(stabilize=False, **kw)
    pids = list(range(0, ctx.n_patches, 5))
    ncd = [ctx.patch_info(p)["n_coarse"] for p in pids]
    G = [sf.family("truncation", k - 1, 0, 1, R=min(2, k - 1))[0] for k in ncd]
    M = [sf.random_minv(k, rng) for k in ncd]
    c, dg = ctx_lod.debug_select(pids, G, M)
    for i in range(len(pids)):
        for d in range(2):
            assert np.array_equal(c[i][d], M[i][:, d])
    assert not dg[..., :7].any()
    ref = ctx.debug_select(pids, G, M)
    monkeypatch.setenv("SLOD_CHUNK", "3")
    chunked = pkg.SlodContext(stabilize=True, **kw).debug_select(pids, G, M)
    assert all(np.array_equal(a, b) for a, b in zip(ref[0], chunked[0])) and np.array_equal(ref[1], chunked[1])


def _all_diag(ctx):
    return np.array([[ctx.diagnostics(p, d) for d in range(ctx.s)] for p in range(ctx.n_patches)])


def test_debug_select_leaves_handle_state(monkeypatch):
    """slod_debug_select writes only scratch: basis, A basis, K, M_H, every patch's diagnostics and status words are
    bit-identical before and after, and a later slod_compute_basis gives the same basis."""
    kw = dict(dim=2, spacedim=1, n_global_refinements=4, oversampling=2)
    ctx = _handle(kw, monkeypatch)
    ctx.set_coefficient(0, 5, make_tables(2, 1, 5, "uniform100", 4)[0])
    ctx.compute_basis()
    ctx.assemble_coarse()
    ctx.assemble_coarse_mass()
    before = ([x.copy() for x in ctx.all_basis()], ctx.coarse_csr()[2].copy(), ctx.coarse_mass_csr()[2].copy(),
              _all_diag(ctx))
    pids = list(range(0, ctx.n_patches, 7))
    G = [sf.family("truncation", ctx.patch_info(p)["n_coarse"] - 1, 0, 2, R=1)[0] for p in pids]
    ctx.debug_select(pids, G, [np.eye(g.shape[0]) for g in G])
    after = ([x.copy() for x in ctx.all_basis()], ctx.coarse_csr()[2], ctx.coarse_mass_csr()[2], _all_diag(ctx))
    assert all(np.array_equal(a, b) for a, b in zip(before[0], after[0]))
    assert all(np.array_equal(a, b) for a, b in zip(before[1:], after[1:]))
    ctx.compute_basis()
    assert all(np.array_equal(a, b) for a, b in zip(before[0], ctx.all_basis()))


# the parity configurations: (kwargs, coefficient refinement, table kind)
REAL = {
    "2d_l2": (dict(dim=2, spacedim=1, n_global_refinements=4, n_subdivisions=2, oversampling=2), 5, "uniform100"),
    "2d_l4": (dict(dim=2, spacedim=1, n_global_refinements=4, n_subdivisions=2, oversampling=4), 5, "uniform100"),
    "2d_l5": (dict(dim=2, spacedim=1, n_global_refinements=4, n_subdivisions=2, oversampling=5), 5, "uniform100"),
    "elast_l1": (dict(dim=2, spacedim=2, n_global_refinements=3, n_subdivisions=2, oversampling=1, problem=1), 4,
                 "uniform100"),
    "elast_l3": (dict(dim=2, spacedim=2, n_global_refinements=4, n_subdivisions=2, oversampling=3, problem=1), 5,
                 "uniform100"),
    "3d_l1": (dict(dim=3, spacedim=1, n_global_refinements=2, n_subdivisions=2, oversampling=1), 3, "uniform100"),
    "3d_l2_split": (dict(dim=3, spacedim=1, n_global_refinements=3, n_subdivisions=2, oversampling=2), 4, "uniform1e4"),
    "2d_n8_simt": (dict(dim=2, spacedim=1, n_global_refinements=4, n_subdivisions=8, oversampling=2), 7, "uniform100"),
}
PER_CLASS = 8   # patches sampled per class (interior / face / edge / corner): a quarter of the class, at most 8


def _sample(ctx, ell, slod):
    """A quarter (at most PER_CLASS) of the SLOD patches of each class: the number of axes along which the patch is cut
    by the domain boundary (0 interior, 1 face, 2 edge, 3 corner; 2-D corners are class 2)."""
    classes = {}
    for p in range(ctx.n_patches):
        if slod[p]:
            cut = sum(m < 2 * ell + 1 for m in ctx.patch_info(p)["m"])
            classes.setdefault(cut, []).append(p)
    out = []
    for cut, ps in sorted(classes.items()):
        k = min(PER_CLASS, max(1, len(ps) // 4))
        out += [ps[i] for i in np.linspace(0, len(ps) - 1, k).astype(int)]
    return out


@pytest.mark.parametrize("case", list(REAL))
def test_real_patches(case, monkeypatch):
    """The GPU's own Gram matrices (slod_debug_patch_stages) through slod_debug_select: the diagnostics of
    slod_compute_basis are reproduced bit for bit (the harness runs production code on production input) and
    normalize(X c) is the pipeline's phi to 1e-13 times the cancellation |X| |c| / |X c| of the product.  On that same G:
    path-1 items pass the backward-error test, sigma_0 agrees on the eigen paths, and where the reference's margins are
    safe the step count is exact, d is within the forward bound and the smallest kept sigma within Weyl's bound."""
    kw, r, kind = REAL[case]
    ctx = _handle(kw, monkeypatch)
    for f, t in enumerate(make_tables(kw["dim"], kw["spacedim"], r, kind, 1234)):
        ctx.set_coefficient(f, r, t)
    ctx.compute_basis()
    s = ctx.s
    prod = _all_diag(ctx)
    pids = _sample(ctx, kw["oversampling"], prod[:, 0, 5] != 0)
    phis = {p: [ctx.basis(p, d)[0] for d in range(s)] for p in pids}
    stages = {p: ctx.debug_stages(p) for p in pids}
    c, dg = ctx.debug_select(pids, [stages[p][2] for p in pids], [stages[p][1] for p in pids])
    c_id, dg_id = ctx.debug_select(pids, [stages[p][2] for p in pids], [np.eye(stages[p][2].shape[0]) for p in pids])
    assert np.array_equal(dg[..., :7], prod[pids][..., :7])
    assert np.array_equal(dg_id, dg)
    n_safe = 0
    worst_b = worst_f = 0.0
    for i, p in enumerate(pids):
        X, Minv, G = stages[p]
        interior = ctx.patch_dof_class(p, 0)
        ncd = G.shape[0]
        n = ncd - 1
        for d in range(s):
            v = X @ c[i][d]
            tol = 1e-13 * max(1.0, np.linalg.norm(np.abs(X) @ np.abs(c[i][d])) / np.linalg.norm(v))
            assert np.linalg.norm(v / np.linalg.norm(v) - phis[p][d][interior]) <= tol, (p, d)
            other = [k for k in range(ncd) if k != d]
            x = c_id[i][d][other]
            ref = sr.select(G, np.eye(ncd), d)
            what = (case, p, d, dg[i, d].tolist())
            path = int(dg[i, d, 5])
            if path == 1:
                berr, bb = _backward_ok(G, d, x, ref)
                assert berr <= bb, (what, berr, bb)
                worst_b = max(worst_b, berr / bb)
                assert ref["sigma0"] / n * (1 - 1e-13) <= dg[i, d, 2] <= ref["sigma0"] * (1 + 1e-13), what
                assert dg[i, d, 3] >= ref["sigma"][-1] - 8 * n * EPS * ref["sigma0"], what
            else:
                assert abs(dg[i, d, 2] - ref["sigma0"]) <= 1e-13 * ref["sigma0"], what
            if not sr.margins_safe(ref):
                continue
            n_safe += 1
            assert int(dg[i, d, 1]) == ref["steps"], what
            fb = sr.forward_bound(ref)
            ferr = np.linalg.norm(x - ref["d"])
            assert ferr <= fb, (what, ferr, fb)
            worst_f = max(worst_f, ferr / fb if fb > 0 else 0.0)
            if path != 1:
                assert abs(dg[i, d, 3] - ref["kept_min"]) <= 8 * n * EPS * ref["sigma0"], what
                berr, bb = _backward_ok(G, d, x, ref)
                assert berr <= bb, (what, berr, bb)
                worst_b = max(worst_b, berr / bb)
    print(f"\nSELECT-REAL {case}: {len(pids) * s} items from {len(pids)} patches, {n_safe} margin-safe, "
          f"paths {np.bincount(dg[..., 5].astype(int).ravel(), minlength=4).tolist()}, "
          f"max backward/bound {worst_b:.2e}, max forward/bound {worst_f:.2e}")


def test_multi_round_eigen_pipeline(monkeypatch):
    """The eigen pipeline in rounds (SLOD_EIG_CAP): on the cfg-4 shape (3-D, oversampling 2, high contrast) with more
    eigen items than the forced cap, basis, A basis, K and every diagnostic are bit-identical to the one-round run."""
    kw = dict(dim=3, spacedim=1, n_global_refinements=3, n_subdivisions=2, oversampling=2)
    tab = make_tables(3, 1, 4, "uniform1e4", 3001)[0]
    runs = []
    cap = None
    for forced in (False, True):
        ctx = _handle(kw, monkeypatch, **({"SLOD_EIG_CAP": cap} if forced else {}))
        ctx.set_coefficient(0, 4, tab)
        ctx.compute_basis()
        ctx.assemble_coarse()
        diag = _all_diag(ctx)
        if not forced:
            n_eig = int((diag[..., 5] == 3).sum())
            cap = 64 if n_eig > 3 * 64 else max(1, n_eig // 3)
            print(f"\nSELECT-ROUNDS {n_eig} eigen items, cap {cap}")
            assert n_eig > 2 * cap     # at least three rounds
        runs.append(([x.copy() for x in ctx.all_basis()], ctx.coarse_csr()[2].copy(), diag))
    (b0, k0, d0), (b1, k1, d1) = runs
    assert all(np.array_equal(a, b) for a, b in zip(b0, b1))
    assert np.array_equal(k0, k1) and np.array_equal(d0, d1)
