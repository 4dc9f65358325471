"""The kernel plan slod_create derives from the patch shape (slod_get_plan), checked on maps-only handles: no GPU needed,
the plan is made for a device with 227 KB of shared memory per block.

Each row states the plan the selection code in slod_create gives, with the reason in the comment:
* solver: rb = ceil((half band width + 8) / 8) row blocks and nw = ceil(Ncd / 8) column warps pick the tensor-core
  variant 0 (rb <= 13, nw <= 16 and rb > 4 or nw > 8; ldx 128), 1 (rb, nw <= 4; ldx 32) or 2 (rb <= 4, nw <= 8; ldx 64);
  a variant whose shared-memory plan does not fit leaves the SIMT solver (-1), with its windows in global memory when
  even that does not fit;
* dense stage: ntile = 4 / 8 / 16 for ceil(Ncd / 8) <= 4 / 8 / 16, kept only behind a tensor-core solver with
  ldx = 8 ntile and with at most 27 nodes per coarse cell ((n + 1)^dim); else the SIMT dense stage;
* 3-D diffusion with variant 0 and a tensor-core dense stage runs the split solver unless SLOD_FUSED_SOLVER is set."""
import importlib

import pytest

pkg = importlib.import_module("dealii-slod_b200")
KEYS = pkg.PLAN_KEYS


@pytest.fixture(scope="module", autouse=True)
def lib():
    pkg.build_library()
    return pkg.load_library()


def _ctx(dim, s, ref, n, ell, **kw):
    return pkg.SlodContext(dim=dim, spacedim=s, n_global_refinements=ref, n_subdivisions=n, oversampling=ell,
                           problem=1 if s > 1 else 0, stabilize=True, device=-2, **kw)


# (dim, s, ref, n, ell, env) -> (mma_variant, split_solver, dense_ntile, gmem_window, dense_coef_gmem, coarse_blocked,
#                                use_ql, gauss_coef)
PLANS = [
    ((2, 1, 4, 2, 1, None), (1, 0, 4, 0, 0, 1, 1, 0)),    # 9 coarse dofs: variant 1, ldx 32 = 8 * 4
    ((2, 1, 4, 2, 3, None), (2, 0, 8, 0, 0, 1, 1, 0)),    # 49: nw 7 -> variant 2, ldx 64 = 8 * 8
    ((2, 1, 4, 2, 4, None), (0, 0, 16, 0, 0, 1, 1, 0)),   # 81: nw 11 -> variant 0, ldx 128 = 8 * 16
    ((2, 1, 4, 2, 5, None), (0, 0, 16, 0, 0, 1, 1, 0)),   # 121: nw 16
    ((2, 2, 4, 2, 2, None), (2, 0, 8, 0, 0, 1, 1, 0)),    # elasticity, 50
    ((2, 2, 4, 2, 3, None), (0, 0, 16, 0, 0, 1, 1, 0)),   # elasticity, 98: nw 13
    ((2, 1, 4, 4, 3, None), (0, 0, 0, 0, 0, 1, 1, 0)),    # 49, wide band (rb > 4): variant 0, but ntile 8 != 128 / 8
    ((2, 2, 4, 4, 2, None), (0, 0, 0, 0, 0, 1, 1, 0)),    # elasticity, 50: the same
    ((2, 1, 4, 4, 4, None), (0, 0, 16, 0, 0, 1, 1, 0)),   # 81 with 4 subdivisions: variant 0 + ntile 16
    ((2, 1, 4, 4, 5, None), (-1, 0, 0, 0, 0, 1, 1, 0)),   # 121: variant 0's shared memory does not fit -> SIMT
    ((2, 2, 4, 4, 3, None), (-1, 0, 0, 0, 0, 1, 1, 0)),   # elasticity, 98: the same
    ((2, 1, 4, 8, 1, None), (1, 0, 0, 0, 0, 1, 1, 0)),    # 81 nodes per coarse cell > 27: SIMT dense stage
    ((2, 1, 4, 8, 2, None), (-1, 0, 0, 0, 0, 1, 1, 0)),   # 8 subdivisions: the coefficient window leaves no variant
    ((2, 1, 4, 8, 4, None), (-1, 0, 0, 1, 1, 1, 1, 0)),   # 81: SIMT windows and dense coefficients in global memory
    ((2, 2, 4, 8, 2, None), (-1, 0, 0, 0, 0, 0, 1, 0)),   # elasticity: the blocked coarse kernel's box does not fit
    ((3, 1, 3, 2, 0, None), (1, 0, 4, 0, 0, 1, 1, 0)),    # 3-D, one-cell patches
    ((3, 1, 3, 2, 1, None), (0, 0, 0, 0, 0, 1, 1, 0)),    # 27, rb > 4: variant 0, ntile 4 != 128 / 8
    ((3, 1, 3, 2, 2, None), (0, 1, 16, 0, 0, 1, 1, 0)),   # 125: split solver, z-major columns
    ((3, 1, 3, 2, 2, "SLOD_FUSED_SOLVER"), (0, 0, 16, 0, 0, 1, 1, 0)),
    ((3, 1, 2, 4, 2, None), (-1, 0, 0, 1, 0, 0, 1, 0)),   # half band width 241: SIMT windows in global memory
    ((3, 1, 3, 4, 2, None), (-1, 0, 0, 1, 1, 0, 1, 0)),   # 125 coarse dofs too: dense coefficients in global memory
    ((2, 1, 4, 2, 4, "SLOD_FORCE_GMEM_SOLVER"), (-1, 0, 0, 1, 1, 1, 1, 0)),
    ((2, 1, 4, 2, 4, "SLOD_FORCE_SIMT_DENSE"), (0, 0, 0, 0, 0, 1, 1, 0)),
    ((2, 1, 4, 2, 4, "SLOD_SIMPLE_COARSE"), (0, 0, 16, 0, 0, 0, 1, 0)),
    ((2, 1, 4, 2, 4, "SLOD_FORCE_JACOBI"), (0, 0, 16, 0, 0, 1, 0, 0)),
]


@pytest.mark.parametrize("cfg,want", PLANS, ids=[f"dim{c[0]}-s{c[1]}-ref{c[2]}-n{c[3]}-ell{c[4]}-{c[5]}" for c, _ in PLANS])
def test_plan_by_shape(cfg, want, monkeypatch):
    *shape, env = cfg
    if env:
        monkeypatch.setenv(env, "1")   # read by slod_create
    ctx = _ctx(*shape)
    assert ctx.plan() == dict(zip(KEYS, want))
    ctx.close()


GRAM = "coarse dofs per patch exceed the Gram register tile"
SMEM = "patch too large for the shared-memory resident solver"
# (dim, s, ref, n): the largest accepted oversampling, the smallest refused one and the refusal
ENVELOPE = [
    ((2, 1, 4, 2), 5, 6, GRAM),   # 121 / 169 coarse dofs
    ((2, 2, 4, 2), 3, 4, GRAM),   # 98 / 162
    ((3, 1, 3, 2), 2, 3, GRAM),   # 125 / 343
    ((2, 1, 4, 4), 5, 6, GRAM),
    ((2, 2, 4, 4), 3, 4, GRAM),
    # 8 subdivisions: the coefficient window (room for one value per Gauss point) of k_patch_finish and of the SIMT
    # solver no longer fits shared memory
    ((2, 1, 4, 8), 4, 5, SMEM),   # 81 coarse dofs accepted
    ((2, 2, 4, 8), 2, 3, SMEM),
]


@pytest.mark.parametrize("cfg,ok,bad,msg", ENVELOPE, ids=[f"dim{c[0]}-s{c[1]}-n{c[3]}" for c, *_ in ENVELOPE])
def test_envelope_boundary(cfg, ok, bad, msg):
    """slod.h: any oversampling whose patches have at most 128 coarse dofs, except where the shared-memory plan of
    8 subdivisions runs out first.  The largest accepted oversampling builds a plan; the next one is refused with
    SLOD_ERR_UNSUPPORTED and the reason."""
    dim, s, ref, n = cfg
    ctx = _ctx(dim, s, ref, n, ok)
    info = [ctx.patch_info(p)["n_coarse"] for p in range(ctx.n_patches)]
    assert max(info) == s * (2 * ok + 1) ** dim      # some patch has the full size
    ctx.close()
    with pytest.raises(pkg.SlodError) as e:
        _ctx(dim, s, ref, n, bad)
    assert e.value.code == 2 and msg in str(e.value)


@pytest.mark.parametrize("cfg", [(2, 1, 4, 8, 4), (2, 1, 4, 4, 5), (2, 2, 4, 4, 3)], ids=["n8-ell4", "n4-ell5", "elast-n4-ell3"])
def test_simt_dense_stage_above_64_coarse_dofs(cfg):
    """2-D patches with 65 .. 128 coarse dofs whose dense stage is the SIMT kernel (32 Gram entries per thread) are
    accepted: its CTA has 512 threads there, as in 3-D."""
    ctx = _ctx(*cfg)
    dim, s, _, _, ell = cfg
    assert s * (2 * ell + 1) ** dim > 64
    assert ctx.plan()["dense_ntile"] == 0
    ctx.close()


def test_plan_arguments():
    ctx = _ctx(2, 1, 3, 2, 1)
    assert ctx.lib.slod_get_plan(ctx.h, None) == 1
    assert ctx.lib.slod_get_plan(None, None) == 1
    ctx.close()
