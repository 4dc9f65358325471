"""CPU checks of the batched online entry points: a handle without a device refuses them, and the binding rejects
blocks of the wrong shape before it calls the library."""
import ctypes as C
import importlib

import numpy as np
import pytest

pkg = importlib.import_module("dealii-slod_b200")


@pytest.fixture(scope="module")
def ctx():
    pkg.build_library()
    c = pkg.SlodContext(dim=2, n_global_refinements=3, device=-2)
    yield c
    c.close()


def test_maps_only_handle_refuses_batch_calls(ctx):
    nf, nc = ctx.n_fine, ctx.n_patches * ctx.s
    for call in (lambda: ctx.coarse_rhs_batch(np.ones((3, nf))),
                 lambda: ctx.coarse_solve_batch(np.ones((3, nc))),
                 lambda: ctx.prolongate_batch(np.ones((3, nc)))):
        with pytest.raises(pkg.SlodError) as e:
            call()
        assert e.value.code == 3 and "without a device" in str(e.value)
    # through the C ABI directly, n_rhs = 0 included: the missing device is reported first
    buf = np.zeros(max(nf, nc))
    dp = buf.ctypes.data_as(C.POINTER(C.c_double))
    assert ctx.lib.slod_coarse_rhs_batch(ctx.h, 0, dp, dp) == 3
    assert ctx.lib.slod_coarse_solve_batch(ctx.h, 1, dp, dp, 10, 0.0, 1e-10, None, None) == 3
    assert ctx.lib.slod_prolongate_batch(ctx.h, 1, dp, dp) == 3


def test_batch_shapes_are_checked(ctx):
    nf, nc = ctx.n_fine, ctx.n_patches * ctx.s
    bad = {
        ctx.coarse_rhs_batch: [np.ones(nf), np.ones((2, nf + 1)), np.ones((0, nf)), np.ones((2, nf, 1)),
                               np.ones((2, nc))],
        ctx.coarse_solve_batch: [np.ones(nc), np.ones((2, nc - 1)), np.ones((0, nc)), np.ones((2, nf))],
        ctx.prolongate_batch: [np.ones(nc), np.ones((3, nc + 2)), np.ones((0, nc)), np.ones((1, nf))],
    }
    for call, arrays in bad.items():
        for a in arrays:
            with pytest.raises(ValueError):
                call(a)
