"""ctypes binding of ``libslod_b200.so`` (include/slod.h).

This is plumbing for the Python tests and ``bench.py``; the product is the shared library.  There is
no fallback: if the library is missing or no CUDA device is usable every entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SLOD_LIB") or os.path.join(_HERE, "libslod_b200.so")   # SLOD_LIB: instrumented build (tools/)

SLOD_OK = 0
ERRORS = {1: "SLOD_ERR_INVALID", 2: "SLOD_ERR_UNSUPPORTED", 3: "SLOD_ERR_CUDA", 4: "SLOD_ERR_STATE",
          5: "SLOD_ERR_NUMERIC"}
PROBLEM_DIFFUSION, PROBLEM_ELASTICITY = 0, 1

# every symbol include/slod.h declares (tests check that the library exports all of them)
EXPORTS = [
    "slod_create", "slod_destroy", "slod_last_error", "slod_last_create_error", "slod_set_coefficient",
    "slod_patch_count", "slod_get_patch_info", "slod_get_patch_cells", "slod_get_patch_fine_dofs",
    "slod_get_patch_local_dofs", "slod_get_patch_dof_class", "slod_compute_basis", "slod_get_basis",
    "slod_basis_stride", "slod_get_all_basis", "slod_assemble_coarse", "slod_get_coarse_csr",
    "slod_get_patch_diagnostics", "slod_debug_patch_stages", "slod_get_timings", "slod_compute_basis_device",
    "slod_assemble_coarse_device", "slod_ell_width", "slod_ell_to_csr", "slod_launch_count", "slod_alloc_host",
    "slod_free_host", "slod_fine_size", "slod_coarse_rhs", "slod_coarse_solve", "slod_prolongate",
    "slod_fem_solve", "slod_fine_norms", "slod_synchronize", "slod_measure_fp64_peak", "slod_owned_range",
    "slod_comm_unique_id", "slod_comm_init", "slod_offline_distributed", "slod_save_state", "slod_load_state",
    "slod_fine_norms_reference", "slod_set_host_outputs", "slod_coarse_rhs_batch", "slod_coarse_solve_batch",
    "slod_prolongate_batch", "slod_assemble_coarse_mass", "slod_get_coarse_mass_csr", "slod_l2_project_batch",
    "slod_heat_solve", "slod_heat_solve_batch", "slod_fem_heat_solve", "slod_get_plan", "slod_debug_select",
    "slod_update_basis", "slod_heat_theta_solve", "slod_heat_theta_solve_batch", "slod_fem_heat_theta_solve",
]
# slod_get_plan entries, in order
PLAN_KEYS = ["mma_variant", "split_solver", "dense_ntile", "gmem_window", "dense_coef_gmem", "coarse_blocked", "use_ql",
             "gauss_coef"]


class SlodParams(C.Structure):
    _fields_ = [("dim", C.c_int), ("spacedim", C.c_int), ("n_global_refinements", C.c_int),
                ("n_subdivisions", C.c_int), ("oversampling", C.c_int), ("stabilize", C.c_int),
                ("problem", C.c_int), ("quirk_presaved", C.c_int), ("device", C.c_int), ("n_gpus", C.c_int)]


class SlodError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"{ERRORS.get(code, code)}: {msg}")
        self.code = code


_libs = {}


def load_library(path=None):
    """Load libslod_b200.so (built in-tree by ``__graft_entry__.build()``); fails loudly when absent.
    ``path``: another implementation of include/slod.h -- only the test / baseline infrastructure passes one (the C++
    CPU restatement under oracle/); symbols such a library does not export raise AttributeError when called."""
    path = path or LIB_PATH
    if path in _libs:
        return _libs[path]
    if not os.path.exists(path):
        raise ImportError(f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(the CUDA library is the product; there is no CPU fallback)")
    lib = _Lib(C.CDLL(path), partial=(path != LIB_PATH))
    P = C.POINTER
    vp, i64, i32, dbl = C.c_void_p, C.c_int64, C.c_int32, C.c_double
    lib.slod_create.argtypes = [P(SlodParams), P(vp)]
    lib.slod_destroy.argtypes = [vp]
    lib.slod_destroy.restype = None
    lib.slod_last_error.argtypes = [vp]
    lib.slod_last_error.restype = C.c_char_p
    lib.slod_last_create_error.restype = C.c_char_p
    lib.slod_set_coefficient.argtypes = [vp, C.c_int, C.c_int, P(dbl), C.c_size_t]
    lib.slod_patch_count.argtypes = [vp, P(i64)]
    lib.slod_get_plan.argtypes = [vp, P(i32)]
    lib.slod_fine_size.argtypes = [vp, P(i64)]
    lib.slod_coarse_rhs.argtypes = [vp, P(dbl), P(dbl)]
    lib.slod_coarse_solve.argtypes = [vp, P(dbl), P(dbl), i32, dbl, dbl, P(i32), P(dbl)]
    lib.slod_prolongate.argtypes = [vp, P(dbl), P(dbl)]
    lib.slod_coarse_rhs_batch.argtypes = [vp, i32, P(dbl), P(dbl)]
    lib.slod_coarse_solve_batch.argtypes = [vp, i32, P(dbl), P(dbl), i32, dbl, dbl, P(i32), P(dbl)]
    lib.slod_prolongate_batch.argtypes = [vp, i32, P(dbl), P(dbl)]
    lib.slod_fem_solve.argtypes = [vp, P(dbl), P(dbl), i32, dbl, dbl, P(i32), P(dbl)]
    lib.slod_assemble_coarse_mass.argtypes = [vp]
    lib.slod_get_coarse_mass_csr.argtypes = [vp, P(i64), P(i64), P(dbl), P(i64), P(i64)]
    lib.slod_l2_project_batch.argtypes = [vp, i32, P(dbl), P(dbl), i32, dbl, dbl, P(i32), P(dbl)]
    lib.slod_heat_solve.argtypes = [vp, P(dbl), P(dbl), dbl, i32, i32, P(dbl), i32, dbl, dbl, P(i32)]
    lib.slod_heat_solve_batch.argtypes = [vp, i32, P(dbl), P(dbl), dbl, i32, i32, P(dbl), i32, dbl, dbl, P(i32)]
    lib.slod_fem_heat_solve.argtypes = [vp, P(dbl), P(dbl), dbl, i32, i32, P(dbl), i32, dbl, dbl, P(i32)]
    theta = [dbl, dbl, i32, i32, i32, i32, P(dbl), P(dbl), P(dbl), P(dbl), i32, dbl, dbl, P(i32)]
    lib.slod_heat_theta_solve.argtypes = [vp] + theta
    lib.slod_heat_theta_solve_batch.argtypes = [vp, i32] + theta
    lib.slod_fem_heat_theta_solve.argtypes = [vp] + theta
    lib.slod_fine_norms.argtypes = [vp, P(dbl), P(dbl), P(dbl), P(dbl)]
    lib.slod_get_patch_info.argtypes = [vp, i64] + [P(i32)] * 6 + [P(i32), P(i32)]
    lib.slod_get_patch_cells.argtypes = [vp, i64, P(C.c_uint32), P(i32)]
    lib.slod_get_patch_fine_dofs.argtypes = [vp, i64, P(C.c_uint64), P(i32)]
    lib.slod_get_patch_local_dofs.argtypes = [vp, i64, P(C.c_uint32), P(i32)]
    lib.slod_get_patch_dof_class.argtypes = [vp, i64, C.c_int, P(C.c_uint32), P(i32)]
    lib.slod_compute_basis.argtypes = [vp]
    lib.slod_update_basis.argtypes = [vp, P(i64), P(i64)]
    lib.slod_get_basis.argtypes = [vp, i64, C.c_int, P(dbl), P(dbl)]
    lib.slod_basis_stride.argtypes = [vp, P(i64)]
    lib.slod_get_all_basis.argtypes = [vp, P(dbl), P(dbl)]
    lib.slod_assemble_coarse.argtypes = [vp]
    lib.slod_get_coarse_csr.argtypes = [vp, P(i64), P(i64), P(dbl), P(i64), P(i64)]
    lib.slod_get_patch_diagnostics.argtypes = [vp, i64, C.c_int, P(dbl)]
    lib.slod_debug_patch_stages.argtypes = [vp, i64, P(dbl), P(dbl), P(dbl)]
    lib.slod_debug_select.argtypes = [vp, i64, P(i64), P(dbl), P(dbl), P(dbl), P(dbl)]
    lib.slod_get_timings.argtypes = [vp, P(dbl), C.c_int]
    lib.slod_compute_basis_device.argtypes = [vp, i64, i64, vp, vp, vp]
    lib.slod_assemble_coarse_device.argtypes = [vp, i64, i64, vp, vp, vp, vp]
    lib.slod_ell_width.argtypes = [vp, P(i64)]
    lib.slod_ell_to_csr.argtypes = [vp, P(dbl), P(i64), P(i64), P(dbl), P(i64), P(i64)]
    lib.slod_launch_count.argtypes = [vp, P(i64)]
    lib.slod_alloc_host.argtypes = [C.c_size_t, P(vp)]
    lib.slod_free_host.argtypes = [vp]
    lib.slod_synchronize.argtypes = [vp]
    lib.slod_fine_norms_reference.argtypes = [vp, P(dbl), P(dbl), P(dbl), P(dbl)]
    lib.slod_save_state.argtypes = [vp, C.c_char_p]
    lib.slod_load_state.argtypes = [vp, C.c_char_p]
    lib.slod_set_host_outputs.argtypes = [vp, vp, vp, vp]
    lib.slod_owned_range.argtypes = [vp, C.c_int, C.c_int, P(i64), P(i64)]
    lib.slod_comm_unique_id.argtypes = [vp]
    lib.slod_comm_init.argtypes = [vp, C.c_int, C.c_int, vp]
    lib.slod_offline_distributed.argtypes = [vp, vp, vp, vp, C.c_int, C.c_int, vp]
    lib.slod_measure_fp64_peak.argtypes = [vp, P(dbl), P(dbl)]
    _libs[path] = lib
    return lib


class _Missing:
    """Stand-in for a symbol a partial implementation of slod.h does not export: declaring its signature is a no-op,
    calling it fails."""

    def __init__(self, name):
        self._name = name

    def __call__(self, *a):
        raise AttributeError(f"this library does not export {self._name}")


class _Lib:
    def __init__(self, cdll, partial):
        object.__setattr__(self, "_cdll", cdll)
        object.__setattr__(self, "_partial", partial)   # the product library must export everything: strict
        object.__setattr__(self, "_missing", {})

    def __getattr__(self, name):
        try:
            return getattr(self._cdll, name)
        except AttributeError:
            if not self._partial or not name.startswith("slod_"):
                raise
            return self._missing.setdefault(name, _Missing(name))


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


class _PinnedBlock:
    """Owner of one slod_alloc_host block; numpy arrays made from it keep it alive through their ``base`` chain and the
    block is released by slod_free_host when the last of them is collected."""

    def __init__(self, lib, addr, nbytes):
        self._lib, self._addr = lib, addr
        self.__array_interface__ = {"shape": (max(nbytes, 1),), "typestr": "|u1", "data": (addr, False), "version": 3}

    def __del__(self):
        try:
            self._lib.slod_free_host(C.c_void_p(self._addr))
        except Exception:
            pass


class SlodContext:
    """Thin object wrapper over the opaque ``slod_ctx`` handle."""

    def __init__(self, dim=2, spacedim=1, n_global_refinements=2, n_subdivisions=2, oversampling=1,
                 stabilize=False, problem=PROBLEM_DIFFUSION, quirk_presaved=False, device=-1, lib=None, n_gpus=0):
        self.lib = load_library(lib)
        self.par = SlodParams(dim, spacedim, n_global_refinements, n_subdivisions, oversampling,
                              int(bool(stabilize)), problem, int(bool(quirk_presaved)), device, n_gpus)
        self.h = C.c_void_p()
        rc = self.lib.slod_create(C.byref(self.par), C.byref(self.h))
        if rc != SLOD_OK:
            raise SlodError(rc, self.lib.slod_last_create_error().decode())
        self.dim, self.s = dim, spacedim

    def close(self):
        """Destroy the handle.  Arrays returned earlier stay valid: each owns its page-locked block (see _out)."""
        self._reuse = {}
        if getattr(self, "h", None) and self.h.value:
            self.lib.slod_destroy(self.h)
            self.h = C.c_void_p()

    def _out(self, key, shape, dtype=np.float64, reuse=False):
        """Output array in page-locked memory (slod_alloc_host).  The array owns its block: the block is freed when the
        last view of it is garbage collected, never by close().  reuse=False (default): a fresh block per call, so
        results of earlier calls are never overwritten.  reuse=True: the block of the previous call with the same key
        and shape is handed out again (benchmark loops; the caller accepts that the earlier array is overwritten)."""
        if not hasattr(self, "_reuse"):
            self._reuse = {}
        shape = tuple(int(x) for x in np.atleast_1d(shape))
        if reuse:
            arr = self._reuse.get(key)
            if arr is not None and arr.shape == shape and arr.dtype == dtype:
                return arr
        nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        ptr = C.c_void_p()
        if self.par.device == -2 or self.lib.slod_alloc_host(nbytes, C.byref(ptr)) != SLOD_OK:
            arr = np.empty(shape, dtype=dtype)                       # maps-only handle / allocation refused
        else:
            arr = np.asarray(_PinnedBlock(self.lib, ptr.value, nbytes)).view(dtype)[: int(np.prod(shape))].reshape(shape)
        if reuse:
            self._reuse[key] = arr
        return arr

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != SLOD_OK:
            raise SlodError(rc, self.lib.slod_last_error(self.h).decode())

    # -- inputs ----------------------------------------------------------------------------------------
    def set_coefficient(self, field, eta_refinement, values):
        v = np.ascontiguousarray(values, dtype=np.float64).ravel()
        self._ck(self.lib.slod_set_coefficient(self.h, field, eta_refinement, _dp(v), v.size))

    def plan(self):
        """The kernels slod_create chose (slod_get_plan): {key: int} over PLAN_KEYS."""
        out = (C.c_int32 * 8)()
        self._ck(self.lib.slod_get_plan(self.h, out))
        return dict(zip(PLAN_KEYS, (int(x) for x in out)))

    # -- integer maps ----------------------------------------------------------------------------------
    @property
    def n_patches(self):
        n = C.c_int64()
        self._ck(self.lib.slod_patch_count(self.h, C.byref(n)))
        return n.value

    def patch_info(self, patch):
        v = [C.c_int32() for _ in range(6)]
        lo = (C.c_int32 * 3)()
        m = (C.c_int32 * 3)()
        self._ck(self.lib.slod_get_patch_info(self.h, patch, *[C.byref(x) for x in v], lo, m))
        keys = ["n_cells", "n_fine", "n_internal", "n_boundary", "n_domain_boundary", "n_coarse"]
        out = {k: x.value for k, x in zip(keys, v)}
        out["lo"] = tuple(lo)[: self.dim]
        out["m"] = tuple(m)[: self.dim]
        return out

    def patch_cells(self, patch):
        n = C.c_int32()
        self._ck(self.lib.slod_get_patch_cells(self.h, patch, None, C.byref(n)))
        a = np.empty(n.value, dtype=np.uint32)
        self._ck(self.lib.slod_get_patch_cells(self.h, patch, a.ctypes.data_as(C.POINTER(C.c_uint32)), C.byref(n)))
        return a

    def patch_fine_dofs(self, patch):
        n = C.c_int32()
        self._ck(self.lib.slod_get_patch_fine_dofs(self.h, patch, None, C.byref(n)))
        a = np.empty(n.value, dtype=np.uint64)
        self._ck(self.lib.slod_get_patch_fine_dofs(self.h, patch, a.ctypes.data_as(C.POINTER(C.c_uint64)), C.byref(n)))
        return a

    def patch_local_dofs(self, patch):
        n = C.c_int32()
        self._ck(self.lib.slod_get_patch_local_dofs(self.h, patch, None, C.byref(n)))
        a = np.empty(n.value, dtype=np.uint32)
        self._ck(self.lib.slod_get_patch_local_dofs(self.h, patch, a.ctypes.data_as(C.POINTER(C.c_uint32)), C.byref(n)))
        return a

    def patch_dof_class(self, patch, which):
        n = C.c_int32()
        self._ck(self.lib.slod_get_patch_dof_class(self.h, patch, which, None, C.byref(n)))
        a = np.empty(n.value, dtype=np.uint32)
        self._ck(self.lib.slod_get_patch_dof_class(self.h, patch, which, a.ctypes.data_as(C.POINTER(C.c_uint32)),
                                                   C.byref(n)))
        return a

    # -- hot path, host buffers --------------------------------------------------------------------------
    def compute_basis(self):
        self._ck(self.lib.slod_compute_basis(self.h))

    def update_basis(self):
        """Recompute only the patches (and K row blocks) the coefficient change since the last compute_basis /
        update_basis reaches (slod_update_basis).  Returns {"patches": n, "row_blocks": m}."""
        n, m = C.c_int64(), C.c_int64()
        self._ck(self.lib.slod_update_basis(self.h, C.byref(n), C.byref(m)))
        return {"patches": n.value, "row_blocks": m.value}

    def basis(self, patch, comp=0):
        nf = self.patch_info(patch)["n_fine"]
        phi = np.empty(nf)
        aphi = np.empty(nf)
        self._ck(self.lib.slod_get_basis(self.h, patch, comp, _dp(phi), _dp(aphi)))
        return phi, aphi

    @property
    def basis_stride(self):
        n = C.c_int64()
        self._ck(self.lib.slod_basis_stride(self.h, C.byref(n)))
        return n.value

    def all_basis(self, reuse=False, want_aphi=True):
        """(phi, A*phi) of all patches, [n_patches, spacedim, stride]; want_aphi=False skips the second array (None)."""
        shape = (self.n_patches, self.s, self.basis_stride)
        phi = self._out("phi", shape, reuse=reuse)
        aphi = self._out("aphi", shape, reuse=reuse) if want_aphi else None
        self._ck(self.lib.slod_get_all_basis(self.h, _dp(phi), _dp(aphi) if want_aphi else None))
        return phi, aphi

    def assemble_coarse(self):
        self._ck(self.lib.slod_assemble_coarse(self.h))

    def coarse_csr(self, reuse=False):
        return self._csr(self.lib.slod_get_coarse_csr, "", reuse)

    def _csr(self, getter, key, reuse):
        nr, nnz = C.c_int64(), C.c_int64()
        self._ck(getter(self.h, None, None, None, C.byref(nr), C.byref(nnz)))
        rowptr = self._out(key + "rowptr", nr.value + 1, np.int64, reuse=reuse)
        col = self._out(key + "col", nnz.value, np.int64, reuse=reuse)
        val = self._out(key + "val", nnz.value, reuse=reuse)
        i64p = C.POINTER(C.c_int64)
        self._ck(getter(self.h, rowptr.ctypes.data_as(i64p), col.ctypes.data_as(i64p), _dp(val), C.byref(nr),
                        C.byref(nnz)))
        return rowptr, col, val

    # -- online phase (LOD::solve, source/LOD.cc:975-1001; prolongation :1251) --
    @property
    def n_fine(self):
        n = C.c_int64()
        self._ck(self.lib.slod_fine_size(self.h, C.byref(n)))
        return n.value

    def coarse_rhs(self, f_fine):
        f = np.ascontiguousarray(f_fine, dtype=np.float64).ravel()
        if f.size != self.n_fine:
            raise ValueError(f"fine vector has {f.size} entries, expected {self.n_fine}")
        b = np.empty(self.n_patches * self.s)
        self._ck(self.lib.slod_coarse_rhs(self.h, _dp(f), _dp(b)))
        return b

    def coarse_solve(self, rhs, max_steps=10000, tolerance=1e-10, reduction=1e-10):
        """Returns (u, steps, residual); raises SlodError (SLOD_ERR_NUMERIC) when CG does not converge."""
        b = np.ascontiguousarray(rhs, dtype=np.float64).ravel()
        if b.size != self.n_patches * self.s:
            raise ValueError("coarse vector has the wrong size")
        u = np.empty_like(b)
        steps, res = C.c_int32(), C.c_double()
        self._ck(self.lib.slod_coarse_solve(self.h, _dp(b), _dp(u), max_steps, tolerance, reduction,
                                            C.byref(steps), C.byref(res)))
        return u, steps.value, res.value

    def prolongate(self, u_coarse):
        u = np.ascontiguousarray(u_coarse, dtype=np.float64).ravel()
        if u.size != self.n_patches * self.s:
            raise ValueError("coarse vector has the wrong size")
        out = np.empty(self.n_fine)
        self._ck(self.lib.slod_prolongate(self.h, _dp(u), _dp(out)))
        return out

    # -- batched online phase: k vectors per call, one per row of a (k, n) array --
    def _block(self, a, n, what):
        a = np.ascontiguousarray(a, dtype=np.float64)
        if a.ndim != 2 or a.shape[0] < 1 or a.shape[1] != n:
            raise ValueError(f"{what} must be a 2-D array of shape (k, {n}) with k >= 1, got {a.shape}")
        return a

    # reuse: as in all_basis (benchmark loops: the output block of the previous call of the same shape is overwritten)
    def coarse_rhs_batch(self, F, reuse=False):
        """B = C^T F row by row: F (k, n_fine) -> (k, n_coarse)."""
        f = self._block(F, self.n_fine, "fine block")
        b = self._out("rhs_batch", (f.shape[0], self.n_patches * self.s), reuse=reuse)
        self._ck(self.lib.slod_coarse_rhs_batch(self.h, f.shape[0], _dp(f), _dp(b)))
        return b

    def coarse_solve_batch(self, B, max_steps=10000, tolerance=1e-10, reduction=1e-10, reuse=False):
        """Per-row CG: B (k, n_coarse) -> (U (k, n_coarse), steps int32[k], residual[k]); raises SlodError
        (SLOD_ERR_NUMERIC) when a row does not converge."""
        b = self._block(B, self.n_patches * self.s, "coarse block")
        k = b.shape[0]
        u = self._out("u_batch", b.shape, reuse=reuse)
        steps = self._out("steps_batch", k, np.int32, reuse=reuse)
        res = self._out("res_batch", k, reuse=reuse)
        self._ck(self.lib.slod_coarse_solve_batch(self.h, k, _dp(b), _dp(u), max_steps, tolerance, reduction,
                                                  steps.ctypes.data_as(C.POINTER(C.c_int32)), _dp(res)))
        return u, steps, res

    def prolongate_batch(self, U, reuse=False):
        """U_fine = C U row by row: U (k, n_coarse) -> (k, n_fine)."""
        u = self._block(U, self.n_patches * self.s, "coarse block")
        out = self._out("uf_batch", (u.shape[0], self.n_fine), reuse=reuse)
        self._ck(self.lib.slod_prolongate_batch(self.h, u.shape[0], _dp(u), _dp(out)))
        return out

    # -- coarse mass matrix, L2 projection and backward Euler on the SLOD space (an extension of the reference) --
    def assemble_coarse_mass(self):
        self._ck(self.lib.slod_assemble_coarse_mass(self.h))

    def coarse_mass_csr(self, reuse=False):
        """CSR of M_H = C^T M_h C: (rowptr, col, val), the pattern of coarse_csr()."""
        return self._csr(self.lib.slod_get_coarse_mass_csr, "mass_", reuse)

    def l2_project_batch(self, V, max_steps=10000, tolerance=1e-12, reduction=1e-12, reuse=False):
        """M_H u = C^T M_h v row by row: V (k, n_fine) -> (U (k, n_coarse), steps int32[k], residual[k])."""
        v = self._block(V, self.n_fine, "fine block")
        k = v.shape[0]
        u = self._out("l2_u", (k, self.n_patches * self.s), reuse=reuse)
        steps = self._out("l2_steps", k, np.int32, reuse=reuse)
        res = self._out("l2_res", k, reuse=reuse)
        self._ck(self.lib.slod_l2_project_batch(self.h, k, _dp(v), _dp(u), max_steps, tolerance, reduction,
                                                steps.ctypes.data_as(C.POINTER(C.c_int32)), _dp(res)))
        return u, steps, res

    def _vec_or_none(self, a, n, what):
        if a is None:
            return None
        a = np.ascontiguousarray(a, dtype=np.float64).ravel()
        if a.size != n:
            raise ValueError(f"{what} has {a.size} entries, expected {n}")
        return a

    def heat_solve(self, f_fine, u0_coarse, dt, n_steps, out_every=1, max_steps=10000, tolerance=0.0,
                   reduction=1e-12):
        """Backward Euler on the SLOD space (f_fine / u0_coarse may be None: zero).  Returns (U (n_steps // out_every,
        n_coarse), cg_steps int32[n_steps])."""
        nc = self.n_patches * self.s
        f = self._vec_or_none(f_fine, self.n_fine, "fine vector")
        u0 = self._vec_or_none(u0_coarse, nc, "coarse vector")
        out = np.empty((max(n_steps // max(out_every, 1), 1), nc))
        steps = np.zeros(max(n_steps, 1), dtype=np.int32)
        self._ck(self.lib.slod_heat_solve(self.h, None if f is None else _dp(f), None if u0 is None else _dp(u0), dt,
                                          n_steps, out_every, _dp(out), max_steps, tolerance, reduction,
                                          steps.ctypes.data_as(C.POINTER(C.c_int32))))
        return out, steps

    def heat_solve_batch(self, F, U0, dt, n_steps, out_every=1, max_steps=10000, tolerance=0.0, reduction=1e-12):
        """k trajectories at once: F (k, n_fine), U0 (k, n_coarse) (either may be None: zero).  Returns
        (U (n_steps // out_every, k, n_coarse), cg_steps int32 (n_steps, k))."""
        nc = self.n_patches * self.s
        f = None if F is None else self._block(F, self.n_fine, "fine block")
        u0 = None if U0 is None else self._block(U0, nc, "coarse block")
        if f is not None and u0 is not None and f.shape[0] != u0.shape[0]:
            raise ValueError("F and U0 must have the same number of rows")
        if f is None and u0 is None:
            raise ValueError("give F or U0 (the number of trajectories)")
        k = (f if f is not None else u0).shape[0]
        out = np.empty((max(n_steps // max(out_every, 1), 1), k, nc))
        steps = np.zeros((max(n_steps, 1), k), dtype=np.int32)
        self._ck(self.lib.slod_heat_solve_batch(self.h, k, None if f is None else _dp(f),
                                                None if u0 is None else _dp(u0), dt, n_steps, out_every, _dp(out),
                                                max_steps, tolerance, reduction,
                                                steps.ctypes.data_as(C.POINTER(C.c_int32))))
        return out, steps

    def fem_heat_solve(self, f_fine, u0_fine, dt, n_steps, out_every=1, max_steps=200000, tolerance=0.0,
                       reduction=1e-12):
        """The fine-scale reference trajectory.  Returns (U (n_steps // out_every, n_fine), cg_steps int32[n_steps])."""
        f = self._vec_or_none(f_fine, self.n_fine, "fine vector")
        u0 = self._vec_or_none(u0_fine, self.n_fine, "fine vector")
        out = np.empty((max(n_steps // max(out_every, 1), 1), self.n_fine))
        steps = np.zeros(max(n_steps, 1), dtype=np.int32)
        self._ck(self.lib.slod_fem_heat_solve(self.h, None if f is None else _dp(f), None if u0 is None else _dp(u0),
                                              dt, n_steps, out_every, _dp(out), max_steps, tolerance, reduction,
                                              steps.ctypes.data_as(C.POINTER(C.c_int32))))
        return out, steps

    # -- theta scheme with forcing sum_q g_q(t) f_q(x) (slod_heat_theta_solve / _batch, slod_fem_heat_theta_solve) --
    def _fields(self, F, G, n_steps, lead, n):
        """F (*lead, n_fields, n) or None, G (*lead, n_steps + 1, n_fields) or None -> (F, G, n_fields) as C arrays."""
        if F is None:
            return None, None, 1
        F = np.ascontiguousarray(F, dtype=np.float64)
        if F.ndim != len(lead) + 2 or F.shape[:len(lead)] != lead or F.shape[-1] != n or F.shape[-2] < 1:
            raise ValueError(f"fields must have shape {lead + ('n_fields', n)}, got {F.shape}")
        nq = F.shape[-2]
        if G is not None:
            G = np.ascontiguousarray(G, dtype=np.float64)
            if G.shape != lead + (n_steps + 1, nq):
                raise ValueError(f"g must have shape {lead + (n_steps + 1, nq)}, got {G.shape}")
        return F, G, nq

    def heat_theta_solve(self, f_fields, g, u0_coarse, theta, dt, n_steps, out_every=1, n_startup=0, max_steps=10000,
                         tolerance=0.0, reduction=1e-12):
        """The theta scheme on the SLOD space: f_fields (n_fields, n_fine) or None, g (n_steps + 1, n_fields) or None
        (g = 1), u0_coarse or None.  Returns (U (n_steps // out_every, n_coarse), cg_steps int32[n_steps])."""
        nc = self.n_patches * self.s
        f, gg, nq = self._fields(f_fields, g, n_steps, (), self.n_fine)
        u0 = self._vec_or_none(u0_coarse, nc, "coarse vector")
        out = np.empty((max(n_steps // max(out_every, 1), 1), nc))
        steps = np.zeros(max(n_steps, 1), dtype=np.int32)
        self._ck(self.lib.slod_heat_theta_solve(self.h, theta, dt, n_steps, out_every, n_startup, nq,
                                                None if f is None else _dp(f), None if gg is None else _dp(gg),
                                                None if u0 is None else _dp(u0), _dp(out), max_steps, tolerance,
                                                reduction, steps.ctypes.data_as(C.POINTER(C.c_int32))))
        return out, steps

    def heat_theta_solve_batch(self, F, G, U0, theta, dt, n_steps, out_every=1, n_startup=0, max_steps=10000,
                               tolerance=0.0, reduction=1e-12):
        """k trajectories at once: F (k, n_fields, n_fine), G (k, n_steps + 1, n_fields), U0 (k, n_coarse) (each may be
        None).  Returns (U (n_steps // out_every, k, n_coarse), cg_steps int32 (n_steps, k))."""
        nc = self.n_patches * self.s
        if F is None and U0 is None:
            raise ValueError("give F or U0 (the number of trajectories)")
        k = np.shape(F)[0] if F is not None else np.shape(U0)[0]
        f, gg, nq = self._fields(F, G, n_steps, (k,), self.n_fine)
        u0 = None if U0 is None else self._block(U0, nc, "coarse block")
        if u0 is not None and u0.shape[0] != k:
            raise ValueError("F and U0 must have the same number of rows")
        out = np.empty((max(n_steps // max(out_every, 1), 1), k, nc))
        steps = np.zeros((max(n_steps, 1), k), dtype=np.int32)
        self._ck(self.lib.slod_heat_theta_solve_batch(self.h, k, theta, dt, n_steps, out_every, n_startup, nq,
                                                      None if f is None else _dp(f), None if gg is None else _dp(gg),
                                                      None if u0 is None else _dp(u0), _dp(out), max_steps, tolerance,
                                                      reduction, steps.ctypes.data_as(C.POINTER(C.c_int32))))
        return out, steps

    def fem_heat_theta_solve(self, f_fields, g, u0_fine, theta, dt, n_steps, out_every=1, n_startup=0,
                             max_steps=200000, tolerance=0.0, reduction=1e-12):
        """The fine-scale reference of heat_theta_solve.  Returns (U (n_steps // out_every, n_fine), cg_steps)."""
        f, gg, nq = self._fields(f_fields, g, n_steps, (), self.n_fine)
        u0 = self._vec_or_none(u0_fine, self.n_fine, "fine vector")
        out = np.empty((max(n_steps // max(out_every, 1), 1), self.n_fine))
        steps = np.zeros(max(n_steps, 1), dtype=np.int32)
        self._ck(self.lib.slod_fem_heat_theta_solve(self.h, theta, dt, n_steps, out_every, n_startup, nq,
                                                    None if f is None else _dp(f), None if gg is None else _dp(gg),
                                                    None if u0 is None else _dp(u0), _dp(out), max_steps, tolerance,
                                                    reduction, steps.ctypes.data_as(C.POINTER(C.c_int32))))
        return out, steps

    # -- fine-scale reference problem (assemble_and_solve_fem_problem, source/LOD.cc:1004-1094) and norms (:1252) --
    def fem_solve(self, f_fine, max_steps=200000, tolerance=1e-12, reduction=1e-10):
        """Returns (u_fine, steps, residual)."""
        f = np.ascontiguousarray(f_fine, dtype=np.float64).ravel()
        if f.size != self.n_fine:
            raise ValueError(f"fine vector has {f.size} entries, expected {self.n_fine}")
        u = np.empty_like(f)
        steps, res = C.c_int32(), C.c_double()
        self._ck(self.lib.slod_fem_solve(self.h, _dp(f), _dp(u), max_steps, tolerance, reduction,
                                         C.byref(steps), C.byref(res)))
        return u, steps.value, res.value

    def fine_norms(self, v_fine):
        """(L2 norm, H1 seminorm, energy norm) of a fine vector."""
        v = np.ascontiguousarray(v_fine, dtype=np.float64).ravel()
        if v.size != self.n_fine:
            raise ValueError(f"fine vector has {v.size} entries, expected {self.n_fine}")
        l2, h1, en = C.c_double(), C.c_double(), C.c_double()
        self._ck(self.lib.slod_fine_norms(self.h, _dp(v), C.byref(l2), C.byref(h1), C.byref(en)))
        return l2.value, h1.value, en.value

    def fine_norms_reference(self, v_fine):
        """(L2_norm, Linfty_norm, H1_norm) with the reference's quadrature (ParsedConvergenceTable::difference)."""
        v = np.ascontiguousarray(v_fine, dtype=np.float64).ravel()
        if v.size != self.n_fine:
            raise ValueError(f"fine vector has {v.size} entries, expected {self.n_fine}")
        l2, li, h1 = C.c_double(), C.c_double(), C.c_double()
        self._ck(self.lib.slod_fine_norms_reference(self.h, _dp(v), C.byref(l2), C.byref(li), C.byref(h1)))
        return l2.value, li.value, h1.value

    def diagnostics(self, patch, comp=0):
        """8 doubles (slod_get_patch_diagnostics): [0] ||d||_inf before truncation, [1] truncation steps, [5] path
        (0 LOD, 1 Cholesky fast path, 2 Jacobi, 3 QL), [6] QL iterations / Jacobi sweeps, [7] status bits.  [2], [3] by
        path: 0 -> zeros; 1 -> largest diagonal entry of G_o and smallest LDL^T pivot (bounds: sigma_0 / n <= [2] <=
        sigma_0, lambda_min <= [3] <= [2]); 2, 3 -> sigma_0 and the smallest sigma still used."""
        out = np.empty(8)
        self._ck(self.lib.slod_get_patch_diagnostics(self.h, patch, comp, _dp(out)))
        return out

    def debug_stages(self, patch, want_G=True):
        info = self.patch_info(patch)
        ni, ncd = info["n_internal"], info["n_coarse"]
        X = np.empty((ni, ncd))
        Minv = np.empty((ncd, ncd))
        G = np.empty((ncd, ncd)) if want_G else None
        self._ck(self.lib.slod_debug_patch_stages(self.h, patch, _dp(X), _dp(Minv), _dp(G) if want_G else None))
        return X, Minv, G

    def debug_select(self, patches, G, Minv):
        """The selection stage on caller matrices (slod_debug_select).  patches: distinct ids; G, Minv: one
        (n_coarse, n_coarse) array per patch, reference column order.  Returns (c, diag): c a list of (spacedim, n_coarse)
        arrays, diag (len(patches), spacedim, 8) in the layout of diagnostics()."""
        ids = np.ascontiguousarray(patches, dtype=np.int64).ravel()
        if len(G) != ids.size or len(Minv) != ids.size:
            raise ValueError("one G and one Minv per patch")
        ncd = [self.patch_info(int(p))["n_coarse"] for p in ids]
        for k, (g, m) in enumerate(zip(G, Minv)):
            if np.shape(g) != (ncd[k], ncd[k]) or np.shape(m) != (ncd[k], ncd[k]):
                raise ValueError(f"patch {ids[k]}: G and Minv must be {ncd[k]} x {ncd[k]}")
        g = np.concatenate([np.asarray(x, dtype=np.float64).ravel() for x in G]) if ids.size else np.zeros(1)
        m = np.concatenate([np.asarray(x, dtype=np.float64).ravel() for x in Minv]) if ids.size else np.zeros(1)
        c = np.empty(max(1, self.s * sum(ncd)))
        diag = np.empty((ids.size, self.s, 8))
        self._ck(self.lib.slod_debug_select(self.h, ids.size, ids.ctypes.data_as(C.POINTER(C.c_int64)), _dp(g), _dp(m),
                                            _dp(c), _dp(diag)))
        off = np.concatenate([[0], np.cumsum([self.s * k for k in ncd])]).astype(int)
        return [c[off[i]:off[i + 1]].reshape(self.s, ncd[i]) for i in range(ids.size)], diag

    def timings(self):
        out = np.zeros(8)
        self._ck(self.lib.slod_get_timings(self.h, _dp(out), 8))
        return out

    @property
    def launch_count(self):
        n = C.c_int64()
        self._ck(self.lib.slod_launch_count(self.h, C.byref(n)))
        return n.value

    @property
    def ell_width(self):
        n = C.c_int64()
        self._ck(self.lib.slod_ell_width(self.h, C.byref(n)))
        return n.value

    # -- hot path, device buffers (pointers are plain integers, e.g. torch.Tensor.data_ptr()) -----------
    def compute_basis_device(self, p0, p1, d_phi, d_aphi, stream=0):
        self._ck(self.lib.slod_compute_basis_device(self.h, p0, p1, C.c_void_p(d_phi), C.c_void_p(d_aphi),
                                                    C.c_void_p(stream)))

    def assemble_coarse_device(self, p0, p1, d_phi, d_aphi, d_K, stream=0):
        self._ck(self.lib.slod_assemble_coarse_device(self.h, p0, p1, C.c_void_p(d_phi), C.c_void_p(d_aphi),
                                                      C.c_void_p(d_K), C.c_void_p(stream)))

    # -- one handle per GPU, NCCL inside the library ---------------------------------------------------------
    def owned_range(self, rank, world):
        b, e = C.c_int64(), C.c_int64()
        self._ck(self.lib.slod_owned_range(self.h, rank, world, C.byref(b), C.byref(e)))
        return b.value, e.value

    def comm_unique_id(self):
        """128 bytes of an ncclUniqueId (create on one rank, hand to the others)."""
        buf = (C.c_char * 128)()
        rc = self.lib.slod_comm_unique_id(C.cast(buf, C.c_void_p))
        if rc != SLOD_OK:
            raise SlodError(rc, self.lib.slod_last_create_error().decode())
        return bytes(buf)

    def comm_init(self, rank, world, unique_id):
        buf = (C.c_char * 128).from_buffer_copy(unique_id)
        self._ck(self.lib.slod_comm_init(self.h, rank, world, C.cast(buf, C.c_void_p)))

    def offline_distributed(self, d_phi, d_aphi, d_K, gather_phi=False, gather_K=True, stream=0):
        self._ck(self.lib.slod_offline_distributed(self.h, C.c_void_p(d_phi), C.c_void_p(d_aphi), C.c_void_p(d_K),
                                                   int(gather_phi), int(gather_K), C.c_void_p(stream)))

    def save_state(self, path):
        """Checkpoint of the offline phase (basis + coarse matrix) to one binary file."""
        self._ck(self.lib.slod_save_state(self.h, os.fsencode(path)))

    def load_state(self, path):
        self._ck(self.lib.slod_load_state(self.h, os.fsencode(path)))

    def set_host_outputs(self, h_phi=0, h_aphi=0, h_K=0):
        """Host addresses (ints, 0 = none) for the rank's own rows of phi / A*phi / K: slod_offline_distributed copies them
        on the library's own stream as soon as they are final, slod_synchronize waits for the copies."""
        self._ck(self.lib.slod_set_host_outputs(self.h, C.c_void_p(h_phi or None), C.c_void_p(h_aphi or None),
                                                C.c_void_p(h_K or None)))

    def synchronize(self):
        """Wait for the device-buffer calls above; raises SlodError (SLOD_ERR_NUMERIC) if a patch reported a status."""
        self._ck(self.lib.slod_synchronize(self.h))

    def measure_fp64_peak(self):
        """(DFMA, DMMA) TFLOP/s of the handle's device, measured now."""
        a, b = C.c_double(), C.c_double()
        self._ck(self.lib.slod_measure_fp64_peak(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def ell_to_csr(self, h_K):
        h_K = np.ascontiguousarray(h_K, dtype=np.float64)
        nr, nnz = C.c_int64(), C.c_int64()
        self._ck(self.lib.slod_ell_to_csr(self.h, None, None, None, None, C.byref(nr), C.byref(nnz)))
        rowptr = np.empty(nr.value + 1, dtype=np.int64)
        col = np.empty(nnz.value, dtype=np.int64)
        val = np.empty(nnz.value)
        i64p = C.POINTER(C.c_int64)
        self._ck(self.lib.slod_ell_to_csr(self.h, _dp(h_K), rowptr.ctypes.data_as(i64p), col.ctypes.data_as(i64p),
                                          _dp(val), C.byref(nr), C.byref(nnz)))
        return rowptr, col, val
