/*
 * slod.h -- C ABI of the B200-native SLOD offline phase (libslod_b200.so).
 *
 * The reference (camillabelponer/dealii-slod) has no FFI layer: the seam this library replaces is
 * the pair of protected member functions
 *     LOD::compute_basis_function_candidates()   source/LOD.cc:296-768   (declared include/LOD.h:176)
 *     LOD::assemble_global_matrix()              source/LOD.cc:860-973   (declared include/LOD.h:178)
 * called from LOD::run() (source/LOD.cc:1433-1434), together with the integer set-up they depend on
 * (create_patches source/LOD.cc:122-244, create_mesh_for_patch :770-858, fill_dofs_indices_vector
 * include/LODtools.h:334-375) and the PDE hook assemble_stiffness (include/Diffusion.h:111-207,
 * include/Elasticity.h:163-299).  On top of those two, the stages that consume their results are exported as well
 * (SURVEY section 8f rows 1-2): LOD::solve() and the prolongation (source/LOD.cc:975-1001, :1251), the fine FEM reference
 * solve and the error norms (source/LOD.cc:1004-1094, :1252).  INTEGRATION.md shows the reference-side binding.
 *
 * Conventions
 *  - plain C, opaque handle, no exceptions cross the boundary; every call returns an int status
 *    (SLOD_OK == 0) and slod_last_error() gives the message of the last failure on that handle.
 *  - all floating point data is fp64; all buffers are caller-owned.
 *  - host-buffer calls return when their results are complete, with one exception: slod_assemble_coarse only enqueues
 *    (see there).  The device-buffer entry points (slod_*_device) only enqueue on the caller's stream;
 *    slod_synchronize() is their synchronisation point and reports numerical failures of the enqueued patches.
 *  - multi-GPU, two ways, both with NCCL inside the library (libnccl.so.2 is loaded on first use, a single-GPU handle
 *    never needs it): (a) slod_params.n_gpus = N -- one handle, one process, N devices; slod_compute_basis and
 *    slod_assemble_coarse split the patches over the devices and combine the results over NVLink, every other call
 *    behaves as on one device; (b) one process and one handle per GPU (MPI / torchrun style): slod_comm_init joins the
 *    handles into one NCCL communicator and slod_offline_distributed runs the phase with its two all-gathers.
 *    The slod_*_device entry points remain for callers that do their own exchange.
 *  - there is NO CPU fallback: if no CUDA device is usable slod_create fails with SLOD_ERR_CUDA.
 *  - a handle is thread-compatible, not thread-safe (one call at a time per handle).  DIFFERENT handles may be used
 *    concurrently from different host threads and streams, on the same device too: the kernels read their parameters
 *    from one __constant__ block per device, and every call that launches kernels binds its handle's block for its
 *    scope (the calls of different handles on one device enqueue one after the other; the block is re-uploaded,
 *    stream-ordered, only when the resident bytes differ).
 *  - patch size: n_subdivisions >= 2 (with 1 the matrix P^T A^-1 P of some patch is singular: refused with
 *    SLOD_ERR_UNSUPPORTED) and any oversampling whose patches have at most 128 coarse dofs (the Gram register tile of
 *    the dense stage), except 2-D with 8 or more subdivisions once the coefficient window (room for one value per Gauss
 *    point) no longer fits shared memory: diffusion oversampling >= 5, elasticity >= 3 at 8 subdivisions.  Both are
 *    refused by slod_create with SLOD_ERR_UNSUPPORTED.  Patches too large for the shared-memory solvers (3-D,
 *    4 subdivisions, oversampling 2) run through a direct banded solver with its windows in global memory (slower), like
 *    the reference's direct solver (include/LODtools.h:575-580).  slod_get_plan tells which kernels a handle uses.
 *  - patch id == active-cell index of the centre cell after refine_global (Morton / Z-order, x low
 *    bit), exactly as in source/LOD.cc:184-192.
 *  - patch-local fine nodes are numbered lexicographically (x fastest) on the patch's own node box
 *    (p_a = m_a * n_subdivisions + 1 nodes along axis a); a fine DoF is spacedim*node + comp.
 *    slod_get_patch_fine_dofs() maps them to deal.II's global fine DoF numbers,
 *    slod_get_patch_local_dofs() to deal.II's patch-local numbers (Patch::basis_function layout,
 *    include/LOD.h:79).
 */
#ifndef SLOD_B200_H
#define SLOD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct slod_ctx slod_ctx;

enum {
  SLOD_OK = 0,
  SLOD_ERR_INVALID = 1,      /* bad argument / inconsistent parameters                  */
  SLOD_ERR_UNSUPPORTED = 2,  /* configuration outside the implemented envelope           */
  SLOD_ERR_CUDA = 3,         /* CUDA runtime error or no usable device                   */
  SLOD_ERR_STATE = 4,        /* call order violated (e.g. basis requested before compute) */
  SLOD_ERR_NUMERIC = 5       /* a patch problem was not SPD / an eigen-solver or CG did not converge */
};

/* SLOD_PROBLEM_DIFFUSION_TENSOR: -div(A grad u) with a symmetric positive definite dim x dim tensor A per coefficient
 * cell (laminates, fibre composites, layered media), dim 2 or 3, spacedim 1; set with slod_set_coefficient_tensor. */
enum { SLOD_PROBLEM_DIFFUSION = 0, SLOD_PROBLEM_ELASTICITY = 1, SLOD_PROBLEM_DIFFUSION_TENSOR = 2 };
/* slod_params.device: -1 = current CUDA device; SLOD_DEVICE_NONE = no device, integer maps only
 * (patch lists, DoF maps, CSR pattern) -- every compute call on such a handle returns SLOD_ERR_CUDA. */
enum { SLOD_DEVICE_CURRENT = -1, SLOD_DEVICE_NONE = -2 };

/* Mirrors LODParameters (include/LOD.h:85-157) + the template arguments <dim, spacedim>. */
typedef struct {
  int dim;                  /* 2 or 3 (3 only with spacedim 1)                                   */
  int spacedim;             /* 1 diffusion (scalar or tensor), 2 = dim elasticity                 */
  int n_global_refinements; /* "Number of global refinements"                 include/LOD.h:95   */
  int n_subdivisions;       /* "Number of subdivisions" (power of two)        include/LOD.h:94   */
  int oversampling;         /* "Oversampling"                                 include/LOD.h:93   */
  int stabilize;            /* "Stabilize phi_LOD candidates" (SLOD)          include/LOD.h:97   */
  int problem;              /* SLOD_PROBLEM_*                                                     */
  int quirk_presaved;       /* reproduce source/LOD.cc:354-362 ("Constant problem coefficients") */
  int device;               /* CUDA device ordinal, SLOD_DEVICE_CURRENT or SLOD_DEVICE_NONE        */
  int n_gpus;               /* 0 or 1: the handle drives `device` alone.  N > 1: ONE handle drives the N devices
                               device .. device + N - 1 of this process (SLOD_DEVICE_CURRENT counts as 0): the patches
                               are split into contiguous even ranges (the reference's locally_owned_patches,
                               source/LOD.cc:116-118), one host thread and one NCCL rank per device inside the library */
} slod_params;

/* life cycle ------------------------------------------------------------------------------------*/
int slod_create(const slod_params *par, slod_ctx **out);
void slod_destroy(slod_ctx *ctx);
const char *slod_last_error(const slod_ctx *ctx);
/* message of the last failed slod_create (which has no handle to ask) */
const char *slod_last_create_error(void);

/* coefficients: replaces problem_parameter (include/Diffusion.h:7-54).  `cellwise` holds one value
 * per cell of a (2^eta_refinement)^dim grid, lexicographic x fastest.  field 0 = alpha | lambda,
 * field 1 = mu.  If the table is finer than the fine sub-cells (eta < h, as in tests/Poisson_LOD_Example)
 * it is sampled at the Gauss points like the reference does; that mode is available in 2-D. */
int slod_set_coefficient(slod_ctx *ctx, int field, int eta_refinement, const double *cellwise, size_t n);

/* the coefficient of a SLOD_PROBLEM_DIFFUSION_TENSOR handle: `cells` is [n_cells][dim (dim + 1) / 2], one symmetric
 * tensor per cell of the (2^eta_refinement)^dim grid, lexicographic x fastest, each in Voigt order
 *   2-D: a_xx, a_yy, a_xy          3-D: a_xx, a_yy, a_zz, a_yz, a_xz, a_xy.
 * Sub-cell matrices are sum_f a_f K_f with K_f = d_a phi_i d_b phi_j (+ d_b phi_i d_a phi_j for a != b) for component
 * f = (a, b), integrated like the scalar problem's.  Every argument is checked before the device (a maps-only handle
 * checks them too): another problem, n_cells != (2^eta_refinement)^dim, a non-finite entry or a cell that is not
 * positive definite (a Cholesky factorisation with positive pivots) -> SLOD_ERR_INVALID, and slod_last_error names the
 * first offending cell; a table finer than the fine sub-cells (eta < h) -> SLOD_ERR_UNSUPPORTED (the per-Gauss-point mode
 * is scalar only).  slod_set_coefficient on a tensor handle returns SLOD_ERR_INVALID: setting one component at a time
 * could leave an indefinite tensor between calls.  Each component is then stored and expanded onto the sub-cells like a
 * slod_set_coefficient field.  slod_update_basis compares every component (a changed off-diagonal entry marks its
 * cell), and a checkpoint records the problem, so it loads only into a tensor handle.  Where the six-field window of a
 * 3-D patch fits no shared-memory plan (4 subdivisions), the SIMT solver and the finish kernel read it from global
 * memory: such handles have the scalar handle's plan. */
int slod_set_coefficient_tensor(slod_ctx *ctx, int eta_refinement, const double *cells, size_t n_cells);

/* the kernel plan slod_create chose from the largest patch shape (read only; a maps-only handle plans for 227 KB of
 * shared memory per block, as on a B200).  out[8]:
 *   [0] tensor-core patch solver variant 0/1/2 (-1: SIMT banded solver)  [1] split factor + triangular-solve kernels
 *   [2] tensor-core dense stage tiles 4/8/16 (0: SIMT dense stage)  [3] SIMT solver windows in global memory
 *   [4] SIMT dense stage coefficients in global memory  [5] blocked coarse-matrix kernel
 *   [6] tridiagonal-QL eigen path (0: Jacobi only)
 *   [7] coefficients per Gauss point: a table set so far is finer than the fine sub-cells
 * Entries [0]..[6] are 0/1 flags where no count is named. */
int slod_get_plan(const slod_ctx *ctx, int32_t out[8]);

/* integer maps (bit-exact with the reference / the oracle) -----------------------------------------*/
int slod_patch_count(const slod_ctx *ctx, int64_t *n_patches);
/* sizes of one patch: cells, fine DoFs, interior DoFs, patch-boundary DoFs (id 99), domain-boundary
 * DoFs (id 0), coarse DoFs; and the node box m[a] cells / lo[a] first coarse cell per axis. */
int slod_get_patch_info(const slod_ctx *ctx, int64_t patch, int32_t *n_cells, int32_t *n_fine, int32_t *n_internal,
                        int32_t *n_boundary, int32_t *n_domain_boundary, int32_t *n_coarse, int32_t lo[3],
                        int32_t m[3]);
/* Patch::cells (active-cell ids, centre first, x-offset outer)            source/LOD.cc:151-201 */
int slod_get_patch_cells(const slod_ctx *ctx, int64_t patch, uint32_t *cells, int32_t *n);
/* lexicographic patch DoF -> deal.II global fine DoF (dof_handler_fine)    source/LOD.cc:925-929 */
int slod_get_patch_fine_dofs(const slod_ctx *ctx, int64_t patch, uint64_t *global_dofs, int32_t *n);
/* lexicographic patch DoF -> deal.II patch-local DoF (dh_fine_patch)       source/LOD.cc:365-366 */
int slod_get_patch_local_dofs(const slod_ctx *ctx, int64_t patch, uint32_t *local_dofs, int32_t *n);
/* fill_dofs_indices_vector (lexicographic patch numbering, ascending)  include/LODtools.h:334-375
 * which: 0 internal, 1 patch boundary (id 99), 2 domain boundary (id 0). */
int slod_get_patch_dof_class(const slod_ctx *ctx, int64_t patch, int which, uint32_t *dofs, int32_t *n);

/* the hot path, host buffers ------------------------------------------------------------------------*/
/* stages assembly .. premultiply for every patch (source/LOD.cc:345-767), batched on the GPU. */
int slod_compute_basis(slod_ctx *ctx);
/* Patch::basis_function[comp] and basis_function_premultiplied[comp] (include/LOD.h:79-80) in
 * lexicographic patch numbering; either pointer may be NULL. n_fine values each. */
int slod_get_basis(const slod_ctx *ctx, int64_t patch, int comp, double *phi, double *A_phi);
/* all patches at once: arrays [n_patches][spacedim][stride] with stride = slod_basis_stride(). */
int slod_basis_stride(const slod_ctx *ctx, int64_t *stride);
int slod_get_all_basis(const slod_ctx *ctx, double *phi, double *A_phi);
/* global_stiffness_matrix = C^T (A C)  (source/LOD.cc:860-973).  The kernels are enqueued and the call returns: every
 * consumer of the matrix (slod_get_coarse_csr, slod_coarse_solve, ...) is ordered behind them and reports an execution
 * error at its own synchronisation, and slod_get_all_basis, called in between, copies while they run. */
int slod_assemble_coarse(slod_ctx *ctx);
/* CSR of the coarse matrix (rows/cols = spacedim*patch + comp, columns ascending; structural zeros of
 * the sparse product are kept).  Call with rowptr == NULL to query n_rows and nnz. */
int slod_get_coarse_csr(const slod_ctx *ctx, int64_t *rowptr, int64_t *col, double *val, int64_t *n_rows,
                        int64_t *nnz);
/* Bring the basis (and the coarse matrix, if it was assembled) up to date with the coefficient tables set since the
 * last successful slod_compute_basis / slod_update_basis, recomputing only what the change reaches (an extension: the
 * reference recomputes everything).
 * Baseline: the device coefficient array (the tables expanded onto the sub-cells or Gauss points) that the last
 * successful slod_compute_basis or slod_update_basis of this single-device handle read.  Calls that only use the
 * coefficient (slod_fem_solve, slod_fine_norms*, slod_fem_heat_solve) leave it alone.
 * A patch is recomputed iff a value of its coefficient window (the coarse cells of its box; under quirk_presaved, the
 * donor's box for a full-size patch) differs bitwise from the baseline -- any field, sub-cell or Gauss point; 0.0 ->
 * -0.0 counts, a table cell no Gauss point samples does not.  If the array's layout changed (its length, or one value
 * per Gauss point instead of per sub-cell or back), every patch is recomputed.
 * If slod_assemble_coarse ran on the basis being updated, the block-ELL rows of every patch whose own or a structural
 * neighbour's basis changed are recomputed (on the blocked kernel: whole Morton groups of 2^dim patches) and the CSR
 * values refreshed; like slod_assemble_coarse the call may return with those kernels enqueued only.  Otherwise K stays
 * unassembled.
 * Afterwards slod_get_all_basis, slod_get_patch_diagnostics and slod_get_coarse_csr (and the block-ELL rows) are
 * bit-identical to what a fresh handle computes from the same tables with slod_compute_basis (+ slod_assemble_coarse).
 * slod_get_timings [0]..[4] report the update's stages (0 where nothing ran).  If nothing differs, only the comparison
 * kernel runs and both counts are 0.  If any patch is recomputed, M_H is stale as after slod_compute_basis.
 * n_patches_recomputed / n_row_blocks_recomputed (may be NULL): patches and K row blocks (spacedim rows each) recomputed.
 * Errors: no baseline (no basis yet, a basis restored by slod_load_state or computed through the device-buffer
 * entry points, the last compute failed) -> SLOD_ERR_STATE; an n_gpus > 1 handle -> SLOD_ERR_UNSUPPORTED; a recomputed
 * patch with a numerical status -> SLOD_ERR_NUMERIC naming the first one, as slod_compute_basis would, and the handle
 * has no basis and no baseline until the next successful slod_compute_basis. */
int slod_update_basis(slod_ctx *ctx, int64_t *n_patches_recomputed /* may be NULL */,
                      int64_t *n_row_blocks_recomputed /* may be NULL */);

/* ---- online phase on the handle's basis and coarse matrix (SURVEY 8f row 1; replaces LOD::solve(),
 * source/LOD.cc:975-1001, and the prolongation in LOD::compare_lod_with_fem(), source/LOD.cc:1251).
 * Fine vectors are lexicographic: index = node * spacedim + component, node = x + G (y + G z), G = N n + 1 nodes per
 * axis; slod_get_patch_fine_dofs gives the deal.II numbering of the same nodes.  Coarse vectors: spacedim*patch + comp. */
int slod_fine_size(const slod_ctx *ctx, int64_t *n_fine);
/* system_rhs = C^T fem_rhs  (basis_matrix_transposed.Tvmult(system_rhs, fem_rhs), source/LOD.cc:981). */
int slod_coarse_rhs(slod_ctx *ctx, const double *f_fine, double *rhs_coarse);
/* K u = rhs by conjugate gradients from u = 0 (SolverCG, source/LOD.cc:994-998), stopped like deal.II's
 * ReductionControl ("Coarse solver control", include/LOD.h:109): ||r||_2 <= tolerance or ||r||_2 <= reduction * ||r_0||_2.
 * Not converged within max_steps -> SLOD_ERR_NUMERIC (deal.II throws SolverControl::NoConvergence).  The preconditioner
 * is diag(K), not the reference's SSOR(1.2): same solution to the tolerance, different step counts.
 * steps / residual (may be NULL) receive the number of steps taken and the final ||r||_2. */
int slod_coarse_solve(slod_ctx *ctx, const double *rhs_coarse, double *u_coarse, int32_t max_steps, double tolerance,
                      double reduction, int32_t *steps, double *residual);
/* lod_solution = C u  (basis_matrix_transposed.vmult(lod_solution, solution), source/LOD.cc:1251). */
int slod_prolongate(slod_ctx *ctx, const double *u_coarse, double *u_fine);
/* Batched online phase: n_rhs >= 1 vectors per call, each one contiguous ([n_rhs][n_fine] / [n_rhs][n_coarse]).
 * Column j of every result is bit-identical to what the same call computes for that vector alone.
 * The per-vector semantics are those of the three calls above (source/LOD.cc:981, :991-998, :1251): same call-order
 * checks, same device (the first one of an n_gpus > 1 handle), and they serve handles restored by slod_load_state.
 * phi and K are read once per group of columns instead of once per vector.  n_rhs < 1 or a NULL buffer ->
 * SLOD_ERR_INVALID.  The reference solves one system per run; these calls are an extension.
 * slod_coarse_solve_batch runs one CG per column, each with its own step count and ReductionControl test; a column that
 * has stopped is no longer updated.  If any column breaks down or does not converge within max_steps the call returns
 * SLOD_ERR_NUMERIC and slod_last_error names the first such column with its steps and residual; u_coarse, steps and
 * residual (may be NULL, else [n_rhs]) are written for all columns in every case. */
int slod_coarse_rhs_batch(slod_ctx *ctx, int32_t n_rhs, const double *f_fine, double *rhs_coarse);
int slod_coarse_solve_batch(slod_ctx *ctx, int32_t n_rhs, const double *rhs_coarse, double *u_coarse,
                            int32_t max_steps, double tolerance, double reduction,
                            int32_t *steps /* [n_rhs] or NULL */, double *residual /* [n_rhs] or NULL */);
int slod_prolongate_batch(slod_ctx *ctx, int32_t n_rhs, const double *u_coarse, double *u_fine);

/* ---- fine-scale reference problem (SURVEY 8f row 2; the solve of LOD::assemble_and_solve_fem_problem,
 * source/LOD.cc:1004-1094, and the norms of compare_lod_with_fem, source/LOD.cc:1252).  Needs only the coefficient.
 * A u = f on the global Q_iso_Q1 grid with homogeneous Dirichlet conditions (boundary rows of f are ignored, u = 0
 * there), matrix free, by diag-preconditioned conjugate gradients (the reference: CG + AMG) with the same stopping
 * rule and error behaviour as slod_coarse_solve. */
int slod_fem_solve(slod_ctx *ctx, const double *f_fine, double *u_fine, int32_t max_steps, double tolerance,
                   double reduction, int32_t *steps, double *residual);
/* Norms of a fine vector (outputs may be NULL): ||v||_L2 = sqrt(v.Mv) and |v|_H1 = sqrt(v.Lv) with the exact Q1 mass
 * and Laplace matrices of the sub-cell grid, and the energy norm sqrt(v.Av) of the problem's own bilinear form.  The
 * reference integrates |u_fem - u_lod| with a Gauss rule on the coarse cells (ParsedConvergenceTable::difference),
 * which is not exact for Q_iso_Q1 functions; these are the exact values of the same norms. */
int slod_fine_norms(slod_ctx *ctx, const double *v_fine, double *l2, double *h1_semi, double *energy);
/* The same norms the way the reference's error tables compute them (ParsedConvergenceTable::difference,
 * source/LOD.cc:1252; include/LOD.h:111-115): VectorTools::integrate_difference with QGauss((degree + 1) * 2) on the cells
 * of dof_handler_fine, i.e. 2 (n_subdivisions + 1) Gauss points per direction on every COARSE cell; norms of the table's
 * default list: L2_norm, Linfty_norm (maximum over the quadrature points and components), H1_norm (the full norm
 * sqrt(L2^2 + |.|_H1^2)).  Outputs may be NULL. */
int slod_fine_norms_reference(slod_ctx *ctx, const double *v_fine, double *l2, double *linfty, double *h1);

/* ---- the coarse mass matrix and the heat equation on the SLOD space.  The reference solves one elliptic problem and has
 * no time-dependent path: these calls are an extension.  They run on the handle's first device (n_gpus > 1: the one that
 * holds all of phi) and serve handles restored by slod_load_state (the checkpoint does not hold M_H: assemble it again).
 *
 * slod_assemble_coarse_mass: M_H = C^T (M_h C) with M_h the exact Q1 mass matrix of the sub-cell grid, in the block-ELL
 * form and on the structural pattern of the coarse matrix (the same slot convention and CSR pattern).  Needs the basis
 * only.  slod_compute_basis, slod_load_state and slod_assemble_coarse make M_H stale: the calls that need it return
 * SLOD_ERR_STATE until it is assembled again.  Device times of its two kernels: slod_get_timings [6] (M_h phi) and [7]
 * (the product).  slod_get_coarse_mass_csr: the same contract as slod_get_coarse_csr. */
int slod_assemble_coarse_mass(slod_ctx *ctx);
int slod_get_coarse_mass_csr(const slod_ctx *ctx, int64_t *rowptr, int64_t *col, double *val, int64_t *n_rows,
                             int64_t *nnz);
/* L2 projection onto the SLOD space of n_rhs fine fields ([n_rhs][n_fine]): M_H u = C^T M_h v, by one CG on M_H per column
 * (diagonal preconditioner, ReductionControl).  Errors and per-column outputs as in slod_coarse_solve_batch. */
int slod_l2_project_batch(slod_ctx *ctx, int32_t n_rhs, const double *v_fine, double *u_coarse, int32_t max_steps,
                          double tolerance, double reduction, int32_t *steps /* [n_rhs] or NULL */,
                          double *residual /* [n_rhs] or NULL */);
/* Backward Euler for du/dt - div(alpha grad u) = f (elasticity: its operator) on the SLOD space, forcing constant in time:
 * (M_H + dt K) u^k = M_H u^{k-1} + dt C^T f, k = 1 .. n_steps, solved in increment form (r = dt (C^T f - K u^{k-1}),
 * (M_H + dt K) delta = r by CG from zero, u^k = u^{k-1} + delta; the stopping rule applies to each increment).  Needs K
 * and M_H.  f_fine / u0_coarse NULL: zero.  Output o (o = 0 .. n_steps / out_every - 1) is u at step (o + 1) out_every.
 * cg_steps (may be NULL) receives the CG steps of every time step.  M_H + dt K is formed once and kept while dt stays the
 * same.  dt <= 0, n_steps < 1, out_every < 1 or > n_steps -> SLOD_ERR_INVALID.  A time step whose CG breaks down or does
 * not converge -> SLOD_ERR_NUMERIC naming the step (and the column); every output of the steps before it is written.
 * slod_heat_solve_batch: n_rhs trajectories ([n_rhs][n_fine] forcings, [n_rhs][n_coarse] initial values, outputs
 * [n_out][n_rhs][n_coarse], cg_steps [n_steps][n_rhs]); column j is bit-identical whatever n_rhs, its position and its
 * neighbours are, and slod_heat_solve agrees with it to the solver tolerance (slod_coarse_solve / _batch). */
int slod_heat_solve(slod_ctx *ctx, const double *f_fine, const double *u0_coarse, double dt, int32_t n_steps,
                    int32_t out_every, double *u_out, int32_t max_steps, double tolerance, double reduction,
                    int32_t *cg_steps);
int slod_heat_solve_batch(slod_ctx *ctx, int32_t n_rhs, const double *f_fine, const double *u0_coarse, double dt,
                          int32_t n_steps, int32_t out_every, double *u_out, int32_t max_steps, double tolerance,
                          double reduction, int32_t *cg_steps);
/* The fine-scale reference trajectory of the same scheme, the counterpart of slod_fem_solve: (M_h + dt A_h) on the global
 * grid with homogeneous Dirichlet rows (boundary rows of f and u0 are ignored), matrix free, diag-preconditioned CG on
 * each increment.  Needs only the coefficient.  u_out [n_steps / out_every][n_fine]; errors as slod_heat_solve. */
int slod_fem_heat_solve(slod_ctx *ctx, const double *f_fine, const double *u0_fine, double dt, int32_t n_steps,
                        int32_t out_every, double *u_out, int32_t max_steps, double tolerance, double reduction,
                        int32_t *cg_steps);
/* The theta scheme for M_H u' + K u = C^T f(t), theta in [1/2, 1] (1/2: Crank-Nicolson, 1: backward Euler), in the
 * increment form above: (M_H + theta dt K) delta = dt (theta b(t_k) + (1 - theta) b(t_{k-1}) - K u^{k-1}).
 * Forcing: f(x, t) = sum_q g_q(t) f_q(x), q = 0 .. n_fields - 1.  f_fine holds the fields [n_fields][n_fine] (NULL: zero
 * forcing; n_fields and g are then ignored); g holds g_q(t_k) at t_k = k dt as [n_steps + 1][n_fields] (NULL: g = 1).
 * Arbitrary per-step loads are n_fields = n_steps + 1 with g the identity.  C^T f_q is formed once per field and kept
 * on the device (n_fields coarse vectors per trajectory); every step's residual reads all n_fields of them, so the
 * per-step form costs O(n_steps) per step.
 * Rannacher start-up: each of the first n_startup steps is two backward-Euler steps of dt / 2 with the loads
 * (g(t_{k-1}) + g(t_k)) / 2 and g(t_k); cg_steps of such a step is the sum of its two solves.  Crank-Nicolson leaves
 * the stiff modes (dt lambda >> 1) of a non-smooth u0 undamped, with amplification near -1: one or two start-up steps
 * damp them.  M_H + c K is kept for the last coefficient c of K formed (theta dt, or dt / 2 during start-up).
 * At theta = 1, n_fields = 1, g = NULL, n_startup = 0 these are slod_heat_solve / _batch / slod_fem_heat_solve, bit
 * for bit.  Every argument is checked before the device and the call order: theta outside [1/2, 1], n_startup < 0 or
 * > n_steps, n_fields < 1 with fields given, a non-finite entry of g (read only with fields given) and the checks of
 * slod_heat_solve -> SLOD_ERR_INVALID.  Then SLOD_ERR_CUDA (maps-only handle), SLOD_ERR_STATE and SLOD_ERR_NUMERIC as
 * there.
 * slod_heat_theta_solve_batch: f_fine [n_rhs][n_fields][n_fine], g [n_rhs][n_steps + 1][n_fields], u0 [n_rhs][n_coarse],
 * u_out [n_out][n_rhs][n_coarse], cg_steps [n_steps][n_rhs]; columns are independent as in slod_heat_solve_batch.
 * slod_fem_heat_theta_solve: the fine-scale reference of the same scheme (M_h + theta dt A_h, as slod_fem_heat_solve),
 * fine u0 and u_out [n_out][n_fine]. */
int slod_heat_theta_solve(slod_ctx *ctx, double theta, double dt, int32_t n_steps, int32_t out_every,
                          int32_t n_startup, int32_t n_fields, const double *f_fine, const double *g,
                          const double *u0_coarse, double *u_out, int32_t max_steps, double tolerance,
                          double reduction, int32_t *cg_steps);
int slod_heat_theta_solve_batch(slod_ctx *ctx, int32_t n_rhs, double theta, double dt, int32_t n_steps,
                                int32_t out_every, int32_t n_startup, int32_t n_fields, const double *f_fine,
                                const double *g, const double *u0_coarse, double *u_out, int32_t max_steps,
                                double tolerance, double reduction, int32_t *cg_steps);
int slod_fem_heat_theta_solve(slod_ctx *ctx, double theta, double dt, int32_t n_steps, int32_t out_every,
                              int32_t n_startup, int32_t n_fields, const double *f_fine, const double *g,
                              const double *u0_fine, double *u_out, int32_t max_steps, double tolerance,
                              double reduction, int32_t *cg_steps);

/* The wave equation M_H u'' + K u = C^T f(t) on the SLOD space, Newmark time stepping with gamma = 1/2 and beta in
 * [0, 1/2] (0: the explicit central-difference scheme, 1/4: average acceleration, unconditionally stable and energy
 * conserving).  Time points t_k = k dt; the forcing f_fine, g, n_fields is that of slod_heat_theta_solve, step k uses
 * g(t_k).  Each step solves for the acceleration, from zero, with the stopping rule of slod_coarse_solve:
 *   start       M_H a_0 = b(t_0) - K u_0
 *   step k      ut = u_{k-1} + dt v_{k-1} + (1/2 - beta) dt^2 a_{k-1},  (M_H + beta dt^2 K) a_k = b(t_k) - K ut,
 *               u_k = ut + beta dt^2 a_k,  v_k = v_{k-1} + dt/2 (a_{k-1} + a_k)
 * The explicit scheme is stable for dt^2 lambda_max(M_H^-1 K) <= 4 (for beta < 1/4: <= 4 / (1 - 4 beta)); the SLOD
 * space holds no fine-scale modes, so that step is set by the coarse mesh, not by the fine one.
 * u0_coarse, v0_coarse NULL: zero.  u_out [n_out][n_coarse] with n_out = n_steps / out_every, output o the state at step
 * (o + 1) out_every; v_out (NULL: not written) the same for v; energy_out [n_out + 1] (NULL: not computed) the energy
 * E = 1/2 v^T M_H v + 1/2 u^T K u at t_0 and at the outputs; cg_steps [n_steps + 1], entry 0 the start solve.
 * M_H + beta dt^2 K is formed in the cache of the heat calls (beta = 0 solves with M_H itself).
 * Every argument is checked before the device and the call order: beta outside [0, 1/2] or NaN, n_fields < 1 with fields
 * given, a non-finite entry of g (read only with fields given) and the checks of slod_heat_solve -> SLOD_ERR_INVALID.
 * Then SLOD_ERR_CUDA (maps-only handle), SLOD_ERR_STATE (slod_assemble_coarse / slod_assemble_coarse_mass have not run)
 * and SLOD_ERR_NUMERIC when an acceleration solve fails, naming the step (0: the start solve) and the column; the outputs
 * of the earlier steps are written.
 * slod_wave_solve_batch: f_fine [n_rhs][n_fields][n_fine], g [n_rhs][n_steps + 1][n_fields], u0 / v0 [n_rhs][n_coarse],
 * u_out / v_out [n_out][n_rhs][n_coarse], energy_out [n_out + 1][n_rhs], cg_steps [n_steps + 1][n_rhs]; a column is bit
 * for bit the same whatever n_rhs, its position and its neighbours, and agrees with slod_wave_solve to the tolerance.
 * slod_fem_wave_solve: the fine-scale reference of the same scheme (M_h + beta dt^2 A_h, homogeneous Dirichlet rows; the
 * boundary rows of the fields, u0 and v0 are ignored), fine u0 / v0 / u_out / v_out, energy 1/2 v^T M_h v + 1/2 u^T A_h u.
 * Needs only the coefficient. */
int slod_wave_solve(slod_ctx *ctx, double beta, double dt, int32_t n_steps, int32_t out_every, int32_t n_fields,
                    const double *f_fine, const double *g, const double *u0_coarse, const double *v0_coarse,
                    double *u_out, double *v_out, double *energy_out, int32_t max_steps, double tolerance,
                    double reduction, int32_t *cg_steps);
int slod_wave_solve_batch(slod_ctx *ctx, int32_t n_rhs, double beta, double dt, int32_t n_steps, int32_t out_every,
                          int32_t n_fields, const double *f_fine, const double *g, const double *u0_coarse,
                          const double *v0_coarse, double *u_out, double *v_out, double *energy_out,
                          int32_t max_steps, double tolerance, double reduction, int32_t *cg_steps);
int slod_fem_wave_solve(slod_ctx *ctx, double beta, double dt, int32_t n_steps, int32_t out_every, int32_t n_fields,
                        const double *f_fine, const double *g, const double *u0_fine, const double *v0_fine,
                        double *u_out, double *v_out, double *energy_out, int32_t max_steps, double tolerance,
                        double reduction, int32_t *cg_steps);

/* ---- checkpoint of the offline phase (SURVEY 8f row 4; the reference has none: it recomputes every run) ----------
 * slod_save_state writes the parameters, the basis (phi, A*phi) and, if assembled, the coarse matrix to one binary
 * file; slod_load_state restores them into a handle created with the SAME parameters (else SLOD_ERR_INVALID), after
 * which the online entry points (slod_coarse_rhs / _solve / slod_prolongate, slod_get_basis, slod_get_coarse_csr) work
 * without recomputing anything.  The coefficient is not part of the file (slod_fem_solve / slod_fine_norms need it set). */
int slod_save_state(slod_ctx *ctx, const char *path);
int slod_load_state(slod_ctx *ctx, const char *path);

/* Page-locked host memory for the caller-owned output buffers of slod_get_all_basis / slod_get_coarse_csr: copies
 * into pageable memory work too but run at a fraction of the link speed.  No reference counterpart. */
int slod_alloc_host(size_t bytes, void **out);
int slod_free_host(void *p);

/* diagnostics: per patch and component 8 doubles:
 *   [0] ||d||_inf before truncation  [1] truncation steps  [2], [3] see below
 *   [4] reserved  [5] selection path (0 LOD branch, 1 Cholesky fast path, 2 Jacobi fallback, 3 tridiagonal QL)
 *   [6] QL iterations / Jacobi sweeps (0 on paths 0 and 1)  [7] status bits
 * [2] and [3] depend on the path.  G_o is the Gram matrix without row and column d, of size n = n_coarse - 1:
 *   path 0: both 0 (no selection).
 *   path 1: [2] the largest diagonal entry of G_o, [3] the smallest pivot of its LDL^T factorisation.  Bounds, not
 *           eigenvalues: sigma_0 / n <= [2] <= sigma_0 and lambda_min(G_o) <= [3] <= [2].  The path is only taken when
 *           [3] > 1e-12 [2], no pivot is <= 0 and ||d||_inf < 0.49 (then [1] = 0: the truncation loop does not fire).
 *   paths 2, 3: [2] sigma_0 (largest |eigenvalue| of G_o), [3] the smallest sigma still used after the 1e-15 sigma_0
 *           threshold and the [1] truncation steps (sigma_0 when none is left). */
int slod_get_patch_diagnostics(const slod_ctx *ctx, int64_t patch, int comp, double out[8]);
/* stage intermediates of one patch for staged parity tests (recomputed on demand for that patch):
 * X = A_ii^{-1} P_i  (n_internal x n_coarse, row-major), Minv (n_coarse^2), BD^T BD (n_coarse^2). Any may be NULL. */
int slod_debug_patch_stages(slod_ctx *ctx, int64_t patch, double *X, double *Minv, double *G);
/* the same stages for a list of patches, run as one work list in the cost order of slod_compute_basis (the persistent
 * kernels go from one patch to the next as they do there); per patch the results equal slod_debug_patch_stages'.
 *   patches: n distinct patch ids;
 *   X: packed per patch, n_internal x n_coarse, row-major;  Minv, G: packed per patch, n_coarse^2 each, row-major;
 *   reference column order.  G may be NULL; the blocks of LOD-branch patches (no Gram matrix) are set to 0.
 * The handle's basis, coarse matrices, diagnostics and status words are left unchanged.  Repeated or out-of-range patch
 * ids: SLOD_ERR_INVALID, before anything runs; a patch whose solve or dense stage sets status bits: SLOD_ERR_NUMERIC. */
int slod_debug_patch_stages_list(slod_ctx *ctx, int64_t n, const int64_t *patches, double *X, double *Minv, double *G);
/* the selection stage (source/LOD.cc:637-743) run exactly as slod_compute_basis runs it (same kernels, same plan:
 * SLOD_NO_FAST_SELECT, SLOD_FORCE_JACOBI and SLOD_EIG_CAP apply), on caller matrices, for selection tests.
 *   patches: n distinct patch ids (the patch fixes n_coarse and the LOD / SLOD branch);
 *   G, Minv: packed per patch, n_coarse^2 each, row-major, reference column order;
 *   c: packed per patch, [spacedim][n_coarse];  diag: [n][spacedim][8] in the layout of slod_get_patch_diagnostics.
 * The handle's basis, coarse matrices, diagnostics and status words are left unchanged.  Repeated or out-of-range patch
 * ids and non-finite entries: SLOD_ERR_INVALID, before anything runs. */
int slod_debug_select(slod_ctx *ctx, int64_t n, const int64_t *patches, const double *G, const double *Minv, double *c,
                      double *diag);

/* FP64 throughput of the handle's device in TFLOP/s, measured now with two register-resident probe kernels: a DFMA chain
 * and an mma.sync.m8n8k4.f64 chain (the instruction of the tensor-core kernels).  The benchmark's roofline denominator. */
int slod_measure_fp64_peak(slod_ctx *ctx, double *dfma_tflops, double *dmma_tflops);

/* per-kernel device times of the last compute/assemble (CUDA events), ms:
 *   [0] patch solve  [1] dense (M, BD, Gram)  [2] selection (eigen)  [3] finish (phi, A phi)
 *   [4] coarse matrix  [5] factorisation share of [0] (split solver, first chunk)
 *   [6] M_h phi and [7] coarse mass matrix of the last slod_assemble_coarse_mass */
int slod_get_timings(const slod_ctx *ctx, double *ms, int n);

/* the hot path, device buffers (multi-GPU plumbing) ----------------------------------------------------*/
/* Compute the basis of patches [patch_begin, patch_end) into device arrays laid out
 * [n_patches][spacedim][stride]; only the rows of the range are written.  `stream` is a cudaStream_t. */
int slod_compute_basis_device(slod_ctx *ctx, int64_t patch_begin, int64_t patch_end, double *d_phi, double *d_A_phi,
                              void *stream);
/* Coarse-matrix rows of patches [patch_begin, patch_end) in block-ELL form: d_K is
 * [n_patches*spacedim][ell_width] with ell_width = (4*oversampling+3)^dim * spacedim; slot of neighbour
 * offset D and component e is ((Dz+w)*(2w+1)+(Dy+w))*(2w+1)+(Dx+w))*spacedim+e, w = 2*oversampling+1.
 * Needs d_phi of the range and d_A_phi of ALL patches (all-gathered by the caller). */
int slod_assemble_coarse_device(slod_ctx *ctx, int64_t patch_begin, int64_t patch_end, const double *d_phi,
                                const double *d_A_phi, double *d_K, void *stream);
/* Synchronisation point of the two calls above: waits for what they enqueued, makes slod_get_timings valid and returns
 * SLOD_ERR_NUMERIC (first offending patch in slod_last_error) if a patch of the last basis range reported a status
 * (A_ii or M not positive definite, eigen-solver not converged) -- the same mapping slod_compute_basis does. */
int slod_synchronize(slod_ctx *ctx);
int slod_ell_width(const slod_ctx *ctx, int64_t *width);

/* ---- one handle per GPU, NCCL inside the library (multi-process multi-GPU) ---------------------------------------*/
/* [begin, end) of the patch ids owned by `rank` of `world`: create_evenly_distributed_partitioning
 * (source/LOD.cc:116-118) -- contiguous blocks, the first n % world ranks hold one more. */
int slod_owned_range(const slod_ctx *ctx, int rank, int world, int64_t *patch_begin, int64_t *patch_end);
/* 128 bytes of an ncclUniqueId, to be created by one rank and handed to the others by the caller (MPI_Bcast,
 * torch.distributed.broadcast, a file, ...). */
int slod_comm_unique_id(void *id128);
/* Join this handle (its device) into a communicator of `world` ranks. */
int slod_comm_init(slod_ctx *ctx, int rank, int world, const void *id128);
/* The offline phase of this rank on device arrays of the full layout ([n_patches][spacedim][stride] and
 * [n_patches * spacedim][ell_width], as in the *_device calls): basis of the owned range, all-gather of A*phi (and of
 * phi when gather_phi != 0), coarse-matrix rows of the owned range, all-gather of the row blocks when gather_K != 0.
 * Everything is enqueued on `stream`; slod_synchronize() is the synchronisation point. */
int slod_offline_distributed(slod_ctx *ctx, double *d_phi, double *d_A_phi, double *d_K, int gather_phi, int gather_K,
                             void *stream);
/* Host destinations for the rank's OWN rows ([rows of slod_owned_range][spacedim][stride] for phi / A*phi,
 * [rows * spacedim][ell_width] for K; page-locked memory recommended; any pointer may be NULL).  When set,
 * slod_offline_distributed copies the rows on the handle's own stream as soon as the producing kernels are through --
 * phi while the A*phi all-gather and the coarse-matrix kernel still run -- and slod_synchronize waits for the copies. */
int slod_set_host_outputs(slod_ctx *ctx, double *h_phi_rows, double *h_A_phi_rows, double *h_K_rows);
/* convert a host copy of the block-ELL matrix into CSR (same contract as slod_get_coarse_csr) */
int slod_ell_to_csr(const slod_ctx *ctx, const double *h_K, int64_t *rowptr, int64_t *col, double *val,
                    int64_t *n_rows, int64_t *nnz);
/* number of kernels launched by this handle so far */
int slod_launch_count(const slod_ctx *ctx, int64_t *n);

#ifdef __cplusplus
}
#endif
#endif /* SLOD_B200_H */
