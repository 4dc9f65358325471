// Launch interface between the host orchestration (capi.cu) and the kernels (kernels.cu).
#pragma once
#include <cuda_runtime.h>

#include "geom.h"

namespace slod {

constexpr int kSolveNB = 8;  // panel width of the blocked banded Cholesky

struct SolveLayout {
  int threads;
  int R;             // window rows = bw_max + NB
  int ldw;           // band row length = bw_max + 1
  int ldr;           // RHS window leading dimension (>= NcdMax)
  int bw_max;
  int coef_doubles;  // shared doubles reserved for the patch coefficients
  int ldx;           // leading dimension of X rows (NcdMax)
  long long x_stride;     // doubles per patch in Xbuf (NiMax * ldx)
  long long lws_per_cta;  // doubles of L workspace per CTA
  int gmem_window;        // patches too large for shared memory: the band / RHS / panel windows live in the CTA's
  long long gwin_off;     //   slice of the L workspace instead, at this offset (doubles)
};
struct DenseLayout {
  long long w_stride;  // doubles per patch in the flux buffer W
  int threads;
  int ncd_max, nb_max;
  int coef_doubles;
  int ldx;
  long long x_stride;
  long long m_stride;  // ncd_max^2
  int zmajor;          // coarse columns in the z-major order of the split solver (geom.h)
  double *coef_ws;     // SIMT kernel, very large patches: per-CTA coefficient window in global memory (else nullptr)
};
struct FluxLayout {
  int coef_doubles;
  int ldx;             // padded coarse columns (leading dimension of X and W rows)
  int nb_max;
  long long x_stride;
  long long w_stride;  // doubles per patch in Wbuf: round_up(nb_max, 32) * ldx
  int zmajor;          // coarse columns in the z-major order of the split solver (geom.h)
};
struct SelectLayout {
  int threads;
  int fast_path;  // try the Cholesky solve of G d = -g before the eigen-solver
  int ncd_max;
  long long m_stride;
};
struct FinishLayout {
  int ell_width;
  int coef_doubles;
  int nf_max, ncd_max;
  int ldx;
  long long x_stride;
};

cudaError_t upload_params(const Params &p, cudaStream_t st);   // stream-ordered upload of the __constant__ block

cudaError_t launch_patch_solve(int grid, size_t smem, cudaStream_t st, const int *ids, int n_work, const double *coef,
                               double *X, double *Lws, int *status, const SolveLayout &lay);
// tensor-core (mma.sync f64) solver; variant 0: <RBMAX 13, 16 warps> (3-D), 1: <4, 4 warps>, 2: <4, 8 warps> (2-D)
size_t solve_mma_smem(int variant, int coef_doubles, int nip_max, int stw);
cudaError_t launch_patch_solve_mma(int variant, int grid, size_t smem, cudaStream_t st, const int *ids, int n_work,
                                   const double *coef, double *X, double *Lws, int *status, int coef_doubles, int ldx,
                                   long long x_stride, long long lws_per_cta, int nip_max, int stw,
                                   int *work_counter = nullptr);
// split solver for the large 3-D patches (solve_split.cuh): factor records in HBM, then the triangular solves
size_t split_factor_smem(int coef_doubles, int nip_max);
size_t split_trisolve_smem(int nip_max);
long long split_rec_stride(int nip_max);
size_t split_stencil_ws_doubles(int grid, int nip_max);   // per-CTA stencil scratch of k_patch_factor
cudaError_t launch_patch_factor(int grid, size_t smem, cudaStream_t st, const int *ids, int n_work, const double *coef,
                                double *Lrec, double *stencil_ws, int *status, int coef_doubles, int nip_max, int ldx,
                                long long x_stride, int *work_counter);
cudaError_t launch_patch_trisolve(int grid, size_t smem, cudaStream_t st, const int *ids, int n_work, const double *Lrec,
                                  double *X, int coef_doubles, int nip_max, int ldx, long long x_stride, int *work_counter);
cudaError_t launch_patch_dense(int grid, size_t smem, cudaStream_t st, const int *ids, int n_work, const double *coef,
                               const double *X, double *Minv, double *G, double *diag, int *status,
                               const DenseLayout &lay);
// boundary flux W = S_b X - P_b for the tensor-core dense stage
size_t flux_smem(int coef_doubles, int ldx, int nb_max);
cudaError_t launch_patch_flux(int grid, size_t smem, cudaStream_t st, const int *ids, int n_work, const double *coef,
                              const double *X, double *W, const FluxLayout &lay, int *work_counter = nullptr);
// tensor-core dense stage, ntile in {4, 8, 16} (8*ntile >= coarse dofs per patch)
size_t dense_mma_smem(int ntile, int coef_doubles, int nb_max);
cudaError_t launch_patch_dense_mma(int ntile, int grid, size_t smem, cudaStream_t st, const int *ids, int n_work,
                                   const double *coef, const double *X, const double *W, double *Minv, double *G,
                                   double *diag, int *status, const DenseLayout &lay, int *work_counter = nullptr);
// selection pipeline (select.cuh): fast path -> tridiagonalisation + QL (rotation log) -> Jacobi fallback
struct EigLayout {
  int nmax, ldh;
  long long h_stride, v_stride;
  long long log_cap;   // rotations per item
  int ncd_max;
  long long m_stride;
  int cap_items;       // items per round
};
struct SelectPlan {
  SelectLayout lay;
  EigLayout eig;
  int s;        // spacedim: items per patch
  int use_ql;   // 0: everything that fails the fast path goes to the Jacobi kernel
  int grid_fast, grid_tri, grid_ql, grid_fin, grid_jac;
  size_t smem_fast, smem_tri, smem_ql, smem_fin, smem_jac;
};
struct SelectBuffers {
  int *counters;   // [4]: fast-path work counter | eigen items | Jacobi items
  int *eig_list, *jac_list;
  double *H, *V;
  double2 *rot_cs;
  unsigned short *rot_i;
  int *rot_n;
};
size_t select_fast_smem(int ncd_max);
size_t select_jacobi_smem(int ncd_max);
size_t eig_tridiag_smem(int nmax);
size_t eig_ql_smem(int nmax);
size_t eig_finish_smem(int nmax);
cudaError_t launch_select_pipeline(const SelectPlan &pl, cudaStream_t st, const int *ids, int n_work, const double *Minv,
                                   const double *G, double *cvec, double *diag, int *status, const SelectBuffers &b,
                                   int *n_launches);
cudaError_t launch_patch_finish(int grid, size_t smem, cudaStream_t st, const int *ids, int n_work, const double *coef,
                                const double *X, const double *cvec, double *phi, double *aphi,
                                const FinishLayout &lay);
// blocked coarse-matrix kernel: one CTA per Morton-aligned group of 2^dim patches, NU = nodes per axis of the common box.
// groups != nullptr: only the n_groups groups listed (group = patch id >> dim), every row of each; [p0, p1) must then be
// all patches.  The rows of an assembled matrix are rewritten in place.
size_t coarse_blocked_smem(int dim, int s, int NU);
cudaError_t launch_coarse_blocked(int dim, int s, int grid, size_t smem, cudaStream_t st, int p0, int p1,
                                  const double *phi, const double *aphi, double *Kell, const FinishLayout &lay, int NU,
                                  const int *groups = nullptr, int n_groups = 0);
cudaError_t launch_gather(cudaStream_t st, const double *src, const long long *perm, double *dst, long long n);
// incremental update (update.cuh): cell_changed[N^dim] = 1 where a value of the coarse cell's sub-cells differs bitwise
// between the two device coefficient arrays (n doubles each, nq values per sub-cell, n_sub sub-cells per cell and axis)
cudaError_t launch_coef_diff(cudaStream_t st, const double *base, const double *cur, long long n, int dim, int N,
                             int n_sub, int nq, unsigned char *cell_changed);
// online phase (online.cuh): b = C^T f, CG on the block-ELL coarse matrix, u_h = C u
cudaError_t launch_coarse_rhs(cudaStream_t st, int n_patches, int s, const double *phi, const double *f, double *b,
                              int nf_max);
cudaError_t launch_prolongate(cudaStream_t st, long long n_fine, const double *phi, const double *u, double *u_fine,
                              int nf_max);
// fine-grid operators of k_fine_apply (online.cuh)
enum FineOp {
  kFineStiffDirichlet = 0,  // coefficient-weighted stiffness, identity on the domain-boundary rows, boundary columns dropped
  kFineEnergy = 1,          // the same without the boundary treatment: x.y = energy norm^2
  kFineMass = 2,            // mass matrix: x.y = L2 norm^2
  kFineLaplace = 3,         // component-wise unweighted Laplace: x.y = H1 seminorm^2
  kFineHeatDirichlet = 4    // mass + tau * stiffness (theta-scheme step), with the boundary treatment of op 0
};
struct CgOperator {
  const double *Kell;     // block-ELL coarse matrix, or nullptr for a fine Dirichlet operator
  const double *d_coef;   // fine operator: sub-cell coefficients
  long long n_nodes;      // fine operator: nodes of the global grid
  int op = kFineStiffDirichlet;   // fine operator: kFineStiffDirichlet or kFineHeatDirichlet
  double tau = 0.0;               // fine operator kFineHeatDirichlet: the coefficient of the stiffness
};
size_t cg_workspace_doubles(const CgOperator &A, int nrows);
cudaError_t run_cg(cudaStream_t st, int nrows, const CgOperator &A, const double *b, double *x, double *work,
                   int max_steps, double tol, double reduction, int *steps, double *residual, int *flag,
                   long long *launches);
// batched online phase (online_batch.cuh): right-hand sides in groups of at most kBatch columns, interleaved [n][kb].
// 16: the values of one row form one 128-byte line, and the scratch of a group stays small (about 70 MB of fine
// vectors at the 32^3-cell workload) whatever the number of right-hand sides.
constexpr int kBatch = 16;
// [kb][n] <-> [n][kb]; to_interleaved selects the direction
cudaError_t launch_interleave(cudaStream_t st, long long n, int kb, const double *src, double *dst, bool to_interleaved);
cudaError_t launch_coarse_rhs_multi(cudaStream_t st, int n_patches, int s, int kb, const double *phi, const double *F,
                                    double *B, int nf_max);
cudaError_t launch_prolongate_multi(cudaStream_t st, long long n_fine, int kb, const double *phi, const double *U,
                                    double *Uf, int nf_max);
size_t cg_multi_workspace_doubles(int nrows);
// per-column CG on the block-ELL matrix for kb <= kBatch interleaved columns; steps / residual / flag: kb entries each
cudaError_t run_cg_multi(cudaStream_t st, int nrows, const double *Kell, int kb, const double *B, double *X,
                         double *work, int max_steps, double tol, double reduction, int *steps, double *residual,
                         int *flag, long long *launches);
// heat equation on the SLOD space (heat.cuh)
// M_h phi of every patch on its own node box, the [n_patches][s][nf_max] layout of A phi
cudaError_t launch_mass_apply(cudaStream_t st, int n_patches, int s, const double *phi, double *mphi, int nf_max);
// R = tau (sum_q W[q][j] B_q - K U) on the block-ELL matrix for kb <= kBatch interleaved columns (kb = 1: plain
// vectors) and nf >= 1 loads B_q = B + q b_stride in the layout of U; W: nf x kb device weights
cudaError_t launch_ell_residual(cudaStream_t st, int nrows, int kb, const double *Kell, const double *U, int nf,
                                const double *B, long long b_stride, const double *W, double tau, double *R);
// out = sum_q w[q] F[q n .. q n + n) for nf >= 1 (w: nf device doubles)
cudaError_t launch_weighted_sum(cudaStream_t st, long long n, int nf, const double *w, const double *F, double *out);
// z = a x + b y (z may alias x or y)
cudaError_t launch_lincomb(cudaStream_t st, long long n, double a, const double *x, double b, const double *y, double *z);
// y = Op x for a FineOp (tau: kFineHeatDirichlet), no reduction
cudaError_t launch_fine_apply(cudaStream_t st, int op, double tau, long long n_nodes, const double *d_coef,
                              const double *x, double *y);
cudaError_t launch_fine_quadratic_form(cudaStream_t st, int op, long long n_nodes, const double *d_coef, const double *x,
                                       double *partial, int *n_partial);
cudaError_t launch_fine_norms_reference(cudaStream_t st, long long n_cells, int nq, const double *gauss_x,
                                        const double *gauss_w, const double *v, double *partial, int *n_blocks);
cudaError_t run_fp64_probe(int n_sm, double *dfma_tflops, double *dmma_tflops);
// patches != nullptr: the patches patches[p0 .. p1) instead of the range [p0, p1)
cudaError_t launch_coarse(int grid, size_t smem, cudaStream_t st, int p0, int p1, const double *phi, const double *aphi,
                          double *Kell, const FinishLayout &lay, const int *patches = nullptr);

}  // namespace slod
