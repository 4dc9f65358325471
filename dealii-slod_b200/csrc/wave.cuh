// Newmark time stepping (gamma = 1/2, beta in [0, 1/2]) for the wave equation M u'' + K u = b(t), on the SLOD space
// (M = M_H, K the coarse matrix) and on the fine grid (M_h, A_h).  Each step solves for the acceleration:
//   predictor   ut = u_k + dt v_k + (1/2 - beta) dt^2 a_k
//   solve       (M + beta dt^2 K) a_{k+1} = b(t_{k+1}) - K ut          (k_ell_residual with tau = 1, then CG)
//   corrector   u_{k+1} = ut + beta dt^2 a_{k+1},  v_{k+1} = v_k + dt/2 (a_k + a_{k+1})
//
//   k_newmark_update   the corrector, a = a_new and the next predictor in one pass (or the first predictor alone)
//   k_wave_energy      per-block partials of v_j^T M_H v_j + u_j^T K u_j for kb <= kBatch interleaved columns
//   k_wave_energy_sum  E_j = 1/2 (the partials of column j added in block order)
// Included by kernels.cu after heat.cuh.
#pragma once

namespace slod {

// n = kb * nrows values of interleaved columns (or one vector): the update is element-wise, so the layout does not
// matter.  first: only ut = u + dt v + (1/2 - beta) dt^2 a from the state at t_0.
__global__ void __launch_bounds__(256)
k_newmark_update(long long n, int first, double beta, double dt, double *__restrict__ u, double *__restrict__ v,
                 double *__restrict__ a, const double *__restrict__ a_new, double *__restrict__ ut) {
  const double dt2 = dt * dt, c_pred = (0.5 - beta) * dt2, c_corr = beta * dt2, half_dt = 0.5 * dt;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    double ui = u[i], vi = v[i], ai = a[i];
    if (!first) {
      const double an = a_new[i];
      ui = ut[i] + c_corr * an;
      vi = vi + half_dt * (ai + an);
      ai = an;
      u[i] = ui;
      v[i] = vi;
      a[i] = ai;
    }
    ut[i] = ui + dt * vi + c_pred * ai;
  }
}

// One warp per row (grid-stride as k_ell_residual): lane l adds the entries t = l, l + 32, ... of the K row and of the
// M_H row for every column (both matrices have the slot convention of K, so a column is decoded once per entry), one
// warp sum per column and matrix; lane j then adds u_j K u_j + v_j M v_j of the row to its running sum.  Rows of a warp
// come in ascending order and the warps of a block are added in order: partial[block][kBatch], no atomics.  A column's
// arithmetic depends neither on kb nor on the other columns, and the grid depends on nrows only.
__global__ void __launch_bounds__(kCgThreads)
k_wave_energy(int nrows, int kb, const double *__restrict__ Kell, const double *__restrict__ Mell,
              const double *__restrict__ U, const double *__restrict__ V, double *__restrict__ partial) {
  __shared__ int sTab[kCgThreads / 32][3][kCgTab];
  __shared__ double sRed[kCgThreads / 32][kBatch];
  const int s = cP.s, w = cP.w, ww = 2 * w + 1, dim = cP.dim;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool tabulated = ww <= kCgTab;
  double part = 0.0;   // lane j < kb: column j
  for (int row = blockIdx.x * (kCgThreads / 32) + warp; row < nrows; row += gridDim.x * (kCgThreads / 32)) {
    int c[3];
    morton_decode((uint32_t)(row / s), dim, cP.ref, c);
    const double *kr = Kell + (size_t)row * cP.ell_width, *mr = Mell + (size_t)row * cP.ell_width;
    if (tabulated) ell_tabulate(sTab[warp], c, lane);
    double ak[kBatch], am[kBatch];
#pragma unroll
    for (int j = 0; j < kBatch; ++j) ak[j] = am[j] = 0.0;
    for (int t = lane; t < cP.ell_width; t += 32) {
      const double kv = __ldcs(kr + t), mval = __ldcs(mr + t);
      const int col = ell_column(t, sTab[warp], c, tabulated);
      if (col < 0) continue;
      const double *u = U + (size_t)col * kb, *v = V + (size_t)col * kb;
#pragma unroll
      for (int j = 0; j < kBatch; ++j)
        if (j < kb) {
          ak[j] += kv * u[j];
          am[j] += mval * v[j];
        }
    }
    double ku = 0.0, mv = 0.0;   // lane j: (K U)_row and (M V)_row of column j
#pragma unroll
    for (int j = 0; j < kBatch; ++j) {
      if (j >= kb) break;   // kb is uniform
      const double sk = warp_sum(ak[j]), sm = warp_sum(am[j]);
      if (lane == j) {
        ku = sk;
        mv = sm;
      }
    }
    if (lane < kb) {
      const size_t i = (size_t)row * kb + lane;
      part += U[i] * ku + V[i] * mv;
    }
  }
  if (lane < kBatch) sRed[warp][lane] = part;
  __syncthreads();
  if (threadIdx.x < kBatch) {
    double t = 0.0;
    for (int i = 0; i < kCgThreads / 32; ++i) t += sRed[i][threadIdx.x];
    partial[(size_t)blockIdx.x * kBatch + threadIdx.x] = t;
  }
}

// one block: E[j] = 1/2 sum over the n_partial blocks of column j, in block order (column_partial_sums)
__global__ void __launch_bounds__(kCgThreads)
k_wave_energy_sum(int kb, const double *__restrict__ partial, int n_partial, double *__restrict__ E) {
  __shared__ double sOut[kBatch];
  column_partial_sums(partial, n_partial, kb, sOut);
  if (threadIdx.x < kb) E[threadIdx.x] = 0.5 * sOut[threadIdx.x];
}

}  // namespace slod
