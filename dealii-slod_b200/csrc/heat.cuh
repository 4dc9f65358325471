// The coarse mass matrix and theta-scheme time stepping on the SLOD space.
//
//   k_mass_apply     M_h phi       the exact Q1 mass matrix of the sub-cell grid applied to every basis function on its
//                                  own node box; k_coarse_blocked / k_coarse then form M_H = C^T (M_h C) exactly as
//                                  they form K = C^T (A C)
//   k_ell_residual   tau (sum_q W_q B_q - K U)   the right-hand side of one theta-scheme step in increment form
//   k_weighted_sum   sum_q w_q F_q                the load of one step of the fine reference
//   k_lincomb        a x + b y                    S = M_H + c K on the block-ELL arrays, u += delta
//
// On the uniform grid M_h is the tensor product of the 1-D matrices h (1/6, 2/3, 1/6), block diagonal in the
// components.  phi vanishes on the boundary of its node box and outside it, so applying M_h box by box is exact on every
// node of the box, boundary nodes included: the neighbours whose value is missing there are outside the box (zero).
// Included by kernels.cu after online_batch.cuh.
#pragma once

namespace slod {

// one block per row (patch, d), grid-stride over the rows; one thread per entry of the row
__global__ void __launch_bounds__(256)
k_mass_apply(int n_patches, const double *__restrict__ phi, double *__restrict__ mphi, int nf_max) {
  const int s = cP.s, dim = cP.dim;
  const double w_off = cP.h / 6.0, w_diag = 2.0 * cP.h / 3.0;
  for (int row = blockIdx.x; row < n_patches * s; row += gridDim.x) {
    int cc[3], p[3] = {1, 1, 1};   // the node box of the patch (make_geom_at)
    morton_decode((uint32_t)(row / s), dim, cP.ref, cc);
#pragma unroll
    for (int x = 0; x < 3; ++x)
      if (x < dim) p[x] = (min(cc[x] + cP.ell, cP.N - 1) - max(cc[x] - cP.ell, 0) + 1) * cP.n + 1;
    const int nf = p[0] * p[1] * p[2] * s;
    const double *src = phi + (size_t)row * nf_max;
    double *dst = mphi + (size_t)row * nf_max;
    for (int i = threadIdx.x; i < nf_max; i += blockDim.x) {
      if (i >= nf) {
        dst[i] = 0.0;
        continue;
      }
      const int c = i % s, node = i / s;
      const int a[3] = {node % p[0], (node / p[0]) % p[1], node / (p[0] * p[1])};
      double acc = 0.0;
#pragma unroll
      for (int dz = -1; dz <= 1; ++dz) {
        if (dim != 3 && dz != 0) continue;
#pragma unroll
        for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
          for (int dx = -1; dx <= 1; ++dx) {
            const int bx = a[0] + dx, by = a[1] + dy, bz = a[2] + dz;
            if (bx < 0 || bx >= p[0] || by < 0 || by >= p[1] || bz < 0 || bz >= p[2]) continue;
            const double wgt = (dx ? w_off : w_diag) * (dy ? w_off : w_diag) * ((dim != 3) ? 1.0 : dz ? w_off : w_diag);
            acc += wgt * src[((bz * p[1] + by) * p[0] + bx) * s + c];
          }
      }
      dst[i] = acc;
    }
  }
}

// R = tau (sum_q W[q][j] B_q - K U) for kb <= kBatch interleaved columns ([n][kb]; kb = 1: plain vectors) and nf >= 1
// loads B_q = B + q * b_stride, with per-column weights W[nf][kb].  One warp per row (grid-stride as k_cg_spmv); lane l
// adds the entries t = l, l + 32, ... for every column, then one warp sum per column; lane j then sums the nf loads of
// column j.  A column's arithmetic depends neither on kb nor on the other columns.  The load sum starts from its first
// term, so nf = 1 with weight 1.0 gives tau (B - K U) exactly.  Each row reads nf loads per column: with per-step
// forcing (nf = n_steps + 1) a trajectory reads O(n_steps^2) coarse values.
__global__ void __launch_bounds__(kCgThreads)
k_ell_residual(int nrows, int kb, const double *__restrict__ Kell, const double *__restrict__ U, int nf,
               const double *__restrict__ B, long long b_stride, const double *__restrict__ W, double tau,
               double *__restrict__ R) {
  __shared__ int sTab[kCgThreads / 32][3][kCgTab];
  const int s = cP.s, w = cP.w, ww = 2 * w + 1, dim = cP.dim;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool tabulated = ww <= kCgTab;
  for (int row = blockIdx.x * (kCgThreads / 32) + warp; row < nrows; row += gridDim.x * (kCgThreads / 32)) {
    int c[3];
    morton_decode((uint32_t)(row / s), dim, cP.ref, c);
    const double *kr = Kell + (size_t)row * cP.ell_width;
    if (tabulated) ell_tabulate(sTab[warp], c, lane);
    double acc[kBatch];
#pragma unroll
    for (int j = 0; j < kBatch; ++j) acc[j] = 0.0;
    for (int t = lane; t < cP.ell_width; t += 32) {
      const double kv = __ldcs(kr + t);
      const int col = ell_column(t, sTab[warp], c, tabulated);
      if (col < 0) continue;
      const double *u = U + (size_t)col * kb;
#pragma unroll
      for (int j = 0; j < kBatch; ++j)
        if (j < kb) acc[j] += kv * u[j];
    }
    double v = 0.0;   // lane j: the K U entry of column j (warp_sum leaves the same bits in every lane)
#pragma unroll
    for (int j = 0; j < kBatch; ++j) {
      if (j >= kb) break;   // kb is uniform
      const double sj = warp_sum(acc[j]);
      if (lane == j) v = sj;
    }
    if (lane < kb) {   // lane j forms the load of column j, in field order: the columns' sums run side by side
      const size_t i = (size_t)row * kb + lane;
      double load = W[lane] * B[i];
      for (int q = 1; q < nf; ++q) load += W[(size_t)q * kb + lane] * B[q * b_stride + i];
      R[i] = tau * (load - v);
    }
  }
}

// out = sum_q w[q] F_q for nf >= 1 fields F_q = F + q n, summed from the first term in field order
__global__ void __launch_bounds__(256)
k_weighted_sum(long long n, int nf, const double *__restrict__ w, const double *__restrict__ F, double *__restrict__ out) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    double acc = w[0] * F[i];
    for (int q = 1; q < nf; ++q) acc += w[q] * F[q * n + i];
    out[i] = acc;
  }
}

__global__ void __launch_bounds__(256)
k_lincomb(long long n, double a, const double *x, double b, const double *y, double *z) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    z[i] = a * x[i] + b * y[i];
}

}  // namespace slod
