// Batched online phase: C^T F, CG and C U for a block of right-hand sides at once.  Every byte of phi and K is the
// same for all columns, so each kernel reads them once per group of columns instead of once per column.
//
//   k_coarse_rhs_multi     B = C^T F        one warp per coarse row, phi row read once for the group
//   k_cg_*_multi           K X = B          per-column CG (own alpha, beta, ReductionControl test, freeze when done)
//   k_prolongate_multi     U_fine = C U     one thread per fine dof, all columns of the group
//
// Layout: a group of kb <= kBatch columns (kernels.h) is interleaved, [n][kb]: the kb values of one row are contiguous.
//
// Determinism: column j's arithmetic does not depend on kb, on j, or on the other columns.  Thread-to-work maps are
// fixed by kBatch (never by kb), grids are sized from the row counts only, every per-column reduction walks the same
// tree, and lanes / threads of absent columns (j >= kb) only skip their loads and stores.  No atomics.
// Included by kernels.cu after online.cuh.
#pragma once

namespace slod {

constexpr int kVecRows = 256;   // rows per block of the vector kernels (16 per thread row, 16 thread rows)

// dst[i][j] = src[j][i] (i < n, j < kb) and back: the public layout is one contiguous vector per right-hand side
__global__ void __launch_bounds__(256)
k_interleave(long long n, int kb, const double *__restrict__ src, double *__restrict__ dst) {
  const long long total = n * kb;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const long long i = e / kb;
    const int j = (int)(e - i * kb);
    dst[e] = src[(size_t)j * n + i];
  }
}
__global__ void __launch_bounds__(256)
k_deinterleave(long long n, int kb, const double *__restrict__ src, double *__restrict__ dst) {
  const long long total = n * kb;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const int j = (int)(e / n);
    const long long i = e - (long long)j * n;
    dst[e] = src[(size_t)i * kb + j];
  }
}

// one warp per coarse dof (patch, d): lane = column (lane & 15) + 16 * half; half h sums the box positions t = h, h + 2,
// ... of the same sweep as k_coarse_rhs, then the two halves are added.  phi values are read once per group.
__global__ void __launch_bounds__(kCgThreads)
k_coarse_rhs_multi(int n_patches, int kb, const double *__restrict__ phi, const double *__restrict__ F,
                   double *__restrict__ B, int nf_max) {
  const int s = cP.s, n = cP.n;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= n_patches * s) return;
  const int j = lane & (kBatch - 1), half = lane >> 4;
  const bool active = j < kb;
  const int pid = row / s;
  const Geom g = make_geom(cP, pid);
  const int G = cP.nsub + 1;
  const double *pp = phi + (size_t)row * nf_max;
  const int xs = g.p[0] * s;
  const int plane = xs * g.p[1];
  const double *f0 = F + ((((size_t)(g.lo[2] * n) * G + g.lo[1] * n) * G + g.lo[0] * n) * s) * kb + j;
  const size_t fz = (size_t)G * G * s * kb;
  double acc = 0.0;
  if (active) {
    for (int t = half; t < plane; t += 2) {
      const int y = t / xs, x = t - y * xs;
      const double *pl = pp + t;
      const double *fl = f0 + ((size_t)y * G * s + x) * kb;
#pragma unroll 4
      for (int z = 0; z < g.p[2]; ++z) acc += pl[(size_t)z * plane] * fl[z * fz];
    }
  }
  acc += __shfl_down_sync(0xffffffffu, acc, 16);
  if (half == 0 && active) B[(size_t)row * kb + j] = acc;
}

// one thread per fine dof, all columns: the patches and their components in the order of k_prolongate, each phi value
// loaded once and applied to the kb coefficients of its coarse row
__global__ void __launch_bounds__(kCgThreads)
k_prolongate_multi(long long n_fine, int kb, const double *__restrict__ phi, const double *__restrict__ U,
                   double *__restrict__ Uf, int nf_max) {
  const int s = cP.s, n = cP.n, ell = cP.ell, dim = cP.dim;
  const int G = cP.nsub + 1;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < n_fine;
       idx += (long long)gridDim.x * blockDim.x) {
    const int comp = (int)(idx % s);
    long long node = idx / s;
    int a[3];
    a[0] = (int)(node % G);
    node /= G;
    a[1] = (dim >= 2) ? (int)(node % G) : 0;
    a[2] = (dim == 3) ? (int)(node / G) : 0;
    int c0[3] = {0, 0, 0}, c1[3] = {0, 0, 0};
    for (int x = 0; x < dim; ++x) {
      c0[x] = max(0, (a[x] + n - 1) / n - 1 - ell);
      c1[x] = min(cP.N - 1, a[x] / n + ell);
    }
    double acc[kBatch];
#pragma unroll
    for (int j = 0; j < kBatch; ++j) acc[j] = 0.0;
    int c[3];
    for (c[2] = c0[2]; c[2] <= c1[2]; ++c[2])
      for (c[1] = c0[1]; c[1] <= c1[1]; ++c[1])
        for (c[0] = c0[0]; c[0] <= c1[0]; ++c[0]) {
          const Geom g = make_geom_at(cP, c);
          const int pid = (int)morton_fast(c, dim);
          const int loc[3] = {a[0] - g.lo[0] * n, a[1] - g.lo[1] * n, a[2] - g.lo[2] * n};
          const int li = node_index(g, loc) * s + comp;
          for (int d = 0; d < s; ++d) {
            const double ph = phi[((size_t)pid * s + d) * nf_max + li];
            const double *u = U + ((size_t)pid * s + d) * kb;
#pragma unroll
            for (int j = 0; j < kBatch; ++j)
              if (j < kb) acc[j] += u[j] * ph;
          }
        }
    double *out = Uf + (size_t)idx * kb;
#pragma unroll
    for (int j = 0; j < kBatch; ++j)
      if (j < kb) out[j] = acc[j];
  }
}

// ---- per-column conjugate gradients on the block-ELL coarse matrix ----
// Vectors X, R, P, Q are [nrows][kb]; dinv (the diagonal of K) is shared; one CgState per column.  Partial sums are
// [block][kBatch].  A column whose state is done is frozen: its x, r and p are no longer written.

// block j = column j: x = 0, r = b, z = D^-1 r, p = z, ||r_0||^2 and r.z in the order of one 1024-thread block
__global__ void __launch_bounds__(1024)
k_cg_init_multi(int nrows, int kb, const double *__restrict__ Kell, const double *__restrict__ B,
                double *__restrict__ X, double *__restrict__ R, double *__restrict__ P, double *__restrict__ dinv,
                CgState *st, double tol, double reduction) {
  __shared__ double sRed[32];
  const int j = blockIdx.x;
  const int s = cP.s, w = cP.w, ww = 2 * w + 1;
  const int centre = (cP.dim == 3) ? (w * ww + w) * ww + w : w * ww + w;
  double rz = 0.0, rr = 0.0;
  for (int i = threadIdx.x; i < nrows; i += blockDim.x) {
    const int d = i % s;
    const double di = 1.0 / Kell[(size_t)i * cP.ell_width + centre * s + d];
    const double ri = B[(size_t)i * kb + j];
    if (j == 0) dinv[i] = di;
    X[(size_t)i * kb + j] = 0.0;
    R[(size_t)i * kb + j] = ri;
    P[(size_t)i * kb + j] = di * ri;
    rz += ri * di * ri;
    rr += ri * ri;
  }
  rz = block_sum(rz, sRed);
  rr = block_sum(rr, sRed);
  if (threadIdx.x == 0) {
    CgState &c = st[j];
    c.rz[0] = rz;
    c.rz[1] = 0.0;
    c.rr0 = rr;
    c.rr = rr;
    c.tol2 = tol * tol;
    c.red2 = reduction * reduction;
    c.steps = 0;
    c.done = (rr <= tol * tol) ? 1 : 0;
  }
}

// true when every column of the group has stopped (then the kernels of the remaining launches return at once)
__device__ __forceinline__ bool all_done(const CgState *st, int kb) {
  bool all = true;
  for (int j = 0; j < kb; ++j) all = all && st[j].done;
  return all;
}

// Q = K P, one warp per row (grid-stride as k_cg_spmv).  The warp takes the row's entries 32 at a time (four such
// batches per pass, so that four K loads per lane are in flight): lane l computes the column of entry t0 + l once (-1: outside the domain or past the row); then lane (j, h) = (l % 16, l / 16) walks
// the entries e = h, h + 2, ... of the batch, receiving column and value by shuffle, and adds K_e * P[col][j].  Each
// half-warp load reads one 128-byte row of P, so K is read once per step for the whole group and a P row costs one
// L1 wavefront.  The two halves are added at the end of the row.  Per-block partial sums of p.q per column.
__global__ void __launch_bounds__(kCgThreads)
k_cg_spmm(int nrows, int kb, const double *__restrict__ Kell, const double *__restrict__ P, double *__restrict__ Q,
          double *__restrict__ partial, const CgState *st) {
  __shared__ double sRed[kCgThreads / 32][kBatch];
  __shared__ int sTab[kCgThreads / 32][3][kCgTab];
  if (all_done(st, kb)) return;
  const int s = cP.s, w = cP.w, ww = 2 * w + 1, dim = cP.dim;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int j = lane & (kBatch - 1), h = lane >> 4;
  const bool active = j < kb;
  const bool tabulated = ww <= kCgTab;
  double pq = 0.0;   // lane j < kb: column j
  for (int row = blockIdx.x * (kCgThreads / 32) + warp; row < nrows; row += gridDim.x * (kCgThreads / 32)) {
    const int pid = row / s;
    int c[3];
    morton_decode((uint32_t)pid, dim, cP.ref, c);
    const double *kr = Kell + (size_t)row * cP.ell_width;
    if (tabulated) ell_tabulate(sTab[warp], c, lane);
    double acc = 0.0;
    for (int t0 = 0; t0 < cP.ell_width; t0 += 128) {   // four batches of 32 entries: four K loads in flight per lane
      double kv[4];
      int col[4];
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int t = t0 + 32 * b + lane;
        kv[b] = (t < cP.ell_width) ? __ldcs(kr + t) : 0.0;   // K is streamed once per step: keep P in the caches
      }
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int t = t0 + 32 * b + lane;
        col[b] = (t < cP.ell_width) ? ell_column(t, sTab[warp], c, tabulated) : -1;
      }
#pragma unroll
      for (int b = 0; b < 4; ++b)
#pragma unroll
        for (int u = 0; u < 16; ++u) {
          const int ce = __shfl_sync(0xffffffffu, col[b], 2 * u + h);
          const double ke = __shfl_sync(0xffffffffu, kv[b], 2 * u + h);
          if (ce >= 0 && active) acc += ke * P[(size_t)ce * kb + j];
        }
    }
    acc += __shfl_down_sync(0xffffffffu, acc, 16);   // half 0 + half 1
    if (h == 0 && active) {
      Q[(size_t)row * kb + j] = acc;
      pq += acc * P[(size_t)row * kb + j];   // rows of a warp in ascending order: fixed summation order
    }
  }
  if (lane < kBatch) sRed[warp][lane] = pq;
  __syncthreads();
  if (threadIdx.x < kBatch) {
    double t = 0.0;
    for (int i = 0; i < kCgThreads / 32; ++i) t += sRed[i][threadIdx.x];
    partial[(size_t)blockIdx.x * kBatch + threadIdx.x] = t;
  }
}

// Thread (r, j) of a vector kernel (r = threadIdx.x / 16, j = threadIdx.x % 16) owns column j of the rows
// blockIdx.x * kVecRows + r + 16 m, m = 0 .. 15; block sums per column add the 16 thread rows in order.
__device__ __forceinline__ double column_block_sum(double v, double (*sCol)[kBatch]) {
  const int r = threadIdx.x / kBatch, j = threadIdx.x % kBatch;
  __syncthreads();
  sCol[r][j] = v;
  __syncthreads();
  double t = 0.0;
  for (int i = 0; i < kCgThreads / kBatch; ++i) t += sCol[i][j];
  return t;
}
// sum over n_partial blocks of column j of a [block][kBatch] partial array, in block order; every thread of column j
// gets it.  Warp w sums the columns j = w, w + 8 (lanes stride over the blocks, then the butterfly).
__device__ __forceinline__ void column_partial_sums(const double *__restrict__ partial, int n_partial, int kb,
                                                    double *sOut) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int j = warp; j < kBatch; j += kCgThreads / 32) {
    double v = 0.0;
    if (j < kb)
      for (int i = lane; i < n_partial; i += 32) v += partial[(size_t)i * kBatch + j];
    v = warp_sum(v);
    if (lane == 0) sOut[j] = v;
  }
  __syncthreads();
}

// alpha_j = r.z / p.Kp; x += alpha p; r -= alpha q; per-column partial sums of r.D^-1 r and r.r
__global__ void __launch_bounds__(kCgThreads)
k_cg_update_multi(int nrows, int kb, int it, const double *__restrict__ P, const double *__restrict__ Q,
                  const double *__restrict__ dinv, double *__restrict__ X, double *__restrict__ R,
                  const double *__restrict__ partial_pq, int n_partial, double *__restrict__ partial_rz,
                  double *__restrict__ partial_rr, const CgState *st) {
  __shared__ double sPq[kBatch];
  __shared__ double sCol[kCgThreads / kBatch][kBatch];
  if (all_done(st, kb)) return;
  column_partial_sums(partial_pq, n_partial, kb, sPq);
  const int r0 = threadIdx.x / kBatch, j = threadIdx.x % kBatch;
  const bool live = j < kb && !st[j].done;
  const double pq = sPq[j];
  const double alpha = live ? st[j].rz[it & 1] / pq : 0.0;
  double rz = 0.0, rr = 0.0;
  if (live && pq > 0.0) {
    for (int m = 0; m < kVecRows / (kCgThreads / kBatch); ++m) {
      const int i = blockIdx.x * kVecRows + r0 + m * (kCgThreads / kBatch);
      if (i >= nrows) break;
      const size_t e = (size_t)i * kb + j;
      X[e] += alpha * P[e];
      const double ri = R[e] - alpha * Q[e];
      R[e] = ri;
      rz += ri * dinv[i] * ri;
      rr += ri * ri;
    }
  }
  rz = column_block_sum(rz, sCol);
  rr = column_block_sum(rr, sCol);
  if (r0 == 0) {
    partial_rz[(size_t)blockIdx.x * kBatch + j] = (pq > 0.0) ? rz : -1.0;   // negative: breakdown, for the next kernel
    partial_rr[(size_t)blockIdx.x * kBatch + j] = rr;
  }
}

// beta_j = r'.z' / r.z; p = z' + beta p unless the column stops now; block 0 records each column's step and test
__global__ void __launch_bounds__(kCgThreads)
k_cg_direction_multi(int nrows, int kb, int it, const double *__restrict__ R, const double *__restrict__ dinv,
                     double *__restrict__ P, const double *__restrict__ partial_rz,
                     const double *__restrict__ partial_rr, int n_partial, CgState *st) {
  __shared__ double sRz[kBatch], sRr[kBatch];
  if (all_done(st, kb)) return;
  column_partial_sums(partial_rz, n_partial, kb, sRz);
  column_partial_sums(partial_rr, n_partial, kb, sRr);
  const int r0 = threadIdx.x / kBatch, j = threadIdx.x % kBatch;
  bool live = false, breakdown = false, stop = false;
  double rz_new = 0.0, rr = 0.0, rz_old = 1.0;
  if (j < kb) {
    live = !st[j].done;
    breakdown = partial_rz[j] < 0.0;   // block 0's entry carries the flag
    rz_new = sRz[j];
    rr = sRr[j];
    rz_old = st[j].rz[it & 1];
    stop = breakdown || rr <= st[j].tol2 || rr <= st[j].red2 * st[j].rr0;
  }
  __syncthreads();   // every thread of block 0 has read the states before they are advanced
  if (live && !stop) {
    const double beta = rz_new / rz_old;
    for (int m = 0; m < kVecRows / (kCgThreads / kBatch); ++m) {
      const int i = blockIdx.x * kVecRows + r0 + m * (kCgThreads / kBatch);
      if (i >= nrows) break;
      const size_t e = (size_t)i * kb + j;
      P[e] = dinv[i] * R[e] + beta * P[e];
    }
  }
  if (blockIdx.x == 0 && r0 == 0 && live) {
    CgState &c = st[j];
    if (breakdown) {
      c.done = 2;
    } else {
      c.rz[(it + 1) & 1] = rz_new;
      c.rr = rr;
      c.steps = it + 1;
      if (stop) c.done = 1;
    }
  }
}

}  // namespace slod
