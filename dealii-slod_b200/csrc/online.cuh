// Coarse right-hand side, coarse solve and prolongation (SURVEY section 8f row 1): what LOD::solve() and the first
// lines of LOD::compare_lod_with_fem() do with the basis and the coarse matrix the offline phase produced
// (source/LOD.cc:975-1001, :1251).
//
//   k_coarse_rhs   b = C^T f           basis_matrix_transposed.Tvmult(system_rhs, fem_rhs)        source/LOD.cc:981
//   k_cg_*         K u = b             SolverCG + ReductionControl                                source/LOD.cc:991-998
//   k_prolongate   u_h = C u           basis_matrix_transposed.vmult(lod_solution, solution)      source/LOD.cc:1251
//
// C is never formed: column (patch, d) of C is the patch-local vector phi_{patch,d} placed on the patch's node box, so
// both products are box-indexed gathers.  K is used in the block-ELL form k_coarse_blocked wrote (slot = neighbour
// offset, the column index is the Morton code of the neighbour cell).  Fine vectors are lexicographic: node
// (x fastest) * spacedim + component.  Every reduction has a fixed order (no atomics): results are bit-reproducible.
// The preconditioner is the diagonal of K instead of the reference's SSOR(1.2) sweep -- a triangular sweep over a
// matrix with (4 ell + 3)^dim entries per row has no parallelism to speak of, and the stopping rule (residual
// reduction) is the same, so the solutions agree to the tolerance, not the iteration counts.
// Included by kernels.cu.
#pragma once

namespace slod {

constexpr int kCgThreads = 256;

// fixed-order block sum; every thread returns the total.  sRed: blockDim.x / 32 doubles.
__device__ __forceinline__ double block_sum(double v, double *sRed) {
  v = warp_sum(v);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  __syncthreads();
  if (lane == 0) sRed[warp] = v;
  __syncthreads();
  double t = 0.0;
  for (int i = 0; i < nw; ++i) t += sRed[i];
  return t;
}
// sum of a short global array in a fixed order, the same in every block
__device__ __forceinline__ double array_sum(const double *__restrict__ a, int n, double *sRed) {
  double v = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) v += a[i];
  return block_sum(v, sRed);
}

// one warp per coarse dof (patch, d): dot product of phi with f on the patch's node box
__global__ void __launch_bounds__(kCgThreads)
k_coarse_rhs(int n_patches, const double *__restrict__ phi, const double *__restrict__ f, double *__restrict__ b,
             int nf_max) {
  const int s = cP.s, n = cP.n;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= n_patches * s) return;
  const int pid = row / s;
  const Geom g = make_geom(cP, pid);
  const int G = cP.nsub + 1;
  const double *pp = phi + (size_t)row * nf_max;
  const int xs = g.p[0] * s;        // one x line of nodes with their components is contiguous in both arrays
  const int plane = xs * g.p[1];    // lanes sweep an (x, y) plane of the box, the z loop only adds strides
  const double *f0 = f + (((size_t)(g.lo[2] * n) * G + g.lo[1] * n) * G + g.lo[0] * n) * s;
  const size_t fz = (size_t)G * G * s;
  double acc = 0.0;
  for (int t = lane; t < plane; t += 32) {
    const int y = t / xs, x = t - y * xs;
    const double *pl = pp + t;
    const double *fl = f0 + (size_t)y * G * s + x;
#pragma unroll 4
    for (int z = 0; z < g.p[2]; ++z) acc += pl[(size_t)z * plane] * fl[z * fz];
  }
  acc = warp_sum(acc);
  if (lane == 0) b[row] = acc;
}

// one thread per fine dof: sum over the patches whose node box contains the node, in ascending centre order
__global__ void __launch_bounds__(kCgThreads)
k_prolongate(long long n_fine, const double *__restrict__ phi, const double *__restrict__ u,
             double *__restrict__ u_fine, int nf_max) {
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
      c0[x] = max(0, (a[x] + n - 1) / n - 1 - ell);   // first centre whose box reaches the node
      c1[x] = min(cP.N - 1, a[x] / n + ell);
    }
    double acc = 0.0;
    int c[3];
    for (c[2] = c0[2]; c[2] <= c1[2]; ++c[2])
      for (c[1] = c0[1]; c[1] <= c1[1]; ++c[1])
        for (c[0] = c0[0]; c[0] <= c1[0]; ++c[0]) {
          const Geom g = make_geom_at(cP, c);
          const int pid = (int)morton_fast(c, dim);
          const int loc[3] = {a[0] - g.lo[0] * n, a[1] - g.lo[1] * n, a[2] - g.lo[2] * n};
          const int li = node_index(g, loc) * s + comp;
          for (int d = 0; d < s; ++d) acc += u[(size_t)pid * s + d] * phi[((size_t)pid * s + d) * nf_max + li];
        }
    u_fine[idx] = acc;
  }
}

// ---- conjugate gradients on the block-ELL coarse matrix ----
// Device-side scalars: the host only reads them back every few iterations.
struct CgState {
  double rz[2];      // r.z of the current / next iteration (index = iteration parity)
  double rr0;        // ||r_0||^2
  double rr;         // ||r||^2 after the last completed step
  double tol2, red2; // squared absolute tolerance and squared reduction factor (ReductionControl)
  int steps;         // completed steps
  int done;          // 1: converged, 2: breakdown (p.Kp <= 0)
};

// x = 0, r = b, z = D^-1 r, p = z; one block (the vectors are short)
__global__ void __launch_bounds__(1024)
k_cg_init(int nrows, const double *__restrict__ Kell, const double *__restrict__ b, double *__restrict__ x,
          double *__restrict__ r, double *__restrict__ p, double *__restrict__ dinv, CgState *st, double tol,
          double reduction) {
  __shared__ double sRed[32];
  const int s = cP.s, w = cP.w, ww = 2 * w + 1;
  const int centre = (cP.dim == 3) ? (w * ww + w) * ww + w : w * ww + w;
  double rz = 0.0, rr = 0.0;
  for (int i = threadIdx.x; i < nrows; i += blockDim.x) {
    const int d = i % s;
    const double di = Kell ? 1.0 / Kell[(size_t)i * cP.ell_width + centre * s + d] : dinv[i];   // fine operator: preset
    const double ri = b[i];
    dinv[i] = di;
    x[i] = 0.0;
    r[i] = ri;
    p[i] = di * ri;
    rz += ri * di * ri;
    rr += ri * ri;
  }
  rz = block_sum(rz, sRed);
  rr = block_sum(rr, sRed);
  if (threadIdx.x == 0) {
    st->rz[0] = rz;
    st->rz[1] = 0.0;
    st->rr0 = rr;
    st->rr = rr;
    st->tol2 = tol * tol;
    st->red2 = reduction * reduction;
    st->steps = 0;
    st->done = (rr <= tol * tol) ? 1 : 0;
  }
}

// Column decoding of the block-ELL rows, shared by every kernel that multiplies with K (or with a matrix of the same
// slot convention).  The column of entry (dx, dy, dz) is dilate(cx + dx) | dilate(cy + dy) << 1 | dilate(cz + dz) << 2:
// each warp tabulates the 3 (2w+1) dilated coordinates of its row in shared memory (sign bit = outside the domain), so
// an entry costs three table reads and two ORs, and a sweep is bound by the 8 bytes per entry it reads.
constexpr int kCgTab = 32;   // 2w+1 <= 32 (oversampling <= 7); larger stencils take the direct path
__device__ __forceinline__ void ell_tabulate(int (*tab)[kCgTab], const int c[3], int lane) {
  const int w = cP.w, ww = 2 * w + 1, dim = cP.dim;
  __syncwarp();
  for (int i = lane; i < 3 * ww; i += 32) {
    const int a = i / ww, d = i - a * ww, v = c[a] + d - w;
    int code = 0;
    if (a < dim) code = (v >= 0 && v < cP.N) ? (int)(((dim == 3) ? dilate3(v) : dilate2(v)) << a) : (int)0x80000000;
    tab[a][d] = code;
  }
  __syncwarp();
}
// column (coarse dof) of entry t < ell_width of the row whose centre cell is c, -1 outside the domain; `tab` is the
// warp's table (tabulated: 2w+1 <= kCgTab), else the Morton code is computed directly
__device__ __forceinline__ int ell_column(int t, const int (*tab)[kCgTab], const int c[3], bool tabulated) {
  const int s = cP.s, w = cP.w, ww = 2 * w + 1, dim = cP.dim;
  const float inv_ww = 1.0f / (float)ww;   // exact quotients for these small integers
  const int slot = (s == 1) ? t : (t >> 1), e = (s == 1) ? 0 : (t & 1);   // spacedim is 1 or 2
  const int s1 = (int)(((float)slot + 0.5f) * inv_ww), s2 = (int)(((float)s1 + 0.5f) * inv_ww);
  if (tabulated) {
    const int cc = tab[0][slot - s1 * ww] | tab[1][s1 - s2 * ww] | tab[2][s2];
    return (cc >= 0) ? cc * s + e : -1;
  }
  int qc[3] = {c[0] + (slot - s1 * ww) - w, c[1] + (s1 - s2 * ww) - w, (dim == 3) ? c[2] + s2 - w : 0};
  bool valid = true;
#pragma unroll
  for (int x = 0; x < 3; ++x) if (x < dim) valid = valid && (qc[x] >= 0 && qc[x] < cP.N);
  return valid ? (int)morton_fast(qc, dim) * s + e : -1;
}

// q = K p, one warp per row (grid-stride over row groups); per-block partial sums of p.q.
__global__ void __launch_bounds__(kCgThreads)
k_cg_spmv(int nrows, const double *__restrict__ Kell, const double *__restrict__ p, double *__restrict__ q,
          double *__restrict__ partial, const CgState *st) {
  __shared__ double sRed[kCgThreads / 32];
  __shared__ int sTab[kCgThreads / 32][3][kCgTab];
  if (st->done) return;
  const int s = cP.s, w = cP.w, ww = 2 * w + 1, dim = cP.dim;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool tabulated = ww <= kCgTab;
  double pq = 0.0;
  for (int row = blockIdx.x * (kCgThreads / 32) + warp; row < nrows; row += gridDim.x * (kCgThreads / 32)) {
    const int pid = row / s;
    int c[3];
    morton_decode((uint32_t)pid, dim, cP.ref, c);
    const double *kr = Kell + (size_t)row * cP.ell_width;
    double acc = 0.0;
    if (tabulated) {
      ell_tabulate(sTab[warp], c, lane);
      for (int t0 = lane; t0 < cP.ell_width; t0 += 128) {   // four independent entries in flight per lane
        double kv[4];
        int col[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int t = t0 + 32 * u;
          kv[u] = (t < cP.ell_width) ? __ldcs(kr + t) : 0.0;   // K is streamed once per sweep: keep p in the caches
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int t = t0 + 32 * u;
          col[u] = (t < cP.ell_width) ? ell_column(t, sTab[warp], c, true) : -1;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u)
          if (col[u] >= 0) acc += kv[u] * p[col[u]];
      }
    } else {
      for (int t = lane; t < cP.ell_width; t += 32) {
        const int col = ell_column(t, nullptr, c, false);
        if (col >= 0) acc += kr[t] * p[col];
      }
    }
    acc = warp_sum(acc);
    if (lane == 0) q[row] = acc;
    pq += acc * p[row];   // rows of a warp in ascending order: fixed summation order
  }
  if (lane == 0) sRed[warp] = pq;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < kCgThreads / 32; ++i) t += sRed[i];
    partial[blockIdx.x] = t;
  }
}

// alpha = r.z / p.Kp; x += alpha p; r -= alpha q; partial sums of r.D^-1 r and r.r
__global__ void __launch_bounds__(kCgThreads)
k_cg_update(int nrows, int it, const double *__restrict__ p, const double *__restrict__ q,
            const double *__restrict__ dinv, double *__restrict__ x, double *__restrict__ r,
            const double *__restrict__ partial_pq, int n_partial, double *__restrict__ partial_rz,
            double *__restrict__ partial_rr, CgState *st) {
  __shared__ double sRed[kCgThreads / 32];
  if (st->done) return;
  const double pq = array_sum(partial_pq, n_partial, sRed);
  const double alpha = st->rz[it & 1] / pq;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  double rz = 0.0, rr = 0.0;
  if (i < nrows && pq > 0.0) {
    x[i] += alpha * p[i];
    const double ri = r[i] - alpha * q[i];
    r[i] = ri;
    rz = ri * dinv[i] * ri;
    rr = ri * ri;
  }
  rz = block_sum(rz, sRed);
  rr = block_sum(rr, sRed);
  if (threadIdx.x == 0) {
    partial_rz[blockIdx.x] = (pq > 0.0) ? rz : -1.0;   // a negative entry flags the breakdown to k_cg_direction
    partial_rr[blockIdx.x] = rr;
  }
}

// beta = r'.z' / r.z; p = z' + beta p; block 0 records the step and the stopping test
__global__ void __launch_bounds__(kCgThreads)
k_cg_direction(int nrows, int it, const double *__restrict__ r, const double *__restrict__ dinv,
               double *__restrict__ p, const double *__restrict__ partial_rz, const double *__restrict__ partial_rr,
               int n_partial, CgState *st) {
  __shared__ double sRed[kCgThreads / 32];
  if (st->done) return;
  const bool breakdown = partial_rz[0] < 0.0;
  const double rz_new = array_sum(partial_rz, n_partial, sRed);
  const double rr = array_sum(partial_rr, n_partial, sRed);
  const double rz_old = st->rz[it & 1];
  const double rr0 = st->rr0, tol2 = st->tol2, red2 = st->red2;
  __syncthreads();   // every thread of block 0 has read the state before it is advanced
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (!breakdown && i < nrows) p[i] = dinv[i] * r[i] + (rz_new / rz_old) * p[i];
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    if (breakdown) {
      st->done = 2;
    } else {
      st->rz[(it + 1) & 1] = rz_new;
      st->rr = rr;
      st->steps = it + 1;
      if (rr <= tol2 || rr <= red2 * rr0) st->done = 1;
    }
  }
}

// ---- fine-scale operators on the global grid (SURVEY section 8f row 2) ----
// Matrix-free Q_iso_Q1 operators on the (N n + 1)^dim node grid, one thread per node, y = Op x and per-block partial
// sums of x.y.  The node's row is accumulated sub-cell by sub-cell from the same reference matrices the patch kernels
// use (geom.h: Kref / Klam / Kq), so the fine FEM problem of assemble_and_solve_fem_problem (source/LOD.cc:1004-1094)
// is exactly the operator the patch problems restrict.

__device__ __forceinline__ double fine_tensor_entry(const double *__restrict__ d_coef, long long sc, long long fstride,
                                                 int idx) {
  double v = 0.0;
  for (int f = 0; f < tensor_fields(cP.dim); ++f) v += d_coef[f * fstride + sc] * cP.Kq[f][idx];
  return v;
}

__device__ __forceinline__ double fine_stiff_entry(const double *__restrict__ d_coef, long long sc, long long fstride,
                                                   int la, int lb, int ca, int cb) {
  const int dim = cP.dim, s = cP.s;
  const int nl = (1 << dim) * s;
  const int idx = (la * s + ca) * nl + (lb * s + cb);
  if (!cP.gauss_coef) {
    if (cP.problem == 0) return d_coef[sc] * cP.Kref[idx];
    if (cP.problem == kProblemTensor) return fine_tensor_entry(d_coef, sc, fstride, idx);   // never per Gauss point
    return d_coef[fstride + sc] * cP.Kref[idx] + d_coef[sc] * cP.Klam[idx];
  }
  const int nq = 1 << dim;
  double v = 0.0;
  for (int q = 0; q < nq; ++q) {
    if (cP.problem == 0) v += d_coef[sc * nq + q] * cP.Kq[q][idx];
    else v += d_coef[(fstride + sc) * nq + q] * cP.Kq[q][idx] + d_coef[sc * nq + q] * cP.Klamq[q][idx];
  }
  return v;
}

__device__ __forceinline__ double fine_local_entry(int op, double tau, const double *__restrict__ d_coef, long long sc,
                                                   long long fstride, int la, int lb, int ca, int cb) {
  const int dim = cP.dim;
  if (op == kFineHeatDirichlet) {   // mass + tau * stiffness
    double m = (ca == cb) ? 1.0 : 0.0;
    for (int x = 0; x < dim; ++x) m *= (((la >> x) & 1) == ((lb >> x) & 1)) ? cP.h / 3.0 : cP.h / 6.0;
    return m + tau * fine_stiff_entry(d_coef, sc, fstride, la, lb, ca, cb);
  }
  if (op == kFineMass || op == kFineLaplace) {
    if (ca != cb) return 0.0;
    double m[3] = {1.0, 1.0, 1.0};
    int same[3] = {1, 1, 1};
    for (int x = 0; x < dim; ++x) {
      same[x] = (((la >> x) & 1) == ((lb >> x) & 1));
      m[x] = same[x] ? cP.h / 3.0 : cP.h / 6.0;
    }
    if (op == kFineMass) return m[0] * m[1] * m[2];
    double v = 0.0;
    for (int k = 0; k < dim; ++k) {
      double t = (same[k] ? 1.0 : -1.0) / cP.h;
      for (int x = 0; x < dim; ++x) if (x != k) t *= m[x];
      v += t;
    }
    return v;
  }
  return fine_stiff_entry(d_coef, sc, fstride, la, lb, ca, cb);
}

// invdiag != nullptr: write 1 / diagonal of the operator instead of applying it (Jacobi preconditioner).
// tau: the time step of kFineHeatDirichlet, unused by the other operators.
__global__ void __launch_bounds__(kCgThreads)
k_fine_apply(int op, double tau, long long n_nodes, const double *__restrict__ d_coef, const double *__restrict__ x,
             double *__restrict__ y, double *__restrict__ invdiag, double *__restrict__ partial, const CgState *st) {
  __shared__ double sRed[kCgThreads / 32];
  if (st && st->done) return;
  const int dim = cP.dim, s = cP.s, G = cP.nsub + 1, nsub = cP.nsub;
  const bool dirichlet = op == kFineStiffDirichlet || op == kFineHeatDirichlet;
  const long long fstride = (dim == 3) ? (long long)nsub * nsub * nsub : (long long)nsub * nsub;
  const long long node = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  double dot = 0.0;
  if (node < n_nodes) {
    int a[3];
    long long r = node;
    a[0] = (int)(r % G);
    r /= G;
    a[1] = (dim >= 2) ? (int)(r % G) : 0;
    a[2] = (dim == 3) ? (int)(r / G) : 0;
    bool on_boundary = false;
    for (int k = 0; k < dim; ++k) on_boundary = on_boundary || a[k] == 0 || a[k] == G - 1;
    double acc[2] = {0.0, 0.0};
    if (dirichlet && on_boundary) {
      for (int c = 0; c < s; ++c) acc[c] = invdiag ? 1.0 : x[node * s + c];
    } else {
      for (int corner = 0; corner < (1 << dim); ++corner) {   // the sub-cell in which this node is local node `corner`
        int o[3] = {0, 0, 0};
        bool inside = true;
        for (int k = 0; k < dim; ++k) {
          o[k] = a[k] - ((corner >> k) & 1);
          inside = inside && o[k] >= 0 && o[k] < nsub;
        }
        if (!inside) continue;
        const long long sc = ((long long)o[2] * nsub + o[1]) * nsub + o[0];
        for (int lb = 0; lb < (1 << dim); ++lb) {
          int b[3] = {0, 0, 0};
          bool b_boundary = false;
          for (int k = 0; k < dim; ++k) {
            b[k] = o[k] + ((lb >> k) & 1);
            b_boundary = b_boundary || b[k] == 0 || b[k] == G - 1;
          }
          if (dirichlet && b_boundary) continue;
          if (invdiag && lb != corner) continue;
          const long long nb = ((long long)b[2] * G + b[1]) * G + b[0];
          for (int ca = 0; ca < s; ++ca)
            for (int cb = 0; cb < s; ++cb) {
              if (invdiag && cb != ca) continue;
              const double v = fine_local_entry(op, tau, d_coef, sc, fstride, corner, lb, ca, cb);
              acc[ca] += invdiag ? v : v * x[nb * s + cb];
            }
        }
      }
    }
    for (int c = 0; c < s; ++c) {
      if (invdiag) invdiag[node * s + c] = 1.0 / acc[c];
      else {
        if (y) y[node * s + c] = acc[c];
        dot += acc[c] * x[node * s + c];
      }
    }
  }
  dot = block_sum(dot, sRed);
  if (threadIdx.x == 0 && partial) partial[blockIdx.x] = dot;
}

// Norms the way the reference's error tables compute them (ParsedConvergenceTable::difference, source/LOD.cc:1252,
// include/LOD.h:111-115): VectorTools::integrate_difference on the cells of dof_handler_fine -- the COARSE cells, each
// carrying FE_Q_iso_Q1(n) -- with QGauss<dim>((degree + 1) * 2), degree = n, i.e. nq = 2 (n + 1) Gauss points per
// direction and coarse cell, on which the piecewise multilinear function is evaluated sub-cell by sub-cell.  The rule
// is not exact for Q_iso_Q1 functions (kinks inside the cell); slod_fine_norms has the exact values.
// One thread per coarse cell; per block: sum of |v|^2 w, sum of |grad v|^2 w, max |v_c| over the points.
__global__ void __launch_bounds__(kCgThreads)
k_fine_norms_reference(long long n_cells, int nq, const double *__restrict__ gauss_x, const double *__restrict__ gauss_w,
                       const double *__restrict__ v, double *__restrict__ partial) {
  __shared__ double sRed[kCgThreads / 32];
  const int dim = cP.dim, s = cP.s, n = cP.n, N = cP.N, G = cP.nsub + 1;
  const long long cell = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  double l2 = 0.0, h1 = 0.0, linf = 0.0;
  if (cell < n_cells) {
    long long r = cell;
    int c0[3] = {0, 0, 0};
    for (int a = 0; a < dim; ++a) {
      c0[a] = (int)(r % N);
      r /= N;
    }
    const int nqz = (dim == 3) ? nq : 1;
    for (int qz = 0; qz < nqz; ++qz)
      for (int qy = 0; qy < nq; ++qy)
        for (int qx = 0; qx < nq; ++qx) {
          const int q[3] = {qx, qy, qz};
          double w = 1.0, xi[3] = {0, 0, 0};
          int o[3] = {0, 0, 0};
          for (int a = 0; a < dim; ++a) {
            w *= gauss_w[q[a]] * cP.H;
            const double t = gauss_x[q[a]] * n;      // position in sub-cell units inside the coarse cell
            int sub = (int)t;
            if (sub > n - 1) sub = n - 1;
            xi[a] = t - sub;
            o[a] = c0[a] * n + sub;                  // global sub-cell index
          }
          for (int c = 0; c < s; ++c) {
            double val = 0.0, gr[3] = {0, 0, 0};
            for (int l = 0; l < (1 << dim); ++l) {
              const int b[3] = {o[0] + (l & 1), o[1] + ((l >> 1) & 1), o[2] + ((l >> 2) & 1)};
              const long long nb = ((long long)(dim == 3 ? b[2] : 0) * G + b[1]) * G + b[0];
              const double u = v[nb * s + c];
              double sh = 1.0;
              for (int a = 0; a < dim; ++a) sh *= ((l >> a) & 1) ? xi[a] : 1.0 - xi[a];
              val += u * sh;
              for (int a = 0; a < dim; ++a) {
                double g = (((l >> a) & 1) ? 1.0 : -1.0) / cP.h;
                for (int a2 = 0; a2 < dim; ++a2)
                  if (a2 != a) g *= ((l >> a2) & 1) ? xi[a2] : 1.0 - xi[a2];
                gr[a] += u * g;
              }
            }
            l2 += w * val * val;
            for (int a = 0; a < dim; ++a) h1 += w * gr[a] * gr[a];
            linf = fmax(linf, fabs(val));
          }
        }
  }
  l2 = block_sum(l2, sRed);
  __syncthreads();
  h1 = block_sum(h1, sRed);
  __syncthreads();
  // block maximum through the same scratch
  for (int o = 16; o > 0; o >>= 1) linf = fmax(linf, __shfl_xor_sync(0xffffffffu, linf, o));
  if ((threadIdx.x & 31) == 0) sRed[threadIdx.x >> 5] = linf;
  __syncthreads();
  if (threadIdx.x == 0) {
    double m = 0.0;
    for (int i = 0; i < kCgThreads / 32; ++i) m = fmax(m, sRed[i]);
    partial[3 * blockIdx.x + 0] = l2;
    partial[3 * blockIdx.x + 1] = h1;
    partial[3 * blockIdx.x + 2] = m;
  }
}

}  // namespace slod
