// Incremental basis update (slod_update_basis): which coarse cells carry a changed coefficient.
//
// A patch reads the device coefficient array only through load_coef, on the sub-cells of the coarse cells
// [clo, clo + m) of its window.  So a flag per coarse cell -- set when any field, sub-cell or Gauss-point value inside it
// differs -- decides exactly which patches see a different input.  Values are compared as 64-bit integers: a change from
// 0.0 to -0.0 counts, a NaN that keeps its bits does not.
// Included from kernels.cu inside namespace slod.

__global__ void __launch_bounds__(256)
k_coef_diff(const unsigned long long *__restrict__ base, const unsigned long long *__restrict__ cur, long long n,
            int dim, int N, int n_sub, int nq, unsigned char *__restrict__ cell_changed) {
  const long long nsub = (long long)N * n_sub;
  const long long per_field = ((dim == 3) ? nsub * nsub * nsub : nsub * nsub) * nq;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    if (base[i] == cur[i]) continue;
    long long r = (i % per_field) / nq;   // sub-cell, x fastest
    const int x = (int)(r % nsub);
    r /= nsub;
    const int y = (int)(r % nsub), z = (int)(r / nsub);
    // every writer stores the same byte: no atomics needed
    cell_changed[((size_t)(z / n_sub) * N + y / n_sub) * N + x / n_sub] = 1;
  }
}

cudaError_t launch_coef_diff(cudaStream_t st, const double *base, const double *cur, long long n, int dim, int N,
                             int n_sub, int nq, unsigned char *cell_changed) {
  size_t cells = (size_t)N * N * (dim == 3 ? N : 1);
  cudaError_t e = cudaMemsetAsync(cell_changed, 0, cells, st);
  if (e != cudaSuccess) return e;
  long long blocks = (n + 255) / 256;
  if (blocks > 148LL * 8) blocks = 148LL * 8;
  if (blocks < 1) blocks = 1;
  k_coef_diff<<<(int)blocks, 256, 0, st>>>(reinterpret_cast<const unsigned long long *>(base),
                                           reinterpret_cast<const unsigned long long *>(cur), n, dim, N, n_sub, nq,
                                           cell_changed);
  return cudaGetLastError();
}
