// sm_100a kernels of the SLOD offline phase.  One CTA owns one patch at a time; the reference's
// per-patch loop (source/LOD.cc:345-767) becomes five batched kernels:
//
//   k_patch_solve   assemble A_ii (band) + P_i on the fly, blocked banded Cholesky with the multi-RHS
//                   forward substitution fused in, then the backward substitution  -> X = A_ii^{-1} P_i
//                   (replaces assemble_stiffness + Gauss_elimination, source/LOD.cc:433-546)
//   k_patch_dense   M = P^T X / H^d, M^{-1} (in-place Gauss-Jordan like FullMatrix::gauss_jordan),
//                   BD = (S_b X - P_b) M^{-1} streamed in row tiles, G = BD^T BD   (source/LOD.cc:548-553, 609-618, 660)
//   k_patch_select  per component: thresholded pseudo-inverse of G[o,o] by a cyclic Jacobi eigen-solver,
//                   truncation loop, c = M^{-1}(e_d + sum d_k e_k)                  (source/LOD.cc:620-743)
//   k_patch_finish  phi = X c, zero extension, normalisation, A phi                  (source/LOD.cc:745-765)
//   k_coarse        K[(p,d),(q,e)] = phi_{p,d} . (A phi)_{q,e} over shared fine nodes (source/LOD.cc:860-973)
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include "geom.h"
#include "kernels.h"

namespace slod {

__constant__ Params cP;

cudaError_t upload_params(const Params &p, cudaStream_t st) {
  return cudaMemcpyToSymbolAsync(cP, &p, sizeof(Params), 0, cudaMemcpyHostToDevice, st);
}

// ------------------------------------------------------------------------------------------------
// helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int nfields() { return cP.problem == 0 ? 1 : 2; }

// copy the patch's sub-cell coefficients (window origin g.clo) into shared memory, field-major
// t0 / nt: index and number of the threads taking part (default: the whole CTA)
__device__ void load_coef(const Geom &g, const double *__restrict__ d_coef, double *sCoef, int t0 = -1, int nt = 0) {
  if (t0 < 0) { t0 = threadIdx.x; nt = blockDim.x; }
  const int n = cP.n;
  const int msx = g.m[0] * n, msy = g.m[1] * n, msz = (cP.dim == 3) ? g.m[2] * n : 1;
  const int nsubp = msx * msy * msz;
  const long long nsub = cP.nsub;
  const long long fstride = (cP.dim == 3) ? nsub * nsub * nsub : nsub * nsub;
  const int nf = nfields();
  const int nq = cP.gauss_coef ? (1 << cP.dim) : 1;   // values per sub-cell
  for (int idx = t0; idx < nf * nsubp * nq; idx += nt) {
    const int q = idx % nq;
    int r = idx / nq;
    const int f = r / nsubp;
    r -= f * nsubp;
    const int ox = r % msx;
    r /= msx;
    const int oy = r % msy;
    const int oz = r / msy;
    const long long gx = (long long)g.clo[0] * n + ox, gy = (long long)g.clo[1] * n + oy,
                    gz = (cP.dim == 3) ? (long long)g.clo[2] * n + oz : 0;
    sCoef[idx] = d_coef[(f * fstride + (gz * nsub + gy) * nsub + gx) * nq + q];
  }
}

// Morton code of a cell by bit dilation (same value as morton_encode of geom.h, a dozen instructions instead of a loop
// over dim * ref bits)
__device__ __forceinline__ unsigned dilate2(unsigned x) {
  x &= 0xffffu;
  x = (x | (x << 8)) & 0x00ff00ffu;
  x = (x | (x << 4)) & 0x0f0f0f0fu;
  x = (x | (x << 2)) & 0x33333333u;
  x = (x | (x << 1)) & 0x55555555u;
  return x;
}
__device__ __forceinline__ unsigned dilate3(unsigned x) {
  x &= 0x3ffu;
  x = (x | (x << 16)) & 0x030000ffu;
  x = (x | (x << 8)) & 0x0300f00fu;
  x = (x | (x << 4)) & 0x030c30c3u;
  x = (x | (x << 2)) & 0x09249249u;
  return x;
}
__device__ __forceinline__ unsigned morton_fast(const int c[3], int dim) {
  return (dim == 3) ? (dilate3(c[0]) | (dilate3(c[1]) << 1) | (dilate3(c[2]) << 2))
                    : (dilate2(c[0]) | (dilate2(c[1]) << 1));
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// Sums of N (4 or 8) per-lane values over the warp with N + log2(32 / N) + ... shuffles instead of 5 N: at every
// butterfly step a lane keeps one half of its values and hands the other half to its partner.  Afterwards lane L holds
// the total of index warp_sum_index<N>(L) (the four lanes of a quad hold the same one).  Fixed order: deterministic.
template <int N>
__device__ __forceinline__ int warp_sum_index(int lane) {
  return (N == 8) ? (((lane >> 4) & 1) << 2) | (((lane >> 3) & 1) << 1) | ((lane >> 2) & 1)
                  : (((lane >> 4) & 1) << 1) | ((lane >> 3) & 1);
}
__device__ __forceinline__ double warp_sum_packed(const double (&a)[8], int lane) {
  const bool h4 = (lane >> 4) & 1, h3 = (lane >> 3) & 1, h2 = (lane >> 2) & 1;
  double v[4];
#pragma unroll
  for (int j = 0; j < 4; ++j)
    v[j] = (h4 ? a[4 + j] : a[j]) + __shfl_xor_sync(0xffffffffu, h4 ? a[j] : a[4 + j], 16);
  double w[2];
#pragma unroll
  for (int j = 0; j < 2; ++j) w[j] = (h3 ? v[2 + j] : v[j]) + __shfl_xor_sync(0xffffffffu, h3 ? v[j] : v[2 + j], 8);
  double x = (h2 ? w[1] : w[0]) + __shfl_xor_sync(0xffffffffu, h2 ? w[0] : w[1], 4);
  x += __shfl_xor_sync(0xffffffffu, x, 2);
  x += __shfl_xor_sync(0xffffffffu, x, 1);
  return x;
}
__device__ __forceinline__ double warp_sum_packed(const double (&a)[4], int lane) {
  const bool h4 = (lane >> 4) & 1, h3 = (lane >> 3) & 1;
  double v[2];
#pragma unroll
  for (int j = 0; j < 2; ++j)
    v[j] = (h4 ? a[2 + j] : a[j]) + __shfl_xor_sync(0xffffffffu, h4 ? a[j] : a[2 + j], 16);
  double x = (h3 ? v[1] : v[0]) + __shfl_xor_sync(0xffffffffu, h3 ? v[0] : v[1], 8);
  x += __shfl_xor_sync(0xffffffffu, x, 4);
  x += __shfl_xor_sync(0xffffffffu, x, 2);
  x += __shfl_xor_sync(0xffffffffu, x, 1);
  return x;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// interior dof r -> node coords + component
__device__ __forceinline__ void idof_to_node(const Geom &g, int r, int a[3], int &comp) {
  comp = r % cP.s;
  interior_coords(g, r / cP.s, a);
}

// ------------------------------------------------------------------------------------------------
// k_patch_solve
// ------------------------------------------------------------------------------------------------
// Shared-memory plan (doubles): coef | W band window [R][ldw] | RHS window [R][ldr] | Lp [R][NB] |
// Ld [NB][NB] | Linv [NB][NB] | Yd [NB][ldr]
template <int NB>
__global__ void __launch_bounds__(512, 1)
k_patch_solve(const int *__restrict__ patch_ids, int n_work, const double *__restrict__ d_coef,
              double *__restrict__ Xbuf, double *__restrict__ Lws, int *__restrict__ status, SolveLayout lay) {
  extern __shared__ double smem[];
  double *myL = Lws + (size_t)blockIdx.x * lay.lws_per_cta;
  double *sCoef = smem;
  // Large patches (e.g. 3-D, 4 subdivisions, oversampling 2: half band width 381): the three windows do not fit shared
  // memory and live in the CTA's slice of the global workspace (L2 resident); block barriers order the accesses as
  // they do for shared memory.  Slower, but every configuration the reference's direct solver accepts runs.
  double *sW = lay.gmem_window ? myL + lay.gwin_off : sCoef + lay.coef_doubles;
  double *sR = sW + (size_t)lay.R * lay.ldw;
  double *sLp = sR + (size_t)lay.R * lay.ldr;
  double *sLd = lay.gmem_window ? sCoef + lay.coef_doubles : sLp + (size_t)lay.R * NB;
  double *sLinv = sLd + NB * NB;
  double *sYd = sLinv + NB * NB;
  const int tid = threadIdx.x, NT = blockDim.x, lane = tid & 31, warp = tid >> 5;
  const int R = lay.R, ldw = lay.ldw, ldr = lay.ldr;
  const int lstep = NB * NB + lay.bw_max * NB;  // doubles per panel in the L workspace

  for (int w = blockIdx.x; w < n_work; w += gridDim.x) {
    const int pid = patch_ids[w];
    const Geom g = make_geom(cP, pid);
    const int Ni = g.Ni, bw = g.bw, ncd = g.Ncd;
    double *X = Xbuf + (size_t)w * lay.x_stride;
    __syncthreads();
    load_coef(g, d_coef, sCoef);
    __syncthreads();

    // assemble rows [r0, r1) of the band of A_ii and of P_i into the windows
    auto assemble_rows = [&](int r0, int r1) {
      if (r1 > Ni) r1 = Ni;
      if (r0 >= r1) return;
      const int nr = r1 - r0;
      // zero the band rows
      for (int idx = tid; idx < nr * (bw + 1); idx += NT) {
        const int r = r0 + idx / (bw + 1);
        sW[(r % R) * ldw + idx % (bw + 1)] = 0.0;
      }
      // right-hand side P_i (dense row of length ncd)
      for (int idx = tid; idx < nr * ncd; idx += NT) {
        const int r = r0 + idx / ncd, col = idx % ncd;
        int a[3], ca;
        idof_to_node(g, r, a, ca);
        sR[(r % R) * ldr + col] = proj_entry(cP, g, a, ca, col);
      }
    };
    auto assemble_band = [&](int r0, int r1) {
      if (r1 > Ni) r1 = Ni;
      if (r0 >= r1) return;
      const int nr = r1 - r0;
      const int nst = (cP.dim == 3) ? 27 : 9;
      const int per_row = nst * cP.s;
      for (int idx = tid; idx < nr * per_row; idx += NT) {
        const int r = r0 + idx / per_row;
        int e = idx % per_row;
        const int cb = e % cP.s;
        e /= cP.s;
        int dl[3] = {e % 3 - 1, (e / 3) % 3 - 1, (cP.dim == 3) ? (e / 9 - 1) : 0};
        int a[3], ca;
        idof_to_node(g, r, a, ca);
        int b[3] = {a[0] + dl[0], a[1] + dl[1], a[2] + dl[2]};
        bool inside = true;
        _Pragma("unroll") for (int x = 0; x < 3; ++x) if (x < cP.dim) inside = inside && (b[x] >= 1 && b[x] <= g.p[x] - 2);
        if (!inside) continue;
        const int c = interior_index(g, b) * cP.s + cb;
        if (c > r) continue;
        sW[(r % R) * ldw + (c - r + bw)] = stiff_entry(cP, g, sCoef, a, dl, ca, cb);
      }
    };

    assemble_rows(0, NB + bw);
    __syncthreads();
    assemble_band(0, NB + bw);
    __syncthreads();

    int bad = 0;
    // ---------------- factorisation + forward substitution ----------------
    for (int c0 = 0, step = 0; c0 < Ni; c0 += NB, ++step) {
      const int nb = min(NB, Ni - c0);
      const int r1 = min(Ni, c0 + nb + bw);
      const int npr = r1 - (c0 + nb);
      if (warp == 0) {
        for (int idx = lane; idx < NB * NB; idx += 32) {
          const int i = idx / NB, j = idx % NB;
          double v = 0.0;
          if (i < nb && j <= i && i - j <= bw) v = sW[((c0 + i) % R) * ldw + (j - i + bw)];
          sLd[idx] = v;
          sLinv[idx] = 0.0;
        }
        __syncwarp();
        for (int k = 0; k < nb; ++k) {
          const double dkk = sLd[k * NB + k];
          if (!(dkk > 0.0)) bad = 1;
          const double dk = sqrt(dkk);
          __syncwarp();
          if (lane == 0) sLd[k * NB + k] = dk;
          if (lane > k && lane < nb) sLd[lane * NB + k] /= dk;
          __syncwarp();
          for (int idx = lane; idx < nb * nb; idx += 32) {
            const int i = idx / nb, j = idx % nb;
            if (j > k && j <= i) sLd[i * NB + j] -= sLd[i * NB + k] * sLd[j * NB + k];
          }
          __syncwarp();
        }
        if (lane < nb) {  // column `lane` of L_D^{-1}
          const int j = lane;
          double x[NB];
#pragma unroll
          for (int i = 0; i < NB; ++i) {
            if (i >= j && i < nb) {
              double sum = (i == j) ? 1.0 : 0.0;
#pragma unroll
              for (int t = 0; t < NB; ++t)
                if (t >= j && t < i) sum -= sLd[i * NB + t] * x[t];
              x[i] = sum / sLd[i * NB + i];
              sLinv[i * NB + j] = x[i];
            } else {
              x[i] = 0.0;
            }
          }
        }
      }
      __syncthreads();
      // panel  Lp = W[panel rows, c0:c0+nb] * L_D^{-T}
      for (int idx = tid; idx < npr * NB; idx += NT) {
        const int r = idx / NB, k = idx % NB;
        const int i = c0 + nb + r;
        double acc = 0.0;
        if (k < nb) {
          for (int t = 0; t <= k; ++t) {
            const int c = c0 + t;
            if (i - c <= bw) acc += sW[(i % R) * ldw + (c - i + bw)] * sLinv[k * NB + t];
          }
        }
        sLp[idx] = acc;
      }
      // Y_D = L_D^{-1} R_D
      for (int idx = tid; idx < NB * ncd; idx += NT) {
        const int k = idx / ncd, col = idx % ncd;
        double acc = 0.0;
        if (k < nb)
          for (int t = 0; t <= k; ++t) acc += sLinv[k * NB + t] * sR[((c0 + t) % R) * ldr + col];
        sYd[k * ldr + col] = acc;
      }
      __syncthreads();
      // trailing update of the band window
      for (int idx = tid; idx < npr * npr; idx += NT) {
        const int ri = idx / npr, rj = idx % npr;
        if (rj > ri) continue;
        double acc = 0.0;
#pragma unroll
        for (int k = 0; k < NB; ++k) acc += sLp[ri * NB + k] * sLp[rj * NB + k];
        const int i = c0 + nb + ri, j = c0 + nb + rj;
        sW[(i % R) * ldw + (j - i + bw)] -= acc;
      }
      // right-hand side update
      for (int idx = tid; idx < npr * ncd; idx += NT) {
        const int r = idx / ncd, col = idx % ncd;
        double acc = 0.0;
#pragma unroll
        for (int k = 0; k < NB; ++k) acc += sLp[r * NB + k] * sYd[k * ldr + col];
        sR[((c0 + nb + r) % R) * ldr + col] -= acc;
      }
      // spill the panel for the backward substitution, Y_D to X
      {
        double *Ls = myL + (size_t)step * lstep;
        for (int idx = tid; idx < NB * NB; idx += NT) Ls[idx] = sLinv[idx];
        for (int idx = tid; idx < npr * NB; idx += NT) Ls[NB * NB + idx] = sLp[idx];
        for (int idx = tid; idx < nb * ncd; idx += NT) {
          const int k = idx / ncd, col = idx % ncd;
          X[(size_t)(c0 + k) * lay.ldx + col] = sYd[k * ldr + col];
        }
      }
      // slide the window: rows [c0+nb+bw, c0+2nb+bw) take the slots of rows [c0, c0+nb)
      assemble_rows(c0 + nb + bw, c0 + 2 * nb + bw);
      __syncthreads();
      assemble_band(c0 + nb + bw, c0 + 2 * nb + bw);
      __syncthreads();
    }
    if (bad && tid == 0) atomicOr(&status[pid], 1);

    // ---------------- backward substitution:  L^T X = Y ----------------
    const int last = ((Ni - 1) / NB) * NB;
    for (int c0 = last, step = last / NB; c0 >= 0; c0 -= NB, --step) {
      const int nb = min(NB, Ni - c0);
      const int r1 = min(Ni, c0 + nb + bw);
      const int npr = r1 - (c0 + nb);
      const double *Ls = myL + (size_t)step * lstep;
      for (int idx = tid; idx < NB * NB; idx += NT) sLinv[idx] = Ls[idx];
      for (int idx = tid; idx < npr * NB; idx += NT) sLp[idx] = Ls[NB * NB + idx];
      for (int idx = tid; idx < NB * ncd; idx += NT) {
        const int k = idx / ncd, col = idx % ncd;
        sYd[k * ldr + col] = (k < nb) ? X[(size_t)(c0 + k) * lay.ldx + col] : 0.0;
      }
      __syncthreads();
      for (int idx = tid; idx < nb * ncd; idx += NT) {
        const int k = idx / ncd, col = idx % ncd;
        double acc = sYd[k * ldr + col];
        for (int r = 0; r < npr; ++r) acc -= sLp[r * NB + k] * sR[((c0 + nb + r) % R) * ldr + col];
        sYd[k * ldr + col] = acc;
      }
      __syncthreads();
      for (int idx = tid; idx < nb * ncd; idx += NT) {
        const int k = idx / ncd, col = idx % ncd;
        double acc = 0.0;
        for (int t = k; t < nb; ++t) acc += sLinv[t * NB + k] * sYd[t * ldr + col];
        sR[((c0 + k) % R) * ldr + col] = acc;
        X[(size_t)(c0 + k) * lay.ldx + col] = acc;
      }
      __syncthreads();
    }
  }
}

}  // namespace slod
// Persistent kernels fetch their next work item from a global counter (zeroed before the launch) instead of striding by
// the grid size: items are sorted by cost, largest first, and a CTA that starts late -- because another stream's CTAs
// hold its SM -- takes less work instead of finishing late.  The fetch is issued at the top of an item by the last
// thread (its result is only needed at the end of the item); work_counter == nullptr keeps the static stride.
#define SLOD_WORK_LOOP(w, n_work, work_counter, sNext)                                                        \
  for (int w = blockIdx.x; w < (n_work); w = next_work_item(&(sNext)))
__device__ __forceinline__ int next_work_item(int *sNext) {
  __syncthreads();
  const int v = *sNext;
  __syncthreads();   // everybody has read it before the next item's fetch overwrites it
  return v;
}
__device__ __forceinline__ void fetch_work_item(int w, int *work_counter, int *sNext) {
  if (threadIdx.x == blockDim.x - 1)
    *sNext = work_counter ? (int)gridDim.x + atomicAdd(work_counter, 1) : w + (int)gridDim.x;
}

#include "solve_mma.cuh"
#include "solve_split.cuh"
namespace slod {

// ------------------------------------------------------------------------------------------------
// k_patch_dense
// ------------------------------------------------------------------------------------------------
constexpr int kTB = 16;      // boundary rows per tile
constexpr int kGEPT = 32;    // Gram entries per thread (Ncd^2 <= kGEPT * blockDim)

__global__ void __launch_bounds__(512, 1)
k_patch_dense(const int *__restrict__ patch_ids, int n_work, const double *__restrict__ d_coef,
              const double *__restrict__ Xbuf, double *__restrict__ Minv_out, double *__restrict__ G_out,
              double *__restrict__ diag, int *__restrict__ status, DenseLayout lay) {
  extern __shared__ double smem[];
  double *sCoef = lay.coef_ws ? lay.coef_ws + (size_t)blockIdx.x * lay.coef_doubles : smem;
  double *sM = lay.coef_ws ? smem : sCoef + lay.coef_doubles;   // [ncd][ncd]
  double *sT1 = sM + (size_t)lay.ncd_max * lay.ncd_max;  // [kTB][ncd]  W tile
  double *sT2 = sT1 + kTB * lay.ncd_max;                 // [kTB][ncd]  BD tile
  double *sCol = sT2 + kTB * lay.ncd_max;                // [ncd] pivot column
  double *sRow = sCol + lay.ncd_max;                     // [ncd] pivot row
  double *sArow = sRow + lay.ncd_max;                    // [kTB][27*s] stencil row entries
  int *sAnbr = (int *)(sArow + kTB * 27 * 2);            // [kTB][27*s] interior dof of the neighbour or -1
  int *sBlist = sAnbr + kTB * 27 * 2;                    // [NbMax] boundary dofs
  __shared__ int sNb;
  const int tid = threadIdx.x, NT = blockDim.x;

  for (int w = blockIdx.x; w < n_work; w += gridDim.x) {
    const int pid = patch_ids[w];
    const Geom g = make_geom(cP, pid);
    const int ncd = g.Ncd, s = cP.s;
    const double *X = Xbuf + (size_t)w * lay.x_stride;
    __syncthreads();
    load_coef(g, d_coef, sCoef);
    if (tid == 0) sNb = 0;
    __syncthreads();

    // ---- M = P_i^T X / H^d  (source/LOD.cc:548-551); P is the cell-wise weight stencil ----
    const int npc = cP.n + 1;
    const int nloc = (cP.dim == 3) ? npc * npc * npc : npc * npc;
    const double scale = cP.pw / cP.Hd;
    for (int idx = tid; idx < ncd * ncd; idx += NT) {
      const int row = idx / ncd, col = idx % ncd;
      const int comp = row % s;
      int k[3];
      col_to_cell(cP, g, row / s, k);
      double acc = 0.0;
      for (int l = 0; l < nloc; ++l) {
        int t[3] = {l % npc, (l / npc) % npc, (cP.dim == 3) ? l / (npc * npc) : 0};
        int a[3] = {k[0] * cP.n + t[0], k[1] * cP.n + t[1], (cP.dim == 3) ? k[2] * cP.n + t[2] : 0};
        if (node_class(cP, g, a) != 0) continue;
        double wgt = 1.0;
        _Pragma("unroll") for (int x = 0; x < 3; ++x) if (x < cP.dim)
          if (t[x] != 0 && t[x] != cP.n) wgt *= 2.0;
        acc += wgt * X[(size_t)(interior_index(g, a) * s + comp) * lay.ldx + col];
      }
      sM[row * ncd + col] = acc * scale;
    }
    // boundary dof list (order irrelevant for BD^T BD)
    if (g.slod && tid < 32) {  // ascending order (deterministic summation order of BD^T BD)
      int count = 0;
      for (int base = 0; base < g.nnodes; base += 32) {
        const int node = base + tid;
        bool isb = false;
        if (node < g.nnodes) {
          int a[3];
          node_coords(g, node, a);
          isb = (node_class(cP, g, a) & 1) != 0;
        }
        const unsigned mask = __ballot_sync(0xffffffffu, isb);
        if (isb) {
          const int pos = (count + __popc(mask & ((1u << tid) - 1u))) * s;
          for (int c = 0; c < s; ++c) sBlist[pos + c] = node * s + c;
        }
        count += __popc(mask);
      }
      if (tid == 0) sNb = count * s;
    }
    __syncthreads();

    // ---- M^{-1} by in-place Gauss-Jordan sweeps (FullMatrix::gauss_jordan, source/LOD.cc:553) ----
    for (int k = 0; k < ncd; ++k) {
      const double piv = sM[k * ncd + k];
      for (int j = tid; j < ncd; j += NT) {
        sCol[j] = sM[j * ncd + k];
        sRow[j] = sM[k * ncd + j] / piv;
      }
      if (tid == 0) {
        if (!(piv > 0.0)) atomicOr(&status[pid], 2);
      }
      __syncthreads();
      for (int idx = tid; idx < ncd * ncd; idx += NT) {
        const int i = idx / ncd, j = idx % ncd;
        double v;
        if (i == k && j == k) v = 1.0 / piv;
        else if (i == k) v = sRow[j];
        else if (j == k) v = -sCol[i] / piv;
        else v = sM[idx] - sCol[i] * sRow[j];
        sM[idx] = v;
      }
      __syncthreads();
    }
    {
      double *Mo = Minv_out + (size_t)w * lay.m_stride;
      for (int idx = tid; idx < ncd * ncd; idx += NT) Mo[idx] = sM[idx];
    }
    if (!g.slod) continue;

    // ---- BD = (S_b X_i - P_b) M^{-1} in tiles of kTB boundary rows; G += BD^T BD ----
    double gacc[kGEPT];
#pragma unroll
    for (int e = 0; e < kGEPT; ++e) gacc[e] = 0.0;
    const int nbd = sNb;
    const int nst = (cP.dim == 3) ? 27 : 9;
    const int per_row = nst * s;
    for (int t0 = 0; t0 < nbd; t0 += kTB) {
      const int nt = min(kTB, nbd - t0);
      // stencil entries of the boundary rows towards interior dofs
      for (int idx = tid; idx < nt * per_row; idx += NT) {
        const int rb = idx / per_row;
        int e = idx % per_row;
        const int cb = e % s;
        e /= s;
        int dl[3] = {e % 3 - 1, (e / 3) % 3 - 1, (cP.dim == 3) ? (e / 9 - 1) : 0};
        const int dof = sBlist[t0 + rb];
        int a[3];
        node_coords(g, dof / s, a);
        int b[3] = {a[0] + dl[0], a[1] + dl[1], a[2] + dl[2]};
        bool ok = true;
        _Pragma("unroll") for (int x = 0; x < 3; ++x) if (x < cP.dim) ok = ok && (b[x] >= 1 && b[x] <= g.p[x] - 2);
        if (ok) {
          sAnbr[idx] = interior_index(g, b) * s + cb;
          sArow[idx] = stiff_entry(cP, g, sCoef, a, dl, dof % s, cb);
        } else {
          sAnbr[idx] = -1;
          sArow[idx] = 0.0;
        }
      }
      __syncthreads();
      for (int idx = tid; idx < nt * ncd; idx += NT) {
        const int rb = idx / ncd, col = idx % ncd;
        const int dof = sBlist[t0 + rb];
        int a[3];
        node_coords(g, dof / s, a);
        double acc = -proj_entry(cP, g, a, dof % s, col);
        for (int e = 0; e < per_row; ++e) {
          const int nb_ = sAnbr[rb * per_row + e];
          if (nb_ >= 0) acc += sArow[rb * per_row + e] * X[(size_t)nb_ * lay.ldx + col];
        }
        sT1[rb * ncd + col] = acc;
      }
      __syncthreads();
      for (int idx = tid; idx < nt * ncd; idx += NT) {
        const int rb = idx / ncd, col = idx % ncd;
        double acc = 0.0;
        for (int k = 0; k < ncd; ++k) acc += sT1[rb * ncd + k] * sM[k * ncd + col];
        sT2[idx] = acc;
      }
      __syncthreads();
#pragma unroll
      for (int e = 0; e < kGEPT; ++e) {
        const int idx = tid + e * NT;
        if (idx < ncd * ncd) {
          const int i = idx / ncd, j = idx % ncd;
          double acc = gacc[e];
          for (int rb = 0; rb < nt; ++rb) acc += sT2[rb * ncd + i] * sT2[rb * ncd + j];
          gacc[e] = acc;
        }
      }
      __syncthreads();
    }
    {
      double *Go = G_out + (size_t)w * lay.m_stride;
#pragma unroll
      for (int e = 0; e < kGEPT; ++e) {
        const int idx = tid + e * NT;
        if (idx < ncd * ncd) Go[idx] = gacc[e];
      }
    }
  }
}

}  // namespace slod
#include "flux.cuh"
#include "dense_mma.cuh"
namespace slod {

}  // namespace slod
#include "select.cuh"
namespace slod {

// ------------------------------------------------------------------------------------------------
// k_patch_finish : phi = X c (zero on every boundary dof), normalise, A phi
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256, 3)
k_patch_finish(const int *__restrict__ patch_ids, int n_work, const double *__restrict__ d_coef,
               const double *__restrict__ Xbuf, const double *__restrict__ cvec, double *__restrict__ phi_out,
               double *__restrict__ aphi_out, FinishLayout lay) {
  extern __shared__ double smem[];
  double *sCoef = smem;
  double *sPhi = sCoef + lay.coef_doubles;  // [Nf]
  double *sC = sPhi + lay.nf_max;           // [ncd]
  int *sRowDof = (int *)(sC + lay.ncd_max);  // [Ni] patch dof of every interior row
  __shared__ double sRed[32];
  __shared__ double sNorm;
  const int tid = threadIdx.x, NT = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarp = NT >> 5;

  for (int w = blockIdx.x; w < n_work; w += gridDim.x) {
    const int pid = patch_ids[w];
    const Geom g = make_geom(cP, pid);
    const int ncd = g.Ncd, s = cP.s;
    const double *X = Xbuf + (size_t)w * lay.x_stride;
    __syncthreads();
    load_coef(g, d_coef, sCoef);
    for (int r = tid; r < g.Ni; r += NT) {
      int a[3], ca;
      idof_to_node(g, r, a, ca);
      sRowDof[r] = node_index(g, a) * s + ca;
    }
    for (int d = 0; d < s; ++d) {
      __syncthreads();
      for (int i = tid; i < ncd; i += NT) sC[i] = cvec[((size_t)w * s + d) * lay.ncd_max + i];
      for (int i = tid; i < g.Nf; i += NT) sPhi[i] = 0.0;
      __syncthreads();
      double nrm = 0.0;
      if ((lay.ldx & 3) == 0) {
        // eight rows of X per warp iteration, a lane reads 4 consecutive columns of each with two 16-byte loads
        // (16 independent loads in flight per lane) and keeps its 4 entries of c in registers
        double cc[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) cc[q] = (4 * lane + q < ncd) ? sC[4 * lane + q] : 0.0;
        const bool in_row = 4 * lane + 3 < lay.ldx;
        for (int r0 = 8 * warp; r0 < g.Ni; r0 += 8 * nwarp) {
          double acc[8];
          double2 xa[8], xb[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const int r = min(r0 + u, g.Ni - 1);
            const double2 *xp = reinterpret_cast<const double2 *>(X + (size_t)r * lay.ldx + 4 * lane);
            xa[u] = in_row ? xp[0] : make_double2(0.0, 0.0);
            xb[u] = in_row ? xp[1] : make_double2(0.0, 0.0);
          }
#pragma unroll
          for (int u = 0; u < 8; ++u)
            acc[u] = (xa[u].x * cc[0] + xa[u].y * cc[1]) + (xb[u].x * cc[2] + xb[u].y * cc[3]);
          const double tot = warp_sum_packed(acc, lane);   // lane L holds row r0 + warp_sum_index<8>(L)
          const int r = r0 + warp_sum_index<8>(lane);
          if ((lane & 3) == 0 && r < g.Ni) {
            sPhi[sRowDof[r]] = tot;
            nrm += tot * tot;
          }
        }
        nrm = warp_sum(nrm);
      } else {
        // generic layout (SIMT solver): four rows per warp iteration, scalar loads
        for (int r0 = 4 * warp; r0 < g.Ni; r0 += 4 * nwarp) {
          double acc[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int r = min(r0 + u, g.Ni - 1);
#pragma unroll 4
            for (int col = lane; col < ncd; col += 32) acc[u] += X[(size_t)r * lay.ldx + col] * sC[col];
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) acc[u] = warp_sum(acc[u]);
          if (lane == 0) {
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              if (r0 + u < g.Ni) {
                sPhi[sRowDof[r0 + u]] = acc[u];
                nrm += acc[u] * acc[u];
              }
            }
          }
        }
      }
      if (lane == 0) sRed[warp] = nrm;
      __syncthreads();
      if (tid == 0) {
        double t = 0.0;
        for (int i = 0; i < nwarp; ++i) t += sRed[i];
        sNorm = sqrt(t);
      }
      __syncthreads();
      const double inv = 1.0 / sNorm;
      for (int i = tid; i < g.Nf; i += NT) sPhi[i] *= inv;
      __syncthreads();
      double *po = phi_out + ((size_t)pid * s + d) * lay.nf_max;
      double *ao = aphi_out + ((size_t)pid * s + d) * lay.nf_max;
      for (int i = tid; i < lay.nf_max; i += NT) {
        double v = 0.0, av = 0.0;
        if (i < g.Nf) {
          v = sPhi[i];
          int a[3];
          node_coords(g, i / s, a);
          const int ca = i % s;
          if (node_class(cP, g, a) & 2) {
            av = v;  // domain-boundary rows of semi_constrained are identity rows (source/LOD.cc:537-541)
          } else if (cP.dim == 3 && s == 1 && cP.problem == 0 && !cP.gauss_coef) {
            // scalar 3-D problem with one coefficient per sub-cell: the same sums in the same order as the general
            // branch below, fully unrolled -- the 27 phi values around the node are loaded once, the reference-matrix
            // entries are immediate constant-bank operands, sub-cells outside the patch enter with coefficient 0
            const int msx = g.m[0] * cP.n, msy = g.m[1] * cP.n, msz = g.m[2] * cP.n;
            double pn[27];
#pragma unroll
            for (int e = 0; e < 27; ++e) {
              const int bx = a[0] + e % 3 - 1, by = a[1] + (e / 3) % 3 - 1, bz = a[2] + e / 9 - 1;
              const bool in = bx >= 0 && bx < g.p[0] && by >= 0 && by < g.p[1] && bz >= 0 && bz < g.p[2];
              pn[e] = in ? sPhi[(bz * g.p[1] + by) * g.p[0] + bx] : 0.0;
            }
#pragma unroll
            for (int oc = 0; oc < 8; ++oc) {
              const int ox = a[0] - (oc & 1), oy = a[1] - ((oc >> 1) & 1), oz = a[2] - ((oc >> 2) & 1);
              const bool in = ox >= 0 && ox < msx && oy >= 0 && oy < msy && oz >= 0 && oz < msz;
              double racc = 0.0;
#pragma unroll
              for (int lb = 0; lb < 8; ++lb) {
                // vertex lb of the sub-cell with origin node - bits(oc): offset bits(lb) - bits(oc) from the node
                const int ex = (lb & 1) - (oc & 1) + 1, ey = ((lb >> 1) & 1) - ((oc >> 1) & 1) + 1, ez = ((lb >> 2) & 1) - ((oc >> 2) & 1) + 1;
                racc += cP.Kref[oc * 8 + lb] * pn[(ez * 3 + ey) * 3 + ex];
              }
              if (in) av += sCoef[(oz * msy + oy) * msx + ox] * racc;
            }
          } else {
            // sub-cell-wise application of the patch operator: for every sub-cell that contains the node, its local
            // matrix row times the local phi values (include/Diffusion.h:143-193 / include/Elasticity.h:211-284)
            const int dimv = cP.dim, nn = 1 << dimv, nl = nn * s;
            const int msx = g.m[0] * cP.n, msy = g.m[1] * cP.n, msz = (dimv == 3) ? g.m[2] * cP.n : 1;
            const int nsubp = msx * msy * msz;
            for (int oc = 0; oc < nn; ++oc) {
              // sub-cell origin = node - (oc bits); the node is local vertex la = oc of that sub-cell
              const int ox = a[0] - (oc & 1), oy = a[1] - ((oc >> 1) & 1), oz = (dimv == 3) ? a[2] - ((oc >> 2) & 1) : 0;
              if (ox < 0 || ox >= msx || oy < 0 || oy >= msy || oz < 0 || oz >= msz) continue;
              const int sc = (oz * msy + oy) * msx + ox;
              const int rowi = (oc * s + ca) * nl;
              double cacc = 0.0;
              if (!cP.gauss_coef) {
                double racc = 0.0, lacc = 0.0;
                for (int lb = 0; lb < nn; ++lb) {
                  const int nb_ = ((oz + ((lb >> 2) & 1)) * g.p[1] + (oy + ((lb >> 1) & 1))) * g.p[0] + ox + (lb & 1);
                  for (int cb = 0; cb < s; ++cb) {
                    const double pv = sPhi[nb_ * s + cb];
                    racc += cP.Kref[rowi + lb * s + cb] * pv;
                    if (cP.problem != 0) lacc += cP.Klam[rowi + lb * s + cb] * pv;
                  }
                }
                cacc = (cP.problem == 0) ? sCoef[sc] * racc : sCoef[nsubp + sc] * racc + sCoef[sc] * lacc;
              } else {
                for (int q = 0; q < nn; ++q) {
                  double racc = 0.0, lacc = 0.0;
                  for (int lb = 0; lb < nn; ++lb) {
                    const int nb_ = ((oz + ((lb >> 2) & 1)) * g.p[1] + (oy + ((lb >> 1) & 1))) * g.p[0] + ox + (lb & 1);
                    for (int cb = 0; cb < s; ++cb) {
                      const double pv = sPhi[nb_ * s + cb];
                      racc += cP.Kq[q][rowi + lb * s + cb] * pv;
                      if (cP.problem != 0) lacc += cP.Klamq[q][rowi + lb * s + cb] * pv;
                    }
                  }
                  cacc += (cP.problem == 0) ? sCoef[sc * nn + q] * racc
                                            : sCoef[(nsubp + sc) * nn + q] * racc + sCoef[sc * nn + q] * lacc;
                }
              }
              av += cacc;
            }
          }
        }
        po[i] = v;
        ao[i] = av;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// k_coarse : K rows of one patch in block-ELL form.  patch_list == nullptr: the patches [patch_begin, patch_end);
// else the patches patch_list[patch_begin .. patch_end)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_coarse(int patch_begin, int patch_end, const int *__restrict__ patch_list, const double *__restrict__ phi,
         const double *__restrict__ aphi, double *__restrict__ Kell, FinishLayout lay) {
  extern __shared__ double smem[];
  double *sPhi = smem;  // [s][Nf]
  const int tid = threadIdx.x, NT = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarp = NT >> 5;
  const int s = cP.s, n = cP.n, w = cP.w, ww = 2 * w + 1;
  const int nslots = (cP.dim == 3) ? ww * ww * ww : ww * ww;
  for (int it = patch_begin + blockIdx.x; it < patch_end; it += gridDim.x) {
    const int pid = patch_list ? patch_list[it] : it;
    const Geom g = make_geom(cP, pid);
    __syncthreads();
    for (int i = tid; i < s * lay.nf_max; i += NT) sPhi[i] = phi[(size_t)pid * s * lay.nf_max + i];
    __syncthreads();
    int cen[3] = {g.lo[0] + g.cc[0], g.lo[1] + g.cc[1], g.lo[2] + g.cc[2]};
    for (int item = warp; item < nslots * s * s; item += nwarp) {
      const int e = item % s, d = (item / s) % s, slot = item / (s * s);
      int D[3] = {slot % ww - w, (slot / ww) % ww - w, (cP.dim == 3) ? slot / (ww * ww) - w : 0};
      int qc[3] = {cen[0] + D[0], cen[1] + D[1], cen[2] + D[2]};
      double val = 0.0;
      bool valid = true;
      _Pragma("unroll") for (int x = 0; x < 3; ++x) if (x < cP.dim) valid = valid && (qc[x] >= 0 && qc[x] < cP.N);
      if (valid) {
        const int qid = (int)morton_encode(qc, cP.dim, cP.ref);
        const Geom gq = make_geom(cP, qid);
        // overlap box in global node coordinates
        int b0[3], b1[3], cnt = 1;
        for (int x = 0; x < 3; ++x) {
          if (x < cP.dim) {
            b0[x] = max(g.lo[x], gq.lo[x]) * n;
            b1[x] = min(g.lo[x] + g.m[x], gq.lo[x] + gq.m[x]) * n;
            if (b1[x] < b0[x]) valid = false;
          } else {
            b0[x] = 0; b1[x] = 0;
          }
          cnt *= (b1[x] - b0[x] + 1);
        }
        if (valid) {
          const double *aq = aphi + ((size_t)qid * s + e) * lay.nf_max;
          const double *pp = sPhi + d * lay.nf_max;
          const int ex = b1[0] - b0[0] + 1, ey = b1[1] - b0[1] + 1, ez = b1[2] - b0[2] + 1;
          // lanes sweep the (x, y) plane of the overlap box; the z loop only adds plane strides
          const int sp_ = g.p[0] * g.p[1] * s, sq_ = gq.p[0] * gq.p[1] * s;
          const int op = (((b0[2] - g.lo[2] * n) * g.p[1] + (b0[1] - g.lo[1] * n)) * g.p[0] + (b0[0] - g.lo[0] * n)) * s;
          const int oq = (((b0[2] - gq.lo[2] * n) * gq.p[1] + (b0[1] - gq.lo[1] * n)) * gq.p[0] + (b0[0] - gq.lo[0] * n)) * s;
          const int exs = ex * s;
          double acc = 0.0;
          for (int t = lane; t < exs * ey; t += 32) {
            const int iy = t / exs, ix = t - iy * exs;   // ix runs over (node, component)
            const double *p1 = pp + op + iy * g.p[0] * s + ix;
            const double *q1 = aq + oq + iy * gq.p[0] * s + ix;
#pragma unroll 4
            for (int iz = 0; iz < ez; ++iz) acc += p1[iz * sp_] * q1[iz * sq_];
          }
          val = warp_sum(acc);
        }
      }
      if (lane == 0) Kell[((size_t)pid * s + d) * cP.ell_width + slot * s + e] = val;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// k_coarse_blocked : the same rows, one CTA per Morton-aligned group of 2^dim patches.
// The basis functions of the group are staged in shared memory on the group's common node box (zero outside
// each member's own box), so every A*phi value of a neighbour is loaded once per group and multiplied with all
// members' phi at the same shared-memory offset: no per-pair index arithmetic, 2^dim times less L2 traffic.
// LIST = false: the groups that meet [patch_begin, patch_end); true: the n_groups groups of group_list (every member's
// rows are written, [patch_begin, patch_end) must then cover all patches).  Two instantiations keep the code of the
// range path as it was.
// ------------------------------------------------------------------------------------------------
constexpr int kCoarseThreads = 512;
template <int DIM, int S, bool LIST>
__global__ void __launch_bounds__(kCoarseThreads, 1)
k_coarse_blocked(int patch_begin, int patch_end, const int *__restrict__ group_list, int n_groups,
                 const double *__restrict__ phi, const double *__restrict__ aphi, double *__restrict__ Kell,
                 FinishLayout lay, int NU) {
  constexpr int NG = 1 << DIM;   // patches per group
  constexpr int NA = NG * S;     // accumulators per lane and neighbour: (member, component d)
  constexpr int NQ = 4;          // neighbours (adjacent in x) per warp pass (3: no spills but 8.3 instead of 7.7 ms)
  extern __shared__ double smem[];
  const int NUV = (DIM == 3) ? NU * NU * NU : NU * NU;
  double *sU = smem;  // [NA][NUV][S]
  __shared__ int sGeo[NG][8];  // per member: lo[3] (coarse), centre[3] (coarse), pid, in-range flag
  __shared__ int sUlo[3], sUhi[3];
  const int tid = threadIdx.x, NT = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarp = NT >> 5;
  const int n = cP.n, w = cP.w, ww = 2 * w + 1;
  const int g0 = LIST ? 0 : patch_begin >> DIM, g1 = LIST ? n_groups : ((patch_end - 1) >> DIM) + 1;
  for (int it = g0 + blockIdx.x; it < g1; it += gridDim.x) {
    const int grp = LIST ? group_list[it] : it;
    __syncthreads();
    if (tid < NG) {
      const int pid = grp * NG + tid;
      const Geom g = make_geom(cP, pid);
      for (int a = 0; a < 3; ++a) { sGeo[tid][a] = g.lo[a]; sGeo[tid][3 + a] = g.lo[a] + g.cc[a]; }
      sGeo[tid][6] = pid;
      sGeo[tid][7] = (pid >= patch_begin && pid < patch_end) ? 1 : 0;
    }
    for (int idx = tid; idx < NA * NUV * S; idx += NT) sU[idx] = 0.0;
    __syncthreads();
    if (tid == 0) {
      for (int a = 0; a < 3; ++a) {
        int lo = 1 << 30, hi = 0;
        for (int k = 0; k < NG; ++k) {
          const Geom g = make_geom(cP, sGeo[k][6]);
          lo = min(lo, g.lo[a] * n);
          hi = max(hi, (a < DIM) ? (g.lo[a] + g.m[a]) * n : 0);
        }
        sUlo[a] = (a < DIM) ? lo : 0;
        sUhi[a] = hi;
      }
    }
    __syncthreads();
    const int ulo[3] = {sUlo[0], sUlo[1], sUlo[2]}, uhi[3] = {sUhi[0], sUhi[1], sUhi[2]};
    // scatter the members' phi onto the common box
    for (int k = 0; k < NG; ++k) {
      const Geom g = make_geom(cP, sGeo[k][6]);
      const int ox = g.lo[0] * n - ulo[0], oy = g.lo[1] * n - ulo[1], oz = (DIM == 3) ? g.lo[2] * n - ulo[2] : 0;
      for (int d = 0; d < S; ++d) {
        const double *src = phi + ((size_t)sGeo[k][6] * S + d) * lay.nf_max;
        double *dst = sU + (size_t)(k * S + d) * NUV * S;
        for (int i = tid; i < g.Nf; i += NT) {
          const int c = i % S;
          int node = i / S;
          const int ax = node % g.p[0];
          node /= g.p[0];
          const int ay = node % g.p[1], az = node / g.p[1];
          dst[(((az + oz) * NU + (ay + oy)) * NU + (ax + ox)) * S + c] = src[i];
        }
      }
    }
    __syncthreads();
    // neighbour cells of the group: [base - w, base + 1 + w] per axis.  A warp takes NQ neighbours that are adjacent
    // in x at a time: they share the y / z extents of their sweep boxes, so one pass over the union of the boxes loads
    // every staged phi value once for all of them (the kernel is bound by its shared-memory loads: 8 per A*phi value
    // with one neighbour at a time, 8 per NQ values now).
    const int bx = sGeo[0][3], by = sGeo[0][4], bz = sGeo[0][5];  // member 0 = lowest corner of the 2^dim block
    const int span = 2 * w + 2;
    const int ngx = (span + NQ - 1) / NQ;
    const int ngrp = ngx * span * ((DIM == 3) ? span : 1);
    for (int gi = warp; gi < ngrp; gi += nwarp) {
      const int qx0 = bx - w + NQ * (gi % ngx), qy = by - w + (gi / ngx) % span, qz = (DIM == 3) ? bz - w + gi / (ngx * span) : 0;
      if (qy < 0 || qy >= cP.N || qz < 0 || qz >= cP.N) continue;
      // per neighbour: id, x range of the sweep box (global node coordinates), row length; y / z from the first valid one
      int qid[NQ], x0[NQ], x1[NQ], lox[NQ], px[NQ];
      int b0y = 0, b1y = -1, b0z = 0, b1z = -1, loy = 0, loz = 0, py = 1;
      int ux0 = 1 << 30, ux1 = -1;
      bool got = false;
#pragma unroll
      for (int j = 0; j < NQ; ++j) {
        const int qc[3] = {qx0 + j, qy, qz};
        x0[j] = 1; x1[j] = 0; qid[j] = 0; lox[j] = 0; px[j] = 1;
        if (NQ * (gi % ngx) + j >= span || qc[0] < 0 || qc[0] >= cP.N) continue;
        const Geom gq = make_geom_at(cP, qc);
        x0[j] = max(gq.lo[0] * n, ulo[0]);
        x1[j] = min((gq.lo[0] + gq.m[0]) * n, uhi[0]);
        if (x1[j] < x0[j]) continue;
        qid[j] = (int)morton_fast(qc, DIM);
        lox[j] = gq.lo[0] * n;
        px[j] = gq.p[0];
        ux0 = min(ux0, x0[j]);
        ux1 = max(ux1, x1[j]);
        if (!got) {
          got = true;
          b0y = max(gq.lo[1] * n, ulo[1]);
          b1y = min((gq.lo[1] + gq.m[1]) * n, uhi[1]);
          loy = gq.lo[1] * n;
          py = gq.p[1];
          if (DIM == 3) {
            b0z = max(gq.lo[2] * n, ulo[2]);
            b1z = min((gq.lo[2] + gq.m[2]) * n, uhi[2]);
            loz = gq.lo[2] * n;
          } else {
            b0z = 0; b1z = 0; loz = 0;
          }
        }
      }
      if (!got || b1y < b0y || b1z < b0z) continue;
      const int exu = ux1 - ux0 + 1, ey = b1y - b0y + 1, ez = b1z - b0z + 1;
      for (int e = 0; e < S; ++e) {
        double acc[NQ][NA];
#pragma unroll
        for (int j = 0; j < NQ; ++j)
#pragma unroll
          for (int k = 0; k < NA; ++k) acc[j][k] = 0.0;
        for (int t = lane; t < exu * ey; t += 32) {
          const int iy = t / exu, ix = t - iy * exu;
          const int gx = ux0 + ix, gy = b0y + iy;
          const double *u1 = sU + (((b0z - ulo[2]) * NU + (gy - ulo[1])) * NU + (gx - ulo[0])) * S;
          const double *q1[NQ];
          int sq[NQ];
          bool in[NQ];
#pragma unroll
          for (int j = 0; j < NQ; ++j) {
            in[j] = gx >= x0[j] && gx <= x1[j];
            sq[j] = px[j] * py * S;
            q1[j] = aphi + ((size_t)qid[j] * S + e) * lay.nf_max +
                    (((b0z - loz) * py + (gy - loy)) * px[j] + (in[j] ? gx - lox[j] : 0)) * S;
          }
          for (int iz = 0; iz < ez; ++iz) {
#pragma unroll
            for (int c = 0; c < S; ++c) {
              double v[NQ];
#pragma unroll
              for (int j = 0; j < NQ; ++j) v[j] = in[j] ? q1[j][iz * sq[j] + c] : 0.0;
              const double *u = u1 + iz * NU * NU * S + c;
#pragma unroll
              for (int k = 0; k < NA; ++k) {
                const double uk = u[(size_t)k * NUV * S];
#pragma unroll
                for (int j = 0; j < NQ; ++j) acc[j][k] += v[j] * uk;
              }
            }
          }
        }
#pragma unroll
        for (int j = 0; j < NQ; ++j) {
          if (x1[j] < x0[j]) continue;   // warp uniform
          const double val = warp_sum_packed(acc[j], lane);   // lane L holds pair warp_sum_index<NA>(L)
          if ((lane & (NA == 8 ? 3 : 7)) == 0) {
            // pair k = (member k / S, component k % S)
            const int k = warp_sum_index<NA>(lane);
            const int mem = k / S, d = k - mem * S;
            if (sGeo[mem][7]) {
              const int Dx = qx0 + j - sGeo[mem][3], Dy = qy - sGeo[mem][4], Dz = (DIM == 3) ? qz - sGeo[mem][5] : 0;
              if (abs(Dx) <= w && abs(Dy) <= w && abs(Dz) <= w) {
                const int slot = (DIM == 3) ? ((Dz + w) * ww + (Dy + w)) * ww + (Dx + w) : (Dy + w) * ww + (Dx + w);
                Kell[((size_t)sGeo[mem][6] * S + d) * cP.ell_width + slot * S + e] = val;
              }
            }
          }
        }
      }
    }
  }
}
template <int DIM, int S>
static cudaError_t launch_coarse_blocked_t(int grid, size_t smem, cudaStream_t st, int p0, int p1, const double *phi,
                                           const double *aphi, double *Kell, const FinishLayout &lay, int NU,
                                           const int *groups, int n_groups) {
  // a group list rewrites rows of a matrix that was assembled before: the slots the kernel never visits (neighbours
  // outside the domain) are zero already, they depend on the geometry alone.  A range clears its rows first.
  if (groups) {
    cudaError_t e = cudaFuncSetAttribute(k_coarse_blocked<DIM, S, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    k_coarse_blocked<DIM, S, true><<<grid, kCoarseThreads, smem, st>>>(p0, p1, groups, n_groups, phi, aphi, Kell, lay, NU);
    return cudaGetLastError();
  }
  cudaError_t e = cudaFuncSetAttribute(k_coarse_blocked<DIM, S, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  e = cudaMemsetAsync(Kell + (size_t)p0 * S * (lay.ell_width), 0, sizeof(double) * (size_t)(p1 - p0) * S * lay.ell_width, st);
  if (e != cudaSuccess) return e;
  k_coarse_blocked<DIM, S, false><<<grid, kCoarseThreads, smem, st>>>(p0, p1, nullptr, 0, phi, aphi, Kell, lay, NU);
  return cudaGetLastError();
}
size_t coarse_blocked_smem(int dim, int s, int NU) {
  size_t nuv = (dim == 3) ? (size_t)NU * NU * NU : (size_t)NU * NU;
  return sizeof(double) * ((size_t)(1 << dim) * s * nuv * s);
}
cudaError_t launch_coarse_blocked(int dim, int s, int grid, size_t smem, cudaStream_t st, int p0, int p1,
                                  const double *phi, const double *aphi, double *Kell, const FinishLayout &lay, int NU,
                                  const int *groups, int n_groups) {
  if (dim == 3 && s == 1) return launch_coarse_blocked_t<3, 1>(grid, smem, st, p0, p1, phi, aphi, Kell, lay, NU, groups, n_groups);
  if (dim == 2 && s == 1) return launch_coarse_blocked_t<2, 1>(grid, smem, st, p0, p1, phi, aphi, Kell, lay, NU, groups, n_groups);
  if (dim == 2 && s == 2) return launch_coarse_blocked_t<2, 2>(grid, smem, st, p0, p1, phi, aphi, Kell, lay, NU, groups, n_groups);
  return cudaErrorInvalidValue;
}

// ------------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------------
cudaError_t launch_patch_solve(int grid, size_t smem, cudaStream_t st, const int *ids, int n_work, const double *coef,
                               double *X, double *Lws, int *status, const SolveLayout &lay) {
  cudaError_t e = cudaFuncSetAttribute(k_patch_solve<kSolveNB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  k_patch_solve<kSolveNB><<<grid, lay.threads, smem, st>>>(ids, n_work, coef, X, Lws, status, lay);
  return cudaGetLastError();
}
template <int RBMAX, int NW>
static cudaError_t launch_mma_t(int grid, size_t smem, cudaStream_t st, const int *ids, int n_work, const double *coef,
                                double *X, double *Lws, int *status, const SolveMmaLayout &lay, int *work_counter) {
  cudaError_t e = cudaFuncSetAttribute(k_patch_solve_mma<RBMAX, NW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  k_patch_solve_mma<RBMAX, NW><<<grid, 32 * NW, smem, st>>>(ids, n_work, coef, X, Lws, status, lay, work_counter);
  return cudaGetLastError();
}
size_t solve_mma_smem(int variant, int coef_doubles, int nip_max, int stw) {
  const int RBMAX = (variant == 0) ? 13 : 4;
  const int NW = (variant == 0) ? 16 : (variant == 1 ? 4 : 8);
  const int R = 8 * RBMAX, LDWF = (R % 16 == 8) ? R : R + 8, LDP = R + 4;
  return sizeof(double) * ((size_t)coef_doubles + (size_t)R * LDWF + 8 * LDP + kSolveStages * (R * 8 + 64) +
                           (size_t)nip_max * stw) +
         sizeof(int) * ((size_t)nip_max + 8 * NW + RBMAX * (RBMAX - 1) / 2 + 32 + 8);
}
cudaError_t launch_patch_solve_mma(int variant, int grid, size_t smem, cudaStream_t st, const int *ids, int n_work,
                                   const double *coef, double *X, double *Lws, int *status, int coef_doubles, int ldx,
                                   long long x_stride, long long lws_per_cta, int nip_max, int stw, int *work_counter) {
  SolveMmaLayout lay{coef_doubles, nip_max, stw, ldx, x_stride, lws_per_cta};
  if (work_counter) {
    cudaError_t e = cudaMemsetAsync(work_counter, 0, sizeof(int), st);
    if (e != cudaSuccess) return e;
  }
  switch (variant) {
    case 0: return launch_mma_t<13, 16>(grid, smem, st, ids, n_work, coef, X, Lws, status, lay, work_counter);
    case 1: return launch_mma_t<4, 4>(grid, smem, st, ids, n_work, coef, X, Lws, status, lay, work_counter);
    case 2: return launch_mma_t<4, 8>(grid, smem, st, ids, n_work, coef, X, Lws, status, lay, work_counter);
  }
  return cudaErrorInvalidValue;
}

// split solver (solve_split.cuh): factorisation with 8 warps, 2 CTAs per SM; triangular solves with 16 warps
constexpr int kSplitRB = 13, kFactorWarps = 8, kTriWarps = 16;
size_t split_factor_smem(int coef_doubles, int nip_max) {
  const int R = 8 * kSplitRB, LDWF = (R % 16 == 8) ? R : R + 8, LDP = R + 4;
  return sizeof(double) * ((size_t)coef_doubles + (size_t)R * LDWF + 8 * LDP + 2 * 64 + 64) +
         sizeof(int) * ((size_t)nip_max + kSplitRB * (kSplitRB - 1) / 2 + 16 + 8);
}
size_t split_trisolve_smem(int nip_max) {
  return sizeof(double) * ((size_t)kTriStages * kSplitRB * 64) + 2 * kTriStages * sizeof(unsigned long long) +
         sizeof(int) * ((size_t)nip_max + 8 * kTriWarps + kTriWarps + nip_max / 8 + 1 + 8 + 4);
}
long long split_rec_stride(int nip_max) { return (long long)(nip_max / 8) * kSplitRB * 64; }
size_t split_stencil_ws_doubles(int grid, int nip_max) { return (size_t)grid * nip_max * 14; }
cudaError_t launch_patch_factor(int grid, size_t smem, cudaStream_t st, const int *ids, int n_work, const double *coef,
                                double *Lrec, double *stencil_ws, int *status, int coef_doubles, int nip_max, int ldx,
                                long long x_stride, int *work_counter) {
  SplitLayout lay{coef_doubles, nip_max, ldx, x_stride, split_rec_stride(nip_max)};
  cudaError_t e = cudaFuncSetAttribute(k_patch_factor<kSplitRB, kFactorWarps>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  // two CTAs per SM need nearly all of the 228 KB: ask for the largest shared-memory carve-out
  e = cudaFuncSetAttribute(k_patch_factor<kSplitRB, kFactorWarps>, cudaFuncAttributePreferredSharedMemoryCarveout,
                           (int)cudaSharedmemCarveoutMaxShared);
  if (e != cudaSuccess) return e;
  if (getenv("SLOD_PRINT_OCC")) {
    int nb = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_patch_factor<kSplitRB, kFactorWarps>, 32 * kFactorWarps, smem);
    printf("k_patch_factor: %d CTAs/SM, %zu B dynamic shared memory\n", nb, smem);
  }
  if (work_counter && (e = cudaMemsetAsync(work_counter, 0, sizeof(int), st)) != cudaSuccess) return e;
  k_patch_factor<kSplitRB, kFactorWarps><<<grid, 32 * kFactorWarps, smem, st>>>(ids, n_work, coef, Lrec, stencil_ws, status, lay, work_counter);
  return cudaGetLastError();
}
cudaError_t launch_patch_trisolve(int grid, size_t smem, cudaStream_t st, const int *ids, int n_work, const double *Lrec,
                                  double *X, int coef_doubles, int nip_max, int ldx, long long x_stride, int *work_counter) {
  SplitLayout lay{coef_doubles, nip_max, ldx, x_stride, split_rec_stride(nip_max)};
  cudaError_t e = cudaFuncSetAttribute(k_patch_trisolve<kSplitRB, kTriWarps>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  if (work_counter && (e = cudaMemsetAsync(work_counter, 0, sizeof(int), st)) != cudaSuccess) return e;
  k_patch_trisolve<kSplitRB, kTriWarps><<<grid, 32 * kTriWarps, smem, st>>>(ids, n_work, Lrec, X, lay, work_counter);
  return cudaGetLastError();
}

cudaError_t launch_patch_dense(int grid, size_t smem, cudaStream_t st, const int *ids, int n_work, const double *coef,
                               const double *X, double *Minv, double *G, double *diag, int *status,
                               const DenseLayout &lay) {
  cudaError_t e = cudaFuncSetAttribute(k_patch_dense, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  k_patch_dense<<<grid, lay.threads, smem, st>>>(ids, n_work, coef, X, Minv, G, diag, status, lay);
  return cudaGetLastError();
}
template <int NTILE>
static cudaError_t launch_dense_t(int grid, size_t smem, cudaStream_t st, const int *ids, int n_work, const double *coef,
                                  const double *X, const double *W, double *Minv, double *G, double *diag, int *status,
                                  const DenseLayout &lay, int *work_counter) {
  cudaError_t e = cudaFuncSetAttribute(k_patch_dense_mma<NTILE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  k_patch_dense_mma<NTILE><<<grid, 32 * NTILE, smem, st>>>(ids, n_work, coef, X, W, Minv, G, diag, status, lay, work_counter);
  return cudaGetLastError();
}
size_t dense_mma_smem(int ntile, int coef_doubles, int nb_max) {
  (void)nb_max;
  (void)coef_doubles;   // the dense stage needs no coefficients: M comes from X, W from k_patch_flux
  const int NC = 8 * ntile, LDM = NC + 4;
  return sizeof(double) * ((size_t)NC * LDM + 2 * (size_t)kDTB * LDM) + sizeof(int) * ((size_t)NC * 32 + 8);
}
cudaError_t launch_patch_dense_mma(int ntile, int grid, size_t smem, cudaStream_t st, const int *ids, int n_work,
                                   const double *coef, const double *X, const double *W, double *Minv, double *G,
                                   double *diag, int *status, const DenseLayout &lay, int *work_counter) {
  if (work_counter) {
    cudaError_t e = cudaMemsetAsync(work_counter, 0, sizeof(int), st);
    if (e != cudaSuccess) return e;
  }
  switch (ntile) {
    case 4: return launch_dense_t<4>(grid, smem, st, ids, n_work, coef, X, W, Minv, G, diag, status, lay, work_counter);
    case 8: return launch_dense_t<8>(grid, smem, st, ids, n_work, coef, X, W, Minv, G, diag, status, lay, work_counter);
    case 16: return launch_dense_t<16>(grid, smem, st, ids, n_work, coef, X, W, Minv, G, diag, status, lay, work_counter);
  }
  return cudaErrorInvalidValue;
}
size_t flux_smem(int coef_doubles, int ldx, int nb_max) {
  (void)ldx;
  return sizeof(double) * ((size_t)coef_doubles + (size_t)kFTB * kFNB) +
         sizeof(int) * ((size_t)kFTB * kFNB + kFTB + nb_max + 8);
}
cudaError_t launch_patch_flux(int grid, size_t smem, cudaStream_t st, const int *ids, int n_work, const double *coef,
                              const double *X, double *W, const FluxLayout &lay, int *work_counter) {
  cudaError_t e = cudaFuncSetAttribute(k_patch_flux, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  if (work_counter && (e = cudaMemsetAsync(work_counter, 0, sizeof(int), st)) != cudaSuccess) return e;
  k_patch_flux<<<grid, 256, smem, st>>>(ids, n_work, coef, X, W, lay, work_counter);
  return cudaGetLastError();
}

size_t select_fast_smem(int ncd_max) {
  const size_t nbk = (size_t)(ncd_max + 6) / 8;
  return sizeof(double) * (nbk * (nbk + 1) / 2 * 64 + 8 * nbk + 8);
}
size_t select_jacobi_smem(int ncd_max) {
  return sizeof(double) * ((size_t)ncd_max * (ncd_max + 1) / 2 + (size_t)ncd_max * ncd_max + 6 * (size_t)ncd_max) +
         sizeof(int) * (3 * (size_t)ncd_max + 8);
}
size_t eig_tridiag_smem(int nmax) { return sizeof(double) * ((size_t)nmax * (nmax | 1) + 4 * (size_t)nmax); }
size_t eig_ql_smem(int nmax) { return sizeof(double) * 8 * 3 * (size_t)nmax; }
size_t eig_finish_smem(int nmax) {
  return sizeof(double) * ((size_t)nmax * kEigLd + 5 * (size_t)nmax) + sizeof(int) * ((size_t)nmax + 8);
}

cudaError_t launch_select_pipeline(const SelectPlan &pl, cudaStream_t st, const int *ids, int n_work, const double *Minv,
                                   const double *G, double *cvec, double *diag, int *status, const SelectBuffers &b,
                                   int *n_launches) {
  cudaError_t e;
#define SLOD_ATTR(k, sm)                                                                        \
  if ((e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sm))) != cudaSuccess) return e
  SLOD_ATTR(k_select_fast, pl.smem_fast);
  SLOD_ATTR(k_select_jacobi, pl.smem_jac);
  if ((e = cudaMemsetAsync(b.counters, 0, 4 * sizeof(int), st)) != cudaSuccess) return e;
  k_select_fast<<<min(n_work, pl.grid_fast), 256, pl.smem_fast, st>>>(
      ids, n_work, Minv, G, cvec, diag, b.counters, pl.use_ql ? b.eig_list : b.jac_list, pl.use_ql ? 1 : 2, pl.lay);
  ++*n_launches;
  if (pl.use_ql) {
    SLOD_ATTR(k_eig_tridiag<4>, pl.smem_tri);
    SLOD_ATTR(k_eig_tridiag<8>, pl.smem_tri);
    SLOD_ATTR(k_eig_ql, pl.smem_ql);
    SLOD_ATTR(k_eig_finish, pl.smem_fin);
    const long long items_max = (long long)n_work * pl.s;
    for (long long off = 0; off < items_max; off += pl.eig.cap_items) {
      if (pl.eig.nmax - 1 <= 128)   // n = ncd - 1 columns: four per lane are enough
        k_eig_tridiag<4><<<pl.grid_tri, 512, pl.smem_tri, st>>>(ids, b.counters, b.eig_list, (int)off, G, b.H, b.V, pl.eig);
      else
        k_eig_tridiag<8><<<pl.grid_tri, 512, pl.smem_tri, st>>>(ids, b.counters, b.eig_list, (int)off, G, b.H, b.V, pl.eig);
      k_eig_ql<<<pl.grid_ql, 256, pl.smem_ql, st>>>(ids, b.counters, b.eig_list, (int)off, b.V, b.rot_cs, b.rot_i,
                                                   b.rot_n, pl.eig);
      k_eig_finish<<<pl.grid_fin, 128, pl.smem_fin, st>>>(ids, b.counters, b.eig_list, (int)off, Minv, b.H, b.V,
                                                         b.rot_cs, b.rot_i, b.rot_n, cvec, diag, b.jac_list, pl.eig);
      *n_launches += 3;
    }
  }
  k_select_jacobi<<<pl.grid_jac, pl.lay.threads, pl.smem_jac, st>>>(ids, b.counters, b.jac_list, Minv, G, cvec, diag,
                                                                    status, pl.lay);
  ++*n_launches;
#undef SLOD_ATTR
  return cudaGetLastError();
}
cudaError_t launch_patch_finish(int grid, size_t smem, cudaStream_t st, const int *ids, int n_work, const double *coef,
                                const double *X, const double *cvec, double *phi, double *aphi,
                                const FinishLayout &lay) {
  cudaError_t e = cudaFuncSetAttribute(k_patch_finish, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  k_patch_finish<<<grid, 256, smem, st>>>(ids, n_work, coef, X, cvec, phi, aphi, lay);
  return cudaGetLastError();
}
__global__ void __launch_bounds__(256)
k_gather(const double *__restrict__ src, const long long *__restrict__ perm, double *__restrict__ dst, long long n) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    dst[i] = src[perm[i]];
}
cudaError_t launch_gather(cudaStream_t st, const double *src, const long long *perm, double *dst, long long n) {
  if (n <= 0) return cudaSuccess;
  k_gather<<<148 * 8, 256, 0, st>>>(src, perm, dst, n);
  return cudaGetLastError();
}

#include "update.cuh"
}  // namespace slod
#include "online.cuh"
#include "online_batch.cuh"
#include "heat.cuh"
namespace slod {

cudaError_t launch_coarse_rhs(cudaStream_t st, int n_patches, int s, const double *phi, const double *f, double *b,
                              int nf_max) {
  const int rows = n_patches * s, per = kCgThreads / 32;
  k_coarse_rhs<<<(rows + per - 1) / per, kCgThreads, 0, st>>>(n_patches, phi, f, b, nf_max);
  return cudaGetLastError();
}
cudaError_t launch_prolongate(cudaStream_t st, long long n_fine, const double *phi, const double *u, double *u_fine,
                              int nf_max) {
  const long long blocks = (n_fine + kCgThreads - 1) / kCgThreads;
  k_prolongate<<<(int)(blocks < 148 * 16 ? blocks : 148 * 16), kCgThreads, 0, st>>>(n_fine, phi, u, u_fine, nf_max);
  return cudaGetLastError();
}
// a few waves of persistent blocks: short partial-sum arrays for the two vector kernels to reduce
static int cg_apply_blocks(const CgOperator &A, int nrows) {
  if (!A.Kell) return (int)((A.n_nodes + kCgThreads - 1) / kCgThreads);   // fine operator: one thread per node
  const int per = kCgThreads / 32, want = (nrows + per - 1) / per;
  return want < 148 * 8 ? want : 148 * 8;
}
size_t cg_workspace_doubles(const CgOperator &A, int nrows) {
  const int nb_apply = cg_apply_blocks(A, nrows), nb_vec = (nrows + kCgThreads - 1) / kCgThreads;
  // r, p, q, dinv | partial p.q | partial r.z, r.r | state
  return (size_t)4 * nrows + nb_apply + 2 * (size_t)nb_vec + (sizeof(CgState) + 7) / 8;
}
// Runs diag-preconditioned CG until the device-side stopping test fires or max_steps is reached; the host looks at the
// state every `check_every` steps (one 64-byte copy).  A.Kell != nullptr: block-ELL coarse matrix; else the fine
// Dirichlet operator A.op applied matrix free.  Returns the state in *steps / *residual / *flag.
cudaError_t run_cg(cudaStream_t st, int nrows, const CgOperator &A, const double *b, double *x, double *work,
                   int max_steps, double tol, double reduction, int *steps, double *residual, int *flag,
                   long long *launches) {
  const int nb_apply = cg_apply_blocks(A, nrows), nb_vec = (nrows + kCgThreads - 1) / kCgThreads;
  double *r = work, *p = r + nrows, *q = p + nrows, *dinv = q + nrows;
  double *ppq = dinv + nrows, *prz = ppq + nb_apply, *prr = prz + nb_vec;
  CgState *state = reinterpret_cast<CgState *>(prr + nb_vec);
  CgState h{};
  cudaError_t e;
  if (!A.Kell) {
    k_fine_apply<<<nb_apply, kCgThreads, 0, st>>>(A.op, A.tau, A.n_nodes, A.d_coef, nullptr, nullptr, dinv, nullptr,
                                                 nullptr);
    *launches += 1;
  }
  k_cg_init<<<1, 1024, 0, st>>>(nrows, A.Kell, b, x, r, p, dinv, state, tol, reduction);
  *launches += 1;
  const int check_every = A.Kell ? 16 : 64;
  int it = 0;
  for (;;) {
    if ((e = cudaMemcpyAsync(&h, state, sizeof(CgState), cudaMemcpyDeviceToHost, st)) != cudaSuccess) return e;
    if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return e;
    if (h.done || it >= max_steps) break;
    const int upto = (it + check_every < max_steps) ? it + check_every : max_steps;
    for (; it < upto; ++it) {
      if (A.Kell)
        k_cg_spmv<<<nb_apply, kCgThreads, 0, st>>>(nrows, A.Kell, p, q, ppq, state);
      else
        k_fine_apply<<<nb_apply, kCgThreads, 0, st>>>(A.op, A.tau, A.n_nodes, A.d_coef, p, q, nullptr, ppq, state);
      k_cg_update<<<nb_vec, kCgThreads, 0, st>>>(nrows, it, p, q, dinv, x, r, ppq, nb_apply, prz, prr, state);
      k_cg_direction<<<nb_vec, kCgThreads, 0, st>>>(nrows, it, r, dinv, p, prz, prr, nb_vec, state);
      *launches += 3;
    }
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  }
  *steps = h.steps;
  *residual = sqrt(h.rr);
  *flag = h.done;
  return cudaGetLastError();
}
// x . Op x for Op = energy / mass / Laplace (FineOp): per-block partial sums, added up by the caller in block order
cudaError_t launch_fine_quadratic_form(cudaStream_t st, int op, long long n_nodes, const double *d_coef, const double *x,
                                       double *partial, int *n_partial) {
  const int nb = (int)((n_nodes + kCgThreads - 1) / kCgThreads);
  *n_partial = nb;
  if (partial) k_fine_apply<<<nb, kCgThreads, 0, st>>>(op, 0.0, n_nodes, d_coef, x, nullptr, nullptr, partial, nullptr);
  return cudaGetLastError();
}

// ---- batched online phase (online_batch.cuh) ----
cudaError_t launch_interleave(cudaStream_t st, long long n, int kb, const double *src, double *dst, bool to_interleaved) {
  const long long blocks = (n * kb + 255) / 256;
  const int grid = (int)(blocks < 148 * 16 ? blocks : 148 * 16);
  if (to_interleaved) k_interleave<<<grid, 256, 0, st>>>(n, kb, src, dst);
  else k_deinterleave<<<grid, 256, 0, st>>>(n, kb, src, dst);
  return cudaGetLastError();
}
cudaError_t launch_coarse_rhs_multi(cudaStream_t st, int n_patches, int s, int kb, const double *phi, const double *F,
                                    double *B, int nf_max) {
  const int rows = n_patches * s, per = kCgThreads / 32;
  k_coarse_rhs_multi<<<(rows + per - 1) / per, kCgThreads, 0, st>>>(n_patches, kb, phi, F, B, nf_max);
  return cudaGetLastError();
}
cudaError_t launch_prolongate_multi(cudaStream_t st, long long n_fine, int kb, const double *phi, const double *U,
                                    double *Uf, int nf_max) {
  const long long blocks = (n_fine + kCgThreads - 1) / kCgThreads;
  k_prolongate_multi<<<(int)(blocks < 148 * 16 ? blocks : 148 * 16), kCgThreads, 0, st>>>(n_fine, kb, phi, U, Uf,
                                                                                          nf_max);
  return cudaGetLastError();
}
// Grids depend on nrows only (never on kb): the partial-sum arrays, and so every column's sums, have the same shape
// whatever the group holds.
static int cg_multi_apply_blocks(int nrows) {
  const int per = kCgThreads / 32, want = (nrows + per - 1) / per;
  return want < 148 * 8 ? want : 148 * 8;
}
size_t cg_multi_workspace_doubles(int nrows) {
  const size_t nb_apply = cg_multi_apply_blocks(nrows), nb_vec = (nrows + kVecRows - 1) / kVecRows;
  // R, P, Q | dinv | partial p.q | partial r.z, r.r | states
  return 3 * (size_t)kBatch * nrows + nrows + kBatch * (nb_apply + 2 * nb_vec) + (kBatch * sizeof(CgState) + 7) / 8;
}
// The host loop of run_cg for kb columns: every 16 steps it reads the kb states back (kb x 56 bytes) and stops when all
// columns are done or at max_steps.
cudaError_t run_cg_multi(cudaStream_t st, int nrows, const double *Kell, int kb, const double *B, double *X,
                         double *work, int max_steps, double tol, double reduction, int *steps, double *residual,
                         int *flag, long long *launches) {
  const int nb_apply = cg_multi_apply_blocks(nrows), nb_vec = (nrows + kVecRows - 1) / kVecRows;
  const size_t nv = (size_t)kBatch * nrows;
  double *R = work, *P = R + nv, *Q = P + nv, *dinv = Q + nv;
  double *ppq = dinv + nrows, *prz = ppq + (size_t)kBatch * nb_apply, *prr = prz + (size_t)kBatch * nb_vec;
  CgState *state = reinterpret_cast<CgState *>(prr + (size_t)kBatch * nb_vec);
  CgState h[kBatch];
  cudaError_t e;
  k_cg_init_multi<<<kb, 1024, 0, st>>>(nrows, kb, Kell, B, X, R, P, dinv, state, tol, reduction);
  *launches += 1;
  const int check_every = 16;
  int it = 0;
  for (;;) {
    if ((e = cudaMemcpyAsync(h, state, sizeof(CgState) * kb, cudaMemcpyDeviceToHost, st)) != cudaSuccess) return e;
    if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return e;
    bool all = true;
    for (int j = 0; j < kb; ++j) all = all && h[j].done;
    if (all || it >= max_steps) break;
    const int upto = (it + check_every < max_steps) ? it + check_every : max_steps;
    for (; it < upto; ++it) {
      k_cg_spmm<<<nb_apply, kCgThreads, 0, st>>>(nrows, kb, Kell, P, Q, ppq, state);
      k_cg_update_multi<<<nb_vec, kCgThreads, 0, st>>>(nrows, kb, it, P, Q, dinv, X, R, ppq, nb_apply, prz, prr, state);
      k_cg_direction_multi<<<nb_vec, kCgThreads, 0, st>>>(nrows, kb, it, R, dinv, P, prz, prr, nb_vec, state);
      *launches += 3;
    }
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  }
  for (int j = 0; j < kb; ++j) {
    steps[j] = h[j].steps;
    residual[j] = sqrt(h[j].rr);
    flag[j] = h[j].done;
  }
  return cudaGetLastError();
}

// ---- heat equation on the SLOD space (heat.cuh) ----
cudaError_t launch_mass_apply(cudaStream_t st, int n_patches, int s, const double *phi, double *mphi, int nf_max) {
  const int rows = n_patches * s;
  k_mass_apply<<<rows < 148 * 16 ? rows : 148 * 16, 256, 0, st>>>(n_patches, phi, mphi, nf_max);
  return cudaGetLastError();
}
cudaError_t launch_ell_residual(cudaStream_t st, int nrows, int kb, const double *Kell, const double *U, int nf,
                                const double *B, long long b_stride, const double *W, double tau, double *R) {
  k_ell_residual<<<cg_multi_apply_blocks(nrows), kCgThreads, 0, st>>>(nrows, kb, Kell, U, nf, B, b_stride, W, tau, R);
  return cudaGetLastError();
}
cudaError_t launch_weighted_sum(cudaStream_t st, long long n, int nf, const double *w, const double *F, double *out) {
  const long long blocks = (n + 255) / 256;
  k_weighted_sum<<<(int)(blocks < 148 * 16 ? blocks : 148 * 16), 256, 0, st>>>(n, nf, w, F, out);
  return cudaGetLastError();
}
cudaError_t launch_lincomb(cudaStream_t st, long long n, double a, const double *x, double b, const double *y, double *z) {
  const long long blocks = (n + 255) / 256;
  k_lincomb<<<(int)(blocks < 148 * 16 ? blocks : 148 * 16), 256, 0, st>>>(n, a, x, b, y, z);
  return cudaGetLastError();
}
cudaError_t launch_fine_apply(cudaStream_t st, int op, double tau, long long n_nodes, const double *d_coef,
                              const double *x, double *y) {
  const int nb = (int)((n_nodes + kCgThreads - 1) / kCgThreads);
  k_fine_apply<<<nb, kCgThreads, 0, st>>>(op, tau, n_nodes, d_coef, x, y, nullptr, nullptr, nullptr);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// FP64 throughput probes: the denominator of the roofline the benchmark reports (MEASURED_PEAKS.json has no fp64 entry).
// Register-resident chains, 4 CTAs of 512 threads per SM: plain DFMA, and mma.sync m8n8k4 (the instruction of the
// tensor-core kernels above).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(512) k_probe_dfma(double *out, int iters) {
  double a[8];
  const double b = 1.000000001, c = 1e-9;
#pragma unroll
  for (int i = 0; i < 8; ++i) a[i] = threadIdx.x * 1e-3 + i;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < 8; ++i) a[i] = fma(a[i], b, c);
  }
  double s = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) s += a[i];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
__global__ void __launch_bounds__(512) k_probe_dmma(double *out, int iters) {
  double c[4][2];
#pragma unroll
  for (int i = 0; i < 4; ++i) c[i][0] = c[i][1] = 0.0;
  const double a = 1.0 + threadIdx.x * 1e-6, b = 1.0 - threadIdx.x * 1e-6;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < 4; ++i) dmma884(c[i][0], c[i][1], a, b);
  }
  double s = 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) s += c[i][0] + c[i][1];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
// returns TFLOP/s of the DFMA chain and of the DMMA chain on the current device
cudaError_t run_fp64_probe(int n_sm, double *dfma_tflops, double *dmma_tflops) {
  const int grid = n_sm * 4, block = 512, iters = 20000;
  double *out = nullptr;
  cudaError_t e = cudaMalloc(&out, sizeof(double) * grid * block);
  if (e != cudaSuccess) return e;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  const double threads = (double)grid * block, warps = threads / 32;
  double best[2] = {0, 0};
  for (int which = 0; which < 2; ++which)
    for (int rep = 0; rep < 4; ++rep) {   // first repetition = warm-up
      cudaEventRecord(e0, 0);
      if (which == 0) k_probe_dfma<<<grid, block>>>(out, iters);
      else k_probe_dmma<<<grid, block>>>(out, iters);
      cudaEventRecord(e1, 0);
      cudaEventSynchronize(e1);
      float ms = 0;
      cudaEventElapsedTime(&ms, e0, e1);
      const double flop = (which == 0) ? threads * iters * 8 * 2.0 : warps * iters * 4 * (8 * 8 * 4 * 2.0);
      if (rep > 0) best[which] = fmax(best[which], flop / (ms * 1e-3) / 1e12);
    }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(out);
  *dfma_tflops = best[0];
  *dmma_tflops = best[1];
  return cudaGetLastError();
}

cudaError_t launch_fine_norms_reference(cudaStream_t st, long long n_cells, int nq, const double *gauss_x,
                                        const double *gauss_w, const double *v, double *partial, int *n_blocks) {
  const int nb = (int)((n_cells + kCgThreads - 1) / kCgThreads);
  *n_blocks = nb;
  if (partial) k_fine_norms_reference<<<nb, kCgThreads, 0, st>>>(n_cells, nq, gauss_x, gauss_w, v, partial);
  return cudaGetLastError();
}

cudaError_t launch_coarse(int grid, size_t smem, cudaStream_t st, int p0, int p1, const double *phi, const double *aphi,
                          double *Kell, const FinishLayout &lay, const int *patches) {
  cudaError_t e = cudaFuncSetAttribute(k_coarse, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  k_coarse<<<grid, 256, smem, st>>>(p0, p1, patches, phi, aphi, Kell, lay);
  return cudaGetLastError();
}

}  // namespace slod
