// Split patch solver for the large 3-D patches (cfg 4/5: Ni = 729, half band width 91, 125 right-hand sides):
//
//   k_patch_factor    blocked banded Cholesky of A_ii alone.  Small working set (the 104 x 104 circular window), two
//                     CTAs of 8 warps per SM so that the latency-bound look-ahead chain of one patch (8 x 8 diagonal
//                     factorisation + in-register inverse) hides behind the tensor-core trailing update of the other.
//                     The factor leaves the SM as one record per 8-column step: 13 tiles of 8 x 8 (the inverse of the
//                     diagonal factor, then the 12 panel tiles), each stored in mma.m8n8k4 A-FRAGMENT ORDER -- lane l
//                     owns the two doubles {T[g][t], T[g][4+t]} (g = l >> 2, t = l & 3) -- so that the consumer reads
//                     its A operand with one conflict-free 16-byte load per tile (forward sweep) or two conflict-free
//                     8-byte loads (backward sweep: T^T[g][t] = T[t][g] sits at double 8t + 2(g&3) + (g>>2)).
//   k_patch_trisolve  forward and backward substitution with all right-hand sides.  Pure tensor-core streaming: the 16
//                     warps own 8 right-hand-side columns each and never synchronise with each other -- the records
//                     arrive through an 8-stage ring filled by bulk asynchronous copies (cp.async.bulk + mbarrier
//                     transaction counts), every warp waits on the "full" barrier of a stage and releases it through its
//                     "empty" barrier, there is no block-wide barrier inside a patch.  The right-hand-side window lives
//                     in registers as accumulator tiles (as in k_patch_solve_mma).
//
// Together they replace assemble_stiffness + Gauss_elimination of the reference (source/LOD.cc:433-546,
// include/LODtools.h:511-595).  The fused kernel k_patch_solve_mma remains for the small 2-D patches, where one CTA
// holds everything and the factorisation chain is short.  Included by kernels.cu after solve_mma.cuh.
#pragma once
#include <cuda/std/cstdint>

namespace slod {

// ---- mbarrier / bulk-copy primitives (PTX ISA 8.x, sm_90+) ---------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_n(uint64_t *bar, int count) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
// global -> shared bulk copy (TMA engine, no tensor map), completion counted in bytes on `bar`
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// mma.sync.m16n8k8 f64: one instruction = four m8n8k4 (2048 flop), and far more latency tolerant -- a single warp per
// scheduler sustains the tensor pipe with it (tools/dmma_operands.cu: 36.7 TFLOP/s against 31 / 23 with m8n8k4).
// Fragments (g = lane >> 2, t = lane & 3): A a0 (g, t) a1 (g+8, t) a2 (g, t+4) a3 (g+8, t+4); B b0 (t, g) b1 (t+4, g);
// C c0,c1 (g, 2t..2t+1) c2,c3 (g+8, 2t..2t+1).
__device__ __forceinline__ void dmma1688(double &c0, double &c1, double &c2, double &c3, double a0, double a1, double a2,
                                         double a3, double b0, double b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k8.row.col.f64.f64.f64.f64 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
      : "+d"(c0), "+d"(c1), "+d"(c2), "+d"(c3)
      : "d"(a0), "d"(a1), "d"(a2), "d"(a3), "d"(b0), "d"(b1));
}

#ifdef SLOD_PHASE_CLOCKS
#define PHS_DECL(wa, wb, wc) long long ph_acc[12] = {0}; long long ph_last = clock64(); const bool ph_on = (blockIdx.x == 0) && ((threadIdx.x & 31) == 0) && ((threadIdx.x >> 5) == (wa) || (threadIdx.x >> 5) == (wb) || (threadIdx.x >> 5) == (wc));
#else
#define PHS_DECL(wa, wb, wc)
#endif

constexpr int kTriStages = 12;  // ring depth of k_patch_trisolve (12 x 6.5 KB)

struct SplitLayout {
  int coef_doubles;
  int nip_max;            // interior dofs per patch rounded up to 8
  int ldx;                // leading dimension of X rows (8 * NW of the triangular solver)
  long long x_stride;     // doubles per patch in Xbuf
  long long rec_stride;   // doubles per patch in the factor records: (nip_max / 8) * RBMAX * 64
};

// position of element (r, c) of an 8 x 8 tile in A-fragment order
__device__ __forceinline__ int frag_pos(int r, int c) { return 8 * r + 2 * (c & 3) + (c >> 2); }

// Entry of the unconstrained stiffness matrix between interior node a and a + dl (|dl_x| <= 1) for the scalar 3-D problem
// with one coefficient per sub-cell: the sum over the (at most 8) sub-cells that contain both nodes of coefficient times
// reference-matrix entry.  Fully unrolled over the 8 sub-cells around node a with independent loads, so that one entry
// costs one shared-memory round trip, not eight; the 8 x 8 reference matrix comes from shared memory (dynamic indexing
// of __constant__ memory serialises over the distinct addresses of a warp).  a is an INTERIOR node: all 8 sub-cells
// around it exist.
__device__ __forceinline__ double stiff_entry_3d(const Geom &g, const double *sCoef, const double *sK, int n,
                                                 const int a[3], const int dl[3]) {
  const int msx = g.m[0] * n, msy = g.m[1] * n;
  double acc = 0.0;
#pragma unroll
  for (int oc = 0; oc < 8; ++oc) {
    // sub-cell origin = a - (1,1,1) + bits of oc; node a is its local vertex la = 7 - oc (bit set <=> a is the upper node)
    const int bx = oc & 1, by = (oc >> 1) & 1, bz = (oc >> 2) & 1;
    // the other node a + dl is a vertex of the same sub-cell iff dl_x in {0, bx ? +1 : -1} per axis
    const bool ok = (dl[0] == 0 || dl[0] == (bx ? 1 : -1)) && (dl[1] == 0 || dl[1] == (by ? 1 : -1)) &&
                    (dl[2] == 0 || dl[2] == (bz ? 1 : -1));
    const int ox = a[0] - 1 + bx, oy = a[1] - 1 + by, oz = a[2] - 1 + bz;
    const int la = (1 - bx) + 2 * (1 - by) + 4 * (1 - bz);
    const int lb = (1 - bx + dl[0]) + 2 * (1 - by + dl[1]) + 4 * (1 - bz + dl[2]);
    const double c = sCoef[(oz * msy + oy) * msx + ox];
    const double kv = sK[(la * 8 + lb) & 63];
    acc += ok ? c * kv : 0.0;
  }
  return acc;
}

// The tensor problem's lower-stencil entries, components 1 .. 5 (component 0 is in stw already): each one's field through
// the same one-field coefficient window and 8 x 8 reference matrix, added to the entry by the thread that wrote it.  Six
// fields in shared memory would halve k_patch_factor's occupancy; this way its shared-memory plan is the scalar one.
__device__ __forceinline__ void tensor_stencil_components(const Geom &geo, const double *__restrict__ d_coef, double *sCoef,
                                                       double *sK, const int *sRowPk, double *stw, int NBLK) {
  constexpr int nlow = 13;
  for (int f = 1; f < tensor_fields(3); ++f) {
    __syncthreads();
    load_coef<true>(geo, d_coef + (size_t)f * cP.nsub * cP.nsub * cP.nsub, sCoef);
    for (int i = threadIdx.x; i < 64; i += blockDim.x) sK[i] = cP.Kq[f][i];
    __syncthreads();
    for (int item = threadIdx.x; item < NBLK * 8 * (nlow + 1); item += blockDim.x) {
      const int i = item & 7, e = (item % (8 * (nlow + 1))) >> 3;
      const int pk = sRowPk[8 * (item / (8 * (nlow + 1))) + i];
      if (pk >= 0 || !((pk >> (16 + e)) & 1)) continue;   // padding row (keeps its identity entry) or outside the patch
      const int a[3] = {pk & 31, (pk >> 5) & 31, (pk >> 10) & 31};
      int dl[3];
      lower_offset(e, dl);
      __stcg(stw + item, __ldcg(stw + item) + stiff_entry_3d(geo, sCoef, sK, cP.n, a, dl));
    }
  }
}

// =====================================================================================================================
// k_patch_factor
// =====================================================================================================================
template <int RBMAX, int NW>
__global__ void __launch_bounds__(32 * NW, 2)
k_patch_factor(const int *__restrict__ patch_ids, int n_work, const double *__restrict__ d_coef,
               double *__restrict__ Lrec, double *__restrict__ stencil_ws, int *__restrict__ status, SplitLayout lay,
               int *work_counter) {
  constexpr int R = 8 * RBMAX;
  constexpr int LDWF = (R % 16 == 8) ? R : R + 8;  // row stride with LDWF % 16 == 8 : conflict-free C fragments
  constexpr int LDP = R + 4;                        // k-major panel copy
  constexpr int NT = 32 * NW;
  constexpr int LSTEP = RBMAX * 64;                 // doubles per step record
  constexpr int NTT = RBMAX * (RBMAX - 1) / 2;
  extern __shared__ double smem[];
  double *sCoef = smem;
  double *sWf = sCoef + lay.coef_doubles;   // [R][LDWF] circular dense window of the trailing matrix
  double *sLpT = sWf + R * LDWF;            // [8][LDP]  panel, k-major, slot rows
  double *sLinv = sLpT + 8 * LDP;           // [2][64]
  double *sK = sLinv + 2 * 64;              // [64] reference sub-cell matrix
  int *sRowPk = (int *)(sK + 64);           // [nip_max] packed node coords / mask
  int *sTileTab = sRowPk + lay.nip_max;     // [NTT] (offI | offJ << 8) of the trailing-update tiles
  int *sDOff = sTileTab + NTT;              // [16] dof offset of each lower stencil slot
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  constexpr int nlow = 13;                  // lower stencil nodes in 3-D

  for (int tt = tid; tt < NTT; tt += NT) {
    int offI = 1;
    while ((offI + 1) * offI / 2 <= tt) ++offI;
    sTileTab[tt] = offI | ((tt - offI * (offI - 1) / 2 + 1) << 8);
  }
  const bool tensor = cP.problem == kProblemTensor;
  if (!tensor)
    for (int i = tid; i < 64; i += NT) sK[i] = cP.Kref[i];

  unsigned long long table_key = ~0ull;   // shape key (geom.h) of the patch sRowPk / sDOff were built for
  __shared__ int sNextWork;
  SLOD_WORK_LOOP(w, n_work, work_counter, sNextWork) {
    fetch_work_item(w, work_counter, &sNextWork);
    const int pid = patch_ids[w];
    const Geom geo = make_geom(cP, pid);
    const int Ni = geo.Ni, bw = geo.bw, n = cP.n;
    const bool rebuild = (shape_key(geo) != table_key);
    table_key = shape_key(geo);
    const int NBLK = (Ni + 7) >> 3;
    int RB = (bw + 8 + 7) >> 3;
    if (RB > RBMAX) RB = RBMAX;  // host guarantees bw_max fits
    double *rec = Lrec + (size_t)w * lay.rec_stride;
    // lower-stencil entries of every row of this patch, 8 * (nlow + 1) per block row: computed by all threads in the
    // prologue into a per-CTA scratch in global memory (stays in L2), consumed block row by block row as the window
    // slides -- computing them on the fly in the loop put 1.2 k cycles per step on one warp
    double *stw = stencil_ws + (size_t)blockIdx.x * lay.nip_max * (nlow + 1);
    __syncthreads();
    // one coefficient field in the window (the scalar problem's only one, the tensor problem's first component)
    load_coef<true>(geo, d_coef, sCoef);
    if (tensor)
      for (int i = tid; i < 64; i += NT) sK[i] = cP.Kq[0][i];
    if (rebuild)
    for (int r = tid; r < 8 * NBLK; r += NT) {
      int pk = 0;
      if (r < Ni) {
        int a[3];
        interior_coords(geo, r, a);
        int mask = 0;
        for (int e = 0; e <= nlow; ++e) {
          int dl[3];
          lower_offset(e, dl);
          bool inside = true;
#pragma unroll
          for (int x = 0; x < 3; ++x) inside = inside && (a[x] + dl[x] >= 1 && a[x] + dl[x] <= geo.p[x] - 2);
          if (inside) mask |= 1 << e;
        }
        pk = a[0] | (a[1] << 5) | (a[2] << 10) | (mask << 16) | (1 << 31);
      }
      sRowPk[r] = pk;
    }
    if (tid <= nlow) {
      int dl[3];
      lower_offset(tid, dl);
      sDOff[tid] = dl[0] + geo.q[0] * (dl[1] + geo.q[1] * dl[2]);
    }
    __syncthreads();

    auto zero_block_row = [&](int sB) {
      for (int item = tid; item < 32 * RB; item += NT) {
        const int i = item & 7, q = item >> 3;
        *reinterpret_cast<double2 *>(sWf + (8 * sB + i) * LDWF + 2 * q) = make_double2(0.0, 0.0);
      }
    };
    // the (at most 14) lower-stencil entries of each of the 8 rows of block `blk`, computed on the fly from the
    // sub-cell coefficients: item = 8 * e + i is entry e of row i
    auto stencil_item = [&](int blk, int item) -> double {
      const int i = item & 7, e = item >> 3;
      const int pk = sRowPk[8 * blk + i];
      if (pk >= 0) return (e == 0) ? 1.0 : 0.0;       // padding row: identity (flagged through e == 0)
      if (!((pk >> (16 + e)) & 1)) return 0.0;
      const int a[3] = {pk & 31, (pk >> 5) & 31, (pk >> 10) & 31};
      int dl[3];
      lower_offset(e, dl);
      return stiff_entry_3d(geo, sCoef, sK, n, a, dl);
    };
    // ... and the scatter of one of them into block row slot sB of the window
    auto scatter_item = [&](int blk, int sB, int item, double v) {
      const int i = item & 7, e = item >> 3;
      const int r = 8 * blk + i;
      const int pk = sRowPk[r];
      if (pk < 0) {  // bit 31: a real dof row
        if (!((pk >> (16 + e)) & 1)) return;
        const int c = r + sDOff[e];
        int sb = sB - (blk - (c >> 3));
        if (sb < 0) sb += RB;
        sWf[(8 * sB + i) * LDWF + 8 * sb + (c & 7)] = v;
      } else if (e == 0) {
        sWf[(8 * sB + i) * LDWF + 8 * sB + i] = 1.0;
      }
    };

    for (int b = 0; b < RB && b < NBLK; ++b) zero_block_row(b);
    for (int item = tid; item < NBLK * 8 * (nlow + 1); item += NT)
      __stcg(stw + item, stencil_item(item / (8 * (nlow + 1)), item % (8 * (nlow + 1))));
    if (tensor) tensor_stencil_components(geo, d_coef, sCoef, sK, sRowPk, stw, NBLK);
    __syncthreads();
    for (int b = 0; b < RB && b < NBLK; ++b) {   // the first RB block rows of the window
      for (int item = tid; item < 8 * (nlow + 1); item += NT) {
        const double v = __ldcg(stw + b * 8 * (nlow + 1) + item);
        scatter_item(b, b, item, v);
      }
    }
    __syncthreads();
    int bad = 0;
    if (warp == 0) bad |= chol8_inv_reg(sWf, LDWF, lane, sLinv);
    __syncthreads();

    PHS_DECL(0, 3, 4)
    // One step = one full barrier.  Roles:
    //   warp 0        the critical chain: panel tile (k+1, k), update and factorisation of the next diagonal tile --
    //                 started at the top of the step, without waiting for the other panel tiles;
    //   warp 4, ...   (the warps that share warp 0's scheduler, here and in the co-resident CTA) stay off the fp64
    //                 pipe: record tile 0, window slide (zero + refill of the freed block row, next block staged);
    //   other warps   panel tiles 2 .. nl, a named barrier among them and warp 0 (tile 1), trailing tiles.
    constexpr int NTW = NW - NW / 4;          // panel / trailing warps
    constexpr int NBAR = 32 * (NTW + 1);      // named barrier 1: those warps (sync) + warp 0 (arrive)
    constexpr int NBAR2 = 32 * (NTW + 2);     // named barrier 2: the same warps arrive, warp 4 waits (never the other way round)
    constexpr bool kW4Tiles = (RBMAX == 13 && NTW == 6);
    constexpr int NIT = (8 * (nlow + 1) + 31) / 32;
    // warp 4: lower-stencil entries of the block entering the window at the NEXT step, fetched from the L2-resident
    // scratch one step ahead so that the load latency is never on the step's critical path
    double vnext[NIT];
#pragma unroll
    for (int j = 0; j < NIT; ++j)
      vnext[j] = (warp == 4 && RB < NBLK && lane + 32 * j < 8 * (nlow + 1)) ? __ldcg(stw + RB * 8 * (nlow + 1) + lane + 32 * j) : 0.0;
    for (int k = 0, kslot = 0; k < NBLK; ++k, kslot = (kslot + 1 == RB) ? 0 : kslot + 1) {
      PH(0)
      const int cur = k & 1;
      const double *Linv = sLinv + cur * 64;
      int nl = NBLK - 1 - k;  // live panel blocks below the diagonal block
      if (nl > RB - 1) nl = RB - 1;
      double *Ls = rec + (size_t)k * LSTEP;
      const int ntile = nl * (nl + 1) / 2;
      const double binv0 = Linv[g * 8 + t], binv1 = Linv[g * 8 + 4 + t];  // B[k][n] = Linv[n][k]
      auto panel_tile = [&](int off) {   // Lp_I = W[I, D] * Linv^T, I = k + off
        int sI = kslot + off;
        if (sI >= RB) sI -= RB;
        const double *wt = sWf + (8 * sI + g) * LDWF + 8 * kslot;
        double p0 = 0.0, p1 = 0.0;
        dmma884(p0, p1, wt[t], binv0);
        dmma884(p0, p1, wt[4 + t], binv1);
        sLpT[(2 * t) * LDP + 8 * sI + g] = p0;
        sLpT[(2 * t + 1) * LDP + 8 * sI + g] = p1;
        double *dst = Ls + 64 * off;      // element (g, 2t) and (g, 2t + 1) in fragment order
        dst[frag_pos(g, 2 * t)] = p0;
        dst[frag_pos(g, 2 * t + 1)] = p1;
      };
      // W[I, J] -= Lp_I Lp_J^T for the tiles J = jlo .. jhi of block row I = k + offI (three at a time)
      auto sweep_row = [&](int offI, int jlo, int jhi) {
        if (offI > nl) return;
        int sI = kslot + offI;
        if (sI >= RB) sI -= RB;
        const double a0 = -sLpT[t * LDP + 8 * sI + g], a1 = -sLpT[(4 + t) * LDP + 8 * sI + g];
        double *rowp = sWf + (8 * sI + g) * LDWF + 2 * t;
        for (int offJ = jlo; offJ <= jhi; offJ += 3) {
          double2 c[3];
          double b0[3], b1[3];
          int sJ[3];
#pragma unroll
          for (int u = 0; u < 3; ++u) {
            const int oj = (offJ + u <= jhi) ? offJ + u : offJ;
            sJ[u] = kslot + oj;
            if (sJ[u] >= RB) sJ[u] -= RB;
            c[u] = *reinterpret_cast<double2 *>(rowp + 8 * sJ[u]);
            b0[u] = sLpT[t * LDP + 8 * sJ[u] + g];
            b1[u] = sLpT[(4 + t) * LDP + 8 * sJ[u] + g];
          }
#pragma unroll
          for (int u = 0; u < 3; ++u) dmma884(c[u].x, c[u].y, a0, b0[u]);
#pragma unroll
          for (int u = 0; u < 3; ++u) dmma884(c[u].x, c[u].y, a1, b1[u]);
#pragma unroll
          for (int u = 0; u < 3; ++u)
            if (offJ + u <= jhi) *reinterpret_cast<double2 *>(rowp + 8 * sJ[u]) = c[u];
        }
      };
      if (warp == 0) {
        if (nl >= 1) {
          panel_tile(1);
          __syncwarp();
          asm volatile("bar.arrive 1, %0;" ::"n"(NBAR) : "memory");   // tile 1 is in sLpT
          if (kW4Tiles) asm volatile("bar.arrive 2, %0;" ::"n"(NBAR2) : "memory");
          int sI = kslot + 1;
          if (sI >= RB) sI -= RB;
          double *ct = sWf + (8 * sI + g) * LDWF + 8 * sI + 2 * t;
          double2 c = *reinterpret_cast<double2 *>(ct);
          const double a0 = -sLpT[t * LDP + 8 * sI + g], a1 = -sLpT[(4 + t) * LDP + 8 * sI + g];
          dmma884(c.x, c.y, a0, -a0);
          dmma884(c.x, c.y, a1, -a1);
          *reinterpret_cast<double2 *>(ct) = c;
          __syncwarp();
          PH(6)
          bad |= chol8_inv_reg(sWf + (8 * sI) * LDWF + 8 * sI, LDWF, lane, sLinv + (cur ^ 1) * 64);
          PH(7)
        }
      } else if ((warp & 3) == 0) {
        if (warp == 4) {
          // tile 0 of the record: Linv in fragment order
          *reinterpret_cast<double2 *>(Ls + 2 * lane) = make_double2(Linv[g * 8 + t], Linv[g * 8 + 4 + t]);
          // Block row kslot (block k) is dead: only its diagonal tile was still needed, by the factorisation of the
          // previous step, and nothing of it is read in this step.  Clear it and refill it with block k + RB from the
          // stencil scratch.
          if (k + RB < NBLK) {
            double v[NIT];
#pragma unroll
            for (int j = 0; j < NIT; ++j) {
              v[j] = vnext[j];
              vnext[j] = (k + RB + 1 < NBLK && lane + 32 * j < 8 * (nlow + 1))
                             ? __ldcg(stw + (k + RB + 1) * 8 * (nlow + 1) + lane + 32 * j) : 0.0;
            }
            for (int item = lane; item < 32 * RB; item += 32) {
              const int i = item & 7, q = item >> 3;
              *reinterpret_cast<double2 *>(sWf + (8 * kslot + i) * LDWF + 2 * q) = make_double2(0.0, 0.0);
            }
            __syncwarp();
#pragma unroll
            for (int j = 0; j < NIT; ++j)
              if (lane + 32 * j < 8 * (nlow + 1)) scatter_item(k + RB, kslot, lane + 32 * j, v[j]);
          }
          PH(8)
          if (RBMAX == 13 && NTW == 6) {
            if (nl >= 1) asm volatile("bar.sync 2, %0;" ::"n"(NBAR2) : "memory");   // the panel tiles are in sLpT
            PH(9)
            // diagonal tiles (r, r) of the rows 12 .. 7, three independent tiles at a time: W -= Lp_r Lp_r^T
#pragma unroll 1
            for (int r0 = RBMAX - 1; r0 >= RBMAX - 6; r0 -= 3) {
              double *ct[3];
              double2 c[3];
              double a0[3], a1[3];
#pragma unroll
              for (int u = 0; u < 3; ++u) {
                int sI = kslot + (r0 - u);
                if (sI >= RB) sI -= RB;
                ct[u] = sWf + (8 * sI + g) * LDWF + 8 * sI + 2 * t;
                c[u] = *reinterpret_cast<double2 *>(ct[u]);
                a0[u] = -sLpT[t * LDP + 8 * sI + g];
                a1[u] = -sLpT[(4 + t) * LDP + 8 * sI + g];
              }
#pragma unroll
              for (int u = 0; u < 3; ++u) dmma884(c[u].x, c[u].y, a0[u], -a0[u]);
#pragma unroll
              for (int u = 0; u < 3; ++u) dmma884(c[u].x, c[u].y, a1[u], -a1[u]);
#pragma unroll
              for (int u = 0; u < 3; ++u)
                if (r0 - u <= nl) *reinterpret_cast<double2 *>(ct[u]) = c[u];
            }
          }
        }
      } else {
        const int wrank = warp - 1 - (warp >> 2);  // 0 .. NTW-1
        for (int off = 2 + wrank; off <= nl; off += NTW) panel_tile(off);
        PH(1)
        if (nl >= 1 && kW4Tiles) {
          __syncwarp();
          asm volatile("bar.arrive 2, %0;" ::"n"(NBAR2) : "memory");
        }
        if (nl >= 1) asm volatile("bar.sync 1, %0;" ::"n"(NBAR) : "memory");
        PH(3)
        // Trailing tiles by block row: the pair (off, RBMAX - off) has RBMAX tiles for every off, so with RBMAX = 13 the six
        // panel warps take one pair each (the diagonal tile (1, 1) belongs to warp 0).  A warp keeps the A fragments of
        // its row and sweeps the columns three tiles at a time -- no tile table, half the operand loads.  The diagonal
        // tiles of the long rows 7 .. 12 are left to warp 4 (sweep_row below), which has the fourth scheduler's tensor
        // pipe to itself.
        if (RBMAX == 13 && NTW == 6) {
          sweep_row(1 + wrank, (wrank == 0) ? 2 : 1, 1 + wrank);
          sweep_row(RBMAX - 1 - wrank, 1, RBMAX - 2 - wrank);
        } else
        for (int tt = 1 + wrank; tt < ntile; tt += 3 * NTW) {
          double *ct[3];
          double2 c[3];
          double a0[3], a1[3], b0[3], b1[3];
#pragma unroll
          for (int u = 0; u < 3; ++u) {
            const int tu = tt + u * NTW;
            const int tab = sTileTab[tu < ntile ? tu : tt];
            const int offI = tab & 0xff, offJ = tab >> 8;
            int sI = kslot + offI, sJ = kslot + offJ;
            if (sI >= RB) sI -= RB;
            if (sJ >= RB) sJ -= RB;
            ct[u] = sWf + (8 * sI + g) * LDWF + 8 * sJ + 2 * t;
            c[u] = *reinterpret_cast<double2 *>(ct[u]);
            a0[u] = -sLpT[t * LDP + 8 * sI + g];
            a1[u] = -sLpT[(4 + t) * LDP + 8 * sI + g];
            b0[u] = sLpT[t * LDP + 8 * sJ + g];
            b1[u] = sLpT[(4 + t) * LDP + 8 * sJ + g];
          }
#pragma unroll
          for (int u = 0; u < 3; ++u) dmma884(c[u].x, c[u].y, a0[u], b0[u]);
#pragma unroll
          for (int u = 0; u < 3; ++u) dmma884(c[u].x, c[u].y, a1[u], b1[u]);
#pragma unroll
          for (int u = 0; u < 3; ++u)
            if (tt + u * NTW < ntile) *reinterpret_cast<double2 *>(ct[u]) = c[u];
        }
      }
      PH(4)
      __syncthreads();
      PH(5)
    }
    PH_PRINT("factor")
    if (bad && lane == 0) atomicOr(&status[pid], 1);
  }
}

// =====================================================================================================================
// k_patch_trisolve
// =====================================================================================================================
template <int RBMAX, int NW>
__global__ void __launch_bounds__(32 * NW, 1)
k_patch_trisolve(const int *__restrict__ patch_ids, int n_work, const double *__restrict__ Lrec,
                 double *__restrict__ Xbuf, SplitLayout lay, int *work_counter) {
  constexpr int NT = 32 * NW;
  constexpr int NC = 8 * NW;
  constexpr int LSTEP = RBMAX * 64;
  constexpr int NSTG = kTriStages;
  extern __shared__ __align__(128) double smem[];
  double *sRing = smem;                                      // [NSTG][LSTEP]
  uint64_t *sFull = reinterpret_cast<uint64_t *>(sRing + NSTG * LSTEP);   // [NSTG]
  uint64_t *sEmpty = sFull + NSTG;                            // [NSTG]
  int *sRowPk = reinterpret_cast<int *>(sEmpty + NSTG);       // [nip_max] packed node coords of each interior dof
  int *sColCell = sRowPk + lay.nip_max;                       // [NC] packed cell coords of each coarse column (or -1)
  int *sKstart = sColCell + NC;                               // [NW] first forward step of each warp
  int *sNskip = sKstart + NW;                                 // [nip_max / 8 + 1] warps that sit out forward step k; last: backward
  volatile uint32_t *sProgress = reinterpret_cast<volatile uint32_t *>(sNskip + lay.nip_max / 8 + 1);   // records issued so far
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int tpos = 8 * t + 2 * (g & 3) + (g >> 2);           // T^T fragment position, k-step 0 (+32 for k-step 1)
  // Column group (8 columns) of this warp.  With the z-major column order the groups start their forward substitution
  // at different rows (group 0-3 at row 0, 13-15 at 3/4 of the rows of a full patch); the map spreads early and late
  // groups evenly over the four schedulers (warp mod 4).
  const int grp = (NW == 16) ? (warp < 8 ? ((0x86543210u >> (4 * warp)) & 15) : ((0xCFED9BA7u >> (4 * (warp - 8))) & 15))
                             : warp;
  // The ring producer is lane 0 of the warp that owns the LAST column group: with the z-major order its forward
  // substitution starts at 3/4 of the rows (or never, on clipped patches where the group is padding), so it fills the
  // ring ahead of the others instead of adding its bookkeeping to the critical path of a full-work warp.
  const bool is_prod = (grp == NW - 1) && (lane == 0);

  if (tid == 0) {
    for (int s = 0; s < NSTG; ++s) {
      mbar_init(sFull + s, 1);
      mbar_init(sEmpty + s, NW);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    *sProgress = 0;
  }
  __syncthreads();
  uint32_t rec_base = 0;   // records consumed so far by this CTA (ring position and barrier phases follow from it)
  unsigned long long table_key = ~0ull;   // shape key (geom.h) the tables in shared memory were built for

  __shared__ int sNextWork;
  SLOD_WORK_LOOP(w, n_work, work_counter, sNextWork) {
    fetch_work_item(w, work_counter, &sNextWork);
    const int pid = patch_ids[w];
    const Geom geo = make_geom(cP, pid);
    const int Ni = geo.Ni, bw = geo.bw, ncd = geo.Ncd;
    const int NBLK = (Ni + 7) >> 3;
    int RB = (bw + 8 + 7) >> 3;
    if (RB > RBMAX) RB = RBMAX;
    double *X = Xbuf + (size_t)w * lay.x_stride;
    const double *rec = Lrec + (size_t)w * lay.rec_stride;
    const bool rebuild = (shape_key(geo) != table_key);   // block-uniform: integer tables are per shape, not per patch
    table_key = shape_key(geo);
    __syncthreads();   // the tables of the previous patch are dead
    if (rebuild)
    for (int r = tid; r < 8 * NBLK; r += NT) {
      int pk = 0;
      if (r < Ni) {
        int a[3];
        interior_coords(geo, r, a);
        pk = a[0] | (a[1] << 5) | (a[2] << 10) | (1 << 31);
      }
      sRowPk[r] = pk;
    }
    if (rebuild)
    for (int col = tid; col < NC; col += NT) {
      int v = -1;
      if (col < ncd) {
        int kc[3];
        zcol_to_cell(geo, col, kc);   // z-major internal column order (geom.h)
        v = kc[0] | (kc[1] << 5) | (kc[2] << 10);
      }
      sColCell[col] = v;
    }
    __syncthreads();
    const int mycc0 = sColCell[8 * grp + 2 * t], mycc1 = sColCell[8 * grp + 2 * t + 1];
    const int n = cP.n;
    // Block rows in which the columns of this warp have right-hand-side entries: the fine nodes of a cell with z
    // coordinate kz lie in the node planes n kz .. n kz + n.  Before the first of them the forward substitution of these
    // columns is identically zero and is skipped; outside the range the incoming right-hand-side tiles are zero.
    int kstart, kend;
    {
      int first = 1 << 30, last = -1;
      const int cc = sColCell[8 * grp + (lane & 7)];
      if (cc >= 0) {
        const int kz = (cc >> 10) & 31;
        int plo = n * kz, phi_ = n * kz + n;          // node planes of the cell
        if (plo < 1) plo = 1;
        if (phi_ > geo.p[2] - 2) phi_ = geo.p[2] - 2;  // interior planes only
        first = (plo - 1) * geo.q[0] * geo.q[1];
        last = phi_ * geo.q[0] * geo.q[1] - 1;
      }
#pragma unroll
      for (int o = 4; o > 0; o >>= 1) {
        first = min(first, __shfl_xor_sync(0xffffffffu, first, o));
        last = max(last, __shfl_xor_sync(0xffffffffu, last, o));
      }
      kstart = (last < 0) ? NBLK : first >> 3;       // last < 0: padding columns only, nothing to solve
      kend = last >> 3;
      if (lane == 0) sKstart[warp] = kstart;
    }
    __syncthreads();
    // warps that do not take part in a step do not touch the ring: the producer arrives for them (below)
    if (rebuild)
    for (int k = tid; k <= NBLK; k += NT) {
      int cnt = 0;
      for (int w2 = 0; w2 < NW; ++w2) cnt += (k < NBLK) ? (sKstart[w2] > k) : (sKstart[w2] >= NBLK);
      sNskip[k] = cnt;
    }
    __syncthreads();
    const int pw_hi = __double2hiint(cP.pw), pw_lo = __double2loint(cP.pw);
    // right-hand-side tile (C layout) of block blk for this warp's columns: P_i entries from the tables.  The weight
    // pw * 2^(number of axes on which the node is interior to the cell) is put together from the exponent bits: no
    // fp64 instruction competes with the tensor pipe.
    auto rhs_tile = [&](int blk, double &c0, double &c1) {
      if (blk < kstart || blk > kend) {
        c0 = c1 = 0.0;
        return;
      }
      const int pk = sRowPk[8 * blk + g];
      int hi[2];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int cc = h ? mycc1 : mycc0;
        bool in = (pk < 0) && (cc >= 0);
        int cnt = 0;
#pragma unroll
        for (int x = 0; x < 3; ++x) {
          const int tt = ((pk >> (5 * x)) & 31) - n * ((cc >> (5 * x)) & 31);
          in = in && (tt >= 0) && (tt <= n);
          cnt += (tt != 0 && tt != n) ? 1 : 0;
        }
        hi[h] = in ? pw_hi + (cnt << 20) : 0;
      }
      c0 = __hiloint2double(hi[0], hi[0] ? pw_lo : 0);
      c1 = __hiloint2double(hi[1], hi[1] ? pw_lo : 0);
    };

    // ---- record stream of this patch: forward steps 0 .. NBLK-1, then backward steps NBLK-1 .. 0 ----
    const int total = 2 * NBLK;
    int issued = 0;   // producer state (thread 0 only)
    auto step_of = [&](int i) { return i < NBLK ? i : 2 * NBLK - 1 - i; };
    auto top_up = [&](int upto) {   // thread 0: keep the ring filled up to record `upto` (exclusive)
      if (upto > total) upto = total;
      while (issued < upto) {
        const uint32_t r = rec_base + issued;
        const int slot = r % NSTG;
        const uint32_t use = r / NSTG;
        if (use > 0) mbar_wait(sEmpty + slot, (use - 1) & 1);   // every warp is through with the previous occupant
        const int k = step_of(issued);
        int nl = NBLK - 1 - k;
        if (nl > RB - 1) nl = RB - 1;
        const uint32_t bytes = 8u * 64u * (1 + nl);
        mbar_expect_tx(sFull + slot, bytes);
        bulk_g2s(sRing + slot * LSTEP, rec + (size_t)k * LSTEP, bytes, sFull + slot);
        const int nskip = sNskip[issued < NBLK ? k : NBLK];   // "empty" arrivals of the warps that skip this record
        if (nskip > 0) mbar_arrive_n(sEmpty + slot, nskip);
        ++issued;
        // No fence: once the wait on "empty" above has passed, the slot's "full" barrier is already in the phase of
        // this record, so a consumer that sees the new count early still blocks until the bytes have landed.
        *sProgress = rec_base + issued;
      }
    };
    if (is_prod) top_up(NSTG - 1);
    // Wait for record r in its ring slot.  The parity test of an mbarrier only tells the current phase from the one
    // before it, and a warp that sat out the earlier uses of the slot may be several phases ahead of it: the record
    // must have been ISSUED (then the slot's barrier is in the phase of this record, or past it) before the test.
    auto wait_record = [&](uint32_t r, int slot) {
      while ((int32_t)(*sProgress - r) <= 0) __nanosleep(100);
      mbar_wait(sFull + slot, (r / NSTG) & 1);
    };

    // =============================== forward substitution  L Y = P_i ===============================
    double cr[RBMAX][2];   // cr[off]: right-hand-side tile of block k + off (rotating register window)
#pragma unroll
    for (int off = 0; off < RBMAX; ++off) {
      cr[off][0] = cr[off][1] = 0.0;
      if (off < RB && kstart + off < NBLK) rhs_tile(kstart + off, cr[off][0], cr[off][1]);
    }
    PHS_DECL(0, 5, NW - 1)
    // the producer's idle steps: fill the ring as far as the consumers free it (the waits inside top_up pace it)
    if (is_prod) top_up(min(kstart, NBLK) + NSTG - 1);
    for (int k = kstart; k < NBLK; ++k) {
      PH(0)
      const uint32_t r = rec_base + k;
      const int slot = r % NSTG;
      int nl = NBLK - 1 - k;
      if (nl > RB - 1) nl = RB - 1;
      // independent of the record: the B fragments of the current right-hand-side tile, the tile entering the window
      const double b0 = c_to_b(cr[0][0], cr[0][1], lane, 0), b1 = c_to_b(cr[0][0], cr[0][1], lane, 1);
      double n0 = 0.0, n1 = 0.0;
      if (k + RB < NBLK) rhs_tile(k + RB, n0, n1);
      PH(2)
      wait_record(r, slot);
      PH(3)
      const double2 *F = reinterpret_cast<const double2 *>(sRing + slot * LSTEP);
      double y0 = 0.0, y1 = 0.0;
      {
        const double2 li = F[lane];
        dmma884(y0, y1, li.x, b0);
        dmma884(y0, y1, li.y, b1);
      }
      *reinterpret_cast<double2 *>(X + (size_t)(8 * k + g) * lay.ldx + 8 * grp + 2 * t) = make_double2(y0, y1);
      const double yb0 = -c_to_b(y0, y1, lane, 0), yb1 = -c_to_b(y0, y1, lane, 1);
      // R_{k+off} -= Lp_off Y_k with m8n8k4: the short instruction keeps the wait of the NEXT step's dependent pair of
      // Linv multiplications behind the other warps' tensor instructions short (m16n8k8 here: forward sweep 12 % slower)
#pragma unroll
      for (int o4 = 1; o4 < RBMAX; o4 += 4) {
        double2 a[4];
#pragma unroll
        for (int u = 0; u < 4; ++u)
          if (o4 + u < RBMAX && o4 + u <= nl) a[u] = F[32 * (o4 + u) + lane];
#pragma unroll
        for (int u = 0; u < 4; ++u)
          if (o4 + u < RBMAX && o4 + u <= nl) dmma884(cr[o4 + u][0], cr[o4 + u][1], a[u].x, yb0);
#pragma unroll
        for (int u = 0; u < 4; ++u)
          if (o4 + u < RBMAX && o4 + u <= nl) dmma884(cr[o4 + u][0], cr[o4 + u][1], a[u].y, yb1);
      }
      // the producer refills the ring while the tensor pipe works through the instructions just issued
      if (is_prod) top_up(k + NSTG - 1);
      PH(1)
      __syncwarp();
      if (lane == 0) mbar_arrive(sEmpty + slot);
      PH(4)
      // the register window moves up by one block
#pragma unroll
      for (int off = 0; off < RBMAX - 1; ++off) {
        cr[off][0] = (off == RB - 1) ? n0 : cr[off + 1][0];
        cr[off][1] = (off == RB - 1) ? n1 : cr[off + 1][1];
      }
      if (RB == RBMAX) { cr[RBMAX - 1][0] = n0; cr[RBMAX - 1][1] = n1; }
    }

    // =============================== backward substitution  L^T X = Y ===============================
    // xr[off]: NEGATED B fragments of the solved block k + off
    double xr[RBMAX][2];
#pragma unroll
    for (int off = 0; off < RBMAX; ++off) xr[off][0] = xr[off][1] = 0.0;
    auto y_tile = [&](int k) -> double2 {   // Y_k of the forward sweep (zero, and never stored, before kstart)
      return (k >= kstart) ? *reinterpret_cast<const double2 *>(X + (size_t)(8 * k + g) * lay.ldx + 8 * grp + 2 * t)
                           : make_double2(0.0, 0.0);
    };
    if (kstart >= NBLK) {
      // padding columns only: X = 0 (finite values for the consumers), no arithmetic, no part in the ring -- but the
      // producer keeps feeding it
      if (is_prod) top_up(total);
      for (int k = 0; k < NBLK; ++k)
        *reinterpret_cast<double2 *>(X + (size_t)(8 * k + g) * lay.ldx + 8 * grp + 2 * t) = make_double2(0.0, 0.0);
      rec_base += (uint32_t)total;
      continue;
    }
    // Two block rows per iteration (k and k - 1): X_{k+off} contributes to row k with panel tile off of step k and to
    // row k - 1 with panel tile off + 1 of step k - 1 -- one m16n8k8 with the two transposed tiles stacked as A and the X
    // block as B.  The one term of row k - 1 that needs X_k itself follows with m8n8k4.
    double2 ya = y_tile(NBLK - 1), yb = y_tile(NBLK - 2);
    for (int k = NBLK - 1; k >= 0; k -= 2) {
      PH(5)
      const bool two = (k >= 1);
      const int i = 2 * NBLK - 1 - k;   // record index of step k; step k - 1 is record i + 1
      const uint32_t r = rec_base + i;
      const int slot = r % NSTG, slot2 = (r + 1) % NSTG;
      int nl = NBLK - 1 - k;
      if (nl > RB - 1) nl = RB - 1;
      int nl2 = NBLK - k;   // live panel tiles of step k - 1
      if (nl2 > RB - 1) nl2 = RB - 1;
      const double2 yna = y_tile(k - 2), ynb = y_tile(k - 3);
      wait_record(r, slot);
      if (two) wait_record(r + 1, slot2);
      PH(7)
      const double *F = sRing + slot * LSTEP, *F2 = sRing + slot2 * LSTEP;
      double c[2][4] = {{ya.x, ya.y, yb.x, yb.y}, {0.0, 0.0, 0.0, 0.0}};   // two accumulation chains: rows k | k - 1
#pragma unroll
      for (int off = 1; off < RBMAX; ++off) {
        // A = [Lp_off(k)^T ; Lp_{off+1}(k-1)^T] : A[m][kk] = Lp[kk][m]
        const bool lo_on = (off <= nl), hi_on = two && (off + 1 <= nl2) && (off + 1 < RBMAX);
        if (lo_on || hi_on) {
          const double a0 = lo_on ? F[64 * off + tpos] : 0.0, a2 = lo_on ? F[64 * off + 32 + tpos] : 0.0;
          const double a1 = hi_on ? F2[64 * (off + 1 < RBMAX ? off + 1 : off) + tpos] : 0.0;
          const double a3 = hi_on ? F2[64 * (off + 1 < RBMAX ? off + 1 : off) + 32 + tpos] : 0.0;
          dmma1688(c[off & 1][0], c[off & 1][1], c[off & 1][2], c[off & 1][3], a0, a1, a2, a3, xr[off][0], xr[off][1]);
        }
      }
      if (is_prod) top_up(i + NSTG - 3);   // slots of the pair before the previous one: the producer never waits for a straggler
      PH(6)
      const double c0 = c[0][0] + c[1][0], c1 = c[0][1] + c[1][1];
      double p0 = c[0][2] + c[1][2], p1 = c[0][3] + c[1][3];
      PH(8)
      // X_k = Linv_k^T T
      const double tb0 = c_to_b(c0, c1, lane, 0), tb1 = c_to_b(c0, c1, lane, 1);
      double x0 = 0.0, x1 = 0.0;
      dmma884(x0, x1, F[tpos], tb0);
      dmma884(x0, x1, F[32 + tpos], tb1);
      __syncwarp();
      if (lane == 0) mbar_arrive(sEmpty + slot);
      *reinterpret_cast<double2 *>(X + (size_t)(8 * k + g) * lay.ldx + 8 * grp + 2 * t) = make_double2(x0, x1);
      const double nb0 = -c_to_b(x0, x1, lane, 0), nb1 = -c_to_b(x0, x1, lane, 1);
      double mb0 = 0.0, mb1 = 0.0;
      if (two) {
        // row k - 1: the term with X_k (panel tile 1 of step k - 1), then X_{k-1} = Linv_{k-1}^T T
        dmma884(p0, p1, F2[64 + tpos], nb0);
        dmma884(p0, p1, F2[64 + 32 + tpos], nb1);
        const double ub0 = c_to_b(p0, p1, lane, 0), ub1 = c_to_b(p0, p1, lane, 1);
        double z0 = 0.0, z1 = 0.0;
        dmma884(z0, z1, F2[tpos], ub0);
        dmma884(z0, z1, F2[32 + tpos], ub1);
        __syncwarp();
        if (lane == 0) mbar_arrive(sEmpty + slot2);
        *reinterpret_cast<double2 *>(X + (size_t)(8 * (k - 1) + g) * lay.ldx + 8 * grp + 2 * t) = make_double2(z0, z1);
        mb0 = -c_to_b(z0, z1, lane, 0);
        mb1 = -c_to_b(z0, z1, lane, 1);
      }
      // the register window moves down by two block rows
#pragma unroll
      for (int off = RBMAX - 1; off >= 3; --off) { xr[off][0] = xr[off - 2][0]; xr[off][1] = xr[off - 2][1]; }
      if (RBMAX > 2) { xr[2][0] = nb0; xr[2][1] = nb1; }
      xr[1][0] = mb0;
      xr[1][1] = mb1;
      ya = yna;
      yb = ynb;
      PH(9)
    }
    PH_PRINT("trisolve")
    rec_base += (uint32_t)total;
  }
}

}  // namespace slod
