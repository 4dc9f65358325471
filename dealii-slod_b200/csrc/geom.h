// Patch geometry and matrix-free operator entries shared by host and device code.
//
// Everything a patch needs is derived from its id: the reference builds a Triangulation, two
// DoFHandlers, a sparsity pattern and four index vectors per patch (source/LOD.cc:365-431,
// :770-858, include/LODtools.h:334-375); on a structured unit-cube mesh all of that is closed-form
// index arithmetic, evaluated on the fly inside the kernels.
#pragma once
#include <cstdint>

#if defined(__CUDACC__)
#define SLOD_HD __host__ __device__ __forceinline__
#else
#define SLOD_HD inline
#endif

namespace slod {

constexpr int kMaxLocal = 8;  // (2^dim * spacedim) <= 8 : 2-D elasticity, 3-D diffusion
constexpr int kProblemTensor = 2;   // SLOD_PROBLEM_DIFFUSION_TENSOR (include/slod.h)

// coefficient fields of the tensor problem: the components of a symmetric dim x dim tensor in Voigt order
SLOD_HD int tensor_fields(int dim) { return dim * (dim + 1) / 2; }

struct Params {
  int dim, s, ref, n, ell, N;  // N = 2^ref coarse cells per axis
  int nsub;                    // N * n fine sub-cells per axis
  int problem, stabilize, quirk_presaved;
  int pmax;                    // n * (2 ell + 1) + 1 nodes per axis of a full patch
  int nnodes_max;              // pmax^dim
  int NfMax, NiMax, NcdMax;    // strides of the per-patch arrays
  int w;                       // 2 ell + 1 : |neighbour offset| <= w shares a fine node
  int ell_width;               // (2w+1)^dim * s
  int presaved_lo[3];          // quirk B: coefficient window of the first full-size patch
  int has_presaved;
  double H, h, Hd, pw;         // pw = h^dim / 2^dim (projection weight), Hd = H^dim
  // reference sub-cell matrices, local dof = s * (lx + 2 ly + 4 lz) + comp
  double Kref[kMaxLocal * kMaxLocal];   // diffusion: Laplace * h^(d-2);  elasticity: 2 eps:eps
  double Klam[kMaxLocal * kMaxLocal];   // elasticity: div div
  // coefficient finer than the sub-cells (eta < h, e.g. tests/Poisson_LOD_Example): one value per Gauss
  // point of QIterated(QGauss<1>(2), n) and the per-Gauss-point matrices (q = qx + 2 qy + 4 qz).
  // Tensor problem (never per Gauss point): Kq[f] is the matrix of Voigt component f, whose coefficient is field f.
  int gauss_coef;
  double Kq[kMaxLocal][kMaxLocal * kMaxLocal];
  double Klamq[kMaxLocal][kMaxLocal * kMaxLocal];
};

struct Geom {
  int lo[3], m[3], p[3], q[3], cc[3], clo[3];
  int domlo[3], domhi[3];
  int nnodes, Nf, Ni, Nc, Ncd, bw, tc;
  int full, slod;
};

SLOD_HD void morton_decode(uint32_t code, int dim, int ref, int idx[3]) {
  idx[0] = idx[1] = idx[2] = 0;
  for (int b = 0; b < ref; ++b)
    for (int a = 0; a < dim; ++a) idx[a] |= ((code >> (dim * b + a)) & 1u) << b;
}
SLOD_HD uint32_t morton_encode(const int idx[3], int dim, int ref) {
  uint32_t code = 0;
  for (int b = 0; b < ref; ++b)
    for (int a = 0; a < dim; ++a) code |= (uint32_t)((idx[a] >> b) & 1) << (dim * b + a);
  return code;
}

// patch geometry from the coordinates of its centre cell
SLOD_HD Geom make_geom_at(const Params &P, const int c[3]) {
  Geom g;
  g.full = 1;
  g.Nc = 1;
  g.nnodes = 1;
  int ni = 1;
  for (int a = 0; a < 3; ++a) {
    if (a < P.dim) {
      int lo = c[a] - P.ell;
      if (lo < 0) lo = 0;
      int hi = c[a] + P.ell;
      if (hi > P.N - 1) hi = P.N - 1;
      g.lo[a] = lo;
      g.m[a] = hi - lo + 1;
      g.p[a] = g.m[a] * P.n + 1;
      g.q[a] = g.p[a] - 2;
      g.cc[a] = c[a] - lo;
      g.domlo[a] = (lo == 0);
      g.domhi[a] = (hi == P.N - 1);
      if (g.m[a] != 2 * P.ell + 1) g.full = 0;
    } else {
      g.lo[a] = 0; g.m[a] = 1; g.p[a] = 1; g.q[a] = 1; g.cc[a] = 0; g.domlo[a] = 0; g.domhi[a] = 0;
    }
    g.Nc *= g.m[a];
    g.nnodes *= g.p[a];
    ni *= g.q[a];
  }
  g.Nf = P.s * g.nnodes;
  g.Ni = P.s * ni;
  g.Ncd = P.s * g.Nc;
  // lexicographic half bandwidth of A_ii (interior nodes x fastest, component fastest of all)
  int nb = (P.dim == 3) ? (g.q[0] * g.q[1] + g.q[0] + 1) : (g.q[0] + 1);
  g.bw = P.s * nb + (P.s - 1);
  if (g.bw > g.Ni - 1) g.bw = g.Ni - 1;
  // position of the centre cell in the x-outer sweep (source/LOD.cc:156-178)
  g.tc = (P.dim == 3) ? ((g.cc[0] * g.m[1] + g.cc[1]) * g.m[2] + g.cc[2]) : (g.cc[0] * g.m[1] + g.cc[1]);
  // source/LOD.cc:563-564
  int total = 1;
  for (int a = 0; a < P.dim; ++a) total *= P.N;
  g.slod = (P.stabilize && P.ell > 0 && g.Nc != total) ? 1 : 0;
  for (int a = 0; a < 3; ++a) g.clo[a] = g.lo[a];
  if (P.quirk_presaved && g.full && P.has_presaved)
    for (int a = 0; a < 3; ++a) g.clo[a] = P.presaved_lo[a];
  return g;
}
SLOD_HD Geom make_geom(const Params &P, int pid) {
  int c[3];
  morton_decode((uint32_t)pid, P.dim, P.ref, c);
  return make_geom_at(P, c);
}

// Everything integer about a patch (index tables, boundary lists, column order) depends only on its per-axis extents,
// the position of the centre cell and which sides lie on the domain boundary: patches with the same key share it.
// The work lists are sorted by cost, so a persistent CTA sees long runs of equal keys and rebuilds its tables rarely.
SLOD_HD unsigned long long shape_key(const Geom &g) {
  unsigned long long k = 0;
  for (int a = 0; a < 3; ++a)
    k = (k << 20) | (unsigned long long)((g.m[a] << 10) | (g.cc[a] << 2) | (g.domlo[a] << 1) | g.domhi[a]);   // m, cc < 256
  return k;
}

// list position (coarse column / spacedim) of patch cell k (relative coordinates)
SLOD_HD int cell_to_col(const Params &P, const Geom &g, const int k[3]) {
  int t = (P.dim == 3) ? ((k[0] * g.m[1] + k[1]) * g.m[2] + k[2]) : (k[0] * g.m[1] + k[1]);
  return t == g.tc ? 0 : (t < g.tc ? t + 1 : t);
}
SLOD_HD void col_to_cell(const Params &P, const Geom &g, int pos, int k[3]) {
  int t = (pos == 0) ? g.tc : (pos <= g.tc ? pos - 1 : pos);
  if (P.dim == 3) {
    k[2] = t % g.m[2];
    t /= g.m[2];
    k[1] = t % g.m[1];
    k[0] = t / g.m[1];
  } else {
    k[1] = t % g.m[1];
    k[0] = t / g.m[1];
    k[2] = 0;
  }
}

// Internal column order of the split solver path (3-D): the centre cell first (the selection addresses it as column 0,
// like the reference order does), then the other cells sorted by their z coordinate (x outer, y inner inside a z
// layer).  A coarse column is nonzero in P_i only on the fine nodes of its cell, so with this order the 8 columns a
// warp of the triangular solver owns start at about the same row of the forward substitution and everything above is
// skipped.  X, W, M^-1, G and c use it consistently between the solver and k_patch_finish; nothing the C ABI returns
// is in this order (slod_debug_patch_stages permutes back).
SLOD_HD int zcell_to_col(const Geom &g, const int k[3]) {
  const int t = (k[2] * g.m[0] + k[0]) * g.m[1] + k[1];
  const int tcz = (g.cc[2] * g.m[0] + g.cc[0]) * g.m[1] + g.cc[1];
  return t == tcz ? 0 : (t < tcz ? t + 1 : t);
}
SLOD_HD void zcol_to_cell(const Geom &g, int pos, int k[3]) {
  const int tcz = (g.cc[2] * g.m[0] + g.cc[0]) * g.m[1] + g.cc[1];
  int t = (pos == 0) ? tcz : (pos <= tcz ? pos - 1 : pos);
  k[1] = t % g.m[1];
  t /= g.m[1];
  k[0] = t % g.m[0];
  k[2] = t / g.m[0];
}

SLOD_HD void node_coords(const Geom &g, int node, int a[3]) {
  a[0] = node % g.p[0];
  node /= g.p[0];
  a[1] = node % g.p[1];
  a[2] = node / g.p[1];
}
SLOD_HD int node_index(const Geom &g, const int a[3]) { return (a[2] * g.p[1] + a[1]) * g.p[0] + a[0]; }
SLOD_HD void interior_coords(const Geom &g, int idx, int a[3]) {
  a[0] = idx % g.q[0] + 1;
  idx /= g.q[0];
  a[1] = idx % g.q[1] + 1;
  a[2] = (g.p[2] > 1) ? (idx / g.q[1] + 1) : 0;
}
SLOD_HD int interior_index(const Geom &g, const int a[3]) {
  int z = (g.p[2] > 1) ? (a[2] - 1) : 0;
  return (z * g.q[1] + (a[1] - 1)) * g.q[0] + (a[0] - 1);
}
// node classes (source/LOD.cc:830-843 + include/LODtools.h:355-373); bit0 = patch boundary (id 99),
// bit1 = domain boundary (id 0); 0 = internal.  Both bits may be set.
SLOD_HD int node_class(const Params &P, const Geom &g, const int a[3]) {
  int cls = 0;
  _Pragma("unroll") for (int x = 0; x < 3; ++x) if (x < P.dim) {
    if (a[x] == 0) cls |= g.domlo[x] ? 2 : 1;
    if (a[x] == g.p[x] - 1) cls |= g.domhi[x] ? 2 : 1;
  }
  return cls;
}

// P^T entry for fine dof (node a, comp ca) and coarse column col (source/LOD.cc:329-342, 470-496).
SLOD_HD double proj_entry(const Params &P, const Geom &g, const int a[3], int ca, int col) {
  if (col % P.s != ca) return 0.0;
  int k[3];
  col_to_cell(P, g, col / P.s, k);
  double wgt = P.pw;
  _Pragma("unroll") for (int x = 0; x < 3; ++x) if (x < P.dim) {
    int t = a[x] - P.n * k[x];
    if (t < 0 || t > P.n) return 0.0;
    if (t != 0 && t != P.n) wgt *= 2.0;
  }
  return wgt;
}

// Entry idx of the tensor problem's matrix of sub-cell sc: the sum over the Voigt components
template <typename CoefT>
SLOD_HD double tensor_subcell_entry(const Params &P, const CoefT *coef, int nsubp, int sc, int idx) {
  double acc = 0.0;
  for (int f = 0; f < tensor_fields(P.dim); ++f) acc += (double)coef[f * nsubp + sc] * P.Kq[f][idx];
  return acc;
}

// Entry of the unconstrained patch stiffness matrix between (node a, comp ca) and (node a+dl, comp cb)
// (include/Diffusion.h:143-193 / include/Elasticity.h:211-284 summed over the sub-cells containing both
// nodes).  `coef` holds the patch's sub-cell coefficients, field-major, x fastest.
template <typename CoefT>
SLOD_HD double stiff_entry(const Params &P, const Geom &g, const CoefT *coef, const int a[3], const int dl[3],
                           int ca, int cb) {
  int o0[3], o1[3];
  int msub[3];
  for (int x = 0; x < 3; ++x) {
    msub[x] = (x < P.dim) ? g.m[x] * P.n : 1;
    if (x >= P.dim) { o0[x] = 0; o1[x] = 0; continue; }
    int lo_o = (dl[x] == 1) ? a[x] : a[x] - 1;
    int hi_o = (dl[x] == -1) ? a[x] - 1 : a[x];
    if (lo_o < 0) lo_o = 0;
    if (hi_o > msub[x] - 1) hi_o = msub[x] - 1;
    o0[x] = lo_o; o1[x] = hi_o;
  }
  const int nsubp = msub[0] * msub[1] * msub[2];
  const int nl = (1 << P.dim) * P.s;
  double acc = 0.0;
  for (int oz = o0[2]; oz <= o1[2]; ++oz)
    for (int oy = o0[1]; oy <= o1[1]; ++oy)
      for (int ox = o0[0]; ox <= o1[0]; ++ox) {
        const int sc = (oz * msub[1] + oy) * msub[0] + ox;
        const int la = (a[0] - ox) + 2 * (a[1] - oy) + ((P.dim == 3) ? 4 * (a[2] - oz) : 0);
        const int lb = (a[0] + dl[0] - ox) + 2 * (a[1] + dl[1] - oy) + ((P.dim == 3) ? 4 * (a[2] + dl[2] - oz) : 0);
        const int idx = (la * P.s + ca) * nl + (lb * P.s + cb);
        if (P.problem == kProblemTensor) {
          acc += tensor_subcell_entry(P, coef, nsubp, sc, idx);
        } else if (!P.gauss_coef) {
          if (P.problem == 0)
            acc += (double)coef[sc] * P.Kref[idx];
          else
            acc += (double)coef[nsubp + sc] * P.Kref[idx] + (double)coef[sc] * P.Klam[idx];
        } else {
          const int nq = 1 << P.dim;
          for (int q = 0; q < nq; ++q) {
            if (P.problem == 0)
              acc += (double)coef[sc * nq + q] * P.Kq[q][idx];
            else
              acc += (double)coef[(nsubp + sc) * nq + q] * P.Kq[q][idx] + (double)coef[sc * nq + q] * P.Klamq[q][idx];
          }
        }
      }
  return acc;
}

}  // namespace slod
