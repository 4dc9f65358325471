// C ABI (include/slod.h) and host-side orchestration of the batched patch kernels.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>   // types only: libnccl.so.2 is loaded with dlopen on the first multi-GPU call

#include <algorithm>
#include <array>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <numeric>
#include <string>
#include <thread>
#include <vector>

#include "../../include/slod.h"
#include "geom.h"
#include "kernels.h"

using namespace slod;

namespace {

std::string g_create_error;

struct Timings {
  double ms[8] = {0, 0, 0, 0, 0, 0, 0, 0};
};

}  // namespace

struct slod_ctx {
  slod_params par{};
  Params P{};
  int device = 0;
  int n_sm = 148;
  int64_t n_patches = 0;
  int n_fields = 1;                   // 1 diffusion, 2 elasticity, dim (dim + 1) / 2 tensor diffusion
  static constexpr int kMaxFields = 6;
  bool coef_set[kMaxFields] = {};
  std::vector<double> coef_table[kMaxFields];  // caller's cell-wise tables
  int coef_r[kMaxFields] = {};
  bool coef_dirty = true;
  double *d_coef = nullptr;  // [n_fields][nsub^dim]
  size_t d_coef_elems = 0;
  size_t coef_field_elems = 0;
  // results owned by the handle (host-buffer API)
  double *d_phi = nullptr, *d_aphi = nullptr, *d_Kell = nullptr, *d_diag = nullptr;
  int *d_status = nullptr;
  int *d_counter = nullptr;
  int *d_work_counter = nullptr;   // next work item of the persistent solver / flux / dense kernels
  bool basis_done = false, coarse_done = false;
  // chunk workspaces
  int chunk = 0;
  bool chunk_limited = false;
  int64_t ids_cap = 0;   // capacity of d_ids (patches of one range)
  int *d_ids = nullptr;
  double *d_X = nullptr, *d_Minv = nullptr, *d_G = nullptr, *d_cvec = nullptr, *d_Lws = nullptr, *d_W = nullptr, *d_coefws = nullptr;
  double *d_coefws_finish = nullptr;
  bool finish_coef_gmem = false;  // k_patch_finish keeps the patch coefficients in a global scratch (very large patches)
  FluxLayout xl{};
  size_t smem_flux = 0;
  int grid_flux = 0;
  int solve_grid = 0;
  int dense_ntile = 0;   // 0: generic SIMT dense stage, else tensor-core variant
  int mma_variant = -1;  // -1: generic SIMT solver, else tensor-core solver variant
  bool dense_coef_gmem = false;   // SIMT dense kernel keeps the patch coefficients in a global scratch (very large patches)
  int mma_threads = 0;
  int mma_nip = 0, mma_stw = 0;
  bool split_solver = false;      // factor + triangular-solve kernels instead of the fused solver (large 3-D patches)
  size_t smem_factor = 0, smem_tri = 0;
  int split_coef_doubles = 0;     // coefficient window of k_patch_factor: one field
  double *d_Lrec = nullptr;       // factor records of a chunk
  double *d_stw = nullptr;        // per-CTA stencil scratch of k_patch_factor
  cudaEvent_t ev_split = nullptr;
  float split_factor_ms = 0;
  long long mma_lws_per_cta = 0;
  SolveLayout sl{};
  DenseLayout dl{};
  SelectPlan sp{};
  SelectBuffers sb{};
  FinishLayout fl{};
  size_t smem_solve = 0, smem_dense = 0, smem_finish = 0, smem_coarse = 0, smem_coarse_blk = 0;
  int coarse_nu = 0;   // > 0: blocked coarse kernel with this common-box width
  int grid_solve = 0, grid_dense = 0, grid_finish = 0, grid_coarse = 0;
  int bw_max = 0, nb_max = 0;
  cudaEvent_t ev[12]{};   // [8]..[10]: the coarse mass matrix (slod_get_timings [6], [7])
  std::vector<cudaEvent_t> chunk_ev;   // 5 per chunk of the last run_basis
  size_t chunks_pending = 0;
  bool basis_pending = false;
  int64_t pending_p0 = 0, pending_p1 = 0;
  int *h_status = nullptr;   // page-locked copy of d_status
  Timings tm;
  int64_t launches = 0;
  std::vector<int> ids;   // cost-sorted work list of the last patch range
  int64_t ids_p0 = -1, ids_p1 = -1;
  mutable std::string err;
  // host caches
  mutable std::vector<int64_t> fine_numbering;  // global node -> deal.II dof of comp 0
  // CSR pattern of the coarse matrix (integer geometry: built once per handle) and the compacted values
  bool csr_ready = false;
  std::vector<int64_t> csr_rowptr, csr_col;
  long long *d_perm = nullptr;   // CSR entry -> position in the block-ELL array
  cudaStream_t copy_stream = nullptr;   // non-blocking: result read-back overlaps the coarse-matrix kernels
  bool coarse_timing_pending = false;
  double *d_online = nullptr;    // scratch of the online / fine-problem entry points, allocated on first use
  size_t online_doubles = 0;
  double *d_batch = nullptr;     // scratch of the batched online entry points (one group of kBatch columns)
  size_t batch_doubles = 0;
  double *d_val = nullptr;
  int64_t csr_nnz = 0;
  // heat equation on the SLOD space: M_H in block-ELL form and its CSR values, S = M_H + c K for the coefficient c of K
  // last formed (s_coef == 0: not formed), and the scratch of the time steppers
  double *d_Mell = nullptr, *d_Mval = nullptr, *d_Sell = nullptr;
  bool mass_done = false;
  double s_coef = 0.0;
  double *d_heat = nullptr;
  size_t heat_doubles = 0;
  // multi-GPU: (a) n_gpus > 1: this handle is rank 0 and owns one sub-handle per further device; (b) slod_comm_init
  std::vector<slod_ctx *> subs;   // sub-handles of ranks 1 .. n_gpus-1 (owned)
  ncclComm_t comm = nullptr;
  int comm_rank = 0, comm_world = 1;
  double *h_out_phi = nullptr, *h_out_aphi = nullptr, *h_out_K = nullptr;   // slod_set_host_outputs
  cudaEvent_t ev_out[2]{};       // basis rows ready | coarse rows ready
  bool out_pending = false;
  // slod_update_basis: the device coefficient array the handle's basis was computed from (its baseline), and whether
  // d_Kell holds the coarse matrix of that basis
  double *d_coef_base = nullptr;
  size_t base_elems = 0;
  int base_gauss = 0;
  bool have_base = false, base_coarse = false;
  unsigned char *d_cell_changed = nullptr;   // [n_patches]: one flag per coarse cell
  int *d_rows = nullptr;                     // coarse rows (patches or Morton groups) to recompute
  size_t rows_cap = 0;
  std::vector<int> update_ids, update_rows;
};

namespace {

int fail(const slod_ctx *c, int code, const std::string &msg) {
  if (c) c->err = msg;
  return code;
}
#define NEED_DEVICE()                                                                               \
  do {                                                                                             \
    if (ctx->device == SLOD_DEVICE_NONE)                                                           \
      return fail(ctx, SLOD_ERR_CUDA, "handle was created without a device (maps only); no CPU fallback"); \
  } while (0)
#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e__ = (call);                                                                      \
    if (e__ != cudaSuccess)                                                                        \
      return fail(ctx, SLOD_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));        \
  } while (0)


// ---- the kernels' parameter block ----------------------------------------------------------------------------------
// The kernels read one __constant__ Params block per device.  A call that launches kernels binds the handle's block for
// its scope: the device's binding mutex is held (calls of different handles on one device enqueue one after the other,
// never interleaved), the block is uploaded on the call's stream only if the resident bytes differ, and such an upload
// first waits for the last kernels that were enqueued under the previous contents (an event recorded when a binding
// ends).  Several handles with different parameters can therefore share a device and compute from different host
// threads and streams; handles with equal parameters never cause an upload.
struct DeviceParams {
  std::recursive_mutex mu;   // recursive: an entry point may call another one that binds again
  bool valid = false;
  Params resident;
  cudaEvent_t busy = nullptr;
};
DeviceParams &device_params(int device) {
  static DeviceParams table[64];
  return table[(device >= 0 && device < 64) ? device : 0];
}
struct ParamBinding {
  DeviceParams &dp;
  cudaStream_t st;
  cudaError_t err = cudaSuccess;
  ParamBinding(const slod_ctx *ctx, cudaStream_t stream) : dp(device_params(ctx->device)), st(stream) {
    dp.mu.lock();
    if (dp.valid && std::memcmp(&dp.resident, &ctx->P, sizeof(Params)) == 0) return;
    dp.valid = false;
    if (dp.busy && (err = cudaStreamWaitEvent(st, dp.busy, 0)) != cudaSuccess) return;
    if ((err = upload_params(ctx->P, st)) != cudaSuccess) return;
    std::memcpy(&dp.resident, &ctx->P, sizeof(Params));
    dp.valid = true;
  }
  ~ParamBinding() {
    if (!dp.busy) cudaEventCreateWithFlags(&dp.busy, cudaEventDisableTiming);
    if (dp.busy) cudaEventRecord(dp.busy, st);
    dp.mu.unlock();
  }
  ParamBinding(const ParamBinding &) = delete;
  ParamBinding &operator=(const ParamBinding &) = delete;
};
#define BIND_PARAMS(stream)            \
  ParamBinding bound__(ctx, (stream)); \
  CK(bound__.err)

// ---- NCCL, loaded on demand ---------------------------------------------------------------------------------------
struct NcclApi {
  void *lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommInitAll)(ncclComm_t *, int, const int *) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*CommAbort)(ncclComm_t) = nullptr;
  ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Broadcast)(const void *, void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  const char *(*GetErrorString)(ncclResult_t) = nullptr;
  std::string err;
};
NcclApi *nccl_api() {
  static NcclApi api;
  static std::once_flag once;
  std::call_once(once, []() {
    for (const char *name : {"libnccl.so.2", "libnccl.so"}) {
      api.lib = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
      if (api.lib) break;
    }
    if (!api.lib) {
      api.err = std::string("cannot load libnccl.so.2: ") + dlerror();
      return;
    }
    auto sym = [&](const char *n) {
      void *p = dlsym(api.lib, n);
      if (!p) api.err = std::string("libnccl misses ") + n;
      return p;
    };
    api.GetUniqueId = (decltype(api.GetUniqueId))sym("ncclGetUniqueId");
    api.CommInitRank = (decltype(api.CommInitRank))sym("ncclCommInitRank");
    api.CommInitAll = (decltype(api.CommInitAll))sym("ncclCommInitAll");
    api.CommDestroy = (decltype(api.CommDestroy))sym("ncclCommDestroy");
    api.CommAbort = (decltype(api.CommAbort))sym("ncclCommAbort");
    api.AllGather = (decltype(api.AllGather))sym("ncclAllGather");
    api.Broadcast = (decltype(api.Broadcast))sym("ncclBroadcast");
    api.GroupStart = (decltype(api.GroupStart))sym("ncclGroupStart");
    api.GroupEnd = (decltype(api.GroupEnd))sym("ncclGroupEnd");
    api.GetErrorString = (decltype(api.GetErrorString))sym("ncclGetErrorString");
  });
  return &api;
}
#define NK(call)                                                                                   \
  do {                                                                                             \
    ncclResult_t r__ = (call);                                                                     \
    if (r__ != ncclSuccess)                                                                        \
      return fail(ctx, SLOD_ERR_CUDA, std::string(#call) + ": " + nccl_api()->GetErrorString(r__)); \
  } while (0)

void owned_range(int64_t n, int rank, int world, int64_t *b, int64_t *e) {
  const int64_t base = n / world, rem = n % world;
  *b = rank * base + std::min<int64_t>(rank, rem);
  *e = *b + base + (rank < rem ? 1 : 0);
}

// In-place all-gather of the row blocks of `buf` ([n_patches * rows][row_doubles]): rank r contributes the rows of its
// patch range.  Equal ranges: one ncclAllGather; ragged ranges: one broadcast per rank in a group (the blocks are
// disjoint, nothing is reduced).
int gather_blocks(slod_ctx *ctx, double *buf, size_t doubles_per_patch, cudaStream_t st) {
  NcclApi *nc = nccl_api();
  const int W = ctx->comm_world;
  int64_t b, e;
  owned_range(ctx->n_patches, ctx->comm_rank, W, &b, &e);
  if (ctx->n_patches % W == 0) {
    NK(nc->AllGather(buf + (size_t)b * doubles_per_patch, buf, (size_t)(e - b) * doubles_per_patch, ncclDouble, ctx->comm, st));
  } else {
    NK(nc->GroupStart());
    for (int r = 0; r < W; ++r) {
      int64_t rb, re;
      owned_range(ctx->n_patches, r, W, &rb, &re);
      if (re > rb)
        NK(nc->Broadcast(buf + (size_t)rb * doubles_per_patch, buf + (size_t)rb * doubles_per_patch,
                         (size_t)(re - rb) * doubles_per_patch, ncclDouble, r, ctx->comm, st));
    }
    NK(nc->GroupEnd());
  }
  return SLOD_OK;
}

int ipow(int b, int e) {
  int r = 1;
  for (int i = 0; i < e; ++i) r *= b;
  return r;
}

// Voigt order of the tensor components: 2-D a_xx, a_yy, a_xy; 3-D a_xx, a_yy, a_zz, a_yz, a_xz, a_xy
constexpr int kVoigt[2][6][2] = {{{0, 0}, {1, 1}, {0, 1}}, {{0, 0}, {1, 1}, {2, 2}, {1, 2}, {0, 2}, {0, 1}}};

// Reference sub-cell matrices with the 2-point Gauss rule per axis (QIterated(QGauss<1>(2), n),
// source/LOD.cc:91-92); local dof = s * (lx + 2 ly + 4 lz) + comp.
void reference_matrices(Params &P) {
  const int dim = P.dim, s = P.s, nn = 1 << dim, nl = nn * s;
  const double h = P.h, g = 0.5 / std::sqrt(3.0);
  const double pts[2] = {0.5 - g, 0.5 + g};
  const double jxw = std::pow(h / 2.0, dim);
  std::fill(P.Kref, P.Kref + kMaxLocal * kMaxLocal, 0.0);
  std::fill(P.Klam, P.Klam + kMaxLocal * kMaxLocal, 0.0);
  std::memset(P.Kq, 0, sizeof(P.Kq));
  std::memset(P.Klamq, 0, sizeof(P.Klamq));
  for (int q = 0; q < nn; ++q) {
    double x[3] = {pts[q & 1], pts[(q >> 1) & 1], pts[(q >> 2) & 1]};
    double G[8][3];
    for (int i = 0; i < nn; ++i) {
      int nd[3] = {i & 1, (i >> 1) & 1, (i >> 2) & 1};
      for (int a = 0; a < dim; ++a) {
        double v = 1.0;
        for (int b = 0; b < dim; ++b) {
          if (b == a) v *= (nd[b] ? 1.0 : -1.0) / h;
          else v *= nd[b] ? x[b] : (1.0 - x[b]);
        }
        G[i][a] = v;
      }
    }
    if (P.problem == SLOD_PROBLEM_DIFFUSION) {
      for (int i = 0; i < nn; ++i)
        for (int j = 0; j < nn; ++j) {
          double d = 0;
          for (int a = 0; a < dim; ++a) d += G[i][a] * G[j][a];
          P.Kref[i * nl + j] += d * jxw;
          P.Kq[q][i * nl + j] = d * jxw;
        }
    } else if (P.problem == SLOD_PROBLEM_DIFFUSION_TENSOR) {
      // Kq[f]: the matrix of Voigt component f = (a, b), d_a phi_i d_b phi_j (+ d_b phi_i d_a phi_j for a != b)
      for (int f = 0; f < tensor_fields(dim); ++f) {
        const int a = kVoigt[dim - 2][f][0], b = kVoigt[dim - 2][f][1];
        for (int i = 0; i < nn; ++i)
          for (int j = 0; j < nn; ++j)
            P.Kq[f][i * nl + j] += (a == b ? G[i][a] * G[j][a] : G[i][a] * G[j][b] + G[i][b] * G[j][a]) * jxw;
      }
    } else {
      // 2 eps(phi_i):eps(phi_j) and div phi_i div phi_j   (include/Elasticity.h:236-250)
      for (int i = 0; i < nn; ++i)
        for (int ci = 0; ci < s; ++ci)
          for (int j = 0; j < nn; ++j)
            for (int cj = 0; cj < s; ++cj) {
              double ee = 0.0;
              for (int a = 0; a < dim; ++a)
                for (int b = 0; b < dim; ++b) {
                  const double ei = 0.5 * ((a == ci ? G[i][b] : 0.0) + (b == ci ? G[i][a] : 0.0));
                  const double ej = 0.5 * ((a == cj ? G[j][b] : 0.0) + (b == cj ? G[j][a] : 0.0));
                  ee += ei * ej;
                }
              P.Kref[(i * s + ci) * nl + (j * s + cj)] += 2.0 * ee * jxw;
              P.Klam[(i * s + ci) * nl + (j * s + cj)] += G[i][ci] * G[j][cj] * jxw;
              P.Kq[q][(i * s + ci) * nl + (j * s + cj)] = 2.0 * ee * jxw;
              P.Klamq[q][(i * s + ci) * nl + (j * s + cj)] = G[i][ci] * G[j][cj] * jxw;
            }
    }
  }
}

// cell-local node multi-indices in deal.II's hierarchical order (vertices, lines, quads, interior)
std::vector<std::array<int, 3>> cell_walk(int dim, int n) {
  std::vector<std::array<int, 3>> out;
  const int e[2] = {0, n};
  if (dim == 2) {
    for (int v = 0; v < 4; ++v) out.push_back({e[v & 1], e[(v >> 1) & 1], 0});
    for (int t = 1; t < n; ++t) out.push_back({0, t, 0});
    for (int t = 1; t < n; ++t) out.push_back({n, t, 0});
    for (int t = 1; t < n; ++t) out.push_back({t, 0, 0});
    for (int t = 1; t < n; ++t) out.push_back({t, n, 0});
    for (int y = 1; y < n; ++y)
      for (int x = 1; x < n; ++x) out.push_back({x, y, 0});
  } else {
    for (int v = 0; v < 8; ++v) out.push_back({e[v & 1], e[(v >> 1) & 1], e[(v >> 2) & 1]});
    for (int z = 0; z < 2; ++z) {
      for (int t = 1; t < n; ++t) out.push_back({0, t, e[z]});
      for (int t = 1; t < n; ++t) out.push_back({n, t, e[z]});
      for (int t = 1; t < n; ++t) out.push_back({t, 0, e[z]});
      for (int t = 1; t < n; ++t) out.push_back({t, n, e[z]});
    }
    for (int v = 0; v < 4; ++v)
      for (int t = 1; t < n; ++t) out.push_back({e[v & 1], e[(v >> 1) & 1], t});
    for (int f = 0; f < 2; ++f)  // x = 0, x = 1 : free axes y (fast), z
      for (int z = 1; z < n; ++z)
        for (int y = 1; y < n; ++y) out.push_back({e[f], y, z});
    for (int f = 0; f < 2; ++f)  // y faces: free axes x (fast), z
      for (int z = 1; z < n; ++z)
        for (int x = 1; x < n; ++x) out.push_back({x, e[f], z});
    for (int f = 0; f < 2; ++f)  // z faces: free axes x (fast), y
      for (int y = 1; y < n; ++y)
        for (int x = 1; x < n; ++x) out.push_back({x, y, e[f]});
    for (int z = 1; z < n; ++z)
      for (int y = 1; y < n; ++y)
        for (int x = 1; x < n; ++x) out.push_back({x, y, z});
  }
  return out;
}

// DoFHandler::distribute_dofs restated: walk `cells`, number unnumbered nodes in hierarchical order
template <typename CellFn>
void numbering_walk(int dim, int s, int n, size_t n_cells, CellFn cell_at, const int shape[3], const int origin[3],
                    std::vector<int64_t> &num) {
  const auto walk = cell_walk(dim, n);
  num.assign((size_t)shape[0] * shape[1] * shape[2], -1);
  int64_t next = 0;
  for (size_t c = 0; c < n_cells; ++c) {
    int cc[3];
    cell_at(c, cc);
    for (const auto &loc : walk) {
      const int gx = n * (cc[0] - origin[0]) + loc[0], gy = n * (cc[1] - origin[1]) + loc[1],
                gz = (dim == 3) ? n * (cc[2] - origin[2]) + loc[2] : 0;
      int64_t &slot = num[((size_t)gz * shape[1] + gy) * shape[0] + gx];
      if (slot < 0) {
        slot = next;
        next += s;
      }
    }
  }
}

void patch_cells_rel(const Params &P, const Geom &g, std::vector<std::array<int, 3>> &cells) {
  cells.resize(g.Nc);
  for (int pos = 0; pos < g.Nc; ++pos) {
    int k[3];
    col_to_cell(P, g, pos, k);
    cells[pos] = {k[0], k[1], k[2]};
  }
}

// M_H and S are derived from the basis and from K: a new basis, a restored checkpoint or a new K make them stale
void invalidate_mass(slod_ctx *c) {
  c->mass_done = false;
  c->s_coef = 0.0;
}

int check_patch(const slod_ctx *ctx, int64_t patch) {
  if (!ctx) return SLOD_ERR_INVALID;
  if (patch < 0 || patch >= ctx->n_patches) return fail(ctx, SLOD_ERR_INVALID, "patch id out of range");
  return SLOD_OK;
}

// Grow-only device scratch: afterwards p holds at least `need` elements (a regrown block does not keep its contents)
template <class T>
int grow(slod_ctx *ctx, T *&p, size_t &cap, size_t need) {
  if (cap >= need) return SLOD_OK;
  if (p) cudaFree(p);
  p = nullptr;
  cap = 0;
  CK(cudaMalloc(&p, sizeof(T) * need));
  cap = need;
  return SLOD_OK;
}

void free_workspace(slod_ctx *c);
void free_dev(slod_ctx *c) {
  auto F = [](auto *&p) {
    if (p) cudaFree(p);
    p = nullptr;
  };
  F(c->d_coef); F(c->d_phi); F(c->d_aphi); F(c->d_Kell); F(c->d_diag); F(c->d_status);
  F(c->d_perm); F(c->d_val); F(c->d_online); F(c->d_batch);
  F(c->d_Mell); F(c->d_Mval); F(c->d_Sell); F(c->d_heat);
  F(c->d_coef_base); F(c->d_cell_changed); F(c->d_rows);
  free_workspace(c);
}

// Expand the caller's tables (problem_parameter::value, include/Diffusion.h:40-53) onto the fine sub-cell
// grid: one value per sub-cell when eta >= h, one per Gauss point of the 2-point rule when eta < h.
int prepare_coefficients(slod_ctx *ctx) {
  Params &P = ctx->P;
  if (!ctx->coef_dirty) return SLOD_OK;
  int gauss = 0;
  for (int f = 0; f < ctx->n_fields; ++f) {
    if (!ctx->coef_set[f]) return fail(ctx, SLOD_ERR_STATE, "coefficient field not set");
    if ((1 << ctx->coef_r[f]) > P.nsub) gauss = 1;
  }
  const int nq = gauss ? (1 << P.dim) : 1;
  const int mfull = std::min(2 * P.ell + 1, P.N);
  const size_t need = (size_t)ctx->n_fields * ipow(P.n * mfull, P.dim) * nq;
  if ((int)need > ctx->sl.coef_doubles)
    return fail(ctx, SLOD_ERR_UNSUPPORTED,
                "coefficient finer than the fine sub-cells (eta < h) needs per-Gauss-point storage that does not "
                "fit the shared-memory plan of this configuration");
  const int ns = P.nsub, nz = (P.dim == 3) ? ns : 1;
  const size_t per_field = (size_t)ns * ns * nz * nq;
  std::vector<double> fine(per_field * ctx->n_fields);
  const double gp[2] = {0.5 - 0.5 / std::sqrt(3.0), 0.5 + 0.5 / std::sqrt(3.0)};
  for (int f = 0; f < ctx->n_fields; ++f) {
    const int nl = 1 << ctx->coef_r[f];
    const std::vector<double> &tab = ctx->coef_table[f];
    double *out = fine.data() + (size_t)f * per_field;
    auto lookup = [&](int sub, int qbit) -> int {
      if (nl <= ns) return sub / (ns / nl);
      // floor(x / eta) with x = (sub + gp) h and eta = h / ratio
      const int ratio = nl / ns;
      return sub * ratio + (int)std::floor(gp[qbit] * ratio);
    };
    if (nl == ns && nq == 1) {   // one table cell per fine sub-cell: the table is the fine array
      std::copy(tab.begin(), tab.end(), out);
      continue;
    }
    for (int z = 0; z < nz; ++z)
      for (int y = 0; y < ns; ++y)
        for (int x = 0; x < ns; ++x)
          for (int q = 0; q < nq; ++q) {
            const int ix = lookup(x, q & 1), iy = lookup(y, (q >> 1) & 1), iz = (P.dim == 3) ? lookup(z, (q >> 2) & 1) : 0;
            out[(((size_t)z * ns + y) * ns + x) * nq + q] = tab[((size_t)iz * nl + iy) * nl + ix];
          }
  }
  if (ctx->d_coef && ctx->d_coef_elems != fine.size()) {
    cudaFree(ctx->d_coef);
    ctx->d_coef = nullptr;
  }
  if (!ctx->d_coef) CK(cudaMalloc(&ctx->d_coef, sizeof(double) * fine.size()));
  ctx->d_coef_elems = fine.size();
  CK(cudaMemcpy(ctx->d_coef, fine.data(), sizeof(double) * fine.size(), cudaMemcpyHostToDevice));
  P.gauss_coef = gauss;
  ctx->coef_dirty = false;
  return SLOD_OK;
}

void free_workspace(slod_ctx *c) {
  auto F = [](auto *&p) {
    if (p) cudaFree(p);
    p = nullptr;
  };
  F(c->d_counter); F(c->d_work_counter); F(c->d_ids); F(c->d_X); F(c->d_Minv); F(c->d_G); F(c->d_cvec); F(c->d_Lws); F(c->d_W); F(c->d_coefws); F(c->d_coefws_finish);
  c->dl.coef_ws = nullptr;
  c->fl.coef_ws = nullptr;
  F(c->d_Lrec); F(c->d_stw);
  F(c->sb.eig_list); F(c->sb.jac_list); F(c->sb.H); F(c->sb.V); F(c->sb.rot_cs); F(c->sb.rot_i); F(c->sb.rot_n);
  c->chunk = 0;
  c->ids_cap = 0;
}

// Per-patch workspaces for `chunk` patches at a time and the work list of a whole range.  The chunk is sized for the
// range actually computed (a rank of an N-GPU run owns 1/N of the patches), capped by half of the free memory; a later
// call with a larger range reallocates.  ctx->chunk is committed only after every allocation has succeeded: a failed
// allocation leaves the handle without a workspace (chunk == 0) instead of with dangling null pointers.
// SLOD_CHUNK (environment) forces a small chunk: the multi-chunk loop is exercised by tests/test_parity_gpu.py.
// SLOD_EIG_CAP forces few eigen items per round of the selection pipeline: the round loop is exercised by
// tests/test_select_gpu.py.
int ensure_workspace(slod_ctx *ctx, int64_t n_range) {
  const Params &P = ctx->P;
  n_range = std::max<int64_t>(1, std::min<int64_t>(n_range, ctx->n_patches));
  const size_t per_patch = ((size_t)ctx->sl.x_stride + 2 * (size_t)ctx->dl.m_stride + (size_t)P.s * P.NcdMax +
                            (ctx->dense_ntile ? (size_t)ctx->xl.w_stride : 0) +
                            (ctx->split_solver ? (size_t)split_rec_stride(ctx->mma_nip) : 0)) * 8 + 4;
  int64_t forced = 0;
  if (const char *env = getenv("SLOD_CHUNK")) forced = std::max(1, atoi(env));
  if (ctx->chunk > 0 && ctx->ids_cap >= n_range && (ctx->chunk >= n_range || ctx->chunk_limited)) return SLOD_OK;
  cudaStreamSynchronize(0);
  cudaDeviceSynchronize();   // the old workspace may still be in use by enqueued kernels
  free_workspace(ctx);
  size_t free_b = 0, total_b = 0;
  CK(cudaMemGetInfo(&free_b, &total_b));
  const size_t budget = std::min<size_t>(free_b / 2, (size_t)96 << 30);   // one chunk for 2^15 3-D patches (53 GB) on a 180 GB part
  int64_t by_mem = std::max<int64_t>(1, (int64_t)(budget / per_patch));
  int64_t chunk = std::min<int64_t>(by_mem, n_range);
  if (forced) chunk = std::min<int64_t>(chunk, forced);
  const bool limited = chunk < n_range;   // memory- or environment-limited: a larger range would not get a larger chunk
  auto body = [&]() -> int {
    CK(cudaMalloc(&ctx->d_ids, sizeof(int) * n_range));
    CK(cudaMalloc(&ctx->d_counter, sizeof(int) * 4));
    CK(cudaMalloc(&ctx->d_work_counter, sizeof(int) * 4));
    CK(cudaMalloc(&ctx->d_X, sizeof(double) * (size_t)ctx->sl.x_stride * chunk));
    CK(cudaMalloc(&ctx->d_Minv, sizeof(double) * (size_t)ctx->dl.m_stride * chunk));
    CK(cudaMalloc(&ctx->d_G, sizeof(double) * (size_t)ctx->dl.m_stride * chunk));
    CK(cudaMalloc(&ctx->d_cvec, sizeof(double) * (size_t)P.s * P.NcdMax * chunk));
    if (ctx->dense_ntile) CK(cudaMalloc(&ctx->d_W, sizeof(double) * (size_t)ctx->xl.w_stride * chunk));
    if (ctx->dense_coef_gmem) {
      CK(cudaMalloc(&ctx->d_coefws, sizeof(double) * (size_t)ctx->dl.coef_doubles * ctx->grid_dense));
      ctx->dl.coef_ws = ctx->d_coefws;
    }
    if (ctx->finish_coef_gmem) {
      CK(cudaMalloc(&ctx->d_coefws_finish, sizeof(double) * (size_t)ctx->fl.coef_doubles * ctx->grid_finish));
      ctx->fl.coef_ws = ctx->d_coefws_finish;
    }
    if (ctx->split_solver)
    {
      CK(cudaMalloc(&ctx->d_Lrec, sizeof(double) * (size_t)split_rec_stride(ctx->mma_nip) * chunk));
      CK(cudaMalloc(&ctx->d_stw, sizeof(double) * split_stencil_ws_doubles(2 * ctx->n_sm, ctx->mma_nip)));
    }
    else
      CK(cudaMalloc(&ctx->d_Lws, sizeof(double) * (size_t)ctx->sl.lws_per_cta * ctx->grid_solve));
    // selection pipeline: work lists for every (patch, component) of a chunk, eigen buffers for one round
    SelectPlan &sp = ctx->sp;
    SelectBuffers &sb = ctx->sb;
    const size_t items = (size_t)chunk * P.s;
    sb.counters = ctx->d_counter;
    CK(cudaMalloc(&sb.eig_list, sizeof(int) * items));
    CK(cudaMalloc(&sb.jac_list, sizeof(int) * items));
    if (sp.use_ql) {
      const size_t per_item = sizeof(double) * ((size_t)sp.eig.h_stride + sp.eig.v_stride) +
                              (size_t)sp.eig.log_cap * (sizeof(double2) + sizeof(unsigned short)) + 2 * sizeof(int);
      size_t cap = std::max<size_t>(64, ((size_t)4 << 30) / per_item);
      if (const char *env = getenv("SLOD_EIG_CAP")) cap = (size_t)std::max(1, atoi(env));
      cap = std::min(cap, items);
      sp.eig.cap_items = (int)cap;
      CK(cudaMalloc(&sb.H, sizeof(double) * (size_t)sp.eig.h_stride * cap));
      CK(cudaMalloc(&sb.V, sizeof(double) * (size_t)sp.eig.v_stride * cap));
      CK(cudaMalloc(&sb.rot_cs, sizeof(double2) * (size_t)sp.eig.log_cap * cap));
      CK(cudaMalloc(&sb.rot_i, sizeof(unsigned short) * (size_t)sp.eig.log_cap * cap));
      CK(cudaMalloc(&sb.rot_n, sizeof(int) * 2 * cap));
      sp.grid_ql = (int)std::min<size_t>((cap + 7) / 8, (size_t)ctx->n_sm * 8);
    }
    return SLOD_OK;
  };
  const int rc = body();
  if (rc != SLOD_OK) {
    free_workspace(ctx);
    cudaGetLastError();
    return rc;
  }
  ctx->chunk = (int)chunk;
  ctx->chunk_limited = limited;
  ctx->ids_cap = n_range;
  ctx->ids_p0 = ctx->ids_p1 = -1;   // the work list on the device went with the old buffer
  return SLOD_OK;
}

// The solve and dense stages of the n_work patches of the device list `ids`, with the kernels the plan chose: split
// factor + triangular solve, tensor-core or SIMT solver; then flux + tensor-core dense, or SIMT dense.  wc: the work
// counter of the persistent kernels (nullptr: static distribution).  diag / status: the per-patch diagnostics and status
// words the kernels write (indexed by patch id).  Optional events: ev_factor behind the factor kernel of the split
// solver, ev_solved between the two stages.
int launch_patch_stages(slod_ctx *ctx, const int *ids, int nw, int *wc, cudaStream_t st, double *diag, int *status,
                        cudaEvent_t ev_factor, cudaEvent_t ev_solved) {
  if (ctx->split_solver) {
    static const int factor_grid_env = getenv("SLOD_FACTOR_GRID") ? atoi(getenv("SLOD_FACTOR_GRID")) : 0;   // experiments
    CK(launch_patch_factor(std::min(nw, factor_grid_env > 0 ? factor_grid_env : 2 * ctx->n_sm), ctx->smem_factor, st, ids, nw, ctx->d_coef, ctx->d_Lrec,
                           ctx->d_stw, status, ctx->split_coef_doubles, ctx->mma_nip, ctx->sl.ldx, ctx->sl.x_stride, wc));
    if (ev_factor) CK(cudaEventRecord(ev_factor, st));
    CK(launch_patch_trisolve(std::min(nw, ctx->n_sm), ctx->smem_tri, st, ids, nw, ctx->d_Lrec, ctx->d_X,
                             ctx->sl.coef_doubles, ctx->mma_nip, ctx->sl.ldx, ctx->sl.x_stride, wc));
  } else if (ctx->mma_variant >= 0)
    CK(launch_patch_solve_mma(ctx->mma_variant, std::min(nw, ctx->grid_solve), ctx->smem_solve, st, ids, nw,
                              ctx->d_coef, ctx->d_X, ctx->d_Lws, status, ctx->sl.coef_doubles, ctx->sl.ldx,
                              ctx->sl.x_stride, ctx->mma_lws_per_cta, ctx->mma_nip, ctx->mma_stw, wc));
  else
    CK(launch_patch_solve(std::min(nw, ctx->grid_solve), ctx->smem_solve, st, ids, nw, ctx->d_coef, ctx->d_X,
                          ctx->d_Lws, status, ctx->sl));
  if (ev_solved) CK(cudaEventRecord(ev_solved, st));
  if (ctx->dense_ntile) {
    CK(launch_patch_flux(std::min(nw, ctx->grid_flux), ctx->smem_flux, st, ids, nw, ctx->d_coef, ctx->d_X,
                         ctx->d_W, ctx->xl, wc));
    CK(launch_patch_dense_mma(ctx->dense_ntile, std::min(nw, ctx->grid_dense), ctx->smem_dense, st, ids, nw,
                              ctx->d_coef, ctx->d_X, ctx->d_W, ctx->d_Minv, ctx->d_G, diag, status, ctx->dl, wc));
  }
  else
    CK(launch_patch_dense(std::min(nw, ctx->grid_dense), ctx->smem_dense, st, ids, nw, ctx->d_coef, ctx->d_X,
                          ctx->d_Minv, ctx->d_G, diag, status, ctx->dl));
  ctx->launches += (ctx->split_solver ? 2 : 1) + (ctx->dense_ntile ? 2 : 1);
  return SLOD_OK;
}

// Work order of the patch kernels: largest patches first (stable, so equal costs keep the given order).
std::vector<int> cost_order(const Params &P, const std::vector<int> &order) {
  std::vector<long long> cost(order.size());
  for (size_t i = 0; i < order.size(); ++i) {
    const Geom g = make_geom(P, order[i]);
    cost[i] = (long long)g.Ni * g.bw * (g.bw + 4LL * g.Ncd) + (long long)g.Ncd * g.Ncd * g.Ncd * 8;
  }
  std::vector<int> perm(order.size());
  std::iota(perm.begin(), perm.end(), 0);
  std::stable_sort(perm.begin(), perm.end(), [&](int a, int b) { return cost[a] > cost[b]; });
  std::vector<int> out(order.size());
  for (size_t i = 0; i < perm.size(); ++i) out[i] = order[perm[i]];
  return out;
}

// Enqueues stages assembly .. premultiply for the patches [p0, p1) on `st` and returns without waiting: the work list
// of the whole range is uploaded once, every chunk has its own timing events, the status words of the range are cleared
// in front of the kernels and copied to page-locked host memory behind them.  wait_basis() is the synchronisation point.
// `list` (ascending patch ids): only these patches are computed, in the same cost order as in a range; the status words
// of [p0, p1) are still cleared and read back, so the caller passes a range that covers the list.
int run_basis(slod_ctx *ctx, int64_t p0, int64_t p1, double *d_phi, double *d_aphi, cudaStream_t st,
              const std::vector<int> *list = nullptr) {
  const Params &P = ctx->P;
  if (p0 < 0 || p1 > ctx->n_patches || p0 > p1) return fail(ctx, SLOD_ERR_INVALID, "bad patch range");
  const int64_t n_work = list ? (int64_t)list->size() : p1 - p0;
  if (n_work == 0) return SLOD_OK;
  int rc = prepare_coefficients(ctx);
  if (rc) return rc;
  rc = ensure_workspace(ctx, n_work);
  if (rc) return rc;
  BIND_PARAMS(st);
  // work order: largest patches first (integer geometry: cached per range, on the host and on the device; a list is not
  // cached, and the next range uploads its own)
  if (list || ctx->ids_p0 != p0 || ctx->ids_p1 != p1) {
    std::vector<int> order = list ? *list : std::vector<int>((size_t)(p1 - p0));
    if (!list) std::iota(order.begin(), order.end(), (int)p0);
    ctx->ids = cost_order(P, order);
    CK(cudaMemcpyAsync(ctx->d_ids, ctx->ids.data(), sizeof(int) * ctx->ids.size(), cudaMemcpyHostToDevice, st));
    CK(cudaStreamSynchronize(st));   // pageable source: the vector may be rebuilt by the next call
    ctx->ids_p0 = list ? -1 : p0;
    ctx->ids_p1 = list ? -1 : p1;
  }
  const size_t n_ids = ctx->ids.size();
  if (!ctx->h_status) CK(cudaHostAlloc(&ctx->h_status, sizeof(int) * (size_t)ctx->n_patches, cudaHostAllocDefault));
  CK(cudaMemsetAsync(ctx->d_status + p0, 0, sizeof(int) * (size_t)(p1 - p0), st));

  static const bool static_stride = getenv("SLOD_STATIC_WORK") != nullptr;   // A/B switch of the work distribution
  int *wc = static_stride ? nullptr : ctx->d_work_counter;
  const size_t n_chunks = (n_ids + ctx->chunk - 1) / ctx->chunk;
  while (ctx->chunk_ev.size() < 5 * n_chunks) {
    cudaEvent_t e;
    CK(cudaEventCreate(&e));
    ctx->chunk_ev.push_back(e);
  }
  ctx->chunks_pending = 0;
  for (size_t off = 0, ci = 0; off < n_ids; off += ctx->chunk, ++ci) {
    const int nw = (int)std::min<size_t>(ctx->chunk, n_ids - off);
    const int *ids = ctx->d_ids + off;
    cudaEvent_t *ev = ctx->chunk_ev.data() + 5 * ci;
    CK(cudaEventRecord(ev[0], st));
    rc = launch_patch_stages(ctx, ids, nw, wc, st, ctx->d_diag, ctx->d_status, ci == 0 ? ctx->ev_split : nullptr,
                             ev[1]);
    if (rc) return rc;
    CK(cudaEventRecord(ev[2], st));
    int nl = 0;
    CK(launch_select_pipeline(ctx->sp, st, ids, nw, ctx->d_Minv, ctx->d_G, ctx->d_cvec, ctx->d_diag,
                              ctx->d_status, ctx->sb, &nl));
    ctx->launches += nl;
    CK(cudaEventRecord(ev[3], st));
    CK(launch_patch_finish(std::min(nw, ctx->grid_finish), ctx->smem_finish, st, ids, nw, ctx->d_coef,
                           ctx->d_X, ctx->d_cvec, d_phi, d_aphi, ctx->fl));
    CK(cudaEventRecord(ev[4], st));
    ctx->launches += 1;
    ++ctx->chunks_pending;
  }
  CK(cudaMemcpyAsync(ctx->h_status + p0, ctx->d_status + p0, sizeof(int) * (size_t)(p1 - p0), cudaMemcpyDeviceToHost, st));
  CK(cudaEventRecord(ctx->ev[7], st));
  ctx->basis_pending = true;
  ctx->pending_p0 = p0;
  ctx->pending_p1 = p1;
  return SLOD_OK;
}

// Synchronisation point of run_basis: waits for the range, adds up the per-chunk stage times and maps the status words
// of the range to SLOD_ERR_NUMERIC (first offending patch in the message).
int wait_basis(slod_ctx *ctx) {
  if (!ctx->basis_pending) return SLOD_OK;
  ctx->basis_pending = false;
  CK(cudaEventSynchronize(ctx->ev[7]));
  float acc[4] = {0, 0, 0, 0};
  for (size_t ci = 0; ci < ctx->chunks_pending; ++ci)
    for (int k = 0; k < 4; ++k) {
      float ms = 0;
      CK(cudaEventElapsedTime(&ms, ctx->chunk_ev[5 * ci + k], ctx->chunk_ev[5 * ci + k + 1]));
      acc[k] += ms;
    }
  for (int k = 0; k < 4; ++k) ctx->tm.ms[k] = acc[k];
  if (ctx->split_solver && ctx->chunks_pending > 0) {   // first chunk: factorisation share of the solve stage
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, ctx->chunk_ev[0], ctx->ev_split));
    ctx->tm.ms[5] = ms;
  }
  for (int64_t i = ctx->pending_p0; i < ctx->pending_p1; ++i)
    if (ctx->h_status[i]) {
      char buf[160];
      snprintf(buf, sizeof buf, "patch %lld: numerical status bits 0x%x (1 A_ii not SPD, 2 M not SPD, 4 Jacobi not converged)",
               (long long)i, ctx->h_status[i]);
      return fail(ctx, SLOD_ERR_NUMERIC, buf);
    }
  return SLOD_OK;
}

// Enqueues the copy of the device coefficient array that the basis just enqueued on stream 0 reads: the baseline of
// slod_update_basis once the basis has succeeded (a few MB, device to device).
int snapshot_coefficients(slod_ctx *ctx) {
  if (ctx->d_coef_base && ctx->base_elems != ctx->d_coef_elems) {
    CK(cudaFree(ctx->d_coef_base));
    ctx->d_coef_base = nullptr;
  }
  if (!ctx->d_coef_base) CK(cudaMalloc(&ctx->d_coef_base, sizeof(double) * ctx->d_coef_elems));
  ctx->base_elems = ctx->d_coef_elems;
  ctx->base_gauss = ctx->P.gauss_coef;
  CK(cudaMemcpyAsync(ctx->d_coef_base, ctx->d_coef, sizeof(double) * ctx->d_coef_elems, cudaMemcpyDeviceToDevice, 0));
  return SLOD_OK;
}

int finish_coarse_timing(slod_ctx *ctx) {
  if (!ctx->coarse_timing_pending) return SLOD_OK;
  ctx->coarse_timing_pending = false;
  CK(cudaEventSynchronize(ctx->ev[6]));
  float ms = 0;
  CK(cudaEventElapsedTime(&ms, ctx->ev[5], ctx->ev[6]));
  ctx->tm.ms[4] = ms;
  return SLOD_OK;
}

// Rows of a coarse matrix C^T (B C) from phi and B phi (A phi for K, M_h phi for M_H) for the patches [p0, p1), or, with
// d_list, for the n_list entries of that device list: Morton groups (patch id >> dim) on the blocked kernel, patches
// otherwise; [p0, p1) is then the whole matrix.
cudaError_t launch_coarse_rows(const slod_ctx *ctx, cudaStream_t st, int64_t p0, int64_t p1, const double *d_phi,
                               const double *d_bphi, double *d_K, const int *d_list = nullptr, int n_list = 0) {
  if (ctx->coarse_nu > 0)
    return launch_coarse_blocked(ctx->P.dim, ctx->P.s, ctx->n_sm, ctx->smem_coarse_blk, st, (int)p0, (int)p1, d_phi,
                                 d_bphi, d_K, ctx->fl, ctx->coarse_nu, d_list, n_list);
  if (d_list)
    return launch_coarse(std::min(n_list, ctx->grid_coarse), ctx->smem_coarse, st, 0, n_list, d_phi, d_bphi, d_K,
                         ctx->fl, d_list);
  return launch_coarse((int)std::min<int64_t>(p1 - p0, ctx->grid_coarse), ctx->smem_coarse, st, (int)p0, (int)p1, d_phi,
                       d_bphi, d_K, ctx->fl);
}

// The rows of K (launch_coarse_rows), timed by ev[5] .. ev[6]
int run_coarse(slod_ctx *ctx, int64_t p0, int64_t p1, const double *d_phi, const double *d_aphi, double *d_K,
               cudaStream_t st, bool wait = true, const int *d_list = nullptr, int n_list = 0) {
  if (p0 < 0 || p1 > ctx->n_patches || p0 > p1) return fail(ctx, SLOD_ERR_INVALID, "bad patch range");
  if (p0 == p1 || (d_list && n_list == 0)) return SLOD_OK;
  BIND_PARAMS(st);
  CK(cudaEventRecord(ctx->ev[5], st));
  CK(launch_coarse_rows(ctx, st, p0, p1, d_phi, d_aphi, d_K, d_list, n_list));
  CK(cudaEventRecord(ctx->ev[6], st));
  ctx->launches += 1;
  ctx->coarse_timing_pending = true;
  if (!wait) return SLOD_OK;
  return finish_coarse_timing(ctx);
}

// block-ELL -> CSR.  The pattern is integer geometry: (p, q) is structural iff the node boxes intersect.
int ell_to_csr(const slod_ctx *ctx, const double *hK, int64_t *rowptr, int64_t *col, double *val, int64_t *n_rows,
               int64_t *nnz, long long *perm = nullptr) {
  const Params &P = ctx->P;
  const int s = P.s, w = P.w, ww = 2 * w + 1;
  const int nslots = (P.dim == 3) ? ww * ww * ww : ww * ww;
  const int64_t np = ctx->n_patches;
  if (n_rows) *n_rows = np * s;
  // per patch: list of (qid, slot) sorted by qid
  std::vector<int64_t> cnt((size_t)np + 1, 0);
  const unsigned nthr = std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
  auto neighbours = [&](int64_t pid, std::vector<std::pair<uint32_t, int>> &nb) {
    nb.clear();
    const Geom g = make_geom(P, (int)pid);
    for (int slot = 0; slot < nslots; ++slot) {
      int D[3] = {slot % ww - w, (slot / ww) % ww - w, (P.dim == 3) ? slot / (ww * ww) - w : 0};
      int qc[3] = {g.lo[0] + g.cc[0] + D[0], g.lo[1] + g.cc[1] + D[1], g.lo[2] + g.cc[2] + D[2]};
      bool valid = true;
      for (int x = 0; x < P.dim; ++x) valid = valid && qc[x] >= 0 && qc[x] < P.N;
      if (!valid) continue;
      const uint32_t qid = morton_encode(qc, P.dim, P.ref);
      const Geom gq = make_geom(P, (int)qid);
      for (int x = 0; x < P.dim; ++x) {
        const int b0 = std::max(g.lo[x], gq.lo[x]), b1 = std::min(g.lo[x] + g.m[x], gq.lo[x] + gq.m[x]);
        if (b1 < b0) valid = false;
      }
      if (valid) nb.emplace_back(qid, slot);
    }
    std::sort(nb.begin(), nb.end());
  };
  {
    std::vector<std::thread> th;
    for (unsigned t = 0; t < nthr; ++t)
      th.emplace_back([&, t]() {
        std::vector<std::pair<uint32_t, int>> nb;
        for (int64_t pid = t; pid < np; pid += nthr) {
          neighbours(pid, nb);
          cnt[pid + 1] = (int64_t)nb.size();
        }
      });
    for (auto &x : th) x.join();
  }
  // rows of patch pid: s rows, each nb.size()*s entries
  std::vector<int64_t> start((size_t)np + 1, 0);
  for (int64_t p = 0; p < np; ++p) start[p + 1] = start[p] + cnt[p + 1] * s * s;
  if (nnz) *nnz = start[np];
  if (!rowptr) return SLOD_OK;
  if (!col || (!perm && (!val || !hK))) return fail(ctx, SLOD_ERR_INVALID, "null output buffer");
  {
    std::vector<std::thread> th;
    for (unsigned t = 0; t < nthr; ++t)
      th.emplace_back([&, t]() {
        std::vector<std::pair<uint32_t, int>> nb;
        for (int64_t pid = t; pid < np; pid += nthr) {
          neighbours(pid, nb);
          const int64_t per_row = (int64_t)nb.size() * s;
          for (int d = 0; d < s; ++d) {
            const int64_t r = pid * s + d;
            int64_t o = start[pid] + d * per_row;
            rowptr[r] = o;
            const double *krow = hK ? hK + (size_t)r * P.ell_width : nullptr;
            for (const auto &q : nb)
              for (int e = 0; e < s; ++e) {
                col[o] = (int64_t)q.first * s + e;
                if (perm) perm[o] = (long long)r * P.ell_width + q.second * s + e;
                else val[o] = krow[q.second * s + e];
                ++o;
              }
          }
        }
      });
    for (auto &x : th) x.join();
  }
  rowptr[np * s] = start[np];
  return SLOD_OK;
}


// ---- one handle, N devices (slod_params.n_gpus > 1): one host thread and one NCCL rank per device ----------------
slod_ctx *rank_ctx(slod_ctx *ctx, int r) { return r == 0 ? ctx : ctx->subs[(size_t)r - 1]; }

template <typename Fn>
int for_each_rank(slod_ctx *ctx, Fn fn) {
  const int N = 1 + (int)ctx->subs.size();
  std::vector<int> rc((size_t)N, SLOD_OK);
  std::vector<std::thread> th;
  for (int r = 0; r < N; ++r)
    th.emplace_back([&, r]() {
      slod_ctx *c = rank_ctx(ctx, r);
      if (cudaSetDevice(c->device) != cudaSuccess) {
        rc[r] = fail(c, SLOD_ERR_CUDA, "cudaSetDevice failed");
        return;
      }
      rc[r] = fn(c, r);
    });
  for (auto &t : th) t.join();
  cudaSetDevice(ctx->device);
  for (int r = 0; r < N; ++r)
    if (rc[r] != SLOD_OK) {
      if (r > 0) ctx->err = "device " + std::to_string(rank_ctx(ctx, r)->device) + ": " + rank_ctx(ctx, r)->err;
      return rc[r];
    }
  return SLOD_OK;
}

int multi_basis(slod_ctx *ctx) {
  const size_t n = (size_t)ctx->n_patches * ctx->P.s * ctx->P.NfMax;
  const size_t per_patch = (size_t)ctx->P.s * ctx->P.NfMax;
  int rc = for_each_rank(ctx, [&](slod_ctx *c, int r) -> int {
    slod_ctx *ctx = c;   // for the CK / NK macros
    if (!c->d_phi) {
      CK(cudaMalloc(&c->d_phi, sizeof(double) * n));
      CK(cudaMalloc(&c->d_aphi, sizeof(double) * n));
    }
    int64_t b, e;
    owned_range(c->n_patches, r, c->comm_world, &b, &e);
    c->basis_done = c->coarse_done = false;
    int rc2 = run_basis(c, b, e, c->d_phi, c->d_aphi, 0);
    if (rc2) return rc2;
    // every device ends up with A*phi (needed by the coarse-matrix rows of its range) and phi (rank 0 serves the
    // host-buffer getters and the online phase) of every patch
    rc2 = gather_blocks(c, c->d_aphi, per_patch, 0);
    if (rc2) return rc2;
    rc2 = gather_blocks(c, c->d_phi, per_patch, 0);
    if (rc2) return rc2;
    rc2 = wait_basis(c);
    CK(cudaStreamSynchronize(0));
    if (rc2) return rc2;
    c->basis_done = true;
    return SLOD_OK;
  });
  for (int k = 0; k < 8; ++k)
    for (slod_ctx *c : ctx->subs) ctx->tm.ms[k] = std::max(ctx->tm.ms[k], c->tm.ms[k]);
  return rc;
}

int multi_coarse(slod_ctx *ctx) {
  const size_t n = (size_t)ctx->n_patches * ctx->P.s * ctx->P.ell_width;
  int rc = for_each_rank(ctx, [&](slod_ctx *c, int r) -> int {
    slod_ctx *ctx = c;
    if (!c->d_Kell) CK(cudaMalloc(&c->d_Kell, sizeof(double) * n));
    int64_t b, e;
    owned_range(c->n_patches, r, c->comm_world, &b, &e);
    int rc2 = run_coarse(c, b, e, c->d_phi, c->d_aphi, c->d_Kell, 0, false);
    if (rc2) return rc2;
    rc2 = gather_blocks(c, c->d_Kell, (size_t)c->P.s * c->P.ell_width, 0);   // disjoint row blocks, everywhere
    if (rc2) return rc2;
    rc2 = finish_coarse_timing(c);
    CK(cudaStreamSynchronize(0));
    return rc2;
  });
  for (slod_ctx *c : ctx->subs) ctx->tm.ms[4] = std::max(ctx->tm.ms[4], c->tm.ms[4]);
  return rc;
}

}  // namespace

// =================================================================================================
extern "C" {

const char *slod_last_create_error(void) { return g_create_error.c_str(); }
const char *slod_last_error(const slod_ctx *ctx) { return ctx ? ctx->err.c_str() : "null handle"; }

int slod_create(const slod_params *par, slod_ctx **out) {
  if (!par || !out) {
    g_create_error = "null argument";
    return SLOD_ERR_INVALID;
  }
  *out = nullptr;
  auto bad = [&](int code, const std::string &m) {
    g_create_error = m;
    return code;
  };
  if (par->dim != 2 && par->dim != 3) return bad(SLOD_ERR_INVALID, "dim must be 2 or 3");
  if (par->problem == SLOD_PROBLEM_DIFFUSION && par->spacedim != 1)
    return bad(SLOD_ERR_INVALID, "diffusion needs spacedim 1");
  if (par->problem == SLOD_PROBLEM_DIFFUSION_TENSOR && par->spacedim != 1)
    return bad(SLOD_ERR_INVALID, "tensor diffusion needs spacedim 1");
  if (par->problem == SLOD_PROBLEM_ELASTICITY && (par->spacedim != par->dim || par->dim != 2))
    return bad(SLOD_ERR_UNSUPPORTED, "elasticity is implemented for dim = spacedim = 2 (as in the reference)");
  if (par->problem != SLOD_PROBLEM_DIFFUSION && par->problem != SLOD_PROBLEM_ELASTICITY &&
      par->problem != SLOD_PROBLEM_DIFFUSION_TENSOR)
    return bad(SLOD_ERR_INVALID, "unknown problem");
  if (par->n_global_refinements < 0 || par->n_global_refinements * par->dim > 30)
    return bad(SLOD_ERR_INVALID, "n_global_refinements out of range");
  if (par->n_subdivisions < 1 || (par->n_subdivisions & (par->n_subdivisions - 1)))
    return bad(SLOD_ERR_INVALID, "n_subdivisions must be a power of two (include/Diffusion.h:76-80)");
  if (par->oversampling < 0) return bad(SLOD_ERR_INVALID, "oversampling < 0");
  if (par->n_gpus < 0) return bad(SLOD_ERR_INVALID, "n_gpus < 0");
  if (par->n_gpus > 1 && par->device == SLOD_DEVICE_NONE) return bad(SLOD_ERR_INVALID, "n_gpus > 1 on a maps-only handle");

  // device == SLOD_DEVICE_NONE: integer maps only (patch lists, DoF maps, CSR pattern); every compute
  // entry point of such a handle fails with SLOD_ERR_CUDA -- there is no CPU fallback.
  const bool maps_only = (par->device == SLOD_DEVICE_NONE);
  int dev = par->device;
  cudaDeviceProp prop{};
  prop.multiProcessorCount = 148;
  prop.sharedMemPerBlockOptin = 227 * 1024;
  prop.sharedMemPerMultiprocessor = 228 * 1024;
  if (!maps_only) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
      return bad(SLOD_ERR_CUDA, "no CUDA device: libslod_b200 has no CPU fallback");
    if (dev < 0 && par->n_gpus > 1) dev = 0;
    if (dev < 0 && cudaGetDevice(&dev) != cudaSuccess) return bad(SLOD_ERR_CUDA, "cudaGetDevice failed");
    if (dev >= ndev) return bad(SLOD_ERR_INVALID, "device ordinal out of range");
    if (par->n_gpus > 1 && dev + par->n_gpus > ndev)
      return bad(SLOD_ERR_INVALID, "n_gpus: not enough CUDA devices after `device`");
    if (cudaSetDevice(dev) != cudaSuccess) return bad(SLOD_ERR_CUDA, "cudaSetDevice failed");
    if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess)
      return bad(SLOD_ERR_CUDA, "cudaGetDeviceProperties failed");
  }

  auto *ctx = new slod_ctx();
  ctx->par = *par;
  ctx->device = dev;
  ctx->n_sm = prop.multiProcessorCount;
  Params &P = ctx->P;
  P.dim = par->dim; P.s = par->spacedim; P.ref = par->n_global_refinements; P.n = par->n_subdivisions;
  P.ell = par->oversampling; P.N = 1 << P.ref; P.nsub = P.N * P.n;
  P.problem = par->problem; P.stabilize = par->stabilize ? 1 : 0; P.quirk_presaved = par->quirk_presaved ? 1 : 0;
  const int mfull = std::min(2 * P.ell + 1, P.N);
  P.pmax = P.n * mfull + 1;
  P.nnodes_max = ipow(P.pmax, P.dim);
  P.NfMax = P.s * P.nnodes_max;
  P.NiMax = P.s * ipow(P.pmax - 2, P.dim);
  P.NcdMax = P.s * ipow(mfull, P.dim);
  P.w = 2 * P.ell + 1;
  P.ell_width = ipow(2 * P.w + 1, P.dim) * P.s;
  P.H = std::ldexp(1.0, -P.ref);
  P.h = P.H / P.n;
  P.Hd = std::pow(P.H, P.dim);
  P.pw = std::pow(P.h, P.dim) / (double)(1 << P.dim);
  P.has_presaved = 0;
  P.gauss_coef = 0;
  ctx->n_patches = (int64_t)ipow(P.N, P.dim);
  ctx->n_fields = (P.problem == SLOD_PROBLEM_DIFFUSION) ? 1
                  : (P.problem == SLOD_PROBLEM_ELASTICITY) ? 2 : tensor_fields(P.dim);
  reference_matrices(P);
  // quirk B: the first full-size patch in patch-id order donates its matrix (source/LOD.cc:446-450)
  {
    Params Q = P;
    Q.quirk_presaved = 0;
    for (int64_t pid = 0; pid < ctx->n_patches; ++pid) {
      const Geom g = make_geom(Q, (int)pid);
      if (g.full) {
        for (int a = 0; a < 3; ++a) P.presaved_lo[a] = g.lo[a];
        P.has_presaved = 1;
        break;
      }
    }
  }
  // maxima over patch shapes
  int bw_max = 0, nb_max = 0;
  {
    // shapes are products of per-axis extents; scanning the patches along the diagonal + full scan for small grids
    for (int64_t pid = 0; pid < ctx->n_patches; ++pid) {
      const Geom g = make_geom(P, (int)pid);
      if (g.Ni <= 0) {   // n_subdivisions = 1 on a one-cell patch: no interior dof, the patch problem is empty
        delete ctx;
        return bad(SLOD_ERR_UNSUPPORTED, "a patch has no interior fine dof (n_subdivisions = 1 with one-cell patches)");
      }
      if (g.Ni < g.Ncd) {
        // M = P_i^T A_ii^{-1} P_i / H^d has rank <= Ni: with fewer interior fine dofs than coarse dofs it is singular and
        // the reference's gauss_jordan (source/LOD.cc:553) has nothing to invert either (n_subdivisions = 1)
        delete ctx;
        return bad(SLOD_ERR_UNSUPPORTED,
                   "a patch has fewer interior fine dofs than coarse dofs: P^T A^-1 P is singular (use n_subdivisions >= 2)");
      }
      bw_max = std::max(bw_max, g.bw);
      int nb = 0;
      // patch-boundary dofs
      int cnt_int = 1, cnt_nob = 1;
      for (int a = 0; a < P.dim; ++a) {
        cnt_int *= g.p[a];
        cnt_nob *= g.p[a] - (g.domlo[a] ? 0 : 1) - (g.domhi[a] ? 0 : 1);
      }
      nb = P.s * (cnt_int - cnt_nob);
      nb_max = std::max(nb_max, nb);
    }
  }
  ctx->bw_max = bw_max;
  ctx->nb_max = nb_max;
  const bool big = (P.dim == 3);
  const int msub = P.n * mfull;
  // room for one value per Gauss point (eta < h) where that is cheap (2-D); 3-D and the tensor problem keep one per
  // sub-cell
  const int coef_doubles =
      ctx->n_fields * ipow(msub, P.dim) * (P.dim == 2 && P.problem != SLOD_PROBLEM_DIFFUSION_TENSOR ? 4 : 1);
  // ---- layouts ----
  SolveLayout &sl = ctx->sl;
  sl.threads = big ? 512 : 128;
  sl.bw_max = bw_max;
  sl.R = bw_max + kSolveNB;
  sl.ldw = bw_max + 1;
  sl.ldr = P.NcdMax;
  sl.coef_doubles = coef_doubles;
  sl.ldx = P.NcdMax;
  sl.x_stride = (long long)P.NiMax * sl.ldx;
  const int steps_max = (P.NiMax + kSolveNB - 1) / kSolveNB;
  sl.lws_per_cta = (long long)steps_max * (kSolveNB * kSolveNB + bw_max * kSolveNB);
  ctx->smem_solve = sizeof(double) * ((size_t)coef_doubles + (size_t)sl.R * sl.ldw + (size_t)sl.R * sl.ldr +
                                      (size_t)sl.R * kSolveNB + 2 * kSolveNB * kSolveNB + (size_t)kSolveNB * sl.ldr);
  sl.gmem_window = 0;
  sl.gmem_coef = 0;
  sl.gcoef_off = 0;
  sl.gwin_off = 0;
  const size_t smem_solve_small = sizeof(double) * ((size_t)coef_doubles + 2 * kSolveNB * kSolveNB + (size_t)kSolveNB * sl.ldr);
  const long long gwin_doubles = (long long)sl.R * sl.ldw + (long long)sl.R * sl.ldr + (long long)sl.R * kSolveNB;
  // tiles of the tensor-core dense stage behind a solver whose X rows have leading dimension ldx (0: SIMT dense stage)
  auto dense_tiles = [&](int variant, int ldx) {
    const int nt_need = (P.NcdMax + 7) / 8;
    int ntile = nt_need <= 4 ? 4 : (nt_need <= 8 ? 8 : (nt_need <= 16 ? 16 : 0));
    if (getenv("SLOD_FORCE_SIMT_DENSE")) ntile = 0;
    // the register/mma dense stage reads X rows with 16-byte loads: needs the padded layout of the mma solver
    if (ntile && (variant < 0 || 8 * ntile != ldx)) ntile = 0;
    if (ipow(P.n + 1, P.dim) > 27) ntile = 0;   // the gather table of M holds 27 local nodes per coarse cell
    if (ntile && dense_mma_smem(ntile, coef_doubles, nb_max) > prop.sharedMemPerBlockOptin) ntile = 0;
    return ntile;
  };
  // tensor-core solver when the window (RB blocks of 8 rows) and the coarse columns (NW warps x 8) fit a variant
  {
    const int rb_need = (bw_max + 8 + 7) / 8, nw_need = (P.NcdMax + 7) / 8;
    int variant = -1, rbmax = 0, nw = 0;
    if (rb_need <= 13 && nw_need <= 16 && (rb_need > 4 || nw_need > 8)) { variant = 0; rbmax = 13; nw = 16; }
    else if (rb_need <= 4 && nw_need <= 4) { variant = 1; rbmax = 4; nw = 4; }
    else if (rb_need <= 4 && nw_need <= 8) { variant = 2; rbmax = 4; nw = 8; }
    if (getenv("SLOD_FORCE_SIMT_SOLVER") || getenv("SLOD_FORCE_GMEM_SOLVER")) variant = -1;
    // split factor + triangular-solve kernels for large 3-D scalar patches.  They keep their columns in z-major order,
    // which only the tensor-core flux / dense kernels understand.  The factor kernel stages one coefficient field at a
    // time (the tensor problem's components one after the other), so its window is one field whatever the problem.
    const bool split = variant == 0 && P.dim == 3 && P.s == 1 &&
                       (P.problem == SLOD_PROBLEM_DIFFUSION || P.problem == SLOD_PROBLEM_DIFFUSION_TENSOR) &&
                       !getenv("SLOD_FUSED_SOLVER") && dense_tiles(variant, 8 * nw) > 0;
    const int solve_coef = split ? coef_doubles / ctx->n_fields : coef_doubles;
    // a variant whose shared-memory plan does not fit (large coefficient windows: many subdivisions or fields) is no
    // variant: the SIMT solver takes over, with its windows in global memory if need be
    if (variant >= 0 && solve_mma_smem(variant, solve_coef, ((P.NiMax + 7) / 8) * 8, P.s * ((P.dim == 3) ? 13 : 4) + P.s) >
                            prop.sharedMemPerBlockOptin)
      variant = -1;
    if (variant >= 0) {
      ctx->mma_variant = variant;
      ctx->mma_threads = 32 * nw;
      sl.ldx = 8 * nw;
      const int nip = ((P.NiMax + 7) / 8) * 8;
      sl.x_stride = (long long)nip * sl.ldx;
      ctx->mma_lws_per_cta = (long long)(nip / 8) * (64 + 8 * (rbmax - 1) * 8);
      sl.lws_per_cta = std::max(sl.lws_per_cta, ctx->mma_lws_per_cta);
      sl.threads = ctx->mma_threads;
      ctx->mma_nip = nip;
      ctx->mma_stw = P.s * ((P.dim == 3) ? 13 : 4) + P.s;
      ctx->smem_solve = solve_mma_smem(variant, solve_coef, ctx->mma_nip, ctx->mma_stw);
      if (split) {
        ctx->split_solver = true;
        ctx->split_coef_doubles = solve_coef;
        ctx->smem_factor = split_factor_smem(solve_coef, nip);
        ctx->smem_tri = split_trisolve_smem(nip);
      }
    }
  }
  if (ctx->mma_variant < 0 && (ctx->smem_solve > prop.sharedMemPerBlockOptin || getenv("SLOD_FORCE_GMEM_SOLVER"))) {
    // the SIMT solver with its windows in global memory: the fall-back for patches of any size
    sl.gmem_window = 1;
    sl.gwin_off = sl.lws_per_cta;
    sl.lws_per_cta += gwin_doubles;
    ctx->smem_solve = smem_solve_small;
    if (ctx->smem_solve > prop.sharedMemPerBlockOptin && P.problem == SLOD_PROBLEM_DIFFUSION_TENSOR) {
      // the coefficient window does not fit either (the tensor problem's six fields on 3-D patches with 4 subdivisions):
      // it goes to the CTA's slice of the workspace as well.  The other problems keep their envelope.
      sl.gmem_coef = 1;
      sl.gcoef_off = sl.lws_per_cta;
      sl.lws_per_cta += coef_doubles;
      ctx->smem_solve -= sizeof(double) * (size_t)coef_doubles;
    }
  }
  DenseLayout &dl = ctx->dl;
  // the SIMT dense stage keeps kGEPT = 32 Gram entries per thread: 2-D patches with more than 64 coarse dofs need the
  // 512-thread CTA that 3-D always uses
  dl.threads = (big || (size_t)P.NcdMax * P.NcdMax > (size_t)32 * 128) ? 512 : 128;
  dl.ncd_max = P.NcdMax; dl.nb_max = nb_max; dl.coef_doubles = coef_doubles; dl.ldx = sl.ldx;
  dl.x_stride = sl.x_stride;
  dl.m_stride = (long long)P.NcdMax * P.NcdMax;
  ctx->smem_dense = sizeof(double) * ((size_t)coef_doubles + (size_t)dl.m_stride + 2 * 16 * (size_t)P.NcdMax +
                                      2 * (size_t)P.NcdMax + 16 * 54) +
                    sizeof(int) * (16 * 54 + (size_t)nb_max + 8);
  if (const int ntile = dense_tiles(ctx->mma_variant, sl.ldx)) {
    ctx->dense_ntile = ntile;
    ctx->smem_dense = dense_mma_smem(ntile, coef_doubles, nb_max);
    dl.threads = 32 * ntile;
  }
  dl.coef_ws = nullptr;
  if (!ctx->dense_ntile && (ctx->smem_dense > prop.sharedMemPerBlockOptin || getenv("SLOD_FORCE_GMEM_SOLVER")) &&
      ctx->smem_dense - sizeof(double) * (size_t)coef_doubles <= prop.sharedMemPerBlockOptin) {
    ctx->dense_coef_gmem = true;   // the pointer is set when the workspace is allocated
    ctx->smem_dense -= sizeof(double) * (size_t)coef_doubles;
  }
  if (ctx->dense_ntile) {
    FluxLayout &xl = ctx->xl;
    xl.coef_doubles = coef_doubles; xl.ldx = sl.ldx; xl.nb_max = nb_max; xl.x_stride = sl.x_stride;
    xl.w_stride = (long long)((nb_max + 31) / 32 * 32) * sl.ldx;
    dl.w_stride = xl.w_stride;
    xl.zmajor = dl.zmajor = ctx->split_solver ? 1 : 0;
    ctx->smem_flux = flux_smem(coef_doubles, sl.ldx, nb_max);
  }
  SelectPlan &sp = ctx->sp;
  sp.s = P.s;
  sp.lay.threads = big ? 512 : 128;
  sp.lay.ncd_max = P.NcdMax; sp.lay.m_stride = dl.m_stride;
  sp.lay.fast_path = getenv("SLOD_NO_FAST_SELECT") ? 0 : 1;
  sp.smem_fast = select_fast_smem(P.NcdMax);
  sp.smem_jac = select_jacobi_smem(P.NcdMax);
  sp.eig.nmax = P.NcdMax; sp.eig.ldh = P.NcdMax;
  sp.eig.h_stride = (long long)P.NcdMax * P.NcdMax;
  sp.eig.v_stride = 6LL * P.NcdMax;
  sp.eig.log_cap = std::max<long long>(3LL * P.NcdMax * P.NcdMax, 1024);
  sp.eig.ncd_max = P.NcdMax; sp.eig.m_stride = dl.m_stride;
  sp.eig.cap_items = 0;
  sp.smem_tri = eig_tridiag_smem(P.NcdMax);
  sp.smem_ql = eig_ql_smem(P.NcdMax);
  sp.smem_fin = eig_finish_smem(P.NcdMax);
  // the tridiagonalisation keeps columns of up to 256 rows in registers and the whole matrix in shared memory
  sp.use_ql = (P.NcdMax - 1 <= 256 && sp.smem_tri <= prop.sharedMemPerBlockOptin && !getenv("SLOD_FORCE_JACOBI")) ? 1 : 0;
  FinishLayout &fl = ctx->fl;
  fl.ell_width = P.ell_width;
  fl.coef_doubles = coef_doubles; fl.nf_max = P.NfMax; fl.ncd_max = P.NcdMax; fl.ldx = sl.ldx; fl.x_stride = sl.x_stride;
  ctx->smem_finish = sizeof(double) * ((size_t)coef_doubles + P.NfMax + P.NcdMax) + sizeof(int) * ((size_t)P.NiMax + 2);
  fl.coef_ws = nullptr;
  if (ctx->smem_finish > prop.sharedMemPerBlockOptin && P.problem == SLOD_PROBLEM_DIFFUSION_TENSOR) {
    // as for the SIMT dense stage: the window in global memory (the tensor problem's six fields; the other problems
    // keep their envelope)
    ctx->finish_coef_gmem = true;   // the pointer is set when the workspace is allocated
    ctx->smem_finish -= sizeof(double) * (size_t)coef_doubles;
  }
  ctx->smem_coarse = sizeof(double) * ((size_t)P.s * P.NfMax);
  const size_t smem_cap = prop.sharedMemPerBlockOptin;
  {
    // blocked coarse kernel: the 2^dim patches of a Morton block share a node box of (2 ell + 2) n + 1 nodes per axis
    const int nu = std::min((2 * P.ell + 2), P.N) * P.n + 1;
    const size_t sm = coarse_blocked_smem(P.dim, P.s, nu);
    if (P.ref >= 1 && sm + 2048 <= smem_cap && !getenv("SLOD_SIMPLE_COARSE")) {
      ctx->coarse_nu = nu;
      ctx->smem_coarse_blk = sm;
    }
  }
  if ((size_t)P.NcdMax * P.NcdMax > (size_t)32 * dl.threads)
    { delete ctx; return bad(SLOD_ERR_UNSUPPORTED, "patch too large: coarse dofs per patch exceed the Gram register tile"); }
  if (ctx->smem_solve > smem_cap || ctx->smem_dense > smem_cap || sp.smem_fast > smem_cap || sp.smem_jac > smem_cap ||
      ctx->smem_finish > smem_cap || ctx->smem_coarse > smem_cap) {
    delete ctx;
    return bad(SLOD_ERR_UNSUPPORTED, "patch too large for the shared-memory resident solver (oversampling/subdivisions)");
  }
  auto per_sm = [&](size_t smem, int threads) {
    int by_smem = (int)std::max<size_t>(1, (prop.sharedMemPerMultiprocessor) / (smem + 1024));
    int by_thr = std::max(1, 2048 / threads);
    return std::max(1, std::min(std::min(by_smem, by_thr), 16));
  };
  ctx->grid_solve = ctx->n_sm * per_sm(ctx->smem_solve, sl.threads);
  ctx->grid_dense = ctx->n_sm * per_sm(ctx->smem_dense, dl.threads);
  sp.grid_fast = ctx->n_sm * std::min(3, per_sm(sp.smem_fast, 256));
  sp.grid_jac = ctx->n_sm * per_sm(sp.smem_jac, sp.lay.threads);
  sp.grid_tri = ctx->n_sm * per_sm(sp.smem_tri, 256);
  sp.grid_fin = ctx->n_sm * per_sm(sp.smem_fin, 128);
  sp.grid_ql = ctx->n_sm * 8;
  ctx->grid_finish = ctx->n_sm * per_sm(ctx->smem_finish, 256);
  ctx->grid_flux = ctx->n_sm * std::min(getenv("SLOD_FLUX_CTAS") ? atoi(getenv("SLOD_FLUX_CTAS")) : 4, per_sm(ctx->smem_flux, 256));   // env: experiments
  ctx->grid_coarse = ctx->n_sm * per_sm(ctx->smem_coarse, 256);

  auto cuda_bad = [&](const char *what, cudaError_t e) {
    g_create_error = std::string(what) + ": " + cudaGetErrorString(e);
    free_dev(ctx);
    delete ctx;
    return SLOD_ERR_CUDA;
  };
  cudaError_t e;
  ctx->coef_field_elems = (size_t)ipow(P.nsub, P.dim);
  if (maps_only) {
    *out = ctx;
    return SLOD_OK;
  }
  if ((e = cudaMalloc(&ctx->d_status, sizeof(int) * ctx->n_patches)) != cudaSuccess) return cuda_bad("cudaMalloc", e);
  if ((e = cudaMalloc(&ctx->d_diag, sizeof(double) * 8 * P.s * ctx->n_patches)) != cudaSuccess)
    return cuda_bad("cudaMalloc", e);
  cudaMemset(ctx->d_status, 0, sizeof(int) * ctx->n_patches);
  cudaMemset(ctx->d_diag, 0, sizeof(double) * 8 * P.s * ctx->n_patches);
  for (auto &ev : ctx->ev)
    if ((e = cudaEventCreate(&ev)) != cudaSuccess) return cuda_bad("cudaEventCreate", e);
  if ((e = cudaEventCreate(&ctx->ev_split)) != cudaSuccess) return cuda_bad("cudaEventCreate", e);
  if (par->n_gpus > 1) {
    // one sub-handle per further device, one NCCL communicator over all of them
    NcclApi *nc = nccl_api();
    if (!nc->err.empty()) {
      g_create_error = nc->err;
      slod_destroy(ctx);
      return SLOD_ERR_CUDA;
    }
    const int N = par->n_gpus;
    slod_params sp1 = *par;
    sp1.n_gpus = 1;
    for (int r = 1; r < N; ++r) {
      sp1.device = dev + r;
      slod_ctx *sub = nullptr;
      const int rc = slod_create(&sp1, &sub);
      if (rc != SLOD_OK) {
        slod_destroy(ctx);
        return rc;
      }
      ctx->subs.push_back(sub);
    }
    std::vector<int> devs((size_t)N);
    for (int r = 0; r < N; ++r) devs[r] = dev + r;
    std::vector<ncclComm_t> comms((size_t)N);
    const ncclResult_t nr = nc->CommInitAll(comms.data(), N, devs.data());
    if (nr != ncclSuccess) {
      g_create_error = std::string("ncclCommInitAll: ") + nc->GetErrorString(nr);
      slod_destroy(ctx);
      return SLOD_ERR_CUDA;
    }
    for (int r = 0; r < N; ++r) {
      slod_ctx *c = rank_ctx(ctx, r);
      c->comm = comms[r];
      c->comm_rank = r;
      c->comm_world = N;
    }
    cudaSetDevice(dev);
  }
  *out = ctx;
  return SLOD_OK;
}

void slod_destroy(slod_ctx *ctx) {
  if (!ctx) return;
  if (ctx->device == SLOD_DEVICE_NONE) {
    delete ctx;
    return;
  }
  for (slod_ctx *sub : ctx->subs) slod_destroy(sub);
  ctx->subs.clear();
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();   // slod_assemble_coarse only enqueues
  // everything this handle enqueued has completed (synchronised above).  Abort instead of Destroy: Destroy waits for
  // the peers, and a handle that is torn down on an error path (one rank failed) must not hang the process
  if (ctx->comm) nccl_api()->CommAbort(ctx->comm);
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  free_dev(ctx);
  for (auto &ev : ctx->ev)
    if (ev) cudaEventDestroy(ev);
  for (auto &ev : ctx->chunk_ev) cudaEventDestroy(ev);
  if (ctx->ev_split) cudaEventDestroy(ctx->ev_split);
  for (auto &ev : ctx->ev_out)
    if (ev) cudaEventDestroy(ev);
  if (ctx->h_status) cudaFreeHost(ctx->h_status);
  delete ctx;
}

namespace {
// field `field` of the handle := the n values cellwise[0], cellwise[stride], ...; prepare_coefficients expands it onto the
// sub-cells before the next computation
void store_coefficient(slod_ctx *ctx, int field, int eta_refinement, const double *cellwise, size_t n, size_t stride) {
  std::vector<double> &tab = ctx->coef_table[field];
  tab.resize(n);
  for (size_t c = 0; c < n; ++c) tab[c] = cellwise[c * stride];
  ctx->coef_r[field] = eta_refinement;
  ctx->coef_set[field] = true;
  ctx->coef_dirty = true;
  ctx->basis_done = ctx->coarse_done = false;
}
}  // namespace

int slod_set_coefficient(slod_ctx *ctx, int field, int eta_refinement, const double *cellwise, size_t n) {
  if (!ctx || !cellwise) return SLOD_ERR_INVALID;
  if (ctx->P.problem == SLOD_PROBLEM_DIFFUSION_TENSOR)
    return fail(ctx, SLOD_ERR_INVALID,
                "a tensor-diffusion handle takes its coefficient as whole tensors: use slod_set_coefficient_tensor");
  NEED_DEVICE();
  const Params &P = ctx->P;
  if (field < 0 || field >= ctx->n_fields) return fail(ctx, SLOD_ERR_INVALID, "coefficient field index out of range");
  if (eta_refinement < 0 || eta_refinement * P.dim > 30)
    return fail(ctx, SLOD_ERR_INVALID, "eta_refinement out of range ((2^r)^dim must stay below 2^31)");
  size_t want = 1;
  for (int a = 0; a < P.dim; ++a) want <<= eta_refinement;
  if (want != n) return fail(ctx, SLOD_ERR_INVALID, "coefficient table size != (2^r)^dim");
  store_coefficient(ctx, field, eta_refinement, cellwise, n, 1);
  for (slod_ctx *sub : ctx->subs) {
    const int rc = slod_set_coefficient(sub, field, eta_refinement, cellwise, n);
    if (rc) return fail(ctx, rc, sub->err);
  }
  return SLOD_OK;
}

int slod_set_coefficient_tensor(slod_ctx *ctx, int eta_refinement, const double *cells, size_t n_cells) {
  if (!ctx || !cells) return SLOD_ERR_INVALID;
  const Params &P = ctx->P;
  if (P.problem != SLOD_PROBLEM_DIFFUSION_TENSOR)
    return fail(ctx, SLOD_ERR_INVALID, "slod_set_coefficient_tensor needs a SLOD_PROBLEM_DIFFUSION_TENSOR handle: use "
                                       "slod_set_coefficient");
  if (eta_refinement < 0 || eta_refinement * P.dim > 30)
    return fail(ctx, SLOD_ERR_INVALID, "eta_refinement out of range ((2^r)^dim must stay below 2^31)");
  size_t want = 1;
  for (int a = 0; a < P.dim; ++a) want <<= eta_refinement;
  if (want != n_cells) return fail(ctx, SLOD_ERR_INVALID, "n_cells != (2^eta_refinement)^dim");
  const int nc = ctx->n_fields;
  for (size_t c = 0; c < n_cells; ++c) {
    const double *t = cells + c * nc;
    for (int f = 0; f < nc; ++f)
      if (!std::isfinite(t[f])) return fail(ctx, SLOD_ERR_INVALID, "tensor of cell " + std::to_string(c) + " is not finite");
    // Cholesky with positive pivots of the symmetric tensor (Voigt order: the diagonal first)
    double A[3][3];
    for (int f = 0; f < nc; ++f) {
      const int a = kVoigt[P.dim - 2][f][0], b = kVoigt[P.dim - 2][f][1];
      A[a][b] = A[b][a] = t[f];
    }
    bool spd = true;
    for (int j = 0; j < P.dim && spd; ++j) {
      double d = A[j][j];
      for (int k = 0; k < j; ++k) d -= A[j][k] * A[j][k];
      if (!(d > 0.0)) {
        spd = false;
        break;
      }
      A[j][j] = std::sqrt(d);
      for (int i = j + 1; i < P.dim; ++i) {
        double v = A[i][j];
        for (int k = 0; k < j; ++k) v -= A[i][k] * A[j][k];
        A[i][j] = v / A[j][j];
      }
    }
    if (!spd) return fail(ctx, SLOD_ERR_INVALID, "tensor of cell " + std::to_string(c) + " is not positive definite");
  }
  if ((1 << eta_refinement) > P.nsub)
    return fail(ctx, SLOD_ERR_UNSUPPORTED, "a tensor table finer than the fine sub-cells (eta < h) is not supported: "
                                           "the per-Gauss-point mode exists for scalar coefficients only");
  NEED_DEVICE();
  // each component is a cell-wise table of its own, expanded like a slod_set_coefficient field
  for (int f = 0; f < nc; ++f) store_coefficient(ctx, f, eta_refinement, cells + f, n_cells, nc);
  for (slod_ctx *sub : ctx->subs) {
    const int rc = slod_set_coefficient_tensor(sub, eta_refinement, cells, n_cells);
    if (rc) return fail(ctx, rc, sub->err);
  }
  return SLOD_OK;
}

int slod_patch_count(const slod_ctx *ctx, int64_t *n) {
  if (!ctx || !n) return SLOD_ERR_INVALID;
  *n = ctx->n_patches;
  return SLOD_OK;
}

int slod_get_plan(const slod_ctx *ctx, int32_t out[8]) {
  if (!ctx || !out) return SLOD_ERR_INVALID;
  // the rule of prepare_coefficients: one value per Gauss point once any table is finer than the sub-cells
  int gauss = 0;
  for (int f = 0; f < ctx->n_fields; ++f)
    if (ctx->coef_set[f] && (1 << ctx->coef_r[f]) > ctx->P.nsub) gauss = 1;
  out[0] = ctx->mma_variant;
  out[1] = ctx->split_solver ? 1 : 0;
  out[2] = ctx->dense_ntile;
  out[3] = ctx->sl.gmem_window;
  out[4] = ctx->dense_coef_gmem ? 1 : 0;
  out[5] = ctx->coarse_nu > 0 ? 1 : 0;
  out[6] = ctx->sp.use_ql;
  out[7] = gauss;
  return SLOD_OK;
}

int slod_get_patch_info(const slod_ctx *ctx, int64_t patch, int32_t *n_cells, int32_t *n_fine, int32_t *n_internal,
                        int32_t *n_boundary, int32_t *n_domain_boundary, int32_t *n_coarse, int32_t lo[3],
                        int32_t m[3]) {
  int rc = check_patch(ctx, patch);
  if (rc) return rc;
  const Params &P = ctx->P;
  const Geom g = make_geom(P, (int)patch);
  int nb = 0, ndb = 0;
  for (int node = 0; node < g.nnodes; ++node) {
    int a[3];
    node_coords(g, node, a);
    const int c = node_class(P, g, a);
    nb += (c & 1) ? P.s : 0;
    ndb += (c & 2) ? P.s : 0;
  }
  if (n_cells) *n_cells = g.Nc;
  if (n_fine) *n_fine = g.Nf;
  if (n_internal) *n_internal = g.Ni;
  if (n_boundary) *n_boundary = nb;
  if (n_domain_boundary) *n_domain_boundary = ndb;
  if (n_coarse) *n_coarse = g.Ncd;
  for (int a = 0; a < 3; ++a) {
    if (lo) lo[a] = g.lo[a];
    if (m) m[a] = g.m[a];
  }
  return SLOD_OK;
}

int slod_get_patch_cells(const slod_ctx *ctx, int64_t patch, uint32_t *cells, int32_t *n) {
  int rc = check_patch(ctx, patch);
  if (rc) return rc;
  const Params &P = ctx->P;
  const Geom g = make_geom(P, (int)patch);
  if (n) *n = g.Nc;
  if (!cells) return SLOD_OK;
  for (int pos = 0; pos < g.Nc; ++pos) {
    int k[3];
    col_to_cell(P, g, pos, k);
    int c[3] = {g.lo[0] + k[0], g.lo[1] + k[1], g.lo[2] + k[2]};
    cells[pos] = morton_encode(c, P.dim, P.ref);
  }
  return SLOD_OK;
}

int slod_get_patch_fine_dofs(const slod_ctx *ctx, int64_t patch, uint64_t *dofs, int32_t *n) {
  int rc = check_patch(ctx, patch);
  if (rc) return rc;
  const Params &P = ctx->P;
  const Geom g = make_geom(P, (int)patch);
  if (n) *n = g.Nf;
  if (!dofs) return SLOD_OK;
  const int G = P.nsub + 1;
  if (ctx->fine_numbering.empty()) {
    const int shape[3] = {G, G, P.dim == 3 ? G : 1};
    const int origin[3] = {0, 0, 0};
    numbering_walk(P.dim, P.s, P.n, (size_t)ctx->n_patches,
                   [&](size_t c, int cc[3]) { morton_decode((uint32_t)c, P.dim, P.ref, cc); }, shape, origin,
                   ctx->fine_numbering);
  }
  for (int node = 0; node < g.nnodes; ++node) {
    int a[3];
    node_coords(g, node, a);
    const size_t gx = (size_t)g.lo[0] * P.n + a[0], gy = (size_t)g.lo[1] * P.n + a[1],
                 gz = (P.dim == 3) ? (size_t)g.lo[2] * P.n + a[2] : 0;
    const int64_t base = ctx->fine_numbering[(gz * G + gy) * G + gx];
    for (int c = 0; c < P.s; ++c) dofs[(size_t)node * P.s + c] = (uint64_t)(base + c);
  }
  return SLOD_OK;
}

int slod_get_patch_local_dofs(const slod_ctx *ctx, int64_t patch, uint32_t *dofs, int32_t *n) {
  int rc = check_patch(ctx, patch);
  if (rc) return rc;
  const Params &P = ctx->P;
  const Geom g = make_geom(P, (int)patch);
  if (n) *n = g.Nf;
  if (!dofs) return SLOD_OK;
  std::vector<std::array<int, 3>> cells;
  patch_cells_rel(P, g, cells);
  std::vector<int64_t> num;
  const int shape[3] = {g.p[0], g.p[1], g.p[2]};
  const int origin[3] = {0, 0, 0};
  numbering_walk(P.dim, P.s, P.n, cells.size(),
                 [&](size_t c, int cc[3]) { cc[0] = cells[c][0]; cc[1] = cells[c][1]; cc[2] = cells[c][2]; }, shape,
                 origin, num);
  for (int node = 0; node < g.nnodes; ++node)
    for (int c = 0; c < P.s; ++c) dofs[(size_t)node * P.s + c] = (uint32_t)(num[node] + c);
  return SLOD_OK;
}

int slod_get_patch_dof_class(const slod_ctx *ctx, int64_t patch, int which, uint32_t *dofs, int32_t *n) {
  int rc = check_patch(ctx, patch);
  if (rc) return rc;
  if (which < 0 || which > 2) return fail(ctx, SLOD_ERR_INVALID, "which must be 0, 1 or 2");
  const Params &P = ctx->P;
  const Geom g = make_geom(P, (int)patch);
  int cnt = 0;
  for (int node = 0; node < g.nnodes; ++node) {
    int a[3];
    node_coords(g, node, a);
    const int c = node_class(P, g, a);
    const bool in = (which == 0) ? (c == 0) : (which == 1 ? (c & 1) : (c & 2));
    if (!in) continue;
    for (int k = 0; k < P.s; ++k) {
      if (dofs) dofs[cnt] = (uint32_t)(node * P.s + k);
      ++cnt;
    }
  }
  if (n) *n = cnt;
  return SLOD_OK;
}

int slod_basis_stride(const slod_ctx *ctx, int64_t *stride) {
  if (!ctx || !stride) return SLOD_ERR_INVALID;
  *stride = ctx->P.NfMax;
  return SLOD_OK;
}
int slod_ell_width(const slod_ctx *ctx, int64_t *width) {
  if (!ctx || !width) return SLOD_ERR_INVALID;
  *width = ctx->P.ell_width;
  return SLOD_OK;
}
int slod_launch_count(const slod_ctx *ctx, int64_t *n) {
  if (!ctx || !n) return SLOD_ERR_INVALID;
  *n = ctx->launches;
  return SLOD_OK;
}

int slod_compute_basis_device(slod_ctx *ctx, int64_t p0, int64_t p1, double *d_phi, double *d_aphi, void *stream) {
  if (!ctx || !d_phi || !d_aphi) return SLOD_ERR_INVALID;
  NEED_DEVICE();
  if (!ctx->subs.empty()) return fail(ctx, SLOD_ERR_UNSUPPORTED, "device-buffer entry points need a single-device handle (n_gpus <= 1)");
  CK(cudaSetDevice(ctx->device));
  ctx->have_base = ctx->base_coarse = false;   // the handle's diagnostics and status words now describe this run
  return run_basis(ctx, p0, p1, d_phi, d_aphi, (cudaStream_t)stream);
}

int slod_assemble_coarse_device(slod_ctx *ctx, int64_t p0, int64_t p1, const double *d_phi, const double *d_aphi,
                                double *d_K, void *stream) {
  if (!ctx || !d_phi || !d_aphi || !d_K) return SLOD_ERR_INVALID;
  NEED_DEVICE();
  if (!ctx->subs.empty()) return fail(ctx, SLOD_ERR_UNSUPPORTED, "device-buffer entry points need a single-device handle (n_gpus <= 1)");
  CK(cudaSetDevice(ctx->device));
  return run_coarse(ctx, p0, p1, d_phi, d_aphi, d_K, (cudaStream_t)stream, false);   // enqueue only, see slod_synchronize
}

int slod_compute_basis(slod_ctx *ctx) {
  if (!ctx) return SLOD_ERR_INVALID;
  NEED_DEVICE();
  CK(cudaSetDevice(ctx->device));
  const size_t n = (size_t)ctx->n_patches * ctx->P.s * ctx->P.NfMax;
  if (!ctx->d_phi) {
    CK(cudaMalloc(&ctx->d_phi, sizeof(double) * n));
    CK(cudaMalloc(&ctx->d_aphi, sizeof(double) * n));
  }
  ctx->basis_done = ctx->coarse_done = false;
  ctx->have_base = ctx->base_coarse = false;
  invalidate_mass(ctx);
  if (!ctx->subs.empty()) return multi_basis(ctx);
  int rc = run_basis(ctx, 0, ctx->n_patches, ctx->d_phi, ctx->d_aphi, 0);
  if (rc) return rc;
  rc = snapshot_coefficients(ctx);
  if (rc) return rc;
  rc = wait_basis(ctx);
  if (rc) return rc;
  ctx->basis_done = ctx->have_base = true;
  return SLOD_OK;
}

int slod_owned_range(const slod_ctx *ctx, int rank, int world, int64_t *b, int64_t *e) {
  if (!ctx || !b || !e) return SLOD_ERR_INVALID;
  if (world < 1 || rank < 0 || rank >= world) return fail(ctx, SLOD_ERR_INVALID, "rank out of range");
  owned_range(ctx->n_patches, rank, world, b, e);
  return SLOD_OK;
}

int slod_comm_unique_id(void *id128) {
  if (!id128) return SLOD_ERR_INVALID;
  NcclApi *nc = nccl_api();
  if (!nc->err.empty()) {
    g_create_error = nc->err;
    return SLOD_ERR_CUDA;
  }
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
  ncclUniqueId id;
  if (nc->GetUniqueId(&id) != ncclSuccess) return SLOD_ERR_CUDA;
  std::memcpy(id128, &id, sizeof id);
  return SLOD_OK;
}

int slod_comm_init(slod_ctx *ctx, int rank, int world, const void *id128) {
  if (!ctx || !id128) return SLOD_ERR_INVALID;
  NEED_DEVICE();
  if (!ctx->subs.empty()) return fail(ctx, SLOD_ERR_STATE, "handle already drives several devices (n_gpus > 1)");
  if (ctx->comm) return fail(ctx, SLOD_ERR_STATE, "communicator already initialised");
  if (world < 1 || rank < 0 || rank >= world) return fail(ctx, SLOD_ERR_INVALID, "rank out of range");
  NcclApi *nc = nccl_api();
  if (!nc->err.empty()) return fail(ctx, SLOD_ERR_CUDA, nc->err);
  CK(cudaSetDevice(ctx->device));
  ncclUniqueId id;
  std::memcpy(&id, id128, sizeof id);
  NK(nc->CommInitRank(&ctx->comm, world, id, rank));
  ctx->comm_rank = rank;
  ctx->comm_world = world;
  return SLOD_OK;
}

int slod_offline_distributed(slod_ctx *ctx, double *d_phi, double *d_aphi, double *d_K, int gather_phi, int gather_K,
                             void *stream) {
  if (!ctx || !d_phi || !d_aphi || !d_K) return SLOD_ERR_INVALID;
  NEED_DEVICE();
  if (!ctx->subs.empty()) return fail(ctx, SLOD_ERR_UNSUPPORTED, "use slod_compute_basis / slod_assemble_coarse on an n_gpus > 1 handle");
  if (ctx->comm_world > 1 && !ctx->comm) return fail(ctx, SLOD_ERR_STATE, "slod_comm_init has not run");
  CK(cudaSetDevice(ctx->device));
  ctx->have_base = ctx->base_coarse = false;   // the handle's diagnostics and status words now describe this run
  cudaStream_t st = (cudaStream_t)stream;
  int64_t b, e;
  owned_range(ctx->n_patches, ctx->comm_rank, ctx->comm_world, &b, &e);
  const size_t per_patch = (size_t)ctx->P.s * ctx->P.NfMax;
  int rc = run_basis(ctx, b, e, d_phi, d_aphi, st);
  if (rc) return rc;
  const bool host_out = ctx->h_out_phi || ctx->h_out_aphi || ctx->h_out_K;
  if (host_out) {
    if (!ctx->copy_stream) CK(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    for (auto &ev : ctx->ev_out)
      if (!ev) CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    CK(cudaEventRecord(ctx->ev_out[0], st));
    CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_out[0], 0));
    const size_t off = (size_t)b * per_patch, cnt = (size_t)(e - b) * per_patch;
    if (ctx->h_out_phi) CK(cudaMemcpyAsync(ctx->h_out_phi, d_phi + off, sizeof(double) * cnt, cudaMemcpyDeviceToHost, ctx->copy_stream));
    if (ctx->h_out_aphi) CK(cudaMemcpyAsync(ctx->h_out_aphi, d_aphi + off, sizeof(double) * cnt, cudaMemcpyDeviceToHost, ctx->copy_stream));
    ctx->out_pending = true;
  }
  if (ctx->comm_world > 1) {
    rc = gather_blocks(ctx, d_aphi, per_patch, st);
    if (rc) return rc;
    if (gather_phi && (rc = gather_blocks(ctx, d_phi, per_patch, st))) return rc;
  }
  rc = run_coarse(ctx, b, e, d_phi, d_aphi, d_K, st, false);
  if (rc) return rc;
  if (host_out && ctx->h_out_K) {
    const size_t per_k = (size_t)ctx->P.s * ctx->P.ell_width;
    CK(cudaEventRecord(ctx->ev_out[1], st));
    CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_out[1], 0));
    CK(cudaMemcpyAsync(ctx->h_out_K, d_K + (size_t)b * per_k, sizeof(double) * (size_t)(e - b) * per_k, cudaMemcpyDeviceToHost,
                       ctx->copy_stream));
  }
  if (ctx->comm_world > 1 && gather_K) rc = gather_blocks(ctx, d_K, (size_t)ctx->P.s * ctx->P.ell_width, st);
  return rc;
}

int slod_set_host_outputs(slod_ctx *ctx, double *h_phi, double *h_aphi, double *h_K) {
  if (!ctx) return SLOD_ERR_INVALID;
  NEED_DEVICE();
  ctx->h_out_phi = h_phi;
  ctx->h_out_aphi = h_aphi;
  ctx->h_out_K = h_K;
  return SLOD_OK;
}

int slod_synchronize(slod_ctx *ctx) {
  if (!ctx) return SLOD_ERR_INVALID;
  NEED_DEVICE();
  CK(cudaSetDevice(ctx->device));
  int rc = wait_basis(ctx);
  if (rc) return rc;
  rc = finish_coarse_timing(ctx);
  if (rc) return rc;
  if (ctx->out_pending) {
    ctx->out_pending = false;
    CK(cudaStreamSynchronize(ctx->copy_stream));
  }
  return SLOD_OK;
}

int slod_get_basis(const slod_ctx *ctx, int64_t patch, int comp, double *phi, double *aphi) {
  int rc = check_patch(ctx, patch);
  if (rc) return rc;
  if (!ctx->basis_done) return fail(ctx, SLOD_ERR_STATE, "slod_compute_basis has not run");
  if (comp < 0 || comp >= ctx->P.s) return fail(ctx, SLOD_ERR_INVALID, "component out of range");
  const Geom g = make_geom(ctx->P, (int)patch);
  const size_t off = ((size_t)patch * ctx->P.s + comp) * ctx->P.NfMax;
  CK(cudaSetDevice(ctx->device));
  if (phi) CK(cudaMemcpy(phi, ctx->d_phi + off, sizeof(double) * g.Nf, cudaMemcpyDeviceToHost));
  if (aphi) CK(cudaMemcpy(aphi, ctx->d_aphi + off, sizeof(double) * g.Nf, cudaMemcpyDeviceToHost));
  return SLOD_OK;
}

int slod_get_all_basis(const slod_ctx *ctx, double *phi, double *aphi) {
  if (!ctx) return SLOD_ERR_INVALID;
  if (!ctx->basis_done) return fail(ctx, SLOD_ERR_STATE, "slod_compute_basis has not run");
  const size_t n = (size_t)ctx->n_patches * ctx->P.s * ctx->P.NfMax;
  CK(cudaSetDevice(ctx->device));
  // slod_compute_basis returned synchronised, so the basis is complete; the copies go through a non-blocking stream and
  // overlap whatever slod_assemble_coarse has in flight
  slod_ctx *c = const_cast<slod_ctx *>(ctx);
  if (!c->copy_stream) CK(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
  if (phi) CK(cudaMemcpyAsync(phi, ctx->d_phi, sizeof(double) * n, cudaMemcpyDeviceToHost, c->copy_stream));
  if (aphi) CK(cudaMemcpyAsync(aphi, ctx->d_aphi, sizeof(double) * n, cudaMemcpyDeviceToHost, c->copy_stream));
  CK(cudaStreamSynchronize(c->copy_stream));
  return SLOD_OK;
}

// CSR pattern + ELL->CSR permutation: integer geometry, built on the first call and kept for the life of the handle
static int build_csr_cache(slod_ctx *ctx) {
  if (ctx->csr_ready) return SLOD_OK;
  int64_t n_rows = 0, nnz = 0;
  int rc = ell_to_csr(ctx, nullptr, nullptr, nullptr, nullptr, &n_rows, &nnz);
  if (rc) return rc;
  ctx->csr_rowptr.resize((size_t)n_rows + 1);
  ctx->csr_col.resize((size_t)nnz);
  std::vector<long long> perm((size_t)nnz);
  rc = ell_to_csr(ctx, nullptr, ctx->csr_rowptr.data(), ctx->csr_col.data(), nullptr, &n_rows, &nnz, perm.data());
  if (rc) return rc;
  CK(cudaMalloc(&ctx->d_perm, sizeof(long long) * std::max<size_t>(1, (size_t)nnz)));
  CK(cudaMalloc(&ctx->d_val, sizeof(double) * std::max<size_t>(1, (size_t)nnz)));
  CK(cudaMemcpy(ctx->d_perm, perm.data(), sizeof(long long) * (size_t)nnz, cudaMemcpyHostToDevice));
  ctx->csr_nnz = nnz;
  ctx->csr_ready = true;
  return SLOD_OK;
}

static void parallel_copy(void *dst, const void *src, size_t bytes) {
  const unsigned nthr = std::max(1u, std::min(8u, std::thread::hardware_concurrency()));
  if (bytes < ((size_t)8 << 20) || nthr == 1) {
    std::memcpy(dst, src, bytes);
    return;
  }
  std::vector<std::thread> th;
  const size_t per = (bytes + nthr - 1) / nthr;
  for (unsigned t = 0; t < nthr; ++t) {
    const size_t off = (size_t)t * per;
    if (off >= bytes) break;
    th.emplace_back([=]() { std::memcpy((char *)dst + off, (const char *)src + off, std::min(per, bytes - off)); });
  }
  for (auto &x : th) x.join();
}

int slod_assemble_coarse(slod_ctx *ctx) {
  if (!ctx) return SLOD_ERR_INVALID;
  NEED_DEVICE();
  if (!ctx->basis_done) return fail(ctx, SLOD_ERR_STATE, "slod_compute_basis has not run");
  CK(cudaSetDevice(ctx->device));
  const size_t n = (size_t)ctx->n_patches * ctx->P.s * ctx->P.ell_width;
  if (!ctx->d_Kell) CK(cudaMalloc(&ctx->d_Kell, sizeof(double) * n));
  // The kernels are only enqueued: slod_get_all_basis (own copy stream) can run while they execute, every consumer of
  // the matrix is stream ordered behind them, and an execution error surfaces at that consumer's synchronisation.
  int rc = build_csr_cache(ctx);   // first call only: host-side integer geometry, before the kernels are in flight
  if (rc) return rc;
  invalidate_mass(ctx);
  if (!ctx->subs.empty())
    rc = multi_coarse(ctx);   // row blocks on N devices + NCCL all-gather; the matrix is complete on return
  else
    rc = run_coarse(ctx, 0, ctx->n_patches, ctx->d_phi, ctx->d_aphi, ctx->d_Kell, 0, false);
  if (rc) return rc;
  CK(launch_gather(0, ctx->d_Kell, ctx->d_perm, ctx->d_val, ctx->csr_nnz));   // compact block-ELL -> CSR values
  ctx->launches += 1;
  ctx->coarse_done = true;
  ctx->base_coarse = ctx->have_base;
  return SLOD_OK;
}

// A patch reads the coefficient window of the coarse cells [clo, clo + m) (load_coef, kernels.cu): it is recomputed iff
// one of those cells holds a value that differs bitwise from the baseline.  A row block of K depends on phi of its patch
// and on A phi of the column patches of its CSR row; the pattern is symmetric, so the rows to recompute are the CSR
// columns of the recomputed patches' rows.
int slod_update_basis(slod_ctx *ctx, int64_t *n_patches_recomputed, int64_t *n_row_blocks_recomputed) {
  if (!ctx) return SLOD_ERR_INVALID;
  if (n_patches_recomputed) *n_patches_recomputed = 0;
  if (n_row_blocks_recomputed) *n_row_blocks_recomputed = 0;
  NEED_DEVICE();
  if (!ctx->subs.empty())
    return fail(ctx, SLOD_ERR_UNSUPPORTED, "slod_update_basis needs a single-device handle: an n_gpus > 1 handle splits "
                "the patches into fixed ranges per device, and a changed region falls into some of them only");
  if (!ctx->have_base)
    return fail(ctx, SLOD_ERR_STATE, "no baseline to update: slod_compute_basis has not succeeded on this handle since "
                "it was created, restored by slod_load_state or used by a device-buffer entry point");
  CK(cudaSetDevice(ctx->device));
  int rc = finish_coarse_timing(ctx);   // the times of an earlier slod_assemble_coarse are collected now, not later
  if (rc) return rc;
  rc = prepare_coefficients(ctx);
  if (rc) return rc;
  BIND_PARAMS((cudaStream_t)0);
  const Params &P = ctx->P;
  const int64_t np = ctx->n_patches;   // = N^dim coarse cells
  std::vector<unsigned char> changed((size_t)np, 1);
  if (ctx->base_elems == ctx->d_coef_elems && ctx->base_gauss == P.gauss_coef) {   // else the layout changed: all cells
    if (!ctx->d_cell_changed) CK(cudaMalloc(&ctx->d_cell_changed, (size_t)np));
    CK(launch_coef_diff(0, ctx->d_coef_base, ctx->d_coef, (long long)ctx->d_coef_elems, P.dim, P.N, P.n,
                        P.gauss_coef ? 1 << P.dim : 1, ctx->d_cell_changed));
    ctx->launches += 1;
    CK(cudaMemcpyAsync(changed.data(), ctx->d_cell_changed, (size_t)np, cudaMemcpyDeviceToHost, 0));
    CK(cudaStreamSynchronize(0));
  }
  // box sums of the flags: S(x, y, z) = changed cells below (x, y, z) on every axis
  const int N = P.N, Nz = (P.dim == 3) ? N : 1;
  std::vector<int> S((size_t)(N + 1) * (N + 1) * (Nz + 1), 0);
  auto at = [&](int x, int y, int z) -> int & { return S[((size_t)z * (N + 1) + y) * (N + 1) + x]; };
  for (int z = 0; z < Nz; ++z)
    for (int y = 0; y < N; ++y)
      for (int x = 0; x < N; ++x)
        at(x + 1, y + 1, z + 1) = changed[((size_t)z * N + y) * N + x] + at(x, y + 1, z + 1) + at(x + 1, y, z + 1) +
                                  at(x + 1, y + 1, z) - at(x, y, z + 1) - at(x, y + 1, z) - at(x + 1, y, z) + at(x, y, z);
  std::vector<int> &ids = ctx->update_ids;
  ids.clear();
  for (int64_t pid = 0; pid < np; ++pid) {
    const Geom g = make_geom(P, (int)pid);
    const int x0 = g.clo[0], y0 = g.clo[1], z0 = g.clo[2], x1 = x0 + g.m[0], y1 = y0 + g.m[1], z1 = z0 + g.m[2];
    const int n_changed = at(x1, y1, z1) - at(x0, y1, z1) - at(x1, y0, z1) - at(x1, y1, z0) + at(x0, y0, z1) +
                          at(x0, y1, z0) + at(x1, y0, z0) - at(x0, y0, z0);
    if (n_changed > 0) ids.push_back((int)pid);
  }
  if (n_patches_recomputed) *n_patches_recomputed = (int64_t)ids.size();
  for (int k = 0; k < 6; ++k) ctx->tm.ms[k] = 0.0;
  if (ids.empty()) {   // the basis (and K, if it was assembled) are those of the current coefficient already
    ctx->basis_done = true;
    ctx->coarse_done = ctx->base_coarse;
    return SLOD_OK;
  }
  ctx->basis_done = ctx->coarse_done = false;
  ctx->have_base = false;
  invalidate_mass(ctx);
  // the status words of every patch are cleared and read back: outside the list they are zero after the basis that
  // set the baseline, so the first nonzero word belongs to the first failing patch of the list, as in slod_compute_basis
  rc = run_basis(ctx, 0, np, ctx->d_phi, ctx->d_aphi, 0, &ids);
  if (rc) return rc;
  rc = snapshot_coefficients(ctx);
  if (rc) return rc;
  rc = wait_basis(ctx);
  if (rc) {
    ctx->base_coarse = false;
    return rc;
  }
  ctx->basis_done = ctx->have_base = true;
  if (!ctx->base_coarse) return SLOD_OK;
  std::vector<unsigned char> row((size_t)np, 0);
  const int s = P.s;
  for (int q : ids)
    for (int64_t k = ctx->csr_rowptr[(size_t)q * s]; k < ctx->csr_rowptr[(size_t)q * s + 1]; k += s)
      row[(size_t)(ctx->csr_col[k] / s)] = 1;
  std::vector<int> &rows = ctx->update_rows;   // Morton groups on the blocked kernel, patches otherwise
  rows.clear();
  const int gsz = (ctx->coarse_nu > 0) ? 1 << P.dim : 1;
  for (int64_t g = 0; g < np / gsz; ++g)
    if (std::any_of(row.begin() + g * gsz, row.begin() + (g + 1) * gsz, [](unsigned char v) { return v != 0; }))
      rows.push_back((int)g);
  rc = grow(ctx, ctx->d_rows, ctx->rows_cap, rows.size());
  if (rc) return rc;
  CK(cudaMemcpyAsync(ctx->d_rows, rows.data(), sizeof(int) * rows.size(), cudaMemcpyHostToDevice, 0));
  rc = run_coarse(ctx, 0, np, ctx->d_phi, ctx->d_aphi, ctx->d_Kell, 0, false, ctx->d_rows, (int)rows.size());
  if (rc) return rc;
  CK(launch_gather(0, ctx->d_Kell, ctx->d_perm, ctx->d_val, ctx->csr_nnz));
  ctx->launches += 1;
  ctx->coarse_done = true;
  if (n_row_blocks_recomputed) *n_row_blocks_recomputed = (int64_t)rows.size() * gsz;
  return SLOD_OK;
}

// CSR of K (mass == false) or of M_H (mass == true): the same pattern, values gathered on the device
static int get_csr(const slod_ctx *cctx, bool mass, int64_t *rowptr, int64_t *col, double *val, int64_t *n_rows,
                   int64_t *nnz) {
  if (!cctx) return SLOD_ERR_INVALID;
  slod_ctx *ctx = const_cast<slod_ctx *>(cctx);   // the pattern cache is filled lazily
  if (!rowptr) {
    if (ctx->csr_ready) {
      if (n_rows) *n_rows = (int64_t)ctx->csr_rowptr.size() - 1;
      if (nnz) *nnz = ctx->csr_nnz;
      return SLOD_OK;
    }
    return ell_to_csr(ctx, nullptr, nullptr, nullptr, nullptr, n_rows, nnz);
  }
  NEED_DEVICE();
  if (!mass && !ctx->coarse_done) return fail(ctx, SLOD_ERR_STATE, "slod_assemble_coarse has not run");
  if (mass && !ctx->mass_done) return fail(ctx, SLOD_ERR_STATE, "slod_assemble_coarse_mass has not run");
  if (!col || !val) return fail(ctx, SLOD_ERR_INVALID, "null output buffer");
  CK(cudaSetDevice(ctx->device));
  if (n_rows) *n_rows = (int64_t)ctx->csr_rowptr.size() - 1;
  if (nnz) *nnz = ctx->csr_nnz;
  CK(cudaMemcpyAsync(val, mass ? ctx->d_Mval : ctx->d_val, sizeof(double) * (size_t)ctx->csr_nnz,
                     cudaMemcpyDeviceToHost, 0));
  std::memcpy(rowptr, ctx->csr_rowptr.data(), sizeof(int64_t) * ctx->csr_rowptr.size());
  parallel_copy(col, ctx->csr_col.data(), sizeof(int64_t) * ctx->csr_col.size());
  CK(cudaStreamSynchronize(0));
  return SLOD_OK;
}

int slod_get_coarse_csr(const slod_ctx *ctx, int64_t *rowptr, int64_t *col, double *val, int64_t *n_rows,
                        int64_t *nnz) {
  return get_csr(ctx, false, rowptr, col, val, n_rows, nnz);
}

// ---- online phase on the handle's own basis and coarse matrix (SURVEY 8f row 1) ----
// One scratch block for all of these entry points (cudaMalloc / cudaFree per call costs milliseconds next to the tens
// of GB the handle has mapped): [2 fine vectors | 2 coarse vectors | CG workspace of the larger problem].
static int online_scratch(slod_ctx *ctx, double **fine_a, double **fine_b, double **coarse_a, double **coarse_b,
                          double **work) {
  int64_t n_fine = 0;
  slod_fine_size(ctx, &n_fine);
  const size_t nc = (size_t)ctx->n_patches * ctx->P.s;
  const CgOperator Ac{reinterpret_cast<const double *>(1), nullptr, 0}, Af{nullptr, nullptr, n_fine / ctx->P.s};
  const size_t wk = std::max(cg_workspace_doubles(Ac, (int)nc), cg_workspace_doubles(Af, (int)n_fine));
  const int rc = grow(ctx, ctx->d_online, ctx->online_doubles, 2 * (size_t)n_fine + 2 * nc + wk + 8);
  if (rc) return rc;
  double *p = ctx->d_online;
  if (fine_a) *fine_a = p;
  if (fine_b) *fine_b = p + n_fine;
  if (coarse_a) *coarse_a = p + 2 * n_fine;
  if (coarse_b) *coarse_b = p + 2 * n_fine + nc;
  if (work) *work = p + 2 * n_fine + 2 * nc;
  return SLOD_OK;
}

static int check_solver_control(slod_ctx *ctx, int32_t max_steps, double tolerance, double reduction) {
  if (max_steps < 0 || !(tolerance >= 0.0) || !(reduction >= 0.0))
    return fail(ctx, SLOD_ERR_INVALID, "solver control: max_steps, tolerance and reduction must be non-negative");
  return SLOD_OK;
}

static int check_n_rhs(slod_ctx *ctx, int32_t n_rhs) {
  return n_rhs < 1 ? fail(ctx, SLOD_ERR_INVALID, "n_rhs must be at least 1") : SLOD_OK;
}

// The end of an online or heat entry point: stream 0 is synchronised unless a step failed already, the call's launches
// are counted, and a CUDA error becomes SLOD_ERR_CUDA under the entry point's name.
static int finish_call(slod_ctx *ctx, const char *name, cudaError_t e, long long n_launch) {
  if (e == cudaSuccess) e = cudaStreamSynchronize(0);
  ctx->launches += n_launch;
  if (e != cudaSuccess) return fail(ctx, SLOD_ERR_CUDA, std::string(name) + ": " + cudaGetErrorString(e));
  return SLOD_OK;
}

// The outcome of one CG run: SLOD_OK if it converged (flag 1), else SLOD_ERR_NUMERIC (where deal.II throws
// SolverControl::NoConvergence) with a message naming the time step (step > 0), the column (column >= 0), the solver and
// its matrix, and the coefficient c of a matrix M + c A (c > 0).
static int cg_outcome(slod_ctx *ctx, int step, int column, const char *label, double c, int flag, int steps,
                      double res) {
  if (flag == 1) return SLOD_OK;
  std::string msg = step > 0 ? "time step " + std::to_string(step) : std::string();
  if (column >= 0) msg += (msg.empty() ? "column " : " column ") + std::to_string(column);
  if (!msg.empty()) msg += ": ";
  msg += label;
  char buf[160];
  if (c > 0) {
    std::snprintf(buf, sizeof buf, " (c = %.6g)", c);
    msg += buf;
  }
  std::snprintf(buf, sizeof buf, " %s after %d steps (residual %.3e)%s", flag == 2 ? "broke down" : "did not converge",
                steps, res, flag == 2 ? ": the matrix is not positive definite" : "");
  return fail(ctx, SLOD_ERR_NUMERIC, msg + buf);
}

int slod_fine_size(const slod_ctx *ctx, int64_t *n_fine) {
  if (!ctx || !n_fine) return SLOD_ERR_INVALID;
  int64_t n = ctx->P.s;
  for (int a = 0; a < ctx->P.dim; ++a) n *= (int64_t)ctx->P.nsub + 1;
  *n_fine = n;
  return SLOD_OK;
}

int slod_coarse_rhs(slod_ctx *ctx, const double *f_fine, double *rhs_coarse) {
  if (!ctx) return SLOD_ERR_INVALID;
  NEED_DEVICE();
  if (!ctx->basis_done) return fail(ctx, SLOD_ERR_STATE, "slod_compute_basis has not run");
  if (!f_fine || !rhs_coarse) return fail(ctx, SLOD_ERR_INVALID, "null buffer");
  CK(cudaSetDevice(ctx->device));
  BIND_PARAMS((cudaStream_t)0);
  int64_t n_fine = 0;
  slod_fine_size(ctx, &n_fine);
  const size_t nc = (size_t)ctx->n_patches * ctx->P.s;
  double *d_f = nullptr, *d_b = nullptr;
  int rc = online_scratch(ctx, &d_f, nullptr, &d_b, nullptr, nullptr);
  if (rc) return rc;
  cudaError_t e = cudaMemcpyAsync(d_f, f_fine, sizeof(double) * (size_t)n_fine, cudaMemcpyHostToDevice, 0);
  if (e == cudaSuccess) e = launch_coarse_rhs(0, (int)ctx->n_patches, ctx->P.s, ctx->d_phi, d_f, d_b, ctx->P.NfMax);
  if (e == cudaSuccess) e = cudaMemcpyAsync(rhs_coarse, d_b, sizeof(double) * nc, cudaMemcpyDeviceToHost, 0);
  return finish_call(ctx, "slod_coarse_rhs", e, 1);
}

int slod_coarse_solve(slod_ctx *ctx, const double *rhs_coarse, double *u_coarse, int32_t max_steps, double tolerance,
                      double reduction, int32_t *steps, double *residual) {
  if (!ctx) return SLOD_ERR_INVALID;
  NEED_DEVICE();
  if (!ctx->coarse_done) return fail(ctx, SLOD_ERR_STATE, "slod_assemble_coarse has not run");
  if (!rhs_coarse || !u_coarse) return fail(ctx, SLOD_ERR_INVALID, "null buffer");
  int rc = check_solver_control(ctx, max_steps, tolerance, reduction);
  if (rc) return rc;
  CK(cudaSetDevice(ctx->device));
  BIND_PARAMS((cudaStream_t)0);
  const int nrows = (int)(ctx->n_patches * ctx->P.s);
  double *d_b = nullptr, *d_x = nullptr, *d_work = nullptr;
  rc = online_scratch(ctx, nullptr, nullptr, &d_b, &d_x, &d_work);
  if (rc) return rc;
  const CgOperator A{ctx->d_Kell, nullptr, 0};
  cudaError_t e = cudaSuccess;
  int st_steps = 0, flag = 0;
  long long n_launch = 0;
  double res = 0.0;
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_b, rhs_coarse, sizeof(double) * nrows, cudaMemcpyHostToDevice, 0);
  if (e == cudaSuccess)
    e = run_cg(0, nrows, A, d_b, d_x, d_work, max_steps, tolerance, reduction, &st_steps, &res, &flag,
                      &n_launch);
  if (e == cudaSuccess) e = cudaMemcpyAsync(u_coarse, d_x, sizeof(double) * nrows, cudaMemcpyDeviceToHost, 0);
  rc = finish_call(ctx, "slod_coarse_solve", e, n_launch);
  if (steps) *steps = st_steps;
  if (residual) *residual = res;
  if (rc) return rc;
  return cg_outcome(ctx, 0, -1, "coarse CG on K", 0.0, flag, st_steps, res);
}

int slod_prolongate(slod_ctx *ctx, const double *u_coarse, double *u_fine) {
  if (!ctx) return SLOD_ERR_INVALID;
  NEED_DEVICE();
  if (!ctx->basis_done) return fail(ctx, SLOD_ERR_STATE, "slod_compute_basis has not run");
  if (!u_coarse || !u_fine) return fail(ctx, SLOD_ERR_INVALID, "null buffer");
  CK(cudaSetDevice(ctx->device));
  BIND_PARAMS((cudaStream_t)0);
  int64_t n_fine = 0;
  slod_fine_size(ctx, &n_fine);
  const size_t nc = (size_t)ctx->n_patches * ctx->P.s;
  double *d_u = nullptr, *d_f = nullptr;
  int rc = online_scratch(ctx, &d_f, nullptr, &d_u, nullptr, nullptr);
  if (rc) return rc;
  cudaError_t e = cudaSuccess;
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_u, u_coarse, sizeof(double) * nc, cudaMemcpyHostToDevice, 0);
  if (e == cudaSuccess) e = launch_prolongate(0, n_fine, ctx->d_phi, d_u, d_f, ctx->P.NfMax);
  if (e == cudaSuccess) e = cudaMemcpyAsync(u_fine, d_f, sizeof(double) * (size_t)n_fine, cudaMemcpyDeviceToHost, 0);
  return finish_call(ctx, "slod_prolongate", e, 1);
}

// ---- batched online phase: groups of at most kBatch right-hand sides (online_batch.cuh) ----
// One scratch block, allocated on first use and regrown when too small; its size depends on kBatch, not on n_rhs:
// [fine staging | fine interleaved | coarse staging | coarse interleaved a | b | CG workspace].  A group's host block
// ([kb][n], contiguous in the caller's [n_rhs][n] array) is copied in one piece to the staging block and transposed on
// the device; results go the other way.
struct BatchScratch {
  double *fine_stage, *fine, *coarse_stage, *coarse_a, *coarse_b, *work;
};
static int batch_scratch(slod_ctx *ctx, BatchScratch *b) {
  int64_t n_fine = 0;
  slod_fine_size(ctx, &n_fine);
  const size_t nc = (size_t)ctx->n_patches * ctx->P.s;
  const int rc = grow(ctx, ctx->d_batch, ctx->batch_doubles,
                      2 * (size_t)kBatch * n_fine + 3 * (size_t)kBatch * nc + cg_multi_workspace_doubles((int)nc) + 8);
  if (rc) return rc;
  double *p = ctx->d_batch;
  b->fine_stage = p;
  b->fine = p + (size_t)kBatch * n_fine;
  b->coarse_stage = b->fine + (size_t)kBatch * n_fine;
  b->coarse_a = b->coarse_stage + (size_t)kBatch * nc;
  b->coarse_b = b->coarse_a + (size_t)kBatch * nc;
  b->work = b->coarse_b + (size_t)kBatch * nc;
  return SLOD_OK;
}

// One group of kb columns of length n between the caller's host block [kb][n] and an interleaved device array [n][kb],
// through the staging block
static cudaError_t upload_group(const double *host, long long n, int kb, double *stage, double *dev) {
  const cudaError_t e = cudaMemcpyAsync(stage, host, sizeof(double) * kb * (size_t)n, cudaMemcpyHostToDevice, 0);
  return e == cudaSuccess ? launch_interleave(0, n, kb, stage, dev, true) : e;
}
static cudaError_t download_group(const double *dev, long long n, int kb, double *stage, double *host) {
  const cudaError_t e = launch_interleave(0, n, kb, dev, stage, false);
  if (e != cudaSuccess) return e;
  return cudaMemcpyAsync(host, stage, sizeof(double) * kb * (size_t)n, cudaMemcpyDeviceToHost, 0);
}

int slod_coarse_rhs_batch(slod_ctx *ctx, int32_t n_rhs, const double *f_fine, double *rhs_coarse) {
  if (!ctx) return SLOD_ERR_INVALID;
  NEED_DEVICE();
  if (!ctx->basis_done) return fail(ctx, SLOD_ERR_STATE, "slod_compute_basis has not run");
  if (!f_fine || !rhs_coarse) return fail(ctx, SLOD_ERR_INVALID, "null buffer");
  int rc = check_n_rhs(ctx, n_rhs);
  if (rc) return rc;
  CK(cudaSetDevice(ctx->device));
  BIND_PARAMS((cudaStream_t)0);
  int64_t n_fine = 0;
  slod_fine_size(ctx, &n_fine);
  const size_t nc = (size_t)ctx->n_patches * ctx->P.s;
  BatchScratch w{};
  rc = batch_scratch(ctx, &w);
  if (rc) return rc;
  cudaError_t e = cudaSuccess;
  long long n_launch = 0;
  for (int j0 = 0; j0 < n_rhs && e == cudaSuccess; j0 += kBatch) {
    const int kb = std::min(kBatch, n_rhs - j0);
    e = upload_group(f_fine + (size_t)j0 * n_fine, n_fine, kb, w.fine_stage, w.fine);
    if (e == cudaSuccess)
      e = launch_coarse_rhs_multi(0, (int)ctx->n_patches, ctx->P.s, kb, ctx->d_phi, w.fine, w.coarse_a, ctx->P.NfMax);
    if (e == cudaSuccess)
      e = download_group(w.coarse_a, (long long)nc, kb, w.coarse_stage, rhs_coarse + (size_t)j0 * nc);
    n_launch += 3;
  }
  return finish_call(ctx, "slod_coarse_rhs_batch", e, n_launch);
}

int slod_coarse_solve_batch(slod_ctx *ctx, int32_t n_rhs, const double *rhs_coarse, double *u_coarse,
                            int32_t max_steps, double tolerance, double reduction, int32_t *steps, double *residual) {
  if (!ctx) return SLOD_ERR_INVALID;
  NEED_DEVICE();
  if (!ctx->coarse_done) return fail(ctx, SLOD_ERR_STATE, "slod_assemble_coarse has not run");
  if (!rhs_coarse || !u_coarse) return fail(ctx, SLOD_ERR_INVALID, "null buffer");
  int rc = check_n_rhs(ctx, n_rhs);
  if (rc) return rc;
  rc = check_solver_control(ctx, max_steps, tolerance, reduction);
  if (rc) return rc;
  CK(cudaSetDevice(ctx->device));
  BIND_PARAMS((cudaStream_t)0);
  const int nrows = (int)(ctx->n_patches * ctx->P.s);
  BatchScratch w{};
  rc = batch_scratch(ctx, &w);
  if (rc) return rc;
  std::vector<int> st_steps(n_rhs, 0), flag(n_rhs, 0);
  std::vector<double> res(n_rhs, 0.0);
  cudaError_t e = cudaSuccess;
  long long n_launch = 0;
  for (int j0 = 0; j0 < n_rhs && e == cudaSuccess; j0 += kBatch) {
    const int kb = std::min(kBatch, n_rhs - j0);
    e = upload_group(rhs_coarse + (size_t)j0 * nrows, nrows, kb, w.coarse_stage, w.coarse_a);
    if (e == cudaSuccess)
      e = run_cg_multi(0, nrows, ctx->d_Kell, kb, w.coarse_a, w.coarse_b, w.work, max_steps, tolerance, reduction,
                       &st_steps[j0], &res[j0], &flag[j0], &n_launch);
    if (e == cudaSuccess) e = download_group(w.coarse_b, nrows, kb, w.coarse_stage, u_coarse + (size_t)j0 * nrows);
    n_launch += 2;
  }
  rc = finish_call(ctx, "slod_coarse_solve_batch", e, n_launch);
  for (int j = 0; j < n_rhs; ++j) {
    if (steps) steps[j] = st_steps[j];
    if (residual) residual[j] = res[j];
  }
  // the first failing column; every column's u / steps / residual is written
  for (int j = 0; j < n_rhs && !rc; ++j)
    rc = cg_outcome(ctx, 0, j, "coarse CG on K", 0.0, flag[j], st_steps[j], res[j]);
  return rc;
}

int slod_prolongate_batch(slod_ctx *ctx, int32_t n_rhs, const double *u_coarse, double *u_fine) {
  if (!ctx) return SLOD_ERR_INVALID;
  NEED_DEVICE();
  if (!ctx->basis_done) return fail(ctx, SLOD_ERR_STATE, "slod_compute_basis has not run");
  if (!u_coarse || !u_fine) return fail(ctx, SLOD_ERR_INVALID, "null buffer");
  int rc = check_n_rhs(ctx, n_rhs);
  if (rc) return rc;
  CK(cudaSetDevice(ctx->device));
  BIND_PARAMS((cudaStream_t)0);
  int64_t n_fine = 0;
  slod_fine_size(ctx, &n_fine);
  const size_t nc = (size_t)ctx->n_patches * ctx->P.s;
  BatchScratch w{};
  rc = batch_scratch(ctx, &w);
  if (rc) return rc;
  cudaError_t e = cudaSuccess;
  long long n_launch = 0;
  for (int j0 = 0; j0 < n_rhs && e == cudaSuccess; j0 += kBatch) {
    const int kb = std::min(kBatch, n_rhs - j0);
    e = upload_group(u_coarse + (size_t)j0 * nc, (long long)nc, kb, w.coarse_stage, w.coarse_a);
    if (e == cudaSuccess) e = launch_prolongate_multi(0, n_fine, kb, ctx->d_phi, w.coarse_a, w.fine, ctx->P.NfMax);
    if (e == cudaSuccess) e = download_group(w.fine, n_fine, kb, w.fine_stage, u_fine + (size_t)j0 * n_fine);
    n_launch += 3;
  }
  return finish_call(ctx, "slod_prolongate_batch", e, n_launch);
}

// ---- fine-scale reference problem and norms (SURVEY 8f row 2) ----
// Homogeneous Dirichlet conditions (source/LOD.cc:1021-1027): the rows of the boundary nodes of the global grid are
// zeroed in the k fine vectors v [k][n_fine]
static void zero_boundary_rows(const Params &P, double *v, int k, int64_t n_fine) {
  const long long G = P.nsub + 1, n_nodes = n_fine / P.s;
  for (long long node = 0; node < n_nodes; ++node) {
    long long r = node;
    bool bd = false;
    for (int a = 0; a < P.dim; ++a) {
      const long long i = r % G;
      r /= G;
      bd = bd || i == 0 || i == G - 1;
    }
    if (bd)
      for (int q = 0; q < k; ++q)
        for (int c = 0; c < P.s; ++c) v[(size_t)q * n_fine + node * P.s + c] = 0.0;
  }
}

int slod_fem_solve(slod_ctx *ctx, const double *f_fine, double *u_fine, int32_t max_steps, double tolerance,
                   double reduction, int32_t *steps, double *residual) {
  if (!ctx) return SLOD_ERR_INVALID;
  NEED_DEVICE();
  if (!f_fine || !u_fine) return fail(ctx, SLOD_ERR_INVALID, "null buffer");
  int rc = check_solver_control(ctx, max_steps, tolerance, reduction);
  if (rc) return rc;
  CK(cudaSetDevice(ctx->device));
  rc = prepare_coefficients(ctx);
  if (rc) return rc;
  BIND_PARAMS((cudaStream_t)0);
  const Params &P = ctx->P;
  int64_t n_fine = 0;
  slod_fine_size(ctx, &n_fine);
  const long long n_nodes = n_fine / P.s;
  std::vector<double> f(f_fine, f_fine + n_fine);   // the boundary rows of the right-hand side are constrained away
  zero_boundary_rows(P, f.data(), 1, n_fine);
  const CgOperator A{nullptr, ctx->d_coef, n_nodes};
  double *d_b = nullptr, *d_x = nullptr, *d_work = nullptr;
  rc = online_scratch(ctx, &d_b, &d_x, nullptr, nullptr, &d_work);
  if (rc) return rc;
  cudaError_t e = cudaSuccess;
  int st_steps = 0, flag = 0;
  long long n_launch = 0;
  double res = 0.0;
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_b, f.data(), sizeof(double) * (size_t)n_fine, cudaMemcpyHostToDevice, 0);
  if (e == cudaSuccess)
    e = run_cg(0, (int)n_fine, A, d_b, d_x, d_work, max_steps, tolerance, reduction, &st_steps, &res, &flag, &n_launch);
  if (e == cudaSuccess) e = cudaMemcpyAsync(u_fine, d_x, sizeof(double) * (size_t)n_fine, cudaMemcpyDeviceToHost, 0);
  rc = finish_call(ctx, "slod_fem_solve", e, n_launch);
  if (steps) *steps = st_steps;
  if (residual) *residual = res;
  if (rc) return rc;
  return cg_outcome(ctx, 0, -1, "fine CG on A_h", 0.0, flag, st_steps, res);
}

int slod_fine_norms(slod_ctx *ctx, const double *v_fine, double *l2, double *h1_semi, double *energy) {
  if (!ctx) return SLOD_ERR_INVALID;
  NEED_DEVICE();
  if (!v_fine) return fail(ctx, SLOD_ERR_INVALID, "null buffer");
  CK(cudaSetDevice(ctx->device));
  int rc = prepare_coefficients(ctx);
  if (rc) return rc;
  BIND_PARAMS((cudaStream_t)0);
  int64_t n_fine = 0;
  slod_fine_size(ctx, &n_fine);
  const long long n_nodes = n_fine / ctx->P.s;
  int nb = 0;
  launch_fine_quadratic_form(0, kFineMass, n_nodes, nullptr, nullptr, nullptr, &nb);
  double *d_v = nullptr, *d_part = nullptr;   // 3 nb <= n_fine: the partial sums fit the second fine vector
  rc = online_scratch(ctx, &d_v, &d_part, nullptr, nullptr, nullptr);
  if (rc) return rc;
  cudaError_t e = cudaSuccess;
  std::vector<double> part(3 * (size_t)nb);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_v, v_fine, sizeof(double) * (size_t)n_fine, cudaMemcpyHostToDevice, 0);
  const int ops[3] = {kFineMass, kFineLaplace, kFineEnergy};
  for (int k = 0; k < 3 && e == cudaSuccess; ++k)
    e = launch_fine_quadratic_form(0, ops[k], n_nodes, ctx->d_coef, d_v, d_part + (size_t)k * nb, &nb);
  if (e == cudaSuccess)
    e = cudaMemcpyAsync(part.data(), d_part, sizeof(double) * part.size(), cudaMemcpyDeviceToHost, 0);
  rc = finish_call(ctx, "slod_fine_norms", e, 3);
  if (rc) return rc;
  double sum[3] = {0, 0, 0};
  for (int k = 0; k < 3; ++k)
    for (int i = 0; i < nb; ++i) sum[k] += part[(size_t)k * nb + i];   // block order: reproducible
  if (l2) *l2 = std::sqrt(std::max(sum[0], 0.0));
  if (h1_semi) *h1_semi = std::sqrt(std::max(sum[1], 0.0));
  if (energy) *energy = std::sqrt(std::max(sum[2], 0.0));
  return SLOD_OK;
}

// Gauss-Legendre rule on [0, 1] (Newton iteration on the Legendre polynomial)
static void gauss_rule(int nq, std::vector<double> &x, std::vector<double> &w) {
  x.resize(nq);
  w.resize(nq);
  for (int i = 0; i < nq; ++i) {
    double z = std::cos(M_PI * (i + 0.75) / (nq + 0.5)), pp = 1.0;
    for (int it = 0; it < 100; ++it) {
      double p1 = 1.0, p2 = 0.0;
      for (int j = 1; j <= nq; ++j) {
        const double p3 = p2;
        p2 = p1;
        p1 = ((2.0 * j - 1.0) * z * p2 - (j - 1.0) * p3) / j;
      }
      pp = nq * (z * p1 - p2) / (z * z - 1.0);
      const double dz = p1 / pp;
      z -= dz;
      if (std::fabs(dz) < 1e-15) break;
    }
    x[nq - 1 - i] = 0.5 * (1.0 + z);
    w[nq - 1 - i] = 1.0 / ((1.0 - z * z) * pp * pp);
  }
}

int slod_fine_norms_reference(slod_ctx *ctx, const double *v_fine, double *l2, double *linfty, double *h1) {
  if (!ctx) return SLOD_ERR_INVALID;
  NEED_DEVICE();
  if (!v_fine) return fail(ctx, SLOD_ERR_INVALID, "null buffer");
  CK(cudaSetDevice(ctx->device));
  BIND_PARAMS((cudaStream_t)0);
  int64_t n_fine = 0;
  slod_fine_size(ctx, &n_fine);
  const int nq = 2 * (ctx->P.n + 1);   // QGauss((fe.degree + 1) * 2), degree of FE_Q_iso_Q1(n) = n
  std::vector<double> gx, gw;
  gauss_rule(nq, gx, gw);
  int nb = 0;
  launch_fine_norms_reference(0, ctx->n_patches, nq, nullptr, nullptr, nullptr, nullptr, &nb);
  double *d_v = nullptr, *d_part = nullptr;   // second fine vector: Gauss rule (2 nq doubles) + 3 nb partial results
  int rc = online_scratch(ctx, &d_v, &d_part, nullptr, nullptr, nullptr);
  if (rc) return rc;
  if ((int64_t)(2 * nq + 3 * (int64_t)nb) > n_fine) return fail(ctx, SLOD_ERR_UNSUPPORTED, "mesh too small for the scratch layout");
  std::vector<double> part(3 * (size_t)nb);
  cudaError_t e = cudaMemcpyAsync(d_v, v_fine, sizeof(double) * (size_t)n_fine, cudaMemcpyHostToDevice, 0);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_part, gx.data(), sizeof(double) * nq, cudaMemcpyHostToDevice, 0);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_part + nq, gw.data(), sizeof(double) * nq, cudaMemcpyHostToDevice, 0);
  if (e == cudaSuccess)
    e = launch_fine_norms_reference(0, ctx->n_patches, nq, d_part, d_part + nq, d_v, d_part + 2 * nq, &nb);
  if (e == cudaSuccess)
    e = cudaMemcpyAsync(part.data(), d_part + 2 * nq, sizeof(double) * part.size(), cudaMemcpyDeviceToHost, 0);
  rc = finish_call(ctx, "slod_fine_norms_reference", e, 1);
  if (rc) return rc;
  double s2 = 0, sh = 0, mx = 0;
  for (int i = 0; i < nb; ++i) {   // block order: reproducible
    s2 += part[3 * (size_t)i];
    sh += part[3 * (size_t)i + 1];
    mx = std::max(mx, part[3 * (size_t)i + 2]);
  }
  if (l2) *l2 = std::sqrt(std::max(s2, 0.0));
  if (linfty) *linfty = mx;
  if (h1) *h1 = std::sqrt(std::max(s2 + sh, 0.0));
  return SLOD_OK;
}

// ---- heat equation on the SLOD space: coarse mass matrix, L2 projection, backward Euler ----
// M_H = C^T (M_h C) is formed like K: k_mass_apply writes M_h phi in the layout of A phi (a temporary the size of A phi)
// and the coarse-matrix kernel takes it in place of A phi.  The time steppers solve (M_H + dt K) u^k = M_H u^{k-1} + dt b
// in increment form, r = dt (b - K u^{k-1}), S delta = r, u^k = u^{k-1} + delta: the CG drivers start from zero, which is
// the previous step here.
int slod_assemble_coarse_mass(slod_ctx *ctx) {
  if (!ctx) return SLOD_ERR_INVALID;
  NEED_DEVICE();
  if (!ctx->basis_done) return fail(ctx, SLOD_ERR_STATE, "slod_compute_basis has not run");
  CK(cudaSetDevice(ctx->device));
  BIND_PARAMS((cudaStream_t)0);
  int rc = build_csr_cache(ctx);
  if (rc) return rc;
  invalidate_mass(ctx);
  const Params &P = ctx->P;
  const size_t nb = (size_t)ctx->n_patches * P.s * P.NfMax, nk = (size_t)ctx->n_patches * P.s * P.ell_width;
  if (!ctx->d_Mell) CK(cudaMalloc(&ctx->d_Mell, sizeof(double) * nk));
  if (!ctx->d_Mval) CK(cudaMalloc(&ctx->d_Mval, sizeof(double) * std::max<size_t>(1, (size_t)ctx->csr_nnz)));
  double *d_mphi = nullptr;
  CK(cudaMalloc(&d_mphi, sizeof(double) * nb));
  cudaError_t e = cudaEventRecord(ctx->ev[8], 0);
  if (e == cudaSuccess) e = launch_mass_apply(0, (int)ctx->n_patches, P.s, ctx->d_phi, d_mphi, P.NfMax);
  if (e == cudaSuccess) e = cudaEventRecord(ctx->ev[9], 0);
  if (e == cudaSuccess) e = launch_coarse_rows(ctx, 0, 0, ctx->n_patches, ctx->d_phi, d_mphi, ctx->d_Mell);
  if (e == cudaSuccess) e = cudaEventRecord(ctx->ev[10], 0);
  if (e == cudaSuccess) e = launch_gather(0, ctx->d_Mell, ctx->d_perm, ctx->d_Mval, ctx->csr_nnz);
  rc = finish_call(ctx, "slod_assemble_coarse_mass", e, 3);
  cudaFree(d_mphi);
  if (rc) return rc;
  float ms[2] = {0, 0};
  CK(cudaEventElapsedTime(&ms[0], ctx->ev[8], ctx->ev[9]));
  CK(cudaEventElapsedTime(&ms[1], ctx->ev[9], ctx->ev[10]));
  ctx->tm.ms[6] = ms[0];
  ctx->tm.ms[7] = ms[1];
  ctx->mass_done = true;
  return SLOD_OK;
}

int slod_get_coarse_mass_csr(const slod_ctx *ctx, int64_t *rowptr, int64_t *col, double *val, int64_t *n_rows,
                             int64_t *nnz) {
  return get_csr(ctx, true, rowptr, col, val, n_rows, nnz);
}

static int check_time_steps(slod_ctx *ctx, double dt, int32_t n_steps, int32_t out_every) {
  if (!(dt > 0.0) || !std::isfinite(dt)) return fail(ctx, SLOD_ERR_INVALID, "dt must be positive and finite");
  if (n_steps < 1) return fail(ctx, SLOD_ERR_INVALID, "n_steps must be at least 1");
  if (out_every < 1 || out_every > n_steps) return fail(ctx, SLOD_ERR_INVALID, "out_every must be in [1, n_steps]");
  return SLOD_OK;
}

// the common preconditions of the two coarse time steppers
static int heat_prepare(slod_ctx *ctx, double dt, int32_t n_steps, int32_t out_every, const double *u_out,
                        int32_t max_steps, double tolerance, double reduction) {
  if (!ctx->coarse_done) return fail(ctx, SLOD_ERR_STATE, "slod_assemble_coarse has not run");
  if (!ctx->mass_done) return fail(ctx, SLOD_ERR_STATE, "slod_assemble_coarse_mass has not run");
  if (!u_out) return fail(ctx, SLOD_ERR_INVALID, "null buffer");
  int rc = check_time_steps(ctx, dt, n_steps, out_every);
  if (rc) return rc;
  return check_solver_control(ctx, max_steps, tolerance, reduction);
}

// S = M_H + coef K, kept until the coefficient of K changes (or M_H / K become stale)
static cudaError_t heat_form_S(slod_ctx *ctx, double coef, long long *launches) {
  if (ctx->s_coef == coef) return cudaSuccess;
  const size_t nk = (size_t)ctx->n_patches * ctx->P.s * ctx->P.ell_width;
  cudaError_t e = ctx->d_Sell ? cudaSuccess : cudaMalloc(&ctx->d_Sell, sizeof(double) * nk);
  if (e == cudaSuccess) e = launch_lincomb(0, (long long)nk, 1.0, ctx->d_Mell, coef, ctx->d_Kell, ctx->d_Sell);
  *launches += 1;
  ctx->s_coef = e == cudaSuccess ? coef : 0.0;
  return e;
}

// The theta-scheme arguments (slod.h); g_count: the entries of g.  g is read only when fields are given.
static int check_theta(slod_ctx *ctx, double theta, int32_t n_steps, int32_t n_startup, int32_t n_fields,
                       const double *f, const double *g, size_t g_count) {
  if (!(theta >= 0.5 && theta <= 1.0)) return fail(ctx, SLOD_ERR_INVALID, "theta must be in [1/2, 1]");
  if (n_startup < 0 || n_startup > n_steps) return fail(ctx, SLOD_ERR_INVALID, "n_startup must be in [0, n_steps]");
  if (f && n_fields < 1) return fail(ctx, SLOD_ERR_INVALID, "n_fields must be at least 1");
  if (f && g)
    for (size_t i = 0; i < g_count; ++i)
      if (!std::isfinite(g[i])) return fail(ctx, SLOD_ERR_INVALID, "g has a non-finite entry");
  return SLOD_OK;
}

// One solve of the time loop: S = M_H + coef K, r = tau (sum_q w_q b_q - K u), S delta = r, u += delta.  A full step k
// of the theta scheme is one stage (coef = theta dt, tau = dt, w_q = theta g_q(t_k) + (1 - theta) g_q(t_{k-1})); a
// Rannacher start-up step is two backward-Euler stages of dt / 2 (w_q = (g_q(t_{k-1}) + g_q(t_k)) / 2, then g_q(t_k)).
// At theta = 1 without start-up coef = tau = dt and w_q = g_q(t_k) exactly: the backward-Euler entry points.
struct ThetaStage {
  int step;         // the time step k = 1 .. n_steps the stage belongs to
  bool ends_step;   // u is u^k after this stage
  double tau, coef;
};
static std::vector<ThetaStage> theta_stages(double theta, double dt, int n_steps, int n_startup) {
  std::vector<ThetaStage> st;
  for (int k = 1; k <= n_steps; ++k) {
    if (k <= n_startup) {
      st.push_back({k, false, 0.5 * dt, 0.5 * dt});
      st.push_back({k, true, 0.5 * dt, 0.5 * dt});
    } else {
      st.push_back({k, true, dt, theta * dt});
    }
  }
  return st;
}
// the weights of every stage of one column, w[stage][nf]; g [n_steps + 1][nf] or NULL (g = 1)
static void theta_weights(double theta, int n_steps, int n_startup, int nf, const double *g, double *w) {
  auto G = [&](int k, int q) { return g ? g[(size_t)k * nf + q] : 1.0; };
  for (int k = 1; k <= n_steps; ++k)
    for (int half = (k <= n_startup ? 0 : 1); half < 2; ++half, w += nf)
      for (int q = 0; q < nf; ++q)
        w[q] = k <= n_startup ? (half ? G(k, q) : 0.5 * (G(k - 1, q) + G(k, q)))
                              : theta * G(k, q) + (1.0 - theta) * G(k - 1, q);
}

int slod_l2_project_batch(slod_ctx *ctx, int32_t n_rhs, const double *v_fine, double *u_coarse, int32_t max_steps,
                          double tolerance, double reduction, int32_t *steps, double *residual) {
  if (!ctx) return SLOD_ERR_INVALID;
  NEED_DEVICE();
  if (!ctx->mass_done) return fail(ctx, SLOD_ERR_STATE, "slod_assemble_coarse_mass has not run");
  if (!v_fine || !u_coarse) return fail(ctx, SLOD_ERR_INVALID, "null buffer");
  int rc = check_n_rhs(ctx, n_rhs);
  if (rc) return rc;
  rc = check_solver_control(ctx, max_steps, tolerance, reduction);
  if (rc) return rc;
  CK(cudaSetDevice(ctx->device));
  BIND_PARAMS((cudaStream_t)0);
  int64_t n_fine = 0;
  slod_fine_size(ctx, &n_fine);
  const long long n_nodes = n_fine / ctx->P.s;
  const int nrows = (int)(ctx->n_patches * ctx->P.s);
  BatchScratch w{};
  rc = batch_scratch(ctx, &w);
  if (rc) return rc;
  std::vector<int> st_steps(n_rhs, 0), flag(n_rhs, 0);
  std::vector<double> res(n_rhs, 0.0);
  cudaError_t e = cudaSuccess;
  long long n_launch = 0;
  for (int j0 = 0; j0 < n_rhs && e == cudaSuccess; j0 += kBatch) {
    const int kb = std::min(kBatch, n_rhs - j0);
    e = cudaMemcpyAsync(w.fine_stage, v_fine + (size_t)j0 * n_fine, sizeof(double) * kb * (size_t)n_fine,
                        cudaMemcpyHostToDevice, 0);
    for (int j = 0; j < kb && e == cudaSuccess; ++j)   // M_h v, column by column, [kb][n_fine]
      e = launch_fine_apply(0, kFineMass, 0.0, n_nodes, nullptr, w.fine_stage + (size_t)j * n_fine,
                            w.fine + (size_t)j * n_fine);
    if (e == cudaSuccess) e = launch_interleave(0, n_fine, kb, w.fine, w.fine_stage, true);
    if (e == cudaSuccess)
      e = launch_coarse_rhs_multi(0, (int)ctx->n_patches, ctx->P.s, kb, ctx->d_phi, w.fine_stage, w.coarse_a,
                                  ctx->P.NfMax);
    if (e == cudaSuccess)
      e = run_cg_multi(0, nrows, ctx->d_Mell, kb, w.coarse_a, w.coarse_b, w.work, max_steps, tolerance, reduction,
                       &st_steps[j0], &res[j0], &flag[j0], &n_launch);
    if (e == cudaSuccess) e = download_group(w.coarse_b, nrows, kb, w.coarse_stage, u_coarse + (size_t)j0 * nrows);
    n_launch += kb + 3;
  }
  rc = finish_call(ctx, "slod_l2_project_batch", e, n_launch);
  for (int j = 0; j < n_rhs; ++j) {
    if (steps) steps[j] = st_steps[j];
    if (residual) residual[j] = res[j];
  }
  for (int j = 0; j < n_rhs && !rc; ++j)
    rc = cg_outcome(ctx, 0, j, "CG on M_H", 0.0, flag[j], st_steps[j], res[j]);
  return rc;
}

// the single-trajectory theta scheme: slod_heat_theta_solve after its argument checks, and slod_heat_solve (theta = 1)
static int heat_theta_single(slod_ctx *ctx, const char *name, double theta, double dt, int32_t n_steps,
                             int32_t out_every, int32_t n_startup, int32_t n_fields, const double *f_fine,
                             const double *g, const double *u0_coarse, double *u_out, int32_t max_steps,
                             double tolerance, double reduction, int32_t *cg_steps) {
  CK(cudaSetDevice(ctx->device));
  BIND_PARAMS((cudaStream_t)0);
  int rc = heat_prepare(ctx, dt, n_steps, out_every, u_out, max_steps, tolerance, reduction);
  if (rc) return rc;
  int64_t n_fine = 0;
  slod_fine_size(ctx, &n_fine);
  const int nrows = (int)(ctx->n_patches * ctx->P.s);
  const int nf = f_fine ? n_fields : 1;   // no forcing: one zero load
  const std::vector<ThetaStage> stages = theta_stages(theta, dt, n_steps, n_startup);
  std::vector<double> w(stages.size() * nf);
  theta_weights(theta, n_steps, n_startup, nf, f_fine ? g : nullptr, w.data());
  double *d_f = nullptr, *d_r = nullptr, *d_delta = nullptr, *d_work = nullptr;
  rc = online_scratch(ctx, &d_f, nullptr, &d_r, &d_delta, &d_work);
  if (rc) return rc;
  // u | b_0 .. b_{nf-1} | weights
  rc = grow(ctx, ctx->d_heat, ctx->heat_doubles, (1 + (size_t)nf) * nrows + w.size());
  if (rc) return rc;
  double *d_u = ctx->d_heat, *d_b = d_u + nrows, *d_w = d_b + (size_t)nf * nrows;
  cudaError_t e = cudaMemcpyAsync(d_w, w.data(), sizeof(double) * w.size(), cudaMemcpyHostToDevice, 0);
  if (f_fine) {
    for (int q = 0; q < nf && e == cudaSuccess; ++q) {   // C^T f_q, one field at a time through the fine scratch
      e = cudaMemcpyAsync(d_f, f_fine + (size_t)q * n_fine, sizeof(double) * (size_t)n_fine, cudaMemcpyHostToDevice, 0);
      if (e == cudaSuccess)
        e = launch_coarse_rhs(0, (int)ctx->n_patches, ctx->P.s, ctx->d_phi, d_f, d_b + (size_t)q * nrows,
                              ctx->P.NfMax);
      ctx->launches += 1;
    }
  } else if (e == cudaSuccess) {
    e = cudaMemsetAsync(d_b, 0, sizeof(double) * nrows, 0);
  }
  if (e == cudaSuccess)
    e = u0_coarse ? cudaMemcpyAsync(d_u, u0_coarse, sizeof(double) * nrows, cudaMemcpyHostToDevice, 0)
                  : cudaMemsetAsync(d_u, 0, sizeof(double) * nrows, 0);
  long long n_launch = 0;
  int failed_step = 0, flag = 0, st_steps = 0, step_cg = 0;
  double res = 0.0, failed_coef = 0.0;
  for (size_t i = 0; i < stages.size() && e == cudaSuccess; ++i) {
    const ThetaStage &sg = stages[i];
    const int k = sg.step;
    e = heat_form_S(ctx, sg.coef, &n_launch);
    if (e == cudaSuccess)
      e = launch_ell_residual(0, nrows, 1, ctx->d_Kell, d_u, nf, d_b, nrows, d_w + i * nf, sg.tau, d_r);
    const CgOperator S{ctx->d_Sell, nullptr, 0};   // after heat_form_S: the first call allocates d_Sell
    if (e == cudaSuccess)
      e = run_cg(0, nrows, S, d_r, d_delta, d_work, max_steps, tolerance, reduction, &st_steps, &res, &flag, &n_launch);
    if (e != cudaSuccess) break;
    step_cg = (i > 0 && stages[i - 1].step == k ? step_cg : 0) + st_steps;
    if (cg_steps) cg_steps[k - 1] = step_cg;
    if (flag != 1) {
      failed_step = k;
      failed_coef = sg.coef;
      break;
    }
    e = launch_lincomb(0, nrows, 1.0, d_u, 1.0, d_delta, d_u);
    if (e == cudaSuccess && sg.ends_step && k % out_every == 0)
      e = cudaMemcpyAsync(u_out + (size_t)(k / out_every - 1) * nrows, d_u, sizeof(double) * nrows,
                          cudaMemcpyDeviceToHost, 0);
    n_launch += 2;
  }
  rc = finish_call(ctx, name, e, n_launch);
  if (rc || !failed_step) return rc;
  return cg_outcome(ctx, failed_step, -1, "CG on M_H + c K", failed_coef, flag, st_steps, res);
}

// n_rhs trajectories in groups of kBatch interleaved columns: slod_heat_theta_solve_batch after its argument checks,
// and slod_heat_solve_batch (theta = 1)
static int heat_theta_batch(slod_ctx *ctx, const char *name, int32_t n_rhs, double theta, double dt, int32_t n_steps,
                            int32_t out_every, int32_t n_startup, int32_t n_fields, const double *f_fine,
                            const double *g, const double *u0_coarse, double *u_out, int32_t max_steps,
                            double tolerance, double reduction, int32_t *cg_steps) {
  CK(cudaSetDevice(ctx->device));
  BIND_PARAMS((cudaStream_t)0);
  int rc = heat_prepare(ctx, dt, n_steps, out_every, u_out, max_steps, tolerance, reduction);
  if (rc) return rc;
  int64_t n_fine = 0;
  slod_fine_size(ctx, &n_fine);
  const int nrows = (int)(ctx->n_patches * ctx->P.s);
  const int n_groups = (n_rhs + kBatch - 1) / kBatch;
  const size_t gsz = (size_t)kBatch * nrows;   // one interleaved group
  const int nf = f_fine ? n_fields : 1;        // no forcing: one zero load
  const std::vector<ThetaStage> stages = theta_stages(theta, dt, n_steps, n_startup);
  const size_t ns = stages.size(), wg = ns * nf * kBatch;   // weights of one group: [stage][q][kb]
  std::vector<double> w((size_t)n_groups * wg, 0.0), wj(ns * nf);
  for (int j = 0; j < n_rhs; ++j) {
    const double *gj = f_fine && g ? g + (size_t)j * ((size_t)n_steps + 1) * nf : nullptr;
    theta_weights(theta, n_steps, n_startup, nf, gj, wj.data());
    const int grp = j / kBatch, jj = j % kBatch, kb = std::min(kBatch, n_rhs - grp * kBatch);
    for (size_t i = 0; i < ns * nf; ++i) w[grp * wg + i * kb + jj] = wj[i];
  }
  BatchScratch ws{};
  rc = batch_scratch(ctx, &ws);
  if (rc) return rc;
  // [group][nrows][kb] states | loads C^T f_q, [q][group][nrows][kb] | weights [group][wg]
  rc = grow(ctx, ctx->d_heat, ctx->heat_doubles, (1 + (size_t)nf) * n_groups * gsz + w.size());
  if (rc) return rc;
  const size_t b_stride = (size_t)n_groups * gsz;
  double *d_U = ctx->d_heat, *d_B = d_U + b_stride, *d_W = d_B + nf * b_stride;
  cudaError_t e = cudaMemcpyAsync(d_W, w.data(), sizeof(double) * w.size(), cudaMemcpyHostToDevice, 0);
  long long n_launch = 0;
  for (int grp = 0; grp < n_groups && e == cudaSuccess; ++grp) {
    const int j0 = grp * kBatch, kb = std::min(kBatch, n_rhs - j0);
    double *U = d_U + grp * gsz, *B = d_B + grp * gsz;
    if (f_fine) {
      for (int q = 0; q < nf && e == cudaSuccess; ++q) {
        // field q of the group's columns, one copy per column: the host rows are nf n_fine doubles apart, which can
        // exceed the largest pitch of a 2-D copy
        for (int c = 0; c < kb && e == cudaSuccess; ++c)
          e = cudaMemcpyAsync(ws.fine_stage + (size_t)c * n_fine, f_fine + ((size_t)(j0 + c) * nf + q) * n_fine,
                              sizeof(double) * (size_t)n_fine, cudaMemcpyHostToDevice, 0);
        if (e == cudaSuccess) e = launch_interleave(0, n_fine, kb, ws.fine_stage, ws.fine, true);
        if (e == cudaSuccess)
          e = launch_coarse_rhs_multi(0, (int)ctx->n_patches, ctx->P.s, kb, ctx->d_phi, ws.fine, B + q * b_stride,
                                      ctx->P.NfMax);
        n_launch += 2;
      }
    } else if (e == cudaSuccess) {
      e = cudaMemsetAsync(B, 0, sizeof(double) * kb * (size_t)nrows, 0);
    }
    if (e == cudaSuccess && u0_coarse) {
      e = upload_group(u0_coarse + (size_t)j0 * nrows, nrows, kb, ws.coarse_stage, U);
      n_launch += 1;
    } else if (e == cudaSuccess) {
      e = cudaMemsetAsync(U, 0, sizeof(double) * kb * (size_t)nrows, 0);
    }
  }
  std::vector<int> st_steps(n_rhs, 0), flag(n_rhs, 0), step_cg(n_rhs, 0);
  std::vector<double> res(n_rhs, 0.0);
  int failed_step = 0, failed_col = -1;
  double failed_coef = 0.0;
  for (size_t i = 0; i < ns && e == cudaSuccess && !failed_step; ++i) {
    const ThetaStage &sg = stages[i];
    const int k = sg.step;
    const bool first = i == 0 || stages[i - 1].step != k;
    e = heat_form_S(ctx, sg.coef, &n_launch);
    for (int grp = 0; grp < n_groups && e == cudaSuccess; ++grp) {
      const int j0 = grp * kBatch, kb = std::min(kBatch, n_rhs - j0);
      double *U = d_U + grp * gsz, *B = d_B + grp * gsz;
      e = launch_ell_residual(0, nrows, kb, ctx->d_Kell, U, nf, B, (long long)b_stride, d_W + grp * wg + i * nf * kb,
                              sg.tau, ws.coarse_a);
      if (e == cudaSuccess)
        e = run_cg_multi(0, nrows, ctx->d_Sell, kb, ws.coarse_a, ws.coarse_b, ws.work, max_steps, tolerance, reduction,
                         &st_steps[j0], &res[j0], &flag[j0], &n_launch);
      if (e != cudaSuccess) break;
      for (int j = j0; j < j0 + kb; ++j) {
        step_cg[j] = (first ? 0 : step_cg[j]) + st_steps[j];
        if (cg_steps) cg_steps[(size_t)(k - 1) * n_rhs + j] = step_cg[j];
        if (flag[j] != 1 && !failed_step) {
          failed_step = k;
          failed_col = j;
          failed_coef = sg.coef;
        }
      }
      if (failed_step) break;
      e = launch_lincomb(0, (long long)kb * nrows, 1.0, U, 1.0, ws.coarse_b, U);
      n_launch += 2;
    }
    if (e != cudaSuccess || failed_step || !sg.ends_step || k % out_every != 0) continue;
    for (int grp = 0; grp < n_groups && e == cudaSuccess; ++grp) {
      const int j0 = grp * kBatch, kb = std::min(kBatch, n_rhs - j0);
      e = download_group(d_U + grp * gsz, nrows, kb, ws.coarse_stage,
                         u_out + ((size_t)(k / out_every - 1) * n_rhs + j0) * nrows);
      n_launch += 1;
    }
  }
  rc = finish_call(ctx, name, e, n_launch);
  if (rc || !failed_step) return rc;
  return cg_outcome(ctx, failed_step, failed_col, "CG on M_H + c K", failed_coef, flag[failed_col],
                    st_steps[failed_col], res[failed_col]);
}

// the fine-scale reference trajectory: the same scheme with M_h + coef A_h on the global grid (homogeneous Dirichlet
// rows); slod_fem_heat_theta_solve after its argument checks, and slod_fem_heat_solve (theta = 1)
static int fem_heat_theta(slod_ctx *ctx, const char *name, double theta, double dt, int32_t n_steps, int32_t out_every,
                          int32_t n_startup, int32_t n_fields, const double *f_fine, const double *g,
                          const double *u0_fine, double *u_out, int32_t max_steps, double tolerance, double reduction,
                          int32_t *cg_steps) {
  if (!u_out) return fail(ctx, SLOD_ERR_INVALID, "null buffer");
  int rc = check_time_steps(ctx, dt, n_steps, out_every);
  if (rc) return rc;
  rc = check_solver_control(ctx, max_steps, tolerance, reduction);
  if (rc) return rc;
  CK(cudaSetDevice(ctx->device));
  rc = prepare_coefficients(ctx);
  if (rc) return rc;
  BIND_PARAMS((cudaStream_t)0);
  int64_t n_fine = 0;
  slod_fine_size(ctx, &n_fine);
  const long long n_nodes = n_fine / ctx->P.s;
  const int nf = f_fine ? n_fields : 1;   // no forcing: one zero field
  const std::vector<ThetaStage> stages = theta_stages(theta, dt, n_steps, n_startup);
  std::vector<double> w(stages.size() * nf);
  theta_weights(theta, n_steps, n_startup, nf, f_fine ? g : nullptr, w.data());
  // homogeneous Dirichlet conditions: the boundary rows of the fields and of u0 are zero
  std::vector<double> f((size_t)nf * n_fine, 0.0), u0(n_fine, 0.0);
  if (f_fine) std::copy(f_fine, f_fine + (size_t)nf * n_fine, f.begin());
  if (u0_fine) std::copy(u0_fine, u0_fine + n_fine, u0.begin());
  zero_boundary_rows(ctx->P, f.data(), nf, n_fine);
  zero_boundary_rows(ctx->P, u0.data(), 1, n_fine);
  double *d_r = nullptr, *d_delta = nullptr, *d_work = nullptr;
  rc = online_scratch(ctx, &d_r, &d_delta, nullptr, nullptr, &d_work);
  if (rc) return rc;
  // fields | u | A u | load | weights
  rc = grow(ctx, ctx->d_heat, ctx->heat_doubles, (3 + (size_t)nf) * n_fine + w.size());
  if (rc) return rc;
  double *d_F = ctx->d_heat, *d_u = d_F + (size_t)nf * n_fine, *d_q = d_u + n_fine, *d_load = d_q + n_fine;
  double *d_w = d_load + n_fine;
  CgOperator A{nullptr, ctx->d_coef, n_nodes};
  A.op = kFineHeatDirichlet;
  cudaError_t e = cudaMemcpyAsync(d_F, f.data(), sizeof(double) * f.size(), cudaMemcpyHostToDevice, 0);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_u, u0.data(), sizeof(double) * (size_t)n_fine, cudaMemcpyHostToDevice, 0);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_w, w.data(), sizeof(double) * w.size(), cudaMemcpyHostToDevice, 0);
  long long n_launch = 0;
  int failed_step = 0, flag = 0, st_steps = 0, step_cg = 0;
  double res = 0.0, failed_coef = 0.0;
  for (size_t i = 0; i < stages.size() && e == cudaSuccess; ++i) {
    const ThetaStage &sg = stages[i];
    const int k = sg.step;
    A.tau = sg.coef;
    e = launch_fine_apply(0, kFineStiffDirichlet, 0.0, n_nodes, ctx->d_coef, d_u, d_q);
    if (e == cudaSuccess) e = launch_weighted_sum(0, n_fine, nf, d_w + i * nf, d_F, d_load);
    if (e == cudaSuccess) e = launch_lincomb(0, n_fine, sg.tau, d_load, -sg.tau, d_q, d_r);   // tau (load - A u)
    if (e == cudaSuccess)
      e = run_cg(0, (int)n_fine, A, d_r, d_delta, d_work, max_steps, tolerance, reduction, &st_steps, &res, &flag,
                 &n_launch);
    if (e != cudaSuccess) break;
    step_cg = (i > 0 && stages[i - 1].step == k ? step_cg : 0) + st_steps;
    if (cg_steps) cg_steps[k - 1] = step_cg;
    if (flag != 1) {
      failed_step = k;
      failed_coef = sg.coef;
      break;
    }
    e = launch_lincomb(0, n_fine, 1.0, d_u, 1.0, d_delta, d_u);
    if (e == cudaSuccess && sg.ends_step && k % out_every == 0)
      e = cudaMemcpyAsync(u_out + (size_t)(k / out_every - 1) * n_fine, d_u, sizeof(double) * (size_t)n_fine,
                          cudaMemcpyDeviceToHost, 0);
    n_launch += 4;
  }
  rc = finish_call(ctx, name, e, n_launch);
  if (rc || !failed_step) return rc;
  return cg_outcome(ctx, failed_step, -1, "fine CG on M_h + c A_h", failed_coef, flag, st_steps, res);
}

int slod_heat_solve(slod_ctx *ctx, const double *f_fine, const double *u0_coarse, double dt, int32_t n_steps,
                    int32_t out_every, double *u_out, int32_t max_steps, double tolerance, double reduction,
                    int32_t *cg_steps) {
  if (!ctx) return SLOD_ERR_INVALID;
  NEED_DEVICE();
  return heat_theta_single(ctx, "slod_heat_solve", 1.0, dt, n_steps, out_every, 0, 1, f_fine, nullptr, u0_coarse,
                           u_out, max_steps, tolerance, reduction, cg_steps);
}

int slod_heat_solve_batch(slod_ctx *ctx, int32_t n_rhs, const double *f_fine, const double *u0_coarse, double dt,
                          int32_t n_steps, int32_t out_every, double *u_out, int32_t max_steps, double tolerance,
                          double reduction, int32_t *cg_steps) {
  if (!ctx) return SLOD_ERR_INVALID;
  NEED_DEVICE();
  const int rc = check_n_rhs(ctx, n_rhs);
  if (rc) return rc;
  return heat_theta_batch(ctx, "slod_heat_solve_batch", n_rhs, 1.0, dt, n_steps, out_every, 0, 1, f_fine, nullptr,
                          u0_coarse, u_out, max_steps, tolerance, reduction, cg_steps);
}

int slod_fem_heat_solve(slod_ctx *ctx, const double *f_fine, const double *u0_fine, double dt, int32_t n_steps,
                        int32_t out_every, double *u_out, int32_t max_steps, double tolerance, double reduction,
                        int32_t *cg_steps) {
  if (!ctx) return SLOD_ERR_INVALID;
  NEED_DEVICE();
  return fem_heat_theta(ctx, "slod_fem_heat_solve", 1.0, dt, n_steps, out_every, 0, 1, f_fine, nullptr, u0_fine, u_out,
                        max_steps, tolerance, reduction, cg_steps);
}

// The theta-scheme entry points check every argument before the device and the call order, so that a maps-only handle
// reports an invalid argument as such.
static int check_theta_call(slod_ctx *ctx, double theta, double dt, int32_t n_steps, int32_t out_every,
                            int32_t n_startup, int32_t n_fields, const double *f_fine, const double *g, size_t g_rows,
                            const double *u_out, int32_t max_steps, double tolerance, double reduction) {
  if (!u_out) return fail(ctx, SLOD_ERR_INVALID, "null buffer");
  int rc = check_time_steps(ctx, dt, n_steps, out_every);
  if (rc) return rc;
  rc = check_solver_control(ctx, max_steps, tolerance, reduction);
  if (rc) return rc;
  return check_theta(ctx, theta, n_steps, n_startup, n_fields, f_fine, g,
                     n_fields > 0 ? g_rows * ((size_t)n_steps + 1) * n_fields : 0);
}

int slod_heat_theta_solve(slod_ctx *ctx, double theta, double dt, int32_t n_steps, int32_t out_every,
                          int32_t n_startup, int32_t n_fields, const double *f_fine, const double *g,
                          const double *u0_coarse, double *u_out, int32_t max_steps, double tolerance,
                          double reduction, int32_t *cg_steps) {
  if (!ctx) return SLOD_ERR_INVALID;
  int rc = check_theta_call(ctx, theta, dt, n_steps, out_every, n_startup, n_fields, f_fine, g, 1, u_out, max_steps,
                            tolerance, reduction);
  if (rc) return rc;
  NEED_DEVICE();
  return heat_theta_single(ctx, "slod_heat_theta_solve", theta, dt, n_steps, out_every, n_startup, n_fields, f_fine, g,
                           u0_coarse, u_out, max_steps, tolerance, reduction, cg_steps);
}

int slod_heat_theta_solve_batch(slod_ctx *ctx, int32_t n_rhs, double theta, double dt, int32_t n_steps,
                                int32_t out_every, int32_t n_startup, int32_t n_fields, const double *f_fine,
                                const double *g, const double *u0_coarse, double *u_out, int32_t max_steps,
                                double tolerance, double reduction, int32_t *cg_steps) {
  if (!ctx) return SLOD_ERR_INVALID;
  int rc = check_n_rhs(ctx, n_rhs);
  if (rc) return rc;
  rc = check_theta_call(ctx, theta, dt, n_steps, out_every, n_startup, n_fields, f_fine, g, (size_t)n_rhs, u_out,
                        max_steps, tolerance, reduction);
  if (rc) return rc;
  NEED_DEVICE();
  return heat_theta_batch(ctx, "slod_heat_theta_solve_batch", n_rhs, theta, dt, n_steps, out_every, n_startup,
                          n_fields, f_fine, g, u0_coarse, u_out, max_steps, tolerance, reduction, cg_steps);
}

int slod_fem_heat_theta_solve(slod_ctx *ctx, double theta, double dt, int32_t n_steps, int32_t out_every,
                              int32_t n_startup, int32_t n_fields, const double *f_fine, const double *g,
                              const double *u0_fine, double *u_out, int32_t max_steps, double tolerance,
                              double reduction, int32_t *cg_steps) {
  if (!ctx) return SLOD_ERR_INVALID;
  int rc = check_theta_call(ctx, theta, dt, n_steps, out_every, n_startup, n_fields, f_fine, g, 1, u_out, max_steps,
                            tolerance, reduction);
  if (rc) return rc;
  NEED_DEVICE();
  return fem_heat_theta(ctx, "slod_fem_heat_theta_solve", theta, dt, n_steps, out_every, n_startup, n_fields, f_fine,
                        g, u0_fine, u_out, max_steps, tolerance, reduction, cg_steps);
}

// ---- wave equation on the SLOD space: Newmark time stepping (gamma = 1/2) ----
// M_H u'' + K u = b(t), b(t) = sum_q g_q(t) C^T f_q.  Each step solves for the acceleration with S = M_H + beta dt^2 K
// (wave.cuh): the right-hand side b(t_{k+1}) - K ut is k_ell_residual with U = ut and tau = 1, and the CG drivers start
// from zero.  beta = 0 solves with M_H itself: heat_form_S treats a coefficient of 0 as "not formed".
static int check_wave_call(slod_ctx *ctx, double beta, double dt, int32_t n_steps, int32_t out_every, int32_t n_fields,
                           const double *f_fine, const double *g, size_t g_rows, const double *u_out, int32_t max_steps,
                           double tolerance, double reduction) {
  if (!u_out) return fail(ctx, SLOD_ERR_INVALID, "null buffer");
  int rc = check_time_steps(ctx, dt, n_steps, out_every);
  if (rc) return rc;
  rc = check_solver_control(ctx, max_steps, tolerance, reduction);
  if (rc) return rc;
  if (!(beta >= 0.0 && beta <= 0.5)) return fail(ctx, SLOD_ERR_INVALID, "beta must be in [0, 1/2]");
  if (f_fine && n_fields < 1) return fail(ctx, SLOD_ERR_INVALID, "n_fields must be at least 1");
  if (f_fine && g)
    for (size_t i = 0, n = g_rows * ((size_t)n_steps + 1) * n_fields; i < n; ++i)
      if (!std::isfinite(g[i])) return fail(ctx, SLOD_ERR_INVALID, "g has a non-finite entry");
  return SLOD_OK;
}

// the weights g_q(t_k) of one column, w[k][nf] for k = 0 .. n_steps; g [n_steps + 1][nf] or NULL (g = 1)
static void wave_weights(int n_steps, int nf, const double *g, double *w) {
  for (size_t i = 0; i < ((size_t)n_steps + 1) * nf; ++i) w[i] = g ? g[i] : 1.0;
}

// The failure of an acceleration solve: step 0 is the start solve M a_0 = b(t_0) - K u_0.
static int wave_outcome(slod_ctx *ctx, bool fine, int step, int column, double c, int flag, int steps, double res) {
  const char *label = step == 0 ? (fine ? "start solve (step 0): fine CG on M_h" : "start solve (step 0): CG on M_H")
                      : c > 0 ? (fine ? "fine CG on M_h + c A_h" : "CG on M_H + c K")
                              : (fine ? "fine CG on M_h" : "CG on M_H");
  return cg_outcome(ctx, step, column, label, step == 0 ? 0.0 : c, flag, steps, res);
}

// n_rhs trajectories of the coarse scheme in groups of kBatch interleaved columns; batch = false: one trajectory with
// the single-vector kernels (run_cg), which agrees with a one-column batch to the solver tolerance.
static int wave_coarse(slod_ctx *ctx, const char *name, bool batch, int32_t n_rhs, double beta, double dt,
                       int32_t n_steps, int32_t out_every, int32_t n_fields, const double *f_fine, const double *g,
                       const double *u0_coarse, const double *v0_coarse, double *u_out, double *v_out,
                       double *energy_out, int32_t max_steps, double tolerance, double reduction, int32_t *cg_steps) {
  CK(cudaSetDevice(ctx->device));
  BIND_PARAMS((cudaStream_t)0);
  int rc = heat_prepare(ctx, dt, n_steps, out_every, u_out, max_steps, tolerance, reduction);
  if (rc) return rc;
  int64_t n_fine = 0;
  slod_fine_size(ctx, &n_fine);
  const int nrows = (int)(ctx->n_patches * ctx->P.s);
  const int n_groups = batch ? (n_rhs + kBatch - 1) / kBatch : 1;
  const int gmax = batch ? kBatch : 1;          // columns of a full group
  const size_t gsz = (size_t)gmax * nrows;      // one interleaved group
  const int nf = f_fine ? n_fields : 1;         // no forcing: one zero load
  const size_t nk = (size_t)n_steps + 1, wg = nk * nf * gmax;   // weights of one group: [k][q][kb]
  std::vector<double> w((size_t)n_groups * wg, 0.0), wj(nk * nf);
  for (int j = 0; j < n_rhs; ++j) {
    wave_weights(n_steps, nf, f_fine && g ? g + (size_t)j * nk * nf : nullptr, wj.data());
    const int grp = j / gmax, jj = j % gmax, kb = std::min(gmax, n_rhs - grp * gmax);
    for (size_t i = 0; i < nk * nf; ++i) w[grp * wg + i * kb + jj] = wj[i];
  }
  BatchScratch ws{};
  double *d_f = nullptr, *d_r = nullptr, *d_anew = nullptr, *d_work = nullptr;
  if (batch) {
    rc = batch_scratch(ctx, &ws);
    d_r = ws.coarse_a;
    d_anew = ws.coarse_b;
    d_work = ws.work;
  } else {
    rc = online_scratch(ctx, &d_f, nullptr, &d_r, &d_anew, &d_work);
  }
  if (rc) return rc;
  // [group] u | v | a | ut, each [nrows][kb] | loads C^T f_q, [q][group][nrows][kb] | weights | energy partials | E
  const size_t b_stride = (size_t)n_groups * gsz, n_part = wave_energy_workspace_doubles(nrows);
  rc = grow(ctx, ctx->d_heat, ctx->heat_doubles, (4 + (size_t)nf) * b_stride + w.size() + n_part + kBatch);
  if (rc) return rc;
  double *d_state = ctx->d_heat, *d_B = d_state + 4 * b_stride, *d_W = d_B + nf * b_stride;
  double *d_part = d_W + w.size(), *d_E = d_part + n_part;
  auto U = [&](int grp, int which) { return d_state + (size_t)which * b_stride + grp * gsz; };   // 0 u, 1 v, 2 a, 3 ut
  cudaError_t e = cudaMemcpyAsync(d_W, w.data(), sizeof(double) * w.size(), cudaMemcpyHostToDevice, 0);
  long long n_launch = 0;
  for (int grp = 0; grp < n_groups && e == cudaSuccess; ++grp) {
    const int j0 = grp * gmax, kb = std::min(gmax, n_rhs - j0);
    double *B = d_B + grp * gsz;
    if (f_fine) {
      for (int q = 0; q < nf && e == cudaSuccess; ++q) {
        // field q of the group's columns, one copy per column (the host rows are nf n_fine doubles apart)
        for (int c = 0; c < kb && e == cudaSuccess; ++c)
          e = cudaMemcpyAsync((batch ? ws.fine_stage : d_f) + (size_t)c * n_fine, f_fine + ((size_t)(j0 + c) * nf + q) * n_fine,
                              sizeof(double) * (size_t)n_fine, cudaMemcpyHostToDevice, 0);
        if (e == cudaSuccess && batch) e = launch_interleave(0, n_fine, kb, ws.fine_stage, ws.fine, true);
        if (e == cudaSuccess)
          e = batch ? launch_coarse_rhs_multi(0, (int)ctx->n_patches, ctx->P.s, kb, ctx->d_phi, ws.fine,
                                              B + q * b_stride, ctx->P.NfMax)
                    : launch_coarse_rhs(0, (int)ctx->n_patches, ctx->P.s, ctx->d_phi, d_f, B + q * b_stride,
                                        ctx->P.NfMax);
        n_launch += batch ? 2 : 1;
      }
    } else if (e == cudaSuccess) {
      e = cudaMemsetAsync(B, 0, sizeof(double) * kb * (size_t)nrows, 0);
    }
    const double *init[2] = {u0_coarse, v0_coarse};
    for (int which = 0; which < 2 && e == cudaSuccess; ++which) {
      if (!init[which]) {
        e = cudaMemsetAsync(U(grp, which), 0, sizeof(double) * kb * (size_t)nrows, 0);
      } else if (batch) {
        e = upload_group(init[which] + (size_t)j0 * nrows, nrows, kb, ws.coarse_stage, U(grp, which));
        n_launch += 1;
      } else {
        e = cudaMemcpyAsync(U(grp, which), init[which], sizeof(double) * nrows, cudaMemcpyHostToDevice, 0);
      }
    }
  }
  // S = M_H + beta dt^2 K for the steps; the start solve and beta = 0 use M_H
  const double coef = beta * dt * dt;
  if (e == cudaSuccess && coef > 0.0) e = heat_form_S(ctx, coef, &n_launch);
  std::vector<int> st_steps(n_rhs, 0), flag(n_rhs, 0);
  std::vector<double> res(n_rhs, 0.0);
  int failed_step = -1, failed_col = -1;
  for (int k = 0; k <= n_steps && e == cudaSuccess && failed_step < 0; ++k) {
    const double *Sell = (k > 0 && coef > 0.0) ? ctx->d_Sell : ctx->d_Mell;
    const bool out = k == 0 || k % out_every == 0;   // k = 0: only the energy at t_0
    for (int grp = 0; grp < n_groups && e == cudaSuccess; ++grp) {
      const int j0 = grp * gmax, kb = std::min(gmax, n_rhs - j0);
      // k = 0: M a_0 = b(t_0) - K u_0; k > 0: S a_k = b(t_k) - K ut
      e = launch_ell_residual(0, nrows, kb, ctx->d_Kell, U(grp, k == 0 ? 0 : 3), nf, d_B + grp * gsz,
                              (long long)b_stride, d_W + grp * wg + (size_t)k * nf * kb, 1.0, d_r);
      double *x = k == 0 ? U(grp, 2) : d_anew;
      if (e == cudaSuccess) {
        if (batch) {
          e = run_cg_multi(0, nrows, Sell, kb, d_r, x, d_work, max_steps, tolerance, reduction, &st_steps[j0],
                           &res[j0], &flag[j0], &n_launch);
        } else {
          const CgOperator S{Sell, nullptr, 0};
          e = run_cg(0, nrows, S, d_r, x, d_work, max_steps, tolerance, reduction, &st_steps[0], &res[0], &flag[0],
                     &n_launch);
        }
      }
      if (e != cudaSuccess) break;
      for (int j = j0; j < j0 + kb; ++j) {
        if (cg_steps) cg_steps[(size_t)k * n_rhs + j] = st_steps[j];
        if (flag[j] != 1 && failed_step < 0) {
          failed_step = k;
          failed_col = j;
        }
      }
      if (failed_step >= 0) break;
      e = launch_newmark_update(0, (long long)kb * nrows, k == 0, beta, dt, U(grp, 0), U(grp, 1), U(grp, 2), d_anew,
                                U(grp, 3));
      n_launch += 2;
      if (e == cudaSuccess && out && energy_out) {
        e = launch_wave_energy(0, nrows, kb, ctx->d_Kell, ctx->d_Mell, U(grp, 0), U(grp, 1), d_part, d_E);
        if (e == cudaSuccess)
          e = cudaMemcpyAsync(energy_out + (size_t)(k / out_every) * n_rhs + j0, d_E, sizeof(double) * kb,
                              cudaMemcpyDeviceToHost, 0);
        n_launch += 2;
      }
    }
    if (e != cudaSuccess || failed_step >= 0 || k == 0 || k % out_every != 0) continue;
    const int o = k / out_every - 1;
    double *outs[2] = {u_out, v_out};
    for (int which = 0; which < 2; ++which)
      for (int grp = 0; grp < n_groups && e == cudaSuccess && outs[which]; ++grp) {
        const int j0 = grp * gmax, kb = std::min(gmax, n_rhs - j0);
        double *host = outs[which] + ((size_t)o * n_rhs + j0) * nrows;
        if (batch) {
          e = download_group(U(grp, which), nrows, kb, ws.coarse_stage, host);
          n_launch += 1;
        } else {
          e = cudaMemcpyAsync(host, U(grp, which), sizeof(double) * nrows, cudaMemcpyDeviceToHost, 0);
        }
      }
  }
  rc = finish_call(ctx, name, e, n_launch);
  if (rc || failed_step < 0) return rc;
  return wave_outcome(ctx, false, failed_step, batch ? failed_col : -1, coef, flag[failed_col], st_steps[failed_col],
                      res[failed_col]);
}

// the fine-scale reference trajectory: the same scheme with M_h + beta dt^2 A_h on the global grid (homogeneous
// Dirichlet rows: kFineHeatDirichlet with tau = beta dt^2; tau = 0 is M_h with identity boundary rows).  The energy is
// 1/2 v^T M_h v + 1/2 u^T A_h u from the quadratic forms of k_fine_apply, exact because u and v vanish on the boundary.
static int fem_wave(slod_ctx *ctx, double beta, double dt, int32_t n_steps, int32_t out_every, int32_t n_fields,
                    const double *f_fine, const double *g, const double *u0_fine, const double *v0_fine, double *u_out,
                    double *v_out, double *energy_out, int32_t max_steps, double tolerance, double reduction,
                    int32_t *cg_steps) {
  const char *name = "slod_fem_wave_solve";
  CK(cudaSetDevice(ctx->device));
  int rc = prepare_coefficients(ctx);
  if (rc) return rc;
  BIND_PARAMS((cudaStream_t)0);
  int64_t n_fine = 0;
  slod_fine_size(ctx, &n_fine);
  const long long n_nodes = n_fine / ctx->P.s;
  const int nf = f_fine ? n_fields : 1;   // no forcing: one zero field
  std::vector<double> w(((size_t)n_steps + 1) * nf);
  wave_weights(n_steps, nf, f_fine ? g : nullptr, w.data());
  std::vector<double> f((size_t)nf * n_fine, 0.0), x0(2 * (size_t)n_fine, 0.0);   // boundary rows zero
  if (f_fine) std::copy(f_fine, f_fine + (size_t)nf * n_fine, f.begin());
  if (u0_fine) std::copy(u0_fine, u0_fine + n_fine, x0.begin());
  if (v0_fine) std::copy(v0_fine, v0_fine + n_fine, x0.begin() + n_fine);
  zero_boundary_rows(ctx->P, f.data(), nf, n_fine);
  zero_boundary_rows(ctx->P, x0.data(), 2, n_fine);
  int nb = 0;
  launch_fine_quadratic_form(0, kFineMass, n_nodes, nullptr, nullptr, nullptr, &nb);
  double *d_r = nullptr, *d_anew = nullptr, *d_work = nullptr;
  rc = online_scratch(ctx, &d_r, &d_anew, nullptr, nullptr, &d_work);
  if (rc) return rc;
  // fields | u | v | a | ut | A ut | load | weights | energy partials
  rc = grow(ctx, ctx->d_heat, ctx->heat_doubles, (6 + (size_t)nf) * n_fine + w.size() + 2 * (size_t)nb);
  if (rc) return rc;
  double *d_F = ctx->d_heat, *d_u = d_F + (size_t)nf * n_fine, *d_v = d_u + n_fine, *d_a = d_v + n_fine;
  double *d_ut = d_a + n_fine, *d_q = d_ut + n_fine, *d_load = d_q + n_fine, *d_w = d_load + n_fine;
  double *d_part = d_w + w.size();
  CgOperator A{nullptr, ctx->d_coef, n_nodes};
  A.op = kFineHeatDirichlet;
  cudaError_t e = cudaMemcpyAsync(d_F, f.data(), sizeof(double) * f.size(), cudaMemcpyHostToDevice, 0);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_u, x0.data(), sizeof(double) * x0.size(), cudaMemcpyHostToDevice, 0);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_w, w.data(), sizeof(double) * w.size(), cudaMemcpyHostToDevice, 0);
  const double coef = beta * dt * dt;
  std::vector<double> part(2 * (size_t)nb);
  long long n_launch = 0;
  int failed_step = -1, flag = 0, st_steps = 0;
  double res = 0.0;
  for (int k = 0; k <= n_steps && e == cudaSuccess; ++k) {
    A.tau = k == 0 ? 0.0 : coef;
    // k = 0: M a_0 = b(t_0) - A u_0; k > 0: (M + beta dt^2 A) a_k = b(t_k) - A ut
    e = launch_fine_apply(0, kFineStiffDirichlet, 0.0, n_nodes, ctx->d_coef, k == 0 ? d_u : d_ut, d_q);
    if (e == cudaSuccess) e = launch_weighted_sum(0, n_fine, nf, d_w + (size_t)k * nf, d_F, d_load);
    if (e == cudaSuccess) e = launch_lincomb(0, n_fine, 1.0, d_load, -1.0, d_q, d_r);
    if (e == cudaSuccess)
      e = run_cg(0, (int)n_fine, A, d_r, k == 0 ? d_a : d_anew, d_work, max_steps, tolerance, reduction, &st_steps,
                 &res, &flag, &n_launch);
    if (e != cudaSuccess) break;
    if (cg_steps) cg_steps[k] = st_steps;
    if (flag != 1) {
      failed_step = k;
      break;
    }
    e = launch_newmark_update(0, n_fine, k == 0, beta, dt, d_u, d_v, d_a, d_anew, d_ut);
    n_launch += 4;
    if (e != cudaSuccess || (k > 0 && k % out_every != 0)) continue;
    const size_t o = (size_t)(k / out_every);   // k = 0: only the energy at t_0
    if (k > 0 && e == cudaSuccess)
      e = cudaMemcpyAsync(u_out + (o - 1) * n_fine, d_u, sizeof(double) * (size_t)n_fine, cudaMemcpyDeviceToHost, 0);
    if (k > 0 && e == cudaSuccess && v_out)
      e = cudaMemcpyAsync(v_out + (o - 1) * n_fine, d_v, sizeof(double) * (size_t)n_fine, cudaMemcpyDeviceToHost, 0);
    if (e == cudaSuccess && energy_out) {
      e = launch_fine_quadratic_form(0, kFineMass, n_nodes, ctx->d_coef, d_v, d_part, &nb);
      if (e == cudaSuccess) e = launch_fine_quadratic_form(0, kFineEnergy, n_nodes, ctx->d_coef, d_u, d_part + nb, &nb);
      if (e == cudaSuccess)
        e = cudaMemcpyAsync(part.data(), d_part, sizeof(double) * part.size(), cudaMemcpyDeviceToHost, 0);
      if (e == cudaSuccess) e = cudaStreamSynchronize(0);
      n_launch += 2;
      if (e != cudaSuccess) break;
      double sum[2] = {0.0, 0.0};
      for (int i = 0; i < 2; ++i)
        for (int b = 0; b < nb; ++b) sum[i] += part[(size_t)i * nb + b];   // block order: reproducible
      energy_out[o] = 0.5 * sum[0] + 0.5 * sum[1];
    }
  }
  rc = finish_call(ctx, name, e, n_launch);
  if (rc || failed_step < 0) return rc;
  return wave_outcome(ctx, true, failed_step, -1, coef, flag, st_steps, res);
}

int slod_wave_solve(slod_ctx *ctx, double beta, double dt, int32_t n_steps, int32_t out_every, int32_t n_fields,
                    const double *f_fine, const double *g, const double *u0_coarse, const double *v0_coarse,
                    double *u_out, double *v_out, double *energy_out, int32_t max_steps, double tolerance,
                    double reduction, int32_t *cg_steps) {
  if (!ctx) return SLOD_ERR_INVALID;
  int rc = check_wave_call(ctx, beta, dt, n_steps, out_every, n_fields, f_fine, g, 1, u_out, max_steps, tolerance,
                           reduction);
  if (rc) return rc;
  NEED_DEVICE();
  return wave_coarse(ctx, "slod_wave_solve", false, 1, beta, dt, n_steps, out_every, n_fields, f_fine, g, u0_coarse,
                     v0_coarse, u_out, v_out, energy_out, max_steps, tolerance, reduction, cg_steps);
}

int slod_wave_solve_batch(slod_ctx *ctx, int32_t n_rhs, double beta, double dt, int32_t n_steps, int32_t out_every,
                          int32_t n_fields, const double *f_fine, const double *g, const double *u0_coarse,
                          const double *v0_coarse, double *u_out, double *v_out, double *energy_out,
                          int32_t max_steps, double tolerance, double reduction, int32_t *cg_steps) {
  if (!ctx) return SLOD_ERR_INVALID;
  int rc = check_n_rhs(ctx, n_rhs);
  if (rc) return rc;
  rc = check_wave_call(ctx, beta, dt, n_steps, out_every, n_fields, f_fine, g, (size_t)n_rhs, u_out, max_steps,
                       tolerance, reduction);
  if (rc) return rc;
  NEED_DEVICE();
  return wave_coarse(ctx, "slod_wave_solve_batch", true, n_rhs, beta, dt, n_steps, out_every, n_fields, f_fine, g,
                     u0_coarse, v0_coarse, u_out, v_out, energy_out, max_steps, tolerance, reduction, cg_steps);
}

int slod_fem_wave_solve(slod_ctx *ctx, double beta, double dt, int32_t n_steps, int32_t out_every, int32_t n_fields,
                        const double *f_fine, const double *g, const double *u0_fine, const double *v0_fine,
                        double *u_out, double *v_out, double *energy_out, int32_t max_steps, double tolerance,
                        double reduction, int32_t *cg_steps) {
  if (!ctx) return SLOD_ERR_INVALID;
  int rc = check_wave_call(ctx, beta, dt, n_steps, out_every, n_fields, f_fine, g, 1, u_out, max_steps, tolerance,
                           reduction);
  if (rc) return rc;
  NEED_DEVICE();
  return fem_wave(ctx, beta, dt, n_steps, out_every, n_fields, f_fine, g, u0_fine, v0_fine, u_out, v_out, energy_out,
                  max_steps, tolerance, reduction, cg_steps);
}

// ---- checkpoint: parameters + phi + A*phi (+ block-ELL coarse matrix) --------------------------------------------
namespace {
struct StateHeader {
  char magic[8];          // "SLODB200"
  int32_t version;
  int32_t par[8];         // dim, spacedim, ref, n, ell, stabilize, problem, quirk
  int64_t n_patches, stride, ell_width;
  int32_t has_coarse;
  int32_t pad;
};
std::array<int32_t, 8> state_params(const slod_params &p) {
  return {p.dim, p.spacedim, p.n_global_refinements, p.n_subdivisions, p.oversampling, p.stabilize ? 1 : 0, p.problem,
          p.quirk_presaved ? 1 : 0};
}
}  // namespace

int slod_save_state(slod_ctx *ctx, const char *path) {
  if (!ctx || !path) return SLOD_ERR_INVALID;
  NEED_DEVICE();
  if (!ctx->basis_done) return fail(ctx, SLOD_ERR_STATE, "slod_compute_basis has not run");
  CK(cudaSetDevice(ctx->device));
  CK(cudaDeviceSynchronize());
  StateHeader h{};
  std::memcpy(h.magic, "SLODB200", 8);
  h.version = 1;
  const std::array<int32_t, 8> pv = state_params(ctx->par);
  std::memcpy(h.par, pv.data(), sizeof h.par);
  h.n_patches = ctx->n_patches;
  h.stride = ctx->P.NfMax;
  h.ell_width = ctx->P.ell_width;
  h.has_coarse = ctx->coarse_done ? 1 : 0;
  FILE *f = std::fopen(path, "wb");
  if (!f) return fail(ctx, SLOD_ERR_INVALID, std::string("cannot write ") + path);
  bool ok = std::fwrite(&h, sizeof h, 1, f) == 1;
  const size_t nb = (size_t)ctx->n_patches * ctx->P.s * ctx->P.NfMax, nk = (size_t)ctx->n_patches * ctx->P.s * ctx->P.ell_width;
  std::vector<double> buf(std::max(nb, h.has_coarse ? nk : (size_t)0));
  for (const double *src : {(const double *)ctx->d_phi, (const double *)ctx->d_aphi}) {
    if (cudaMemcpy(buf.data(), src, sizeof(double) * nb, cudaMemcpyDeviceToHost) != cudaSuccess) ok = false;
    ok = ok && std::fwrite(buf.data(), sizeof(double), nb, f) == nb;
  }
  if (h.has_coarse) {
    if (cudaMemcpy(buf.data(), ctx->d_Kell, sizeof(double) * nk, cudaMemcpyDeviceToHost) != cudaSuccess) ok = false;
    ok = ok && std::fwrite(buf.data(), sizeof(double), nk, f) == nk;
  }
  ok = (std::fclose(f) == 0) && ok;
  if (!ok) return fail(ctx, SLOD_ERR_INVALID, std::string("write error on ") + path);
  return SLOD_OK;
}

int slod_load_state(slod_ctx *ctx, const char *path) {
  if (!ctx || !path) return SLOD_ERR_INVALID;
  NEED_DEVICE();
  if (!ctx->subs.empty()) return fail(ctx, SLOD_ERR_UNSUPPORTED, "load a checkpoint into a single-device handle");
  CK(cudaSetDevice(ctx->device));
  FILE *f = std::fopen(path, "rb");
  if (!f) return fail(ctx, SLOD_ERR_INVALID, std::string("cannot read ") + path);
  StateHeader h{};
  bool ok = std::fread(&h, sizeof h, 1, f) == 1 && std::memcmp(h.magic, "SLODB200", 8) == 0 && h.version == 1;
  const std::array<int32_t, 8> pv = state_params(ctx->par);
  if (!ok || std::memcmp(h.par, pv.data(), sizeof h.par) != 0 || h.n_patches != ctx->n_patches ||
      h.stride != ctx->P.NfMax || h.ell_width != ctx->P.ell_width) {
    std::fclose(f);
    return fail(ctx, SLOD_ERR_INVALID, "not a checkpoint of a handle with these parameters");
  }
  const size_t nb = (size_t)ctx->n_patches * ctx->P.s * ctx->P.NfMax, nk = (size_t)ctx->n_patches * ctx->P.s * ctx->P.ell_width;
  if (!ctx->d_phi) {
    CK(cudaMalloc(&ctx->d_phi, sizeof(double) * nb));
    CK(cudaMalloc(&ctx->d_aphi, sizeof(double) * nb));
  }
  std::vector<double> buf(std::max(nb, h.has_coarse ? nk : (size_t)0));
  for (double *dst : {ctx->d_phi, ctx->d_aphi}) {
    ok = ok && std::fread(buf.data(), sizeof(double), nb, f) == nb;
    if (ok && cudaMemcpy(dst, buf.data(), sizeof(double) * nb, cudaMemcpyHostToDevice) != cudaSuccess) ok = false;
  }
  ctx->basis_done = ok;
  ctx->coarse_done = false;
  ctx->have_base = ctx->base_coarse = false;   // the checkpoint holds no coefficient
  invalidate_mass(ctx);
  if (ok && h.has_coarse) {
    if (!ctx->d_Kell) CK(cudaMalloc(&ctx->d_Kell, sizeof(double) * nk));
    ok = std::fread(buf.data(), sizeof(double), nk, f) == nk;
    if (ok && cudaMemcpy(ctx->d_Kell, buf.data(), sizeof(double) * nk, cudaMemcpyHostToDevice) != cudaSuccess) ok = false;
    std::fclose(f);
    if (!ok) return fail(ctx, SLOD_ERR_INVALID, std::string("short read on ") + path);
    int rc = build_csr_cache(ctx);
    if (rc) return rc;
    CK(launch_gather(0, ctx->d_Kell, ctx->d_perm, ctx->d_val, ctx->csr_nnz));
    CK(cudaStreamSynchronize(0));
    ctx->launches += 1;
    ctx->coarse_done = true;
    return SLOD_OK;
  }
  std::fclose(f);
  if (!ok) return fail(ctx, SLOD_ERR_INVALID, std::string("short read on ") + path);
  return SLOD_OK;
}

/* pinned host memory for the caller-owned output buffers (device->host copies into pageable memory run at a
 * fraction of the link speed) */
int slod_alloc_host(size_t bytes, void **out) {
  if (!out) return SLOD_ERR_INVALID;
  *out = nullptr;
  return cudaHostAlloc(out, std::max<size_t>(bytes, 1), cudaHostAllocDefault) == cudaSuccess ? SLOD_OK : SLOD_ERR_CUDA;
}
int slod_free_host(void *p) {
  if (!p) return SLOD_OK;
  return cudaFreeHost(p) == cudaSuccess ? SLOD_OK : SLOD_ERR_CUDA;
}

int slod_ell_to_csr(const slod_ctx *ctx, const double *h_K, int64_t *rowptr, int64_t *col, double *val,
                    int64_t *n_rows, int64_t *nnz) {
  if (!ctx) return SLOD_ERR_INVALID;
  return ell_to_csr(ctx, h_K, rowptr, col, val, n_rows, nnz);
}

int slod_get_patch_diagnostics(const slod_ctx *ctx, int64_t patch, int comp, double out[8]) {
  int rc = check_patch(ctx, patch);
  if (rc) return rc;
  NEED_DEVICE();
  if (!out || comp < 0 || comp >= ctx->P.s) return fail(ctx, SLOD_ERR_INVALID, "bad argument");
  CK(cudaSetDevice(ctx->device));
  CK(cudaMemcpy(out, ctx->d_diag + ((size_t)patch * ctx->P.s + comp) * 8, sizeof(double) * 8, cudaMemcpyDeviceToHost));
  int st = 0;
  CK(cudaMemcpy(&st, ctx->d_status + patch, sizeof(int), cudaMemcpyDeviceToHost));
  out[7] = st;
  return SLOD_OK;
}

// reference coarse column of a patch -> the column the patch kernels keep it in: z-major on the split solver (geom.h),
// the same column otherwise
static std::vector<int> internal_columns(const slod_ctx *ctx, const Geom &g) {
  std::vector<int> zpos((size_t)g.Ncd);
  for (int c = 0; c < g.Ncd; ++c) {
    int k[3];
    col_to_cell(ctx->P, g, c, k);
    zpos[c] = ctx->split_solver ? zcell_to_col(g, k) : c;
  }
  return zpos;
}

// X, Minv and G of the patch in workspace slot w to host memory (any may be NULL), in the reference column order
static int copy_stages_out(slod_ctx *ctx, const Geom &g, int w, double *X, double *Minv, double *G) {
  const size_t ms = ctx->dl.m_stride;
  if (X) CK(cudaMemcpy2D(X, sizeof(double) * g.Ncd, ctx->d_X + (size_t)w * ctx->sl.x_stride, sizeof(double) * ctx->sl.ldx,
                         sizeof(double) * g.Ncd, g.Ni, cudaMemcpyDeviceToHost));
  if (Minv) CK(cudaMemcpy(Minv, ctx->d_Minv + w * ms, sizeof(double) * g.Ncd * g.Ncd, cudaMemcpyDeviceToHost));
  if (G) CK(cudaMemcpy(G, ctx->d_G + w * ms, sizeof(double) * g.Ncd * g.Ncd, cudaMemcpyDeviceToHost));
  if (ctx->split_solver) {
    const std::vector<int> zpos = internal_columns(ctx, g);   // back to the reference order
    std::vector<double> tmp;
    if (X) {
      tmp.assign(X, X + (size_t)g.Ni * g.Ncd);
      for (int r = 0; r < g.Ni; ++r)
        for (int c = 0; c < g.Ncd; ++c) X[(size_t)r * g.Ncd + c] = tmp[(size_t)r * g.Ncd + zpos[c]];
    }
    for (double *Mx : {Minv, G})
      if (Mx) {
        tmp.assign(Mx, Mx + (size_t)g.Ncd * g.Ncd);
        for (int r = 0; r < g.Ncd; ++r)
          for (int c = 0; c < g.Ncd; ++c) Mx[(size_t)r * g.Ncd + c] = tmp[(size_t)zpos[r] * g.Ncd + zpos[c]];
      }
  }
  return SLOD_OK;
}

int slod_debug_patch_stages(slod_ctx *ctx, int64_t patch, double *X, double *Minv, double *G) {
  int rc = check_patch(ctx, patch);
  if (rc) return rc;
  NEED_DEVICE();
  CK(cudaSetDevice(ctx->device));
  rc = prepare_coefficients(ctx);
  if (rc) return rc;
  rc = wait_basis(ctx);   // the workspace of an enqueued range is about to be reused
  if (rc) return rc;
  rc = ensure_workspace(ctx, 1);
  if (rc) return rc;
  BIND_PARAMS((cudaStream_t)0);
  ctx->ids_p0 = ctx->ids_p1 = -1;   // the device work list is overwritten below
  const int id = (int)patch;
  CK(cudaMemcpy(ctx->d_ids, &id, sizeof(int), cudaMemcpyHostToDevice));
  rc = launch_patch_stages(ctx, ctx->d_ids, 1, nullptr, 0, ctx->d_diag, ctx->d_status, nullptr, nullptr);
  if (rc) return rc;
  CK(cudaDeviceSynchronize());
  const Geom g = make_geom(ctx->P, id);
  if (G && !g.slod) return fail(ctx, SLOD_ERR_STATE, "patch takes the LOD branch: no Gram matrix");
  return copy_stages_out(ctx, g, 0, X, Minv, G);
}

int slod_debug_patch_stages_list(slod_ctx *ctx, int64_t n, const int64_t *patches, double *X, double *Minv, double *G) {
  if (!ctx) return SLOD_ERR_INVALID;
  if (n < 0 || (n > 0 && (!patches || !X || !Minv))) return fail(ctx, SLOD_ERR_INVALID, "bad argument");
  const Params &P = ctx->P;
  // host checks first: nothing is launched on an invalid list
  std::vector<int64_t> xoff((size_t)n + 1, 0), moff((size_t)n + 1, 0);   // offsets of the packed X / square blocks
  std::vector<int> slot_of((size_t)ctx->n_patches, -1);                   // position of a patch id in `patches`
  for (int64_t i = 0; i < n; ++i) {
    const int64_t p = patches[i];
    if (p < 0 || p >= ctx->n_patches) return fail(ctx, SLOD_ERR_INVALID, "patch id out of range");
    if (slot_of[(size_t)p] >= 0) return fail(ctx, SLOD_ERR_INVALID, "repeated patch id " + std::to_string(p));
    slot_of[(size_t)p] = (int)i;
    const Geom g = make_geom(P, (int)p);
    xoff[i + 1] = xoff[i] + (int64_t)g.Ni * g.Ncd;
    moff[i + 1] = moff[i] + (int64_t)g.Ncd * g.Ncd;
  }
  NEED_DEVICE();
  if (n == 0) return SLOD_OK;
  CK(cudaSetDevice(ctx->device));
  int rc = prepare_coefficients(ctx);
  if (rc) return rc;
  rc = wait_basis(ctx);   // the workspace of an enqueued range is about to be reused
  if (rc) return rc;
  rc = ensure_workspace(ctx, n);
  if (rc) return rc;
  BIND_PARAMS((cudaStream_t)0);
  ctx->ids_p0 = ctx->ids_p1 = -1;   // the device work list is overwritten below
  const std::vector<int> order = cost_order(P, std::vector<int>(patches, patches + n));
  // diagnostics and status words go to scratch copies (indexed by patch id): the handle's own arrays stay untouched
  const size_t n_diag = (size_t)8 * P.s * ctx->n_patches;
  double *d_dg = nullptr;
  int *d_st = nullptr;
  auto body = [&]() -> int {
    CK(cudaMalloc(&d_dg, sizeof(double) * n_diag));
    CK(cudaMalloc(&d_st, sizeof(int) * (size_t)ctx->n_patches));
    CK(cudaMemset(d_st, 0, sizeof(int) * (size_t)ctx->n_patches));
    CK(cudaMemcpy(ctx->d_ids, order.data(), sizeof(int) * order.size(), cudaMemcpyHostToDevice));
    std::vector<int> st((size_t)ctx->n_patches);
    for (int64_t i0 = 0; i0 < n; i0 += ctx->chunk) {
      const int nc = (int)std::min<int64_t>(ctx->chunk, n - i0);
      rc = launch_patch_stages(ctx, ctx->d_ids + i0, nc, ctx->d_work_counter, 0, d_dg, d_st, nullptr, nullptr);
      if (rc) return rc;
      CK(cudaDeviceSynchronize());
      for (int w = 0; w < nc; ++w) {
        const int id = order[(size_t)(i0 + w)];
        const int64_t i = slot_of[(size_t)id];
        const Geom g = make_geom(P, id);
        double *Gi = G ? G + moff[i] : nullptr;
        if (Gi && !g.slod) {   // LOD branch: no Gram matrix
          std::fill(Gi, Gi + (size_t)g.Ncd * g.Ncd, 0.0);
          Gi = nullptr;
        }
        rc = copy_stages_out(ctx, g, w, X + xoff[i], Minv + moff[i], Gi);
        if (rc) return rc;
      }
    }
    CK(cudaMemcpy(st.data(), d_st, sizeof(int) * st.size(), cudaMemcpyDeviceToHost));
    for (int64_t i = 0; i < n; ++i)
      if (st[(size_t)patches[i]])
        return fail(ctx, SLOD_ERR_NUMERIC, "patch " + std::to_string(patches[i]) + ": numerical status bits " +
                                               std::to_string(st[(size_t)patches[i]]));
    return SLOD_OK;
  };
  rc = body();
  if (d_dg) cudaFree(d_dg);
  if (d_st) cudaFree(d_st);
  return rc;
}

int slod_debug_select(slod_ctx *ctx, int64_t n, const int64_t *patches, const double *G, const double *Minv, double *c,
                      double *diag) {
  if (!ctx) return SLOD_ERR_INVALID;
  if (n < 0 || (n > 0 && (!patches || !G || !Minv || !c || !diag))) return fail(ctx, SLOD_ERR_INVALID, "bad argument");
  const Params &P = ctx->P;
  const int s = P.s;
  // host checks first: nothing is launched on an invalid list
  std::vector<int64_t> moff((size_t)n + 1, 0), coff((size_t)n + 1, 0);   // offsets of the packed matrices / c blocks
  std::vector<char> seen((size_t)ctx->n_patches, 0);
  for (int64_t i = 0; i < n; ++i) {
    const int64_t p = patches[i];
    if (p < 0 || p >= ctx->n_patches) return fail(ctx, SLOD_ERR_INVALID, "patch id out of range");
    if (seen[(size_t)p]) return fail(ctx, SLOD_ERR_INVALID, "repeated patch id " + std::to_string(p));
    seen[(size_t)p] = 1;
    const int ncd = make_geom(P, (int)p).Ncd;
    moff[i + 1] = moff[i] + (int64_t)ncd * ncd;
    coff[i + 1] = coff[i] + (int64_t)s * ncd;
  }
  for (int64_t k = 0; k < moff[n]; ++k)
    if (!std::isfinite(G[k]) || !std::isfinite(Minv[k]))
      return fail(ctx, SLOD_ERR_INVALID, "non-finite entry in G or Minv");
  NEED_DEVICE();
  if (n == 0) return SLOD_OK;
  CK(cudaSetDevice(ctx->device));
  int rc = wait_basis(ctx);   // the workspace of an enqueued range is about to be reused
  if (rc) return rc;
  rc = ensure_workspace(ctx, n);
  if (rc) return rc;
  BIND_PARAMS((cudaStream_t)0);
  ctx->ids_p0 = ctx->ids_p1 = -1;   // the device work list is overwritten below
  // the kernels write diagnostics at patch id * s + d and status bits at the patch id: scratch copies of both keep the
  // handle's own arrays untouched
  const size_t n_diag = (size_t)8 * s * ctx->n_patches;
  double *d_dg = nullptr;
  int *d_st = nullptr;
  auto body = [&]() -> int {
    CK(cudaMalloc(&d_dg, sizeof(double) * n_diag));
    CK(cudaMalloc(&d_st, sizeof(int) * (size_t)ctx->n_patches));
    CK(cudaMemset(d_dg, 0, sizeof(double) * n_diag));
    CK(cudaMemset(d_st, 0, sizeof(int) * (size_t)ctx->n_patches));
    const int64_t ms = ctx->dl.m_stride, ldc = P.NcdMax;
    std::vector<double> hG, hM, hc;
    std::vector<int> ids;
    for (int64_t i0 = 0; i0 < n; i0 += ctx->chunk) {
      const int nc = (int)std::min<int64_t>(ctx->chunk, n - i0);
      ids.assign(patches + i0, patches + i0 + nc);
      hG.assign((size_t)nc * ms, 0.0);
      hM.assign((size_t)nc * ms, 0.0);
      for (int w = 0; w < nc; ++w) {
        const Geom g = make_geom(P, ids[w]);
        const int ncd = g.Ncd;
        const double *Gi = G + moff[i0 + w], *Mi = Minv + moff[i0 + w];
        const std::vector<int> zpos = internal_columns(ctx, g);
        for (int r = 0; r < ncd; ++r)
          for (int col = 0; col < ncd; ++col) {
            hG[(size_t)w * ms + (size_t)zpos[r] * ncd + zpos[col]] = Gi[(size_t)r * ncd + col];
            hM[(size_t)w * ms + (size_t)zpos[r] * ncd + zpos[col]] = Mi[(size_t)r * ncd + col];
          }
      }
      CK(cudaMemcpy(ctx->d_ids, ids.data(), sizeof(int) * nc, cudaMemcpyHostToDevice));
      CK(cudaMemcpy(ctx->d_G, hG.data(), sizeof(double) * hG.size(), cudaMemcpyHostToDevice));
      CK(cudaMemcpy(ctx->d_Minv, hM.data(), sizeof(double) * hM.size(), cudaMemcpyHostToDevice));
      int nl = 0;
      CK(launch_select_pipeline(ctx->sp, 0, ctx->d_ids, nc, ctx->d_Minv, ctx->d_G, ctx->d_cvec, d_dg, d_st, ctx->sb, &nl));
      ctx->launches += nl;
      hc.resize((size_t)nc * s * ldc);
      CK(cudaMemcpy(hc.data(), ctx->d_cvec, sizeof(double) * hc.size(), cudaMemcpyDeviceToHost));
      for (int w = 0; w < nc; ++w) {
        const Geom g = make_geom(P, ids[w]);
        const int ncd = g.Ncd;
        const std::vector<int> zpos = internal_columns(ctx, g);
        for (int col = 0; col < ncd; ++col)
          for (int d = 0; d < s; ++d)
            c[coff[i0 + w] + (int64_t)d * ncd + col] = hc[((size_t)w * s + d) * ldc + zpos[col]];
      }
    }
    std::vector<double> hdg(n_diag);
    std::vector<int> hst((size_t)ctx->n_patches);
    CK(cudaMemcpy(hdg.data(), d_dg, sizeof(double) * n_diag, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(hst.data(), d_st, sizeof(int) * hst.size(), cudaMemcpyDeviceToHost));
    for (int64_t i = 0; i < n; ++i)
      for (int d = 0; d < s; ++d) {
        double *out = diag + ((size_t)i * s + d) * 8;
        std::memcpy(out, hdg.data() + ((size_t)patches[i] * s + d) * 8, sizeof(double) * 8);
        out[7] = hst[(size_t)patches[i]];
      }
    return SLOD_OK;
  };
  rc = body();
  if (d_dg) cudaFree(d_dg);
  if (d_st) cudaFree(d_st);
  return rc;
}

int slod_measure_fp64_peak(slod_ctx *ctx, double *dfma_tflops, double *dmma_tflops) {
  if (!ctx || !dfma_tflops || !dmma_tflops) return SLOD_ERR_INVALID;
  NEED_DEVICE();
  CK(cudaSetDevice(ctx->device));
  CK(cudaDeviceSynchronize());
  CK(run_fp64_probe(ctx->n_sm, dfma_tflops, dmma_tflops));
  ctx->launches += 8;
  return SLOD_OK;
}

int slod_get_timings(const slod_ctx *ctx, double *ms, int n) {
  if (!ctx || !ms) return SLOD_ERR_INVALID;
  if (ctx->device != SLOD_DEVICE_NONE && (ctx->coarse_timing_pending || ctx->basis_pending)) {
    slod_ctx *c = const_cast<slod_ctx *>(ctx);
    int rc = wait_basis(c);   // a numerical status is reported here too: the times of a failed run mean nothing
    if (rc) return rc;
    rc = finish_coarse_timing(c);
    if (rc) return rc;
  }
  for (int i = 0; i < n && i < 8; ++i) ms[i] = ctx->tm.ms[i];
  return SLOD_OK;
}

}  // extern "C"
