// rcvd_api.cu -- host driver + C ABI (include/rcvd.h) of the B200 temporal-consistency solver.
//
// Replaces ceres::Solve as called from DepthVideoPoseOptimizer::poseOptimizationStep
// (reference lib/PoseOptimizer.cpp:954-962) and ::normalizeDepth (:1117-1125): Levenberg-
// Marquardt with Ceres' trust-region rules on the host, all arithmetic on the device.
// There is NO CPU fallback: without a CUDA device rcvd_problem_create fails.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <dlfcn.h>
#include <limits>
#include <map>
#include <set>
#include <string>
#include <vector>

#include <cub/device/device_segmented_sort.cuh>
#include "rcvd_eval.cuh"
#include "rcvd_linalg.cuh"
#include "rcvd_update.cuh"
#include "rcvd_dense.cuh"
#include "rcvd_filter.cuh"
#include "rcvd_bilateral.cuh"
#include "rcvd_builder.cuh"
static int64_t g_filter_launches = 0;

using namespace rcvd;

#define RCVD_API extern "C" __attribute__((visibility("default")))

constexpr int kFastSmem = (3 * kTile * kJsLd + 4 * 256) * (int)sizeof(double);
static bool run_path_ok_host(const rcvd_config& c, const Layout& L);
static bool fast_path_ok_host(const rcvd_config& c, const Layout& L) {
  return L.k == 1 && c.spatial_type == RCVD_SPATIAL_IDENTITY && c.intr_opt != RCVD_INTR_SHARED && !c.fix_poses && !c.fix_depth_xforms &&
         !c.fix_spatial_xforms && (c.depth_type != RCVD_DEPTH_GRID || !c.depth_cubic);
}

static bool run_path_ok_host(const rcvd_config& c, const Layout& L) { return fast_path_ok_host(c, L) && c.depth_type == RCVD_DEPTH_GRID && L.G < 65535; }

static thread_local std::string g_err = "";
static int set_err(int code, const char* fmt, ...) {
  char buf[512]; va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof(buf), fmt, ap); va_end(ap);
  g_err = buf; return code;
}
#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return set_err(RCVD_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); } while (0)

// Every entry point works on the device it is given and puts the caller's current device back on exit (the caller may be a PyTorch
// process working on another GPU of the node).
struct DevGuard {
  int prev = -1; cudaError_t err = cudaSuccess;
  explicit DevGuard(int d) { if (cudaGetDevice(&prev) != cudaSuccess) prev = -1; err = cudaSetDevice(d); }
  ~DevGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
#define SET_DEVICE(d) DevGuard dev_guard_(d); if (dev_guard_.err != cudaSuccess) return set_err(RCVD_ERR_CUDA, "cudaSetDevice(%d) failed: %s", (int)(d), cudaGetErrorString(dev_guard_.err))

// ---- NCCL through dlopen (plumbing only; the data path collective is one all-reduce) ----
namespace nccl {
typedef struct { char internal[128]; } UniqueId;
typedef void* Comm;
static void* lib = nullptr;
static int (*GetUniqueId)(UniqueId*) = nullptr;
static int (*CommInitRank)(Comm*, int, UniqueId, int) = nullptr;
static int (*AllReduce)(const void*, void*, size_t, int, int, Comm, cudaStream_t) = nullptr;
static int (*CommDestroy)(Comm) = nullptr;
static const char* (*GetErrorString)(int) = nullptr;
static int (*GroupStart)() = nullptr;
static int (*GroupEnd)() = nullptr;
static int (*Broadcast)(const void*, void*, size_t, int, int, Comm, cudaStream_t) = nullptr;
static int (*Reduce)(const void*, void*, size_t, int, int, int, Comm, cudaStream_t) = nullptr;
static bool load() {
  if (lib) return true;
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  for (const char* n : names) { lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL); if (lib) break; }
  if (!lib) return false;
  GetUniqueId = (int (*)(UniqueId*))dlsym(lib, "ncclGetUniqueId");
  CommInitRank = (int (*)(Comm*, int, UniqueId, int))dlsym(lib, "ncclCommInitRank");
  AllReduce = (int (*)(const void*, void*, size_t, int, int, Comm, cudaStream_t))dlsym(lib, "ncclAllReduce");
  CommDestroy = (int (*)(Comm))dlsym(lib, "ncclCommDestroy");
  GetErrorString = (const char* (*)(int))dlsym(lib, "ncclGetErrorString");
  GroupStart = (int (*)())dlsym(lib, "ncclGroupStart"); GroupEnd = (int (*)())dlsym(lib, "ncclGroupEnd");
  Broadcast = (int (*)(const void*, void*, size_t, int, int, Comm, cudaStream_t))dlsym(lib, "ncclBroadcast");
  Reduce = (int (*)(const void*, void*, size_t, int, int, int, Comm, cudaStream_t))dlsym(lib, "ncclReduce");
  return GetUniqueId && CommInitRank && AllReduce && CommDestroy && GroupStart && GroupEnd && Broadcast && Reduce;
}
constexpr int kFloat64 = 8, kUint8 = 1, kSum = 0, kMax = 2;   // ncclFloat64, ncclUint8, ncclSum, ncclMax
}  // namespace nccl

// ---- small vector kernels of the LM loop ----
enum { SC_COST = 0, SC_CAND = 1, SC_GY = 2, SC_YHY = 3, SC_STEP2 = 4, SC_X2 = 5, SC_GMAX = 6, SC_GDOTD = 7, SC_DMAX = 8, SC_N = 16 };

__global__ void k_extract_diag(const double* __restrict__ H, double* __restrict__ diag, int N, int npad) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N * npad) return;
  const int f = i / npad, l = i % npad;
  diag[i] = H[(size_t)f * npad * npad + (size_t)l * npad + l];
}
__global__ void k_jacobi_scale(const double* __restrict__ diag, double* __restrict__ S, int n, int enable) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) S[i] = enable ? 1.0 / (1.0 + sqrt(diag[i])) : 1.0;
}
// lmdiag = clamp(S^2 diagH) (unless reuse); D2 = lmdiag / radius; gs = S g
__global__ void k_lm_prepare(const double* __restrict__ diagH, const double* __restrict__ S, const double* __restrict__ g, double* __restrict__ lmdiag,
                             double* __restrict__ D2, double* __restrict__ gs, int n, int reuse, double radius, double dmin, double dmax) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double s = S[i];
  double d = lmdiag[i];
  if (!reuse) { d = fmin(fmax(s * s * diagH[i], dmin), dmax); lmdiag[i] = d; }
  D2[i] = d / radius;
  gs[i] = s * g[i];
}
__global__ void k_mul(const double* __restrict__ a, const double* __restrict__ b, double* __restrict__ o, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) o[i] = a[i] * b[i];
}
__device__ __forceinline__ double project_lb(const rcvd_config& c, const Layout& L, const uint8_t* in_range, int f, int l, double v) {
  if (c.depth_lower_bound && l >= L.offD && l < L.offS && ((l - L.offD) % L.k) == 0 && in_range[f]) return fmax(v, 0.0);
  return v;
}
// xc = Plus(x, alpha * (-y*S)) with bounds projection; accumulates |x - xc|^2 over active params,
// g . delta and max|delta| (for the line search).  y, S, g have npad stride; x, xc nf stride.
__global__ void __launch_bounds__(256) k_candidate(rcvd_config cfg, Layout L, const uint8_t* __restrict__ in_range, const uint8_t* __restrict__ active,
                                                    const double* __restrict__ x, const double* __restrict__ y, const double* __restrict__ S,
                                                    const double* __restrict__ g, double alpha, double* __restrict__ xc, double* __restrict__ scal, int N) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  double d2 = 0.0, gd = 0.0, dm = 0.0;
  if (i < N * L.nf) {
    const int f = i / L.nf, l = i % L.nf;
    const size_t v = (size_t)f * L.npad + l;
    const double delta = -y[v] * S[v];
    const double xn = project_lb(cfg, L, in_range, f, l, x[i] + alpha * delta);
    xc[i] = xn;
    if (active[v]) { const double d = x[i] - xn; d2 = d * d; }
    gd = g[v] * delta; dm = fabs(delta);
  }
  d2 = warp_sum(d2); gd = warp_sum(gd);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) dm = fmax(dm, __shfl_xor_sync(0xffffffffu, dm, o));
  if ((threadIdx.x & 31) == 0) {
    red_add(scal + SC_STEP2, d2); red_add(scal + SC_GDOTD, gd);
    atomicMax((unsigned long long*)(scal + SC_DMAX), (unsigned long long)__double_as_longlong(dm));   // dm >= 0: bit pattern is monotone
  }
}
// |x|^2 over active params and max-norm of the projected gradient step x - Plus(x, -g)
__global__ void __launch_bounds__(256) k_state_norms(rcvd_config cfg, Layout L, const uint8_t* __restrict__ in_range, const uint8_t* __restrict__ active,
                                                      const double* __restrict__ x, const double* __restrict__ g, double* __restrict__ scal, int N) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  double x2 = 0.0, gm = 0.0;
  if (i < N * L.nf) {
    const int f = i / L.nf, l = i % L.nf;
    const size_t v = (size_t)f * L.npad + l;
    if (active[v]) {
      x2 = x[i] * x[i];
      gm = fabs(x[i] - project_lb(cfg, L, in_range, f, l, x[i] - g[v]));
    }
  }
  x2 = warp_sum(x2);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) gm = fmax(gm, __shfl_xor_sync(0xffffffffu, gm, o));
  if ((threadIdx.x & 31) == 0) {
    red_add(scal + SC_X2, x2);
    atomicMax((unsigned long long*)(scal + SC_GMAX), (unsigned long long)__double_as_longlong(gm));
  }
}
__global__ void __launch_bounds__(256) k_dot2(const double* __restrict__ a, const double* __restrict__ b, const double* __restrict__ c,
                                               const double* __restrict__ d, int n, double* __restrict__ scal, int s0, int s1) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  double p = 0.0, q = 0.0;
  if (i < n) { p = a[i] * b[i]; q = c[i] * d[i]; }
  p = warp_sum(p); q = warp_sum(q);
  if ((threadIdx.x & 31) == 0) { red_add(scal + s0, p); red_add(scal + s1, q); }
}
__global__ void k_finalize_mask(rcvd_config cfg, Layout L, uint8_t* __restrict__ mask, int N) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N * L.npad) return;
  const int l = i % L.npad;
  if (l >= L.nf || is_const_local(cfg, L, l)) mask[i] = 0;
}
__global__ void k_project_state(rcvd_config cfg, Layout L, const uint8_t* __restrict__ in_range, double* __restrict__ x, int N) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < N * L.nf) x[i] = project_lb(cfg, L, in_range, i / L.nf, i % L.nf, x[i]);
}
__global__ void k_h_to_dense(const double* __restrict__ H, const HBlock* __restrict__ hb, int nblocks, double* __restrict__ out, int N, int nf, int npad, const int* __restrict__ uperm) {
  const int b = blockIdx.y;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= nf * nf) return;
  const int i = e / nf, j = e % nf;
  const HBlock hbk = hb[b];
  if (hbk.r == hbk.c && j > i) return;
  const double v = H[(size_t)b * npad * npad + (size_t)i * npad + j];
  const size_t U = (size_t)N * nf;
  const int ur = uperm[hbk.r], uc = uperm[hbk.c];          // internal -> caller's frame order
  out[((size_t)ur * nf + i) * U + (size_t)uc * nf + j] = v;
  out[((size_t)uc * nf + j) * U + (size_t)ur * nf + i] = v;
}

// ---------------------------------------------------------------------------
struct Level { int frame_off, nframes; int trsm_off, ntrsm; int upd_off, nupd; int upd2_off, nupd2; int fwd_off, nfwd; int it_off, nit, it2_off, nit2; int own_off, nown; };   // frame_off: every frame of the level (substitution); own_off: the frames this rank factors   // upd: targets consumed by the next level; upd2: the rest

struct rcvd_problem {
  rcvd_config cfg; Layout L; int N = 0; int device = 0;
  cudaStream_t stream = nullptr;
  // host inputs
  std::vector<uint8_t> in_range; std::vector<double> median, adaptive;
  std::vector<int32_t> pair_frames; std::vector<int64_t> offsets; std::vector<float> records_h;
  std::vector<int32_t> struct_pairs;   // global frame-pair graph (multi-GPU); empty -> local pairs
  std::vector<int32_t> trip_centers; std::vector<int64_t> trip_offsets; std::vector<float> trip_records;   // smoothness triplets
  float* d_trip_records = nullptr; int32_t *d_trip_tile_center = nullptr, *d_trip_tile_count = nullptr; int64_t* d_trip_tile_begin = nullptr; int num_trip_tiles = 0;
  int first_frame = 0, last_frame = -1;
  // device problem data
  float* d_records = nullptr; int32_t *d_tile_pair = nullptr, *d_tile_count = nullptr, *d_pair_frames = nullptr, *d_blk_of = nullptr;
  int64_t* d_tile_begin = nullptr; uint8_t *d_in_range = nullptr, *d_active = nullptr;
  double *d_median = nullptr, *d_adaptive = nullptr; float* d_scale_locs = nullptr; int nscale = 0;
  int num_tiles = 0; int64_t C = 0;
  // state & vectors
  double *d_x = nullptr, *d_xc = nullptr, *d_xsave = nullptr;
  double *d_g = nullptr, *d_S = nullptr, *d_diagH = nullptr, *d_lmdiag = nullptr, *d_D2 = nullptr, *d_gs = nullptr, *d_rhs = nullptr, *d_ytmp = nullptr,
         *d_y = nullptr, *d_Sy = nullptr, *d_Hy = nullptr, *d_partial = nullptr, *d_scal = nullptr;
  double* h_scal = nullptr;   // pinned
  int npartial = 0;
  // matrices
  double *d_H = nullptr, *d_Lb = nullptr, *d_T = nullptr, *d_invL = nullptr, *d_invT = nullptr;
  int nHblocks = 0, nLoff = 0; HBlock *d_hblocks = nullptr, *d_lblocks = nullptr; int* d_fail = nullptr;
  std::vector<HBlock> hblocks;
  // schedule
  std::vector<Level> levels; int *d_lvl_frames = nullptr; GemmTask *d_trsm_tasks = nullptr, *d_upd_tasks = nullptr; int2 *d_trsm_pairs = nullptr, *d_upd_pairs = nullptr;
  SubTask* d_sub_tasks = nullptr; int n_sub_tasks = 0; int* d_sub_counters = nullptr; int* d_sub_need = nullptr; int fused_subst = 1, sub_first_level = 0;   // k_substitution: levels >= sub_first_level (fused_subst: 0 off, 1 default width limit, > 1 that many tasks per level phase)
  SolveTask *d_fwd_tasks = nullptr, *d_col_tasks = nullptr; int* d_col_ptr = nullptr; TrsmTask* d_trsm_ll = nullptr; bool use_trsm_ll = false, trsm_deep = true;
  cudaGraphExec_t solve_graph = nullptr;
  bool structure_ready = false, constraints_set = false, frames_set = false;
  // multi GPU
  int nranks = 1, rank = 0; nccl::Comm comm = nullptr;
  int64_t launches = 0, graph_launches = 0;
  std::vector<double> h_state; bool state_dirty = false; bool use_fast = true; bool overlap = true; bool trim_gemm = true; bool potrf_chain_warp = true; bool potrf_blocked = true; int side_slice = 0; bool allow_trsm_ll = true; bool sub_solves = false; int order_slack = 4;   // multiple elimination with degree slack 4 (measured at config 2: slack 1..5 -> 13.65 13.11 12.74 12.66 13.09 ms per iteration); -1: greedy minimum degree
  cudaStream_t side_stream = nullptr; cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  double *d_g2 = nullptr, *d_delta = nullptr; int* h_fail = nullptr;
  cudaEvent_t ev[8] = {nullptr};
  std::vector<void*> allocs;
  // kernel-class profiling (rcvd_debug_profile_linear): when set, enqueue_factor_solve records one event per launch
  std::vector<std::pair<int, cudaEvent_t>>* prof = nullptr;
  // distributed factorisation (nranks > 1): ownership, internal frame numbering, broadcast / reduce segments
  bool eval_only = false;   // test / bench hook: only rcvd_evaluate is used (no H, no factor storage)
  bool use_runs = true, records_sorted = false;   // run path of the accumulate kernel (bilinear depth grid): records sorted by cell pair
  bool dist_enabled = true, dist = false, identity_perm = true, graph_warm = false, force_full_H = false; int LB = 0;
  std::vector<int> uperm, iperm, fa_off, fa_cnt, fb_off, fb_cnt, tseg, bseg, hseg;   // *_off/_cnt: per-owner frame ranges (phase A / B); segs: (first, count) pairs
  int *d_lvl_own = nullptr, *d_own_lblocks = nullptr, *d_own_hblocks = nullptr, *d_uperm = nullptr; int n_own_l = 0, n_own_h = 0;
  // TMA-fed persistent update kernel (rcvd_update.cuh)
  UpdItem* d_upd_items = nullptr; CUtensorMap tmapT; bool gemm_tma = true, tmap_ok = false; int upd_rb = 0, upd_neff = 0, num_sms = 148, upd_ipc = 0, upd_dbg = 0, upd_team_items = 1, upd_reserve = 0;   // upd_reserve: SMs kept free by the overlapped updates of narrow levels; upd_team_items: launches of <= that many items per SM take the two-team shape
  std::vector<double> level_ms;   // last rcvd_debug_profile_linear: per level x kernel class
  double upd_flops = 0.0;   // algorithmic flops of the update GEMMs of one factorisation (2 nf^3 per product, nf^2 (nf+1) on symmetric targets)
  rcvd_problem() {}
};

template <class T> static int dalloc(rcvd_problem* p, T** ptr, size_t count) {
  *ptr = nullptr;
  if (count == 0) count = 1;
  // stream-ordered pool allocation: the reference calls the solver once per schedule step, so a handle's
  // gigabytes of factor storage are recycled from the pool instead of paying cudaMalloc/cudaFree per call
  cudaError_t e = cudaMallocAsync((void**)ptr, count * sizeof(T), p->stream);
  if (e != cudaSuccess) return set_err(RCVD_ERR_CUDA, "cudaMallocAsync(%zu bytes) failed: %s", count * sizeof(T), cudaGetErrorString(e));
  p->allocs.push_back(*ptr);
  return RCVD_OK;
}
template <class T> static int upload(rcvd_problem* p, T** ptr, const std::vector<T>& v) {
  int rc = dalloc(p, ptr, v.size()); if (rc) return rc;
  if (!v.empty()) CK(cudaMemcpyAsync(*ptr, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, p->stream));
  return RCVD_OK;
}
static void free_all(rcvd_problem* p) {
  if (p->solve_graph) { cudaGraphExecDestroy(p->solve_graph); p->solve_graph = nullptr; }
  if (p->side_stream) cudaStreamSynchronize(p->side_stream);
  for (void* q : p->allocs) cudaFreeAsync(q, p->stream);
  p->allocs.clear();
  if (p->stream) cudaStreamSynchronize(p->stream);
  if (p->h_scal) { cudaFreeHost(p->h_scal); p->h_scal = nullptr; }
  p->structure_ready = false;
}

static DevProblem dev_problem(const rcvd_problem* p) {
  DevProblem d; d.cfg = p->cfg; d.L = p->L; d.N = p->N; d.num_tiles = p->num_tiles; d.num_constraints = p->C;
  d.records = p->d_records; d.tile_pair = p->d_tile_pair; d.tile_begin = p->d_tile_begin; d.tile_count = p->d_tile_count;
  d.pair_frames = p->d_pair_frames; d.blk_of = p->d_blk_of; d.in_range = p->d_in_range; d.median = p->d_median;
  d.adaptive = p->adaptive.empty() ? nullptr : p->d_adaptive; d.scale_locs = p->d_scale_locs; d.num_scale_locs = p->nscale;
  d.rank = p->rank; d.nranks = p->nranks;
  d.trip_records = p->d_trip_records; d.trip_tile_center = p->d_trip_tile_center; d.trip_tile_begin = p->d_trip_tile_begin; d.trip_tile_count = p->d_trip_tile_count; d.num_trip_tiles = p->num_trip_tiles;
  return d;
}

// ---- structure: block layout, elimination order, level schedule ----
static int build_structure(rcvd_problem* p) {
  free_all(p);
  const int N = p->N; const Layout& L = p->L; const int npad = L.npad; const size_t bs = (size_t)npad * npad;
  CK(cudaSetDevice(p->device));
  // frame graph
  std::vector<std::set<int>> adj(N);
  auto addEdge = [&](int a, int b) { if (a != b) { adj[a].insert(b); adj[b].insert(a); } };
  const std::vector<int32_t>& sp = p->struct_pairs.empty() ? p->pair_frames : p->struct_pairs;
  for (size_t i = 0; i + 1 < sp.size(); i += 2) {
    const int a = sp[i], b = sp[i + 1];
    if (a < 0 || a >= N || b < 0 || b >= N) return set_err(RCVD_ERR_INVALID, "pair frame index out of range");
    addEdge(a, b);
    if (p->cfg.intr_opt == RCVD_INTR_SHARED) { addEdge(a, 0); addEdge(b, 0); }
  }
  if (p->cfg.position_reg > 0.0) for (int f = 0; f + 2 < N; ++f) { addEdge(f, f + 1); addEdge(f, f + 2); addEdge(f + 1, f + 2); }
  for (size_t t = 0; t < p->trip_centers.size(); ++t) {
    const int f = p->trip_centers[t];
    if (f < 1 || f + 1 >= N) return set_err(RCVD_ERR_INVALID, "triplet centre frame out of range");
    addEdge(f - 1, f); addEdge(f - 1, f + 1); addEdge(f, f + 1);
    if (p->cfg.intr_opt == RCVD_INTR_SHARED) { addEdge(f - 1, 0); addEdge(f, 0); addEdge(f + 1, 0); }
  }
  std::vector<std::set<int>> orig = adj;
  // Multiple minimum-degree elimination: each round eliminates a maximal independent set of frames whose current degree is
  // within `slack` of the minimum (ties -> lowest frame id).  slack = 0 is plain greedy minimum degree one frame at a time
  // semantics-wise; a small slack trades a few % more fill for a shallower elimination tree (fewer sequential levels).
  std::vector<int> order, pos(N, -1); std::vector<std::vector<int>> cs(N);
  {
    std::vector<uint8_t> done(N, 0);
    const int slack = p->order_slack;
    while ((int)order.size() < N) {
      size_t md = (size_t)-1;
      for (int f = 0; f < N; ++f) if (!done[f]) md = std::min(md, adj[f].size());
      std::vector<int> cand;
      const size_t lim = md + (size_t)(slack > 0 ? slack : 0);
      for (int f = 0; f < N; ++f) if (!done[f] && adj[f].size() <= lim) cand.push_back(f);
      std::stable_sort(cand.begin(), cand.end(), [&](int a, int b) { return adj[a].size() < adj[b].size(); });
      std::vector<uint8_t> blocked(N, 0); std::vector<int> chosen;
      for (int f : cand) { if (blocked[f]) continue; chosen.push_back(f); blocked[f] = 1; for (int a : adj[f]) blocked[a] = 1; if (slack < 0) break; }
      for (int best : chosen) {
        done[best] = 1; pos[best] = (int)order.size(); order.push_back(best);
        std::vector<int> nb(adj[best].begin(), adj[best].end());
        cs[best] = nb;
        for (int a : nb) adj[a].erase(best);
        for (size_t i = 0; i < nb.size(); ++i) for (size_t j = i + 1; j < nb.size(); ++j) { adj[nb[i]].insert(nb[j]); adj[nb[j]].insert(nb[i]); }
      }
    }
    for (int f = 0; f < N; ++f) std::sort(cs[f].begin(), cs[f].end(), [&](int a, int b) { return pos[a] < pos[b]; });
  }
  // levels
  std::vector<int> lvl(N, 0); int nl = 0;
  for (int k : order) { for (int a : cs[k]) lvl[a] = std::max(lvl[a], lvl[k] + 1); nl = std::max(nl, lvl[k] + 1); }
  std::vector<std::vector<int>> lf(nl);
  for (int k : order) lf[lvl[k]].push_back(k);

  // ---- multi-GPU distribution of the factorisation (DESIGN.md section 5) ----
  // Phase A = the wide early levels (throughput-bound: thousands of block products): every frame (= block column of the factor) has an
  // owner rank that factors it (potrf, trsm) and computes every update INTO its column; after the trsm of a level the new off-diagonal
  // factor blocks X_rk are broadcast from their owners (they are the operands of everybody's updates and of the replicated
  // substitution).  Phase B = the tail of narrow levels (< 3 frames per level: a latency chain that does not shard) is replicated:
  // at the boundary every owner broadcasts its trailing blocks.  H is reduced to the owners only (no all-reduce of the matrix).
  const int R = p->nranks;
  bool dist = R > 1 && p->dist_enabled && p->cfg.intr_opt != RCVD_INTR_SHARED && !(p->cfg.position_reg > 0.0) && p->trip_centers.empty();
  int LB = 0;
  if (dist) { LB = nl; while (LB > 0 && (int)lf[LB - 1].size() < 3) --LB; if (LB == 0) dist = false; }
  p->dist = dist; p->LB = LB;
  std::vector<int> own(N, 0);
  if (dist) {
    // incoming update work of every column over the phase-A levels (block products; symmetric targets count half)
    std::vector<double> tot_in(N, 0.0);
    for (int l = 0; l < LB; ++l) for (int k : lf[l]) { const auto& m = cs[k]; for (size_t a = 0; a < m.size(); ++a) for (size_t b = 0; b <= a; ++b) tot_in[m[b]] += (a == b) ? 0.5 : 1.0; }
    std::vector<double> load(R, 0.0);
    for (int l = 0; l < nl; ++l) {
      std::vector<int> fr = lf[l];
      auto w = [&](int k) { return tot_in[k] + (l < LB ? 0.6 * cs[k].size() + 0.3 : 0.0); };   // + its own trsm / potrf
      std::stable_sort(fr.begin(), fr.end(), [&](int a, int b) { return w(a) > w(b); });
      for (int k : fr) { int q = 0; for (int t = 1; t < R; ++t) if (load[t] < load[q]) q = t; own[k] = q; load[q] += w(k); }
    }
  }
  // internal frame numbering: owner-major, phase-A frames first -- every per-frame array an owner broadcasts / reduces is one contiguous range
  std::vector<int> uperm, iperm(N, -1);
  p->fa_off.assign(R, 0); p->fa_cnt.assign(R, 0); p->fb_off.assign(R, 0); p->fb_cnt.assign(R, 0);
  for (int q = 0; q < R; ++q) for (int ph = 0; ph < 2; ++ph) {
    (ph ? p->fb_off : p->fa_off)[q] = (int)uperm.size();
    for (int f = 0; f < N; ++f) if (own[f] == q && ((lvl[f] >= LB) == (ph == 1))) uperm.push_back(f);
    (ph ? p->fb_cnt : p->fa_cnt)[q] = (int)uperm.size() - (ph ? p->fb_off : p->fa_off)[q];
  }
  for (int i = 0; i < N; ++i) iperm[uperm[i]] = i;
  p->identity_perm = true; for (int i = 0; i < N; ++i) if (uperm[i] != i) p->identity_perm = false;
  p->uperm = uperm; p->iperm = iperm;
  if (!p->identity_perm) {
    auto I = [&](int f) { return iperm[f]; };
    std::vector<int> order2(N), pos2(N), lvl2(N), own2(N); std::vector<std::vector<int>> cs2(N); std::vector<std::set<int>> orig2(N);
    for (int i = 0; i < N; ++i) order2[i] = I(order[i]);
    for (int f = 0; f < N; ++f) { pos2[I(f)] = pos[f]; lvl2[I(f)] = lvl[f]; own2[I(f)] = own[f]; for (int a : cs[f]) cs2[I(f)].push_back(I(a)); for (int a : orig[f]) orig2[I(f)].insert(I(a)); }
    for (auto& v : lf) for (int& k : v) k = I(k);
    order.swap(order2); pos.swap(pos2); lvl.swap(lvl2); own.swap(own2); cs.swap(cs2); orig.swap(orig2);
  }
  // L off-diagonal blocks (r later than c).  Phase A: level-major, owner-major inside a level (what a rank produces in one level is one
  // contiguous range of T); phase B: owner-major (what a rank owns of the trailing matrix is one contiguous range of L).
  std::map<std::pair<int, int>, int> lid; int nLoff = 0;
  std::vector<int> lcol;   // column (earlier-eliminated) frame of each off-diagonal factor block
  auto number_col = [&](int k) { for (int r : cs[k]) { lid[{r, k}] = N + nLoff++; lcol.push_back(k); } };
  p->tseg.assign((size_t)std::max(LB, 0) * R * 2, 0); p->bseg.assign((size_t)R * 2, 0);
  for (int l = 0; l < LB; ++l) for (int q = 0; q < R; ++q) {
    const int first = nLoff;
    for (int k : lf[l]) if (own[k] == q) number_col(k);
    p->tseg[((size_t)l * R + q) * 2] = first; p->tseg[((size_t)l * R + q) * 2 + 1] = nLoff - first;
  }
  for (int q = 0; q < R; ++q) {
    const int first = nLoff;
    for (int l = LB; l < nl; ++l) for (int k : lf[l]) if (own[k] == q) number_col(k);
    p->bseg[(size_t)q * 2] = first; p->bseg[(size_t)q * 2 + 1] = nLoff - first;
  }
  p->nLoff = nLoff;
  // H blocks: diagonal first (internal frame order = owner-major), then original off-diagonals oriented (later, earlier), owner-major
  p->hblocks.clear();
  std::vector<int32_t> blk_of((size_t)N * N, -1);
  for (int f = 0; f < N; ++f) p->hblocks.push_back({f, f, f});
  p->hseg.assign((size_t)R * 2, 0);
  for (int q = 0; q < R; ++q) {
    p->hseg[(size_t)q * 2] = (int)p->hblocks.size();
    for (int a = 0; a < N; ++a) for (int b : orig[a]) if (a < b) {
      const int r = pos[a] > pos[b] ? a : b, c = pos[a] > pos[b] ? b : a;
      if (own[c] != q) continue;
      const int hid = (int)p->hblocks.size();
      p->hblocks.push_back({lid[{r, c}], r, c});
      blk_of[(size_t)r * N + c] = hid * 2 + 1;   // (fa = r) is the row side
      blk_of[(size_t)c * N + r] = hid * 2 + 0;
    }
    p->hseg[(size_t)q * 2 + 1] = (int)p->hblocks.size() - p->hseg[(size_t)q * 2];
  }
  p->nHblocks = (int)p->hblocks.size();
  // all L blocks with their H source (or -1)
  std::vector<HBlock> lblocks(N + nLoff);
  for (int f = 0; f < N; ++f) lblocks[f] = {f, f, f};
  for (auto& kv : lid) lblocks[kv.second] = {-1, kv.first.first, kv.first.second};
  for (int h = N; h < p->nHblocks; ++h) lblocks[p->hblocks[h].lblk].lblk = h;
  // blocks this rank owns: what it loads into the factor and what it multiplies in the model term (all of them without distribution)
  std::vector<int> own_lblocks, own_hblocks;
  for (int b = 0; b < N + nLoff; ++b) { const int c = b < N ? b : lcol[b - N]; if (!dist || own[c] == p->rank) own_lblocks.push_back(b); }
  for (int h = 0; h < p->nHblocks; ++h) if (!dist || own[p->hblocks[h].c] == p->rank) own_hblocks.push_back(h);
  p->n_own_l = (int)own_lblocks.size(); p->n_own_h = (int)own_hblocks.size();
  double upd_flops = 0.0;
  std::vector<int> lvl_frames, lvl_own; std::vector<GemmTask> trsm_tasks, upd_tasks; std::vector<int2> trsm_pairs, upd_pairs;
  std::vector<SolveTask> fwd_tasks, col_tasks; std::vector<int> col_ptr(N + 1, 0); std::vector<TrsmTask> trsm_ll;
  std::vector<UpdItem> upd_items;
  // tile cut of the update targets: kUpdMaxTile-row tiles over the unknowns (rounded to 8)
  const int upd_neff = std::min(npad, (L.nf + 7) / 8 * 8);
  const int upd_nt = (upd_neff + kUpdMaxTile - 1) / kUpdMaxTile;
  const int upd_tile = std::min(kUpdMaxTile, upd_neff);          // 80-row tiles (balanced 5 x 5 units per warp), the remainder last
  p->upd_rb = upd_tile; p->upd_neff = upd_neff;
  p->levels.clear();
  for (int l = 0; l < nl; ++l) {
    Level lv; lv.frame_off = (int)lvl_frames.size(); lv.nframes = (int)lf[l].size(); lv.own_off = (int)lvl_own.size();
    lv.trsm_off = (int)trsm_tasks.size(); lv.upd_off = (int)upd_tasks.size(); lv.fwd_off = (int)fwd_tasks.size();
    std::map<int, std::vector<int2>> upd;   // target L block id -> source pairs
    const bool shared_level = !dist || l >= LB;   // replicated work: every rank does all of it
    for (int k : lf[l]) {
      lvl_frames.push_back(k);
      const bool mine = shared_level || own[k] == p->rank;
      if (mine) lvl_own.push_back(k);
      for (int r : cs[k]) {
        const int id = lid[{r, k}];
        if (mine) {
          trsm_tasks.push_back({id - N, (int)trsm_pairs.size(), 1, 2});
          trsm_pairs.push_back(make_int2(id, k));
          trsm_ll.push_back({id - N, id, k});
        }
        fwd_tasks.push_back({id - N, r, k});
      }
      for (size_t a = 0; a < cs[k].size(); ++a) for (size_t b = 0; b <= a; ++b) {
        const int r = cs[k][a], c = cs[k][b];                     // c is eliminated before r: the target lives in column c
        if (!shared_level && own[c] != p->rank) continue;
        const int target = (r == c) ? r : lid[{r, c}];
        upd[target].push_back(make_int2(lid[{r, k}] - N, lid[{c, k}] - N));
      }
    }
    lv.nown = (int)lvl_own.size() - lv.own_off;
    // targets whose column frame is eliminated in the very next level must be complete before that level starts (critical);
    // all other updates may overlap the next level's potrf / inverse / trsm on a second stream.
    for (int pass = 0; pass < 2; ++pass) {
      if (pass == 1) lv.upd2_off = (int)upd_tasks.size();
      for (auto& kv : upd) {
        const int cframe = kv.first < N ? kv.first : lcol[kv.first - N];
        const bool critical = (lvl[cframe] == l + 1);
        if (critical != (pass == 0)) continue;
        upd_tasks.push_back({kv.first, (int)upd_pairs.size(), (int)kv.second.size(), kv.first < N ? 1 : 0});
        { const double n = (double)L.nf; upd_flops += (double)kv.second.size() * (kv.first < N ? n * n * (n + 1.0) : 2.0 * n * n * n); }
        upd_pairs.insert(upd_pairs.end(), kv.second.begin(), kv.second.end());
      }
    }
    lv.ntrsm = (int)trsm_tasks.size() - lv.trsm_off; lv.nupd = lv.upd2_off - lv.upd_off; lv.nupd2 = (int)upd_tasks.size() - lv.upd2_off; lv.nfwd = (int)fwd_tasks.size() - lv.fwd_off;
    // work items of the persistent update kernel: one per (target tile, source-pair list), heaviest first
    for (int pass = 0; pass < 2; ++pass) {
      const int t0 = pass ? lv.upd2_off : lv.upd_off, tn = pass ? lv.nupd2 : lv.nupd;
      const size_t i0 = upd_items.size();
      for (int q = t0; q < t0 + tn; ++q) {
        const GemmTask& tk = upd_tasks[q];
        for (int ti = 0; ti < upd_nt; ++ti) for (int tj = 0; tj < ((tk.lower_only & 1) ? ti + 1 : upd_nt); ++tj) {
          UpdItem it; it.dst = tk.dst; it.first = tk.first; it.count = tk.count; it.m0 = (short)(ti * upd_tile); it.n0 = (short)(tj * upd_tile);
          it.mrows = (short)std::min(upd_tile, upd_neff - ti * upd_tile); it.ncols = (short)std::min(upd_tile, upd_neff - tj * upd_tile);
          it.flags = ((tk.lower_only & 1) && ti == tj) ? 1 : 0;
          upd_items.push_back(it);
        }
      }
      auto cost = [](const UpdItem& a) { return (long)a.count * (a.mrows / 8) * (a.ncols / 8) * ((a.flags & 1) ? 3 : 4); };
      std::stable_sort(upd_items.begin() + i0, upd_items.end(), [&](const UpdItem& a, const UpdItem& b) { return cost(a) > cost(b); });
      if (pass) { lv.it2_off = (int)i0; lv.nit2 = (int)(upd_items.size() - i0); } else { lv.it_off = (int)i0; lv.nit = (int)(upd_items.size() - i0); }
    }
    p->levels.push_back(lv);
  }
  for (int k = 0; k < N; ++k) { col_ptr[k] = (int)col_tasks.size(); for (int r : cs[k]) col_tasks.push_back({lid[{r, k}] - N, r, k}); }
  col_ptr[N] = (int)col_tasks.size();
  // task list of the fused substitution kernel (k_substitution): forward levels ascending, backward levels descending, every GEMV cut
  // into kSubChunk-row / -column chunks; a task depends only on tasks before it
  std::vector<SubTask> sub_tasks; std::vector<int> sub_need(2 * (size_t)N, 0);
  {
    const int nch = (npad + kSubChunk - 1) / kSubChunk;
    // The wide levels at the bottom of the tree stay level-scheduled launches (thousands of independent GEMVs: a launch spreads them
    // over the machine at once, a persistent CTA works through them one memory latency at a time); the narrow levels above them -- a
    // latency chain of four tiny launches per level -- run as ONE dataflow kernel: forward narrow, backward narrow in a single launch.
    const int limit = p->fused_subst <= 0 ? -1 : (p->fused_subst == 1 ? 4 * p->num_sms : p->fused_subst);
    int LS = (int)p->levels.size();
    while (LS > 0 && (p->levels[LS - 1].nframes + p->levels[LS - 1].nfwd) * nch <= limit) --LS;
    p->sub_first_level = LS;
    for (size_t l = LS; l < p->levels.size(); ++l) {
      const Level& lv = p->levels[l];
      for (int i = 0; i < lv.nframes; ++i) for (int c = 0; c < nch; ++c) sub_tasks.push_back({0, -1, -1, lvl_frames[lv.frame_off + i], c});
      for (int q = 0; q < lv.nfwd; ++q) { const SolveTask& t = fwd_tasks[lv.fwd_off + q]; for (int c = 0; c < nch; ++c) sub_tasks.push_back({1, t.blk, t.r, t.k, c}); sub_need[t.r] += nch; sub_need[N + t.k] += nch; }
    }
    for (int l = (int)p->levels.size() - 1; l >= LS; --l) {
      const Level& lv = p->levels[l];
      for (int q = 0; q < lv.nfwd; ++q) { const SolveTask& t = fwd_tasks[lv.fwd_off + q]; for (int c = 0; c < nch; ++c) sub_tasks.push_back({2, t.blk, t.r, t.k, c}); }
      for (int i = 0; i < lv.nframes; ++i) for (int c = 0; c < nch; ++c) sub_tasks.push_back({3, -1, -1, lvl_frames[lv.frame_off + i], c});
    }
    p->n_sub_tasks = (int)sub_tasks.size();
  }

  // ---- device allocations ----
  int rc;
#define UP(ptr, vec) if ((rc = upload(p, &(ptr), vec))) return rc
  p->upd_flops = upd_flops;
  UP(p->d_blk_of, blk_of); UP(p->d_hblocks, p->hblocks); UP(p->d_lblocks, lblocks); UP(p->d_lvl_frames, lvl_frames); UP(p->d_lvl_own, lvl_own);
  UP(p->d_own_lblocks, own_lblocks); UP(p->d_own_hblocks, own_hblocks); UP(p->d_uperm, p->uperm);
  UP(p->d_trsm_tasks, trsm_tasks); UP(p->d_upd_tasks, upd_tasks); UP(p->d_trsm_pairs, trsm_pairs); UP(p->d_upd_pairs, upd_pairs);
  UP(p->d_sub_tasks, sub_tasks); UP(p->d_sub_need, sub_need); if ((rc = dalloc(p, &p->d_sub_counters, (size_t)4 * N + 4))) return rc;
  UP(p->d_fwd_tasks, fwd_tasks); UP(p->d_col_tasks, col_tasks); UP(p->d_col_ptr, col_ptr); UP(p->d_trsm_ll, trsm_ll); UP(p->d_upd_items, upd_items);
  // tiles
  const int np = (int)(p->pair_frames.size() / 2);
  std::vector<int32_t> tile_pair, tile_count; std::vector<int64_t> tile_begin;
  for (int i = 0; i < np; ++i)
    for (int64_t b = p->offsets[i]; b < p->offsets[i + 1]; b += kTile) { tile_pair.push_back(i); tile_begin.push_back(b); tile_count.push_back((int32_t)std::min<int64_t>(kTile, p->offsets[i + 1] - b)); }
  p->num_tiles = (int)tile_pair.size(); p->C = p->offsets.empty() ? 0 : p->offsets.back();
  UP(p->d_tile_pair, tile_pair); UP(p->d_tile_begin, tile_begin); UP(p->d_tile_count, tile_count);
  {
    std::vector<int32_t> pf_int(p->pair_frames.size());
    for (size_t i = 0; i < pf_int.size(); ++i) pf_int[i] = p->iperm[p->pair_frames[i]];
    UP(p->d_pair_frames, pf_int); UP(p->d_records, p->records_h);
  }
  p->records_sorted = false;
  if (p->use_runs && run_path_ok_host(p->cfg, L) && p->C > 0 && p->C < (int64_t)0x7fffffff) {
    // run path of the accumulate kernel: the records of every pair sorted by (source cell, target cell) -- device segmented sort by pair
    const long long n = p->C;
    unsigned *d_k0 = nullptr, *d_k1 = nullptr; int *d_i0 = nullptr, *d_i1 = nullptr; float* d_sorted = nullptr; int64_t* d_off = nullptr; void* d_tmp = nullptr;
    int rcs;
    if ((rcs = dalloc(p, &d_k0, (size_t)n)) || (rcs = dalloc(p, &d_k1, (size_t)n)) || (rcs = dalloc(p, &d_i0, (size_t)n)) || (rcs = dalloc(p, &d_i1, (size_t)n)) || (rcs = dalloc(p, &d_sorted, (size_t)n * 6)) ||
        (rcs = upload(p, &d_off, p->offsets))) return rcs;
    k_record_keys<<<(unsigned)((n + 255) / 256), 256, 0, p->stream>>>(p->cfg, p->d_records, n, d_k0, d_i0);
    size_t tmp_bytes = 0;
    CK(cub::DeviceSegmentedSort::SortPairs(nullptr, tmp_bytes, d_k0, d_k1, d_i0, d_i1, (int)n, np, d_off, d_off + 1, p->stream));
    CK(cudaMallocAsync(&d_tmp, std::max<size_t>(tmp_bytes, 16), p->stream));
    CK(cub::DeviceSegmentedSort::SortPairs(d_tmp, tmp_bytes, d_k0, d_k1, d_i0, d_i1, (int)n, np, d_off, d_off + 1, p->stream));
    k_gather_records<<<(unsigned)((n * 6 + 255) / 256), 256, 0, p->stream>>>(p->d_records, d_i1, n, d_sorted);
    CK(cudaFreeAsync(d_tmp, p->stream));
    CK(cudaGetLastError());
    p->d_records = d_sorted; p->records_sorted = true;      // (the unsorted copy and the sort buffers go back to the pool with the handle's other allocations)
  }
  {
    std::vector<int32_t> tc, tn; std::vector<int64_t> tb;
    for (size_t i = 0; i < p->trip_centers.size(); ++i)
      for (int64_t b = p->trip_offsets[i]; b < p->trip_offsets[i + 1]; b += kTile) { tc.push_back(p->trip_centers[i]); tb.push_back(b); tn.push_back((int32_t)std::min<int64_t>(kTile, p->trip_offsets[i + 1] - b)); }
    p->num_trip_tiles = (int)tc.size();
    UP(p->d_trip_tile_center, tc); UP(p->d_trip_tile_begin, tb); UP(p->d_trip_tile_count, tn); UP(p->d_trip_records, p->trip_records);
  }
  {
    std::vector<uint8_t> ir(N); std::vector<double> md(N), ad;
    for (int i = 0; i < N; ++i) { ir[i] = p->in_range[p->uperm[i]]; md[i] = p->median[p->uperm[i]]; }
    UP(p->d_in_range, ir); UP(p->d_median, md);
    if (!p->adaptive.empty()) {
      const size_t G = p->adaptive.size() / N; ad.resize(p->adaptive.size());
      for (int i = 0; i < N; ++i) std::copy(p->adaptive.begin() + (size_t)p->uperm[i] * G, p->adaptive.begin() + (size_t)(p->uperm[i] + 1) * G, ad.begin() + (size_t)i * G);
      UP(p->d_adaptive, ad);
    }
  }
  {
    // scale-regulariser lattice in float32, lib/PoseOptimizer.cpp:1382-1385
    std::vector<float> locs; const int gx = p->cfg.scale_grid_x, gy = p->cfg.scale_grid_y;
    for (int y = 0; y < gy; ++y) for (int x = 0; x < gx; ++x) {
      // host code is built without -mfma, so these float ops are not contracted
      const float fx = -1.f + 2.f * x / (gx - 1);
      const float fy = -1.f + 2.f * y / (gy - 1);
      locs.push_back(fx); locs.push_back(fy);
    }
    p->nscale = (int)(locs.size() / 2);
    UP(p->d_scale_locs, locs);
  }
#undef UP
  p->first_frame = 0; p->last_frame = -1;
  { bool any = false; for (int f = 0; f < N; ++f) if (p->in_range[f]) { if (!any) { p->first_frame = f; any = true; } p->last_frame = f; } }
  const size_t Upad = (size_t)N * npad, U = (size_t)N * L.nf;
#define DA(ptr, n) if ((rc = dalloc(p, &(ptr), (n)))) return rc
  DA(p->d_x, U); DA(p->d_xc, U); DA(p->d_xsave, U);
  DA(p->d_g, 2 * Upad + 8); p->d_diagH = p->d_g + Upad + 8;   // [gradient | 8 scalars | diag H]: one packed all-reduce at N > 1
  DA(p->d_S, Upad); DA(p->d_lmdiag, Upad); DA(p->d_D2, Upad); DA(p->d_gs, Upad); DA(p->d_rhs, Upad);
  DA(p->d_g2, Upad + 8); DA(p->d_delta, Upad);
  DA(p->d_ytmp, Upad); DA(p->d_y, Upad); DA(p->d_Sy, Upad); DA(p->d_Hy, Upad); DA(p->d_scal, SC_N); DA(p->d_active, Upad); DA(p->d_fail, 1);
  const RegCounts rcn = reg_counts(p->cfg, L, N, p->nscale);
  p->npartial = p->num_tiles + (rcn.total + 127) / 128 + p->num_trip_tiles + 1;
  DA(p->d_partial, (size_t)p->npartial);
  if (p->eval_only) { DA(p->d_H, 1); DA(p->d_Lb, 1); DA(p->d_T, 1); DA(p->d_invL, 1); DA(p->d_invT, 1); }   // cost / gradient evaluations only: no matrices
  else {
    DA(p->d_H, (size_t)p->nHblocks * bs); DA(p->d_Lb, (size_t)(N + nLoff) * bs); DA(p->d_T, (size_t)std::max(nLoff, 1) * bs);
    DA(p->d_invL, (size_t)N * bs); DA(p->d_invT, (size_t)N * npad * 16);
  }
#undef DA
  {
    // 2-D TMA view of the T buffer (off-diagonal factor blocks X_rk, row-major): inner = k, outer = block * npad + row, box [rb][16], 128-B swizzle
    p->tmap_ok = false;
    cudaDeviceGetAttribute(&p->num_sms, cudaDevAttrMultiProcessorCount, p->device);
    typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                 CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    void* fn = nullptr; cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess && fn && qres == cudaDriverEntryPointSuccess) {
      const cuuint64_t gdim[2] = {(cuuint64_t)npad, (cuuint64_t)std::max(nLoff, 1) * npad};
      const cuuint64_t gstr[1] = {(cuuint64_t)npad * sizeof(double)};
      const cuuint32_t box[2] = {16u, (cuuint32_t)p->upd_rb};
      const cuuint32_t estr[2] = {1u, 1u};
      const CUresult r = ((EncodeFn)fn)(&p->tmapT, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, p->d_T, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                        CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      p->tmap_ok = (r == CUDA_SUCCESS);
    }
    cudaGetLastError();
    if (p->tmap_ok) { CK(cudaFuncSetAttribute(k_update_tma<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)upd_smem_bytes(p->upd_rb, 1))); CK(cudaFuncSetAttribute(k_update_tma<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)upd_smem_bytes(p->upd_rb, 2))); }
    else if (p->gemm_tma) return set_err(RCVD_ERR_CUDA, "cuTensorMapEncodeTiled unavailable or failed: the TMA update kernel cannot run");
  }
  CK(cudaMallocHost((void**)&p->h_scal, (SC_N + 2) * sizeof(double)));
  p->h_fail = (int*)(p->h_scal + SC_N);
  CK(cudaMemsetAsync(p->d_x, 0, U * sizeof(double), p->stream));
  CK(cudaMemsetAsync(p->d_lmdiag, 0, Upad * sizeof(double), p->stream));
  CK(cudaMemsetAsync(p->d_S, 0, Upad * sizeof(double), p->stream));
  // active mask
  CK(cudaMemsetAsync(p->d_active, 0, Upad, p->stream));
  DevProblem d = dev_problem(p);
  if (p->num_tiles > 0) k_mark_static<<<p->num_tiles, kTile, 0, p->stream>>>(d, p->d_active);
  if (rcn.total > 0) {
    DevProblem d1 = d; d1.nranks = 1; d1.rank = 0;   // mark regardless of rank ownership
    k_regularisers<2><<<(rcn.total + 127) / 128, 128, 0, p->stream>>>(d1, rcn, p->d_x, nullptr, nullptr, nullptr, p->d_active, p->first_frame, p->last_frame);
  }
  if (p->num_trip_tiles > 0) k_triplets<2><<<p->num_trip_tiles, kTile, 0, p->stream>>>(d, p->d_x, nullptr, nullptr, nullptr, p->d_active);
  k_finalize_mask<<<(int)((Upad + 255) / 256), 256, 0, p->stream>>>(p->cfg, L, p->d_active, N);
  CK(cudaGetLastError());
  if (p->nranks > 1) {   // the parameter set of the program is the union over the ranks' constraint shards (norms and stopping tests must agree on every rank)
    const int r = nccl::AllReduce(p->d_active, p->d_active, Upad, nccl::kUint8, nccl::kMax, p->comm, p->stream);
    if (r != 0) return set_err(RCVD_ERR_NCCL, "ncclAllReduce(active mask) failed");
  }
  // kernels that need > 48 KB dynamic smem
  if ((npad * 16 + 16 * (npad + 1)) * (int)sizeof(double) > 220 * 1024) return set_err(RCVD_ERR_INVALID, "frame block too large for the panel-inverse kernel (npad=%d)", npad);
  CK(cudaFuncSetAttribute(k_trinv, cudaFuncAttributeMaxDynamicSharedMemorySize, (npad * 16 + 16 * (npad + 1)) * (int)sizeof(double)));
  CK(cudaFuncSetAttribute(k_accumulate_fast, cudaFuncAttributeMaxDynamicSharedMemorySize, kFastSmem));
  CK(cudaFuncSetAttribute(k_accumulate_runs, cudaFuncAttributeMaxDynamicSharedMemorySize, kRunSmem));
  p->use_trsm_ll = p->allow_trsm_ll && trsm_ll_smem_bytes(npad) <= 220 * 1024;
  if (p->use_trsm_ll) { CK(cudaFuncSetAttribute(k_trsm_ll<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)trsm_ll_smem_bytes(npad, 2))); if (trsm_ll_smem_bytes(npad, 4) <= 220 * 1024) CK(cudaFuncSetAttribute(k_trsm_ll<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)trsm_ll_smem_bytes(npad, 4))); }
  if (potrf_smem_bytes(npad) <= 220 * 1024) CK(cudaFuncSetAttribute(k_potrf_smem, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)potrf_smem_bytes(npad)));
  CK(cudaStreamSynchronize(p->stream));
  p->structure_ready = true;
  return RCVD_OK;
}

static int allreduce(rcvd_problem* p, double* buf, size_t count) {
  if (p->nranks <= 1) return RCVD_OK;
  const int r = nccl::AllReduce(buf, buf, count, nccl::kFloat64, nccl::kSum, p->comm, p->stream);
  if (r != 0) return set_err(RCVD_ERR_NCCL, "ncclAllReduce failed: %s", nccl::GetErrorString ? nccl::GetErrorString(r) : "?");
  return RCVD_OK;
}
// One fused NCCL launch: for every rank q, segs[q] = (first, count) in units of `unit` doubles of `base` is broadcast from q (bcast) or
// summed onto q (!bcast), in place.  Every rank passes identical segments.
struct Seg { size_t first, count; };
static int grouped(rcvd_problem* p, double* base, size_t unit, const std::vector<Seg>& segs, bool bcast) {
  int r = nccl::GroupStart();
  for (size_t i = 0; i < segs.size() && r == 0; ++i) {
    if (segs[i].count == 0) continue;
    const int root = (int)(i % (size_t)p->nranks);
    double* ptr = base + segs[i].first * unit;
    r = bcast ? nccl::Broadcast(ptr, ptr, segs[i].count * unit, nccl::kFloat64, root, p->comm, p->stream)
              : nccl::Reduce(ptr, ptr, segs[i].count * unit, nccl::kFloat64, nccl::kSum, root, p->comm, p->stream);
  }
  const int r2 = nccl::GroupEnd();
  if (r == 0) r = r2;
  if (r != 0) return set_err(RCVD_ERR_NCCL, "grouped NCCL %s failed: %s", bcast ? "broadcast" : "reduce", nccl::GetErrorString ? nccl::GetErrorString(r) : "?");
  return RCVD_OK;
}

// Enqueues factorisation of (S H S + D2) and the solve y = A^{-1} gs on p->stream.
static int enqueue_factor_solve(rcvd_problem* p) {
  const Layout& L = p->L; const int N = p->N, npad = L.npad; cudaStream_t st = p->stream;
  const int nL = N + p->nLoff;
  const int tiles = (npad + 63) / 64;
  enum { P_LOAD = 0, P_POTRF, P_TRINV, P_TRSM, P_GEMM, P_SOLVE };
  int prof_level = 0;
  auto mark = [&](int cls) {   // profiling mode only (single stream, not captured)
    if (!p->prof) return;
    cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, st); p->prof->push_back({cls < 0 ? cls : (cls | (prof_level << 8)), e});
  };
  const int neff = p->trim_gemm ? std::min(npad, (L.nf + 7) / 8 * 8) : npad;
  auto gemm = [&](cudaStream_t cs, int ntasks, double* dstp, const double* A, const double* B, const GemmTask* tasks, const int2* prs, double alpha, double beta) {
    // trimming applies to the update products only (beta != 0): the legacy inverse-times-block TRSM must write every padded row of T
    k_gemm_nt<<<dim3(tiles, tiles, ntasks), 128, 0, cs>>>(dstp, A, B, tasks, prs, npad, beta != 0.0 ? neff : npad, alpha, beta);
  };
  mark(-1);
  k_load_factor<<<dim3((npad * npad + 255) / 256, p->dist ? p->n_own_l : nL), 256, 0, st>>>(p->d_H, p->d_Lb, p->d_lblocks, p->d_S, p->d_D2, npad, L.nf, p->dist ? p->d_own_lblocks : nullptr);
  p->launches += 1; mark(P_LOAD);
  // Two-stream schedule (fork/join inside the captured graph): the non-critical update GEMMs of level l run on `side`
  // concurrently with potrf / inverse / trsm of level l+1 on `st`.
  cudaStream_t side = p->side_stream;
  bool side_pending = false, side_used = false;
  const size_t bsz = (size_t)npad * npad;
  // phase boundary of the distributed factorisation: the owners' explicit inverses (for the replicated substitution) and their
  // blocks of the trailing matrix go to everybody; from here on every rank factors the same narrow tail
  auto phase_boundary = [&]() -> int {
    if (side_pending || side_used) { CK(cudaEventRecord(p->ev_join, side)); CK(cudaStreamWaitEvent(st, p->ev_join, 0)); side_pending = false; }
    std::vector<Seg> inv, tr;
    for (int q = 0; q < p->nranks; ++q) inv.push_back({(size_t)p->fa_off[q], (size_t)p->fa_cnt[q]});
    for (int q = 0; q < p->nranks; ++q) tr.push_back({(size_t)p->fb_off[q], (size_t)p->fb_cnt[q]});
    for (int q = 0; q < p->nranks; ++q) tr.push_back({(size_t)N + (size_t)p->bseg[2 * q], (size_t)p->bseg[2 * q + 1]});
    int rc = grouped(p, p->d_invL, bsz, inv, true); if (rc) return rc;
    return grouped(p, p->d_Lb, bsz, tr, true);
  };
  for (size_t li = 0; li < p->levels.size(); ++li) {
    const Level& lv = p->levels[li]; prof_level = (int)li;
    if (p->dist && (int)li == p->LB) { int rc = phase_boundary(); if (rc) return rc; }
    const int* lframes = p->d_lvl_own + lv.own_off; const int nfr = lv.nown;      // the frames this rank factors at this level
    if (nfr > 0) {
    if (potrf_smem_bytes(npad) <= 220 * 1024)
      k_potrf_smem<<<nfr, kPotrfSmemThreads, potrf_smem_bytes(npad), st>>>(p->d_Lb, p->d_invT, lframes, npad, p->d_fail, (p->potrf_chain_warp ? 1 : 0) | (p->potrf_blocked ? 2 : 0));
    else {
      // large blocks: 16-wide panels, panel factor on one CTA per frame, trailing update on the whole machine
      const int nt16 = npad / 16;
      for (int jb = 0; jb < nt16; ++jb) {
        k_potrf_panel<<<nfr, kPotrfThreads, 0, st>>>(p->d_Lb, p->d_invT, lframes, npad, jb, p->d_fail);
        p->launches += 1;
        const int m = npad - (jb + 1) * 16;
        if (m > 0) { const int n64 = (m + 63) / 64; k_potrf_trail<<<dim3(n64 * (n64 + 1) / 2, nfr), 128, 0, st>>>(p->d_Lb, lframes, npad, jb); p->launches += 1; }
      }
      p->launches -= 1;   // (the common increment below)
    }
    p->launches += 1; mark(P_POTRF);
    if (p->use_trsm_ll) {
      // the explicit inverse is only needed by the (much later) substitution phase: compute it off the critical path
      cudaStream_t is = st;
      if (p->overlap) { CK(cudaEventRecord(p->ev_fork, st)); CK(cudaStreamWaitEvent(side, p->ev_fork, 0)); is = side; side_used = true; }
      k_trinv<<<dim3(npad / 16, nfr), 256, (npad * 16 + 16 * (npad + 1)) * sizeof(double), is>>>(p->d_Lb, p->d_invT, p->d_invL, lframes, npad);
      p->launches += 1; mark(P_TRINV);
      if (lv.ntrsm > 0) {
        const int strips = (npad + kTrsmStrip - 1) / kTrsmStrip;
        if (p->trsm_deep && strips * lv.ntrsm <= p->num_sms && trsm_ll_smem_bytes(npad, 4) <= 220 * 1024)   // a single wave: deep panel prefetch, one CTA per SM
          k_trsm_ll<4><<<dim3(strips, lv.ntrsm), 128, trsm_ll_smem_bytes(npad, 4), st>>>(p->d_T, p->d_Lb, p->d_invT, p->d_trsm_ll + lv.trsm_off, npad);
        else
          k_trsm_ll<2><<<dim3(strips, lv.ntrsm), 128, trsm_ll_smem_bytes(npad, 2), st>>>(p->d_T, p->d_Lb, p->d_invT, p->d_trsm_ll + lv.trsm_off, npad);
        p->launches++; mark(P_TRSM);
      }
    } else {
      k_trinv<<<dim3(npad / 16, nfr), 256, (npad * 16 + 16 * (npad + 1)) * sizeof(double), st>>>(p->d_Lb, p->d_invT, p->d_invL, lframes, npad);
      p->launches += 1; mark(P_TRINV);
      if (lv.ntrsm > 0) { gemm(st, lv.ntrsm, p->d_T, p->d_Lb, p->d_invL, p->d_trsm_tasks + lv.trsm_off, p->d_trsm_pairs, 1.0, 0.0); p->launches++; mark(P_TRSM); }
    }
    }
    if (p->dist && (int)li < p->LB) {
      // the off-diagonal factor blocks of this level, from their owners to everybody (one fused NCCL launch)
      std::vector<Seg> segs;
      for (int q = 0; q < p->nranks; ++q) segs.push_back({(size_t)p->tseg[(li * p->nranks + q) * 2], (size_t)p->tseg[(li * p->nranks + q) * 2 + 1]});
      int rc = grouped(p, p->d_T, bsz, segs, true); if (rc) return rc;
    }
    if (lv.nupd2 > 0 && p->overlap) {
      CK(cudaEventRecord(p->ev_fork, st)); CK(cudaStreamWaitEvent(side, p->ev_fork, 0));
    }
    if (side_pending) { CK(cudaStreamWaitEvent(st, p->ev_join, 0)); side_pending = false; }   // U2(l-1) before U1(l)
    auto update = [&](cudaStream_t cs, int off, int n, bool side_launch) {   // persistent TMA-fed update kernel
      if (side_launch && p->upd_reserve > 0 && lv.nframes <= p->upd_reserve) {
        // overlapped updates of a narrow level: one CTA per SM and `upd_reserve` SMs left free, so that the next level's potrf CTAs
        // (a whole SM each) start at once instead of waiting for a persistent CTA of this launch to retire
        k_update_tma<2><<<std::max(1, std::min(n, p->num_sms - p->upd_reserve)), UpdShape<2>::threads, upd_smem_bytes(p->upd_rb, 2), cs>>>(p->tmapT, p->d_Lb, p->d_upd_items + off, n, p->d_upd_pairs, npad, p->upd_neff, p->upd_rb, p->upd_dbg);
        return;
      }
      if (n <= p->num_sms * p->upd_team_items) {   // few items: two DMMA teams per tile, one CTA per SM
        k_update_tma<2><<<std::min(n, p->num_sms), UpdShape<2>::threads, upd_smem_bytes(p->upd_rb, 2), cs>>>(p->tmapT, p->d_Lb, p->d_upd_items + off, n, p->d_upd_pairs, npad, p->upd_neff, p->upd_rb, p->upd_dbg);
      } else {
        int grid = std::min(n, 2 * p->num_sms);
        if (p->upd_ipc > 0) grid = std::max(grid, (n + p->upd_ipc - 1) / p->upd_ipc);
        k_update_tma<1><<<grid, UpdShape<1>::threads, upd_smem_bytes(p->upd_rb, 1), cs>>>(p->tmapT, p->d_Lb, p->d_upd_items + off, n, p->d_upd_pairs, npad, p->upd_neff, p->upd_rb, p->upd_dbg);
      }
    };
    if (p->gemm_tma) {
      if (lv.nit > 0) { update(st, lv.it_off, lv.nit, false); p->launches++; mark(P_GEMM); }
      if (lv.nit2 > 0) {
        update(p->overlap ? side : st, lv.it2_off, lv.nit2, p->overlap); p->launches++; mark(P_GEMM);
        if (p->overlap) { CK(cudaEventRecord(p->ev_join, side)); side_pending = true; side_used = true; }
      }
      continue;
    }
    if (lv.nupd > 0) { gemm(st, lv.nupd, p->d_Lb, p->d_T, p->d_T, p->d_upd_tasks + lv.upd_off, p->d_upd_pairs, -1.0, 1.0); p->launches++; mark(P_GEMM); }
    if (lv.nupd2 > 0) {
      cudaStream_t us = p->overlap ? side : st;
      // sliced so that the grid of one launch is about `side_slice` CTAs: a potrf / trsm CTA of the chain needs most of an SM's
      // shared memory and can only start on an SM that has drained, which a long low-priority grid never lets happen
      const int per = (p->overlap && p->side_slice > 0) ? std::max(1, p->side_slice / (tiles * tiles)) : lv.nupd2;
      for (int o = 0; o < lv.nupd2; o += per) {
        gemm(us, std::min(per, lv.nupd2 - o), p->d_Lb, p->d_T, p->d_T, p->d_upd_tasks + lv.upd2_off + o, p->d_upd_pairs, -1.0, 1.0); p->launches++; mark(P_GEMM);
      }
      if (p->overlap) { CK(cudaEventRecord(p->ev_join, side)); side_pending = true; side_used = true; }
    }
  }
  if (p->dist && p->LB >= (int)p->levels.size()) { int rc = phase_boundary(); if (rc) return rc; }
  if (side_pending || side_used) { CK(cudaEventRecord(p->ev_join, side)); CK(cudaStreamWaitEvent(st, p->ev_join, 0)); }
  CK(cudaMemcpyAsync(p->d_rhs, p->d_gs, (size_t)N * npad * sizeof(double), cudaMemcpyDeviceToDevice, st));
  const bool sub = p->use_trsm_ll && p->sub_solves;
  const int nlv = (int)p->levels.size();
  const int LS = sub ? nlv : p->sub_first_level;       // levels >= LS: the persistent dataflow kernel (rcvd_linalg.cuh, k_substitution)
  for (int l = 0; l < LS; ++l) {
    const Level& lv = p->levels[l];
    if (sub) k_fwd_diag_sub<<<lv.nframes, 256, (npad + 16) * sizeof(double), st>>>(p->d_Lb, p->d_invT, p->d_rhs, p->d_ytmp, p->d_lvl_frames + lv.frame_off, npad);
    else k_fwd_diag<<<dim3((npad + 7) / 8, lv.nframes), 256, 0, st>>>(p->d_invL, p->d_rhs, p->d_ytmp, p->d_lvl_frames + lv.frame_off, npad);
    p->launches++;
    if (lv.nfwd > 0) { k_fwd_update<<<dim3((npad + 7) / 8, lv.nfwd), 256, 0, st>>>(p->d_T, p->d_ytmp, p->d_rhs, p->d_fwd_tasks + lv.fwd_off, npad); p->launches++; }
  }
  if (LS < nlv && p->n_sub_tasks > 0) {
    CK(cudaMemsetAsync(p->d_sub_counters, 0, ((size_t)4 * N + 4) * sizeof(int), st));
    SubCounters cn; cn.ticket = p->d_sub_counters; cn.fin = p->d_sub_counters + 4; cn.fdone = cn.fin + N; cn.bin = cn.fdone + N; cn.bdone = cn.bin + N;
    cn.fin_need = p->d_sub_need; cn.bin_need = p->d_sub_need + N;
    k_substitution<<<std::min(p->n_sub_tasks, p->num_sms), kSubThreads, substitution_smem_bytes(npad), st>>>(p->d_invL, p->d_T, p->d_rhs, p->d_ytmp, p->d_y, p->d_sub_tasks, p->n_sub_tasks, cn, npad);
    p->launches++;
  }
  for (int l = LS - 1; l >= 0; --l) {
    const Level& lv = p->levels[l];
    if (lv.nfwd > 0) { k_bwd_update<<<dim3((npad + 31) / 32, lv.nfwd), 256, 0, st>>>(p->d_T, p->d_y, p->d_ytmp, p->d_fwd_tasks + lv.fwd_off, npad); p->launches++; }
    if (sub) k_bwd_diag_sub<<<lv.nframes, 256, (npad + 16) * sizeof(double), st>>>(p->d_Lb, p->d_invT, p->d_ytmp, p->d_y, p->d_lvl_frames + lv.frame_off, npad);
    else k_bwd_diag<<<dim3((npad + 31) / 32, lv.nframes), 256, 0, st>>>(p->d_invL, p->d_ytmp, p->d_y, p->d_lvl_frames + lv.frame_off, npad);
    p->launches += 1;
  }
  mark(P_SOLVE);
  CK(cudaGetLastError());
  return RCVD_OK;
}

// factor+solve through a CUDA graph (the level schedule is ~5 launches per level)
static int factor_solve(rcvd_problem* p) {
  if (p->nranks > 1 && !p->graph_warm) {   // NCCL establishes its connections lazily on first use: not inside a stream capture
    p->graph_warm = true;
    return enqueue_factor_solve(p);
  }
  if (!p->solve_graph) {
    cudaGraph_t graph;
    const int64_t l0 = p->launches;
    CK(cudaStreamBeginCapture(p->stream, cudaStreamCaptureModeThreadLocal));
    int rc = enqueue_factor_solve(p);
    cudaError_t e = cudaStreamEndCapture(p->stream, &graph);
    if (rc) return rc;
    if (e != cudaSuccess) return set_err(RCVD_ERR_CUDA, "graph capture failed: %s", cudaGetErrorString(e));
    CK(cudaGraphInstantiate(&p->solve_graph, graph, 0));
    cudaGraphDestroy(graph);
    p->graph_launches = p->launches - l0;
    p->launches = l0;
  }
  CK(cudaGraphLaunch(p->solve_graph, p->stream));
  p->launches += p->graph_launches;
  return RCVD_OK;
}

// ---------------------------------------------------------------------------
// Evaluation
// ---------------------------------------------------------------------------

// Cost (-> d_scal[slot]) at state x; optionally gradient (gout, npad stride) and H.
static int enqueue_evaluate(rcvd_problem* p, const double* x, bool wantG, bool wantH, double* gout, int slot) {
  if (wantH && p->eval_only) return set_err(RCVD_ERR_INVALID, "this handle was set to evaluation-only (rcvd_debug_set_eval_only): no normal matrix");
  const Layout& L = p->L; const int N = p->N, npad = L.npad; cudaStream_t st = p->stream;
  const size_t bs = (size_t)npad * npad, Upad = (size_t)N * npad;
  DevProblem d = dev_problem(p);
  const RegCounts rcn = reg_counts(p->cfg, L, N, p->nscale);
  const int regblocks = (rcn.total + 127) / 128;
  if (wantH) CK(cudaMemsetAsync(p->d_H, 0, (size_t)p->nHblocks * bs * sizeof(double), st));
  if (wantG) CK(cudaMemsetAsync(gout, 0, (Upad + 8) * sizeof(double), st));
  if (p->num_tiles > 0) {
    if (wantH && p->use_fast && p->records_sorted) k_accumulate_runs<<<p->num_tiles, kTile, kRunSmem, st>>>(d, x, p->d_H, gout, p->d_partial);
    else if (wantH && p->use_fast && fast_path_ok_host(p->cfg, L)) k_accumulate_fast<<<p->num_tiles, kTile, kFastSmem, st>>>(d, x, p->d_H, gout, p->d_partial);
    else if (wantH) k_accumulate_generic<true><<<p->num_tiles, kTile, 0, st>>>(d, x, p->d_H, gout, p->d_partial);
    else if (wantG) k_accumulate_generic<false><<<p->num_tiles, kTile, 0, st>>>(d, x, nullptr, gout, p->d_partial);
    else k_cost_static<<<p->num_tiles, kTile, 0, st>>>(d, x, p->d_partial);
    p->launches++;
  }
  if (regblocks > 0) {
    double* part = p->d_partial + p->num_tiles;
    if (wantH) k_regularisers<1><<<regblocks, 128, 0, st>>>(d, rcn, x, p->d_H, gout, part, nullptr, p->first_frame, p->last_frame);
    else if (wantG) k_regularisers<3><<<regblocks, 128, 0, st>>>(d, rcn, x, nullptr, gout, part, nullptr, p->first_frame, p->last_frame);
    else k_regularisers<0><<<regblocks, 128, 0, st>>>(d, rcn, x, nullptr, nullptr, part, nullptr, p->first_frame, p->last_frame);
    p->launches++;
  }
  if (p->num_trip_tiles > 0) {
    double* part = p->d_partial + p->num_tiles + regblocks;
    if (wantH) k_triplets<1><<<p->num_trip_tiles, kTile, 0, st>>>(d, x, p->d_H, gout, part, nullptr);
    else if (wantG) k_triplets<3><<<p->num_trip_tiles, kTile, 0, st>>>(d, x, nullptr, gout, part, nullptr);
    else k_triplets<0><<<p->num_trip_tiles, kTile, 0, st>>>(d, x, nullptr, nullptr, part, nullptr);
    p->launches++;
  }
  k_reduce_partials<<<1, 1024, 0, st>>>(p->d_partial, p->num_tiles + regblocks + p->num_trip_tiles, p->d_scal, slot);
  p->launches++;
  CK(cudaGetLastError());
  if (p->nranks > 1) {
    int rc;
    if (wantG) {
      // ONE packed all-reduce: [gradient (Upad) | cost + 7 spare | diagonal of H (Upad, only with H into d_g)]
      CK(cudaMemcpyAsync(gout + Upad, p->d_scal + slot, sizeof(double), cudaMemcpyDeviceToDevice, st));
      size_t cnt = Upad + 8;
      if (wantH && gout == p->d_g) { k_extract_diag<<<(int)((Upad + 255) / 256), 256, 0, st>>>(p->d_H, p->d_diagH, N, npad); p->launches++; cnt = 2 * Upad + 8; }
      if ((rc = allreduce(p, gout, cnt))) return rc;
      CK(cudaMemcpyAsync(p->d_scal + slot, gout + Upad, sizeof(double), cudaMemcpyDeviceToDevice, st));
    } else if ((rc = allreduce(p, p->d_scal + slot, 1))) return rc;
    if (wantH) {
      if (p->dist && !p->force_full_H) {
        // the normal matrix is summed onto the OWNER of every block only (its frames' diagonal blocks, the off-diagonal blocks of its columns)
        std::vector<Seg> segs;
        for (int q = 0; q < p->nranks; ++q) segs.push_back({(size_t)p->fa_off[q], (size_t)(p->fa_cnt[q] + p->fb_cnt[q])});
        for (int q = 0; q < p->nranks; ++q) segs.push_back({(size_t)p->hseg[2 * q], (size_t)p->hseg[2 * q + 1]});
        if ((rc = grouped(p, p->d_H, bs, segs, false))) return rc;
      } else if ((rc = allreduce(p, p->d_H, (size_t)p->nHblocks * bs))) return rc;
    }
  }
  return RCVD_OK;
}

// Frame-major host vectors in the caller's frame order <-> device vectors in the internal (owner-major) order.
static int upload_frames(rcvd_problem* p, double* dst, const double* src_user, int stride_dst, int stride_src, int count) {
  std::vector<double> tmp((size_t)p->N * stride_dst, 0.0);
  for (int i = 0; i < p->N; ++i) memcpy(tmp.data() + (size_t)i * stride_dst, src_user + (size_t)p->uperm[i] * stride_src, (size_t)count * sizeof(double));
  CK(cudaMemcpyAsync(dst, tmp.data(), tmp.size() * sizeof(double), cudaMemcpyHostToDevice, p->stream));
  CK(cudaStreamSynchronize(p->stream));      // tmp goes out of scope
  return RCVD_OK;
}
static int download_frames(rcvd_problem* p, double* dst_user, const double* src, int stride_dst, int stride_src, int count) {
  std::vector<double> tmp((size_t)p->N * stride_src);
  CK(cudaMemcpyAsync(tmp.data(), src, tmp.size() * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
  CK(cudaStreamSynchronize(p->stream));
  for (int i = 0; i < p->N; ++i) memcpy(dst_user + (size_t)p->uperm[i] * stride_dst, tmp.data() + (size_t)i * stride_src, (size_t)count * sizeof(double));
  return RCVD_OK;
}
// device state -> h_state (caller's frame order); used before the structure is rebuilt
static int save_state(rcvd_problem* p) {
  DevGuard g(p->device); cudaStreamSynchronize(p->stream);
  if (p->h_state.size() != (size_t)p->N * p->L.nf) p->h_state.assign((size_t)p->N * p->L.nf, 0.0);
  return download_frames(p, p->h_state.data(), p->d_x, p->L.nf, p->L.nf, p->L.nf);
}

static int ensure_ready(rcvd_problem* p) {
  if (!p->structure_ready) {
    if (p->offsets.empty()) { p->offsets.assign(1, 0); }
    if (p->in_range.empty()) p->in_range.assign(p->N, 1);
    if (p->median.empty()) p->median.assign(p->N, 1.0);
    int rc = build_structure(p); if (rc) return rc;
    p->state_dirty = true;
  }
  if (p->state_dirty) {
    if (p->h_state.size() != (size_t)p->N * p->L.nf) p->h_state.assign((size_t)p->N * p->L.nf, 0.0);
    { int rc = upload_frames(p, p->d_x, p->h_state.data(), p->L.nf, p->L.nf, p->L.nf); if (rc) return rc; }
    p->state_dirty = false;
  }
  return RCVD_OK;
}

static int read_scalars(rcvd_problem* p) {
  CK(cudaMemcpyAsync(p->h_scal, p->d_scal, SC_N * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
  CK(cudaMemcpyAsync(p->h_fail, p->d_fail, sizeof(int), cudaMemcpyDeviceToHost, p->stream));
  CK(cudaStreamSynchronize(p->stream));
  return RCVD_OK;
}

// ---------------------------------------------------------------------------
// Polynomial minimisation for the Armijo line search (ceres/polynomial.cc semantics)
// ---------------------------------------------------------------------------
namespace ls {
struct Sample { double x, value, gradient; bool valueValid, gradValid; };
static double evalPoly(const std::vector<double>& p, double x) { double v = 0; for (double c : p) v = v * x + c; return v; }
static bool solveDense(std::vector<std::vector<double>> A, std::vector<double> b, std::vector<double>& x) {
  const int n = (int)b.size(); std::vector<int> perm(n); for (int i = 0; i < n; ++i) perm[i] = i;
  for (int k = 0; k < n; ++k) {
    int pr = k, pc = k; double best = 0;
    for (int i = k; i < n; ++i) for (int j = k; j < n; ++j) if (std::fabs(A[i][j]) > best) { best = std::fabs(A[i][j]); pr = i; pc = j; }
    if (best == 0) return false;
    std::swap(A[k], A[pr]); std::swap(b[k], b[pr]);
    for (int i = 0; i < n; ++i) std::swap(A[i][k], A[i][pc]);
    std::swap(perm[k], perm[pc]);
    for (int i = k + 1; i < n; ++i) { const double f = A[i][k] / A[k][k]; for (int j = k; j < n; ++j) A[i][j] -= f * A[k][j]; b[i] -= f * b[k]; }
  }
  std::vector<double> y(n);
  for (int i = n - 1; i >= 0; --i) { double s = b[i]; for (int j = i + 1; j < n; ++j) s -= A[i][j] * y[j]; y[i] = s / A[i][i]; }
  x.assign(n, 0.0); for (int i = 0; i < n; ++i) x[perm[i]] = y[i];
  return true;
}
static std::vector<double> realRoots(std::vector<double> p) {
  while (!p.empty() && p[0] == 0.0) p.erase(p.begin());
  std::vector<double> out; const int d = (int)p.size() - 1; if (d < 1) return out;
  if (d == 1) { out.push_back(-p[1] / p[0]); return out; }
  if (d == 2) { const double a = p[0], b = p[1], c = p[2], D = b * b - 4 * a * c; if (D >= 0) { const double sq = std::sqrt(D); out.push_back((-b + sq) / (2 * a)); out.push_back((-b - sq) / (2 * a)); } else { out.push_back(-b / (2 * a)); out.push_back(-b / (2 * a)); } return out; }
  std::vector<std::pair<double, double>> z(d);
  for (int i = 0; i < d; ++i) { const double ang = 2 * M_PI * i / d + 0.4; z[i] = {0.9 * std::cos(ang), 0.9 * std::sin(ang)}; }
  auto cmul = [](std::pair<double, double> a, std::pair<double, double> b) { return std::make_pair(a.first * b.first - a.second * b.second, a.first * b.second + a.second * b.first); };
  auto cdiv = [](std::pair<double, double> a, std::pair<double, double> b) { const double dd = b.first * b.first + b.second * b.second; return std::make_pair((a.first * b.first + a.second * b.second) / dd, (a.second * b.first - a.first * b.second) / dd); };
  for (int it = 0; it < 500; ++it) {
    double mx = 0;
    for (int i = 0; i < d; ++i) {
      std::pair<double, double> v = {p[0], 0.0};
      for (int j = 1; j <= d; ++j) { v = cmul(v, z[i]); v.first += p[j]; }
      std::pair<double, double> den = {p[0], 0.0};
      for (int j = 0; j < d; ++j) if (j != i) den = cmul(den, {z[i].first - z[j].first, z[i].second - z[j].second});
      auto dl = cdiv(v, den); z[i].first -= dl.first; z[i].second -= dl.second;
      mx = std::max(mx, std::fabs(dl.first) + std::fabs(dl.second));
    }
    if (mx < 1e-14) break;
  }
  for (auto& r : z) out.push_back(r.first);
  return out;
}
static double minimizeInterpolating(const std::vector<Sample>& s, double xmin, double xmax) {
  int nc = 0; for (auto& q : s) { if (q.valueValid) ++nc; if (q.gradValid) ++nc; }
  const int deg = nc - 1;
  std::vector<std::vector<double>> A; std::vector<double> b;
  for (auto& q : s) {
    if (q.valueValid) { std::vector<double> row(nc); for (int j = 0; j <= deg; ++j) row[j] = std::pow(q.x, deg - j); A.push_back(row); b.push_back(q.value); }
    if (q.gradValid) { std::vector<double> row(nc); for (int j = 0; j < deg; ++j) row[j] = (deg - j) * std::pow(q.x, deg - j - 1); row[deg] = 0; A.push_back(row); b.push_back(q.gradient); }
  }
  std::vector<double> poly; if (!solveDense(A, b, poly)) return 0.5 * (xmin + xmax);
  double ox = (xmin + xmax) / 2.0, ov = evalPoly(poly, ox);
  const double vmin = evalPoly(poly, xmin); if (vmin < ov) { ov = vmin; ox = xmin; }
  const double vmax = evalPoly(poly, xmax); if (vmax < ov) { ov = vmax; ox = xmax; }
  if (poly.size() <= 2) return ox;
  std::vector<double> der;
  for (int j = 0; j < deg; ++j) der.push_back((deg - j) * poly[j]);
  for (double r : realRoots(der)) { if (r < xmin || r > xmax) continue; const double v = evalPoly(poly, r); if (v < ov) { ov = v; ox = r; } }
  return ox;
}
}  // namespace ls

__global__ void k_make_delta(const double* __restrict__ y, const double* __restrict__ S, double* __restrict__ delta, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) delta[i] = -y[i] * S[i];
}

static inline int nblk(size_t n, int b = 256) { return (int)((n + b - 1) / b); }

// model = gs.y - 1/2 (Sy)^T H (Sy); leaves GY, YHY in d_scal
static int enqueue_model_terms(rcvd_problem* p) {
  const int N = p->N, npad = p->L.npad; const size_t Upad = (size_t)N * npad; cudaStream_t st = p->stream;
  k_mul<<<nblk(Upad), 256, 0, st>>>(p->d_S, p->d_y, p->d_Sy, (int)Upad);
  CK(cudaMemsetAsync(p->d_Hy, 0, Upad * sizeof(double), st));
  k_spmv_sym<<<dim3((npad + 7) / 8, p->dist ? p->n_own_h : p->nHblocks), 256, 0, st>>>(p->d_H, p->d_hblocks, p->d_Sy, p->d_Hy, npad, p->dist ? p->d_own_hblocks : nullptr);
  k_dot2<<<nblk(Upad), 256, 0, st>>>(p->d_gs, p->d_y, p->d_Sy, p->d_Hy, (int)Upad, p->d_scal, SC_GY, SC_YHY);
  if (p->dist) { int rc = allreduce(p, p->d_scal + SC_YHY, 1); if (rc) return rc; }   // every rank multiplied the H blocks it owns
  k_make_delta<<<nblk(Upad), 256, 0, st>>>(p->d_y, p->d_S, p->d_delta, (int)Upad);
  p->launches += 4;
  return RCVD_OK;
}

__global__ void __launch_bounds__(256) k_candidate2(rcvd_config cfg, Layout L, const uint8_t* __restrict__ in_range, const uint8_t* __restrict__ active,
                                                     const double* __restrict__ x, const double* __restrict__ delta, const double* __restrict__ g,
                                                     double alpha, double* __restrict__ xc, double* __restrict__ scal, int N) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  double d2 = 0.0, gd = 0.0, dm = 0.0;
  if (i < N * L.nf) {
    const int f = i / L.nf, l = i % L.nf;
    const size_t v = (size_t)f * L.npad + l;
    const double dl = delta[v];
    const double xn = project_lb(cfg, L, in_range, f, l, x[i] + alpha * dl);
    xc[i] = xn;
    if (active[v]) { const double d = x[i] - xn; d2 = d * d; }
    gd = g[v] * dl; dm = fabs(dl);
  }
  d2 = warp_sum(d2); gd = warp_sum(gd);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) dm = fmax(dm, __shfl_xor_sync(0xffffffffu, dm, o));
  if ((threadIdx.x & 31) == 0) {
    red_add(scal + SC_STEP2, d2); red_add(scal + SC_GDOTD, gd);
    atomicMax((unsigned long long*)(scal + SC_DMAX), (unsigned long long)__double_as_longlong(dm));
  }
}

static int enqueue_candidate(rcvd_problem* p, double alpha, const double* g) {
  const size_t U = (size_t)p->N * p->L.nf;
  k_candidate2<<<nblk(U), 256, 0, p->stream>>>(p->cfg, p->L, p->d_in_range, p->d_active, p->d_x, p->d_delta, g, alpha, p->d_xc, p->d_scal, p->N);
  p->launches++;
  return RCVD_OK;
}

static float ev_ms(cudaEvent_t a, cudaEvent_t b) { float m = 0; cudaEventElapsedTime(&m, a, b); return m; }

// ---------------------------------------------------------------------------
// Levenberg-Marquardt, Ceres semantics (TrustRegionMinimizer::Minimize restated).
// ---------------------------------------------------------------------------
static int lm_solve(rcvd_problem* p, const rcvd_solve_options& o, rcvd_solve_summary& sum) {
  using clk = std::chrono::steady_clock;
  const auto t0 = clk::now();
  memset(&sum, 0, sizeof(sum));
  int rc = ensure_ready(p); if (rc) return rc;
  const Layout& L = p->L; const int N = p->N, npad = L.npad; const size_t Upad = (size_t)N * npad, U = (size_t)N * L.nf; cudaStream_t st = p->stream;
  const int64_t launches0 = p->launches;
  sum.num_constraints = p->C;
  const bool constrained = p->cfg.depth_lower_bound && L.nd > 0;
  for (int i = 0; i < 8; ++i) if (!p->ev[i]) CK(cudaEventCreate(&p->ev[i]));
  if (constrained) { k_project_state<<<nblk(U), 256, 0, st>>>(p->cfg, L, p->d_in_range, p->d_x, N); p->launches++; }
  // user-visible minimum-cost iterate
  CK(cudaMemcpyAsync(p->d_xsave, p->d_x, U * sizeof(double), cudaMemcpyDeviceToDevice, st));

  auto full_eval = [&]() -> int {   // cost, gradient, H, diag, norms at d_x
    CK(cudaMemsetAsync(p->d_scal, 0, SC_N * sizeof(double), st));
    CK(cudaEventRecord(p->ev[0], st));
    int r = enqueue_evaluate(p, p->d_x, true, true, p->d_g, SC_COST); if (r) return r;
    CK(cudaEventRecord(p->ev[1], st));
    if (p->nranks <= 1) k_extract_diag<<<nblk(Upad), 256, 0, st>>>(p->d_H, p->d_diagH, N, npad);
    k_state_norms<<<nblk(U), 256, 0, st>>>(p->cfg, L, p->d_in_range, p->d_active, p->d_x, p->d_g, p->d_scal, N);
    p->launches += 2;
    r = read_scalars(p); if (r) return r;
    sum.eval_ms += ev_ms(p->ev[0], p->ev[1]);
    return RCVD_OK;
  };
  if ((rc = full_eval())) return rc;
  double xCost = p->h_scal[SC_COST], xNorm = std::sqrt(p->h_scal[SC_X2]), gmax = p->h_scal[SC_GMAX];
  sum.initial_cost = xCost;
  k_jacobi_scale<<<nblk(Upad), 256, 0, st>>>(p->d_diagH, p->d_S, (int)Upad, o.jacobi_scaling);
  p->launches++;
  double radius = o.initial_radius, decrease = 2.0; bool reuseDiag = false;
  double minimumCost = xCost;
  int iter = 0, invalid = 0; bool stepSuccessful = true;
  auto finish = [&](int term, const char* msg) { sum.termination = term; snprintf(sum.message, sizeof(sum.message), "%s", msg); };
  finish(RCVD_TERM_NO_CONVERGENCE, "");
  if (o.verbose) fprintf(stderr, "[rcvd] iter      cost      cost_change  |gradient|   |step|    tr_ratio  tr_radius\n[rcvd] %4d %.6e %10.2e %10.2e %10.2e %10.2e %10.2e\n", 0, xCost, 0.0, gmax, 0.0, 0.0, radius);
  for (;;) {
    if (stepSuccessful) {
      ++sum.num_successful_steps;
      if (xCost < minimumCost || iter == 0) { minimumCost = xCost; CK(cudaMemcpyAsync(p->d_xsave, p->d_x, U * sizeof(double), cudaMemcpyDeviceToDevice, st)); }
    } else ++sum.num_unsuccessful_steps;
    if (iter >= o.max_iterations) { finish(RCVD_TERM_NO_CONVERGENCE, "Maximum number of iterations reached."); break; }
    if (stepSuccessful && gmax <= o.gradient_tolerance) { finish(RCVD_TERM_CONVERGENCE, "Gradient tolerance reached."); break; }
    if (radius <= o.min_radius) { finish(RCVD_TERM_CONVERGENCE, "Minimum trust region radius reached."); break; }
    ++iter; stepSuccessful = false;
    // --- ComputeTrustRegionStep + candidate evaluation, one host sync ---
    CK(cudaMemsetAsync(p->d_scal, 0, SC_N * sizeof(double), st));
    CK(cudaMemsetAsync(p->d_fail, 0, sizeof(int), st));
    CK(cudaEventRecord(p->ev[2], st));
    k_lm_prepare<<<nblk(Upad), 256, 0, st>>>(p->d_diagH, p->d_S, p->d_g, p->d_lmdiag, p->d_D2, p->d_gs, (int)Upad, reuseDiag ? 1 : 0, radius, o.min_lm_diagonal, o.max_lm_diagonal);
    p->launches++;
    reuseDiag = true;
    if ((rc = factor_solve(p))) return rc;
    if ((rc = enqueue_model_terms(p))) return rc;
    CK(cudaEventRecord(p->ev[3], st));
    double alpha = 1.0;
    if (!constrained) {
      if ((rc = enqueue_candidate(p, 1.0, p->d_g))) return rc;
      if ((rc = enqueue_evaluate(p, p->d_xc, false, false, nullptr, SC_CAND))) return rc;
      CK(cudaEventRecord(p->ev[4], st));
    }
    if ((rc = read_scalars(p))) return rc;
    sum.linear_ms += ev_ms(p->ev[2], p->ev[3]);
    if (!constrained) sum.cost_ms += ev_ms(p->ev[3], p->ev[4]);
    const double gy = p->h_scal[SC_GY], yHy = p->h_scal[SC_YHY];
    const double modelChange = gy - 0.5 * yHy;
    const bool ok = (*p->h_fail == 0) && std::isfinite(gy) && std::isfinite(yHy);
    if (!(ok && modelChange > 0.0)) {
      if (++invalid >= o.max_consecutive_invalid_steps) { finish(RCVD_TERM_FAILURE, "Number of consecutive invalid steps more than max_num_consecutive_invalid_steps."); break; }
      radius = radius / decrease; decrease *= 2.0; reuseDiag = true;
      if (o.verbose) fprintf(stderr, "[rcvd] %4d invalid step (fail=%d model=%g), radius %.3e\n", iter, *p->h_fail, modelChange, radius);
      continue;
    }
    invalid = 0;
    if (constrained) {
      // DoLineSearch: Armijo with cubic interpolation along the projected path (ceres defaults)
      auto trial = [&](double a, ls::Sample& s) -> int {
        CK(cudaMemsetAsync(p->d_scal, 0, SC_N * sizeof(double), st));
        int r = enqueue_candidate(p, a, p->d_g); if (r) return r;
        r = enqueue_evaluate(p, p->d_xc, true, false, p->d_g2, SC_CAND); if (r) return r;
        k_dot2<<<nblk(Upad), 256, 0, st>>>(p->d_g2, p->d_delta, p->d_g2, p->d_delta, (int)Upad, p->d_scal, SC_GY, SC_YHY);
        p->launches++;
        r = read_scalars(p); if (r) return r;
        s.x = a; s.value = p->h_scal[SC_CAND]; s.valueValid = std::isfinite(s.value);
        s.gradient = p->h_scal[SC_GY]; s.gradValid = s.valueValid && std::isfinite(s.gradient);
        return RCVD_OK;
      };
      ls::Sample cur, prev{0, 0, 0, false, false};
      if ((rc = trial(1.0, cur))) return rc;
      const double gd = p->h_scal[SC_GDOTD], dirMax = p->h_scal[SC_DMAX];
      ls::Sample init{0.0, xCost, gd, true, true};
      int lsIter = 0; bool success = true;
      while (!cur.valueValid || cur.value > xCost + 1e-4 * gd * cur.x) {
        if (++lsIter >= 20) { success = false; break; }
        const double lo = 1e-3 * cur.x, hi = 0.6 * cur.x;
        double ss;
        if (!cur.valueValid) ss = std::min(std::max(cur.x * 0.5, lo), hi);
        else { std::vector<ls::Sample> sm{init, cur}; if (prev.valueValid) sm.push_back(prev); ss = ls::minimizeInterpolating(sm, lo, hi); }
        if (ss * dirMax < 1e-9) { success = false; break; }
        prev = cur;
        if ((rc = trial(ss, cur))) return rc;
      }
      alpha = success ? cur.x : 1.0;
      CK(cudaMemsetAsync(p->d_scal, 0, SC_N * sizeof(double), st));
      if ((rc = enqueue_candidate(p, alpha, p->d_g))) return rc;
      if ((rc = enqueue_evaluate(p, p->d_xc, false, false, nullptr, SC_CAND))) return rc;
      if ((rc = read_scalars(p))) return rc;
    }
    double candCost = p->h_scal[SC_CAND];
    if (!std::isfinite(candCost)) candCost = std::numeric_limits<double>::max();
    const double stepNorm = std::sqrt(p->h_scal[SC_STEP2]);
    if (stepNorm <= o.parameter_tolerance * (xNorm + o.parameter_tolerance)) { finish(RCVD_TERM_CONVERGENCE, "Parameter tolerance reached."); break; }
    const double costChange = xCost - candCost;
    if (std::fabs(costChange) <= o.function_tolerance * xCost) { finish(RCVD_TERM_CONVERGENCE, "Function tolerance reached."); break; }
    const double relDecrease = (candCost >= std::numeric_limits<double>::max()) ? std::numeric_limits<double>::lowest() : costChange / modelChange;
    if (relDecrease > o.min_relative_decrease) {
      std::swap(p->d_x, p->d_xc);
      if ((rc = full_eval())) return rc;
      xCost = p->h_scal[SC_COST]; xNorm = std::sqrt(p->h_scal[SC_X2]); gmax = p->h_scal[SC_GMAX];
      stepSuccessful = true;
      radius = radius / std::max(1.0 / 3.0, 1.0 - std::pow(2.0 * relDecrease - 1.0, 3));
      radius = std::min(o.max_radius, radius); decrease = 2.0; reuseDiag = false;
    } else {
      radius = radius / decrease; decrease *= 2.0; reuseDiag = true;
    }
    if (o.verbose) fprintf(stderr, "[rcvd] %4d %.6e %10.2e %10.2e %10.2e %10.2e %10.2e\n", iter, stepSuccessful ? xCost : candCost, costChange, gmax, stepNorm, relDecrease, radius);
  }
  CK(cudaMemcpyAsync(p->d_x, p->d_xsave, U * sizeof(double), cudaMemcpyDeviceToDevice, st));
  CK(cudaStreamSynchronize(st));
  sum.iterations = iter; sum.final_cost = minimumCost;
  sum.gpu_launches = p->launches - launches0;
  sum.total_ms = std::chrono::duration<double, std::milli>(clk::now() - t0).count();
  return RCVD_OK;
}

// ---------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------
RCVD_API const char* rcvd_last_error(void) { return g_err.c_str(); }
RCVD_API int32_t rcvd_abi_version(void) { return 1; }
RCVD_API int32_t rcvd_frame_stride(const rcvd_config* c) { Layout L; return (c && make_layout(*c, L)) ? L.nf : -1; }
RCVD_API int32_t rcvd_depth_param_offset(const rcvd_config* c) { Layout L; return (c && make_layout(*c, L)) ? L.offD : -1; }
RCVD_API int32_t rcvd_spatial_param_offset(const rcvd_config* c) { Layout L; return (c && make_layout(*c, L)) ? L.offS : -1; }
RCVD_API void rcvd_default_solve_options(rcvd_solve_options* o) {
  o->max_iterations = 1000; o->verbose = 0; o->function_tolerance = 1e-6; o->gradient_tolerance = 1e-10; o->parameter_tolerance = 1e-8;
  o->initial_radius = 1e4; o->max_radius = 1e16; o->min_radius = 1e-32; o->min_relative_decrease = 1e-3; o->min_lm_diagonal = 1e-6;
  o->max_lm_diagonal = 1e32; o->max_consecutive_invalid_steps = 5; o->jacobi_scaling = 1;
}

RCVD_API int32_t rcvd_problem_create(const rcvd_config* cfg, int32_t device, rcvd_problem** out) {
  if (!cfg || !out) return set_err(RCVD_ERR_INVALID, "null argument");
  Layout L;
  if (!make_layout(*cfg, L) || cfg->num_frames <= 0) return set_err(RCVD_ERR_INVALID, "unsupported transform configuration");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev)
    return set_err(RCVD_ERR_NO_DEVICE, "no usable CUDA device (%s); this library has no CPU fallback", e != cudaSuccess ? cudaGetErrorString(e) : "device ordinal out of range");
  SET_DEVICE(device);
  {  // keep freed blocks in the device's default pool (released only on cudaDeviceReset / explicit trim)
    cudaMemPool_t pool; unsigned long long keep = ~0ull;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
  }
  rcvd_problem* p = new rcvd_problem();
  p->cfg = *cfg; p->L = L; p->N = cfg->num_frames; p->device = device;
  // the critical chain (potrf -> trsm -> next-level updates) runs at the highest priority, the overlapped updates at the lowest,
  // so that a freed SM goes to the chain first
  int prio_lo = 0, prio_hi = 0; cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
  e = cudaStreamCreateWithPriority(&p->stream, cudaStreamNonBlocking, prio_hi);
  if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&p->side_stream, cudaStreamNonBlocking, prio_lo);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&p->ev_fork, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&p->ev_join, cudaEventDisableTiming);
  if (e != cudaSuccess) { delete p; return set_err(RCVD_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e)); }
  *out = p; return RCVD_OK;
}
RCVD_API void rcvd_problem_destroy(rcvd_problem* p) {
  if (!p) return;
  DevGuard dev_guard_(p->device);
  free_all(p);
  for (int i = 0; i < 8; ++i) if (p->ev[i]) cudaEventDestroy(p->ev[i]);
  if (p->comm && nccl::CommDestroy) nccl::CommDestroy(p->comm);
  if (p->ev_fork) cudaEventDestroy(p->ev_fork);
  if (p->ev_join) cudaEventDestroy(p->ev_join);
  if (p->side_stream) cudaStreamDestroy(p->side_stream);
  if (p->stream) cudaStreamDestroy(p->stream);
  delete p;
}
RCVD_API int32_t rcvd_problem_set_frames(rcvd_problem* p, const uint8_t* in_range, const double* median, const double* adaptive) {
  if (!p) return set_err(RCVD_ERR_INVALID, "null problem");
  if (in_range) p->in_range.assign(in_range, in_range + p->N); else p->in_range.assign(p->N, 1);
  if (median) p->median.assign(median, median + p->N); else p->median.assign(p->N, 1.0);
  if (adaptive && p->cfg.depth_type == RCVD_DEPTH_GRID) p->adaptive.assign(adaptive, adaptive + (size_t)p->N * p->cfg.depth_grid_x * p->cfg.depth_grid_y); else p->adaptive.clear();
  if (p->cfg.adaptive_deform > 0.0 && p->adaptive.empty()) return set_err(RCVD_ERR_INVALID, "adaptive deformation cost requires node weights");
  if (p->structure_ready) { int rc_ = save_state(p); if (rc_) return rc_; }
  p->structure_ready = false;
  return RCVD_OK;
}
RCVD_API int32_t rcvd_problem_set_constraints(rcvd_problem* p, int32_t np, const int32_t* pf, const int64_t* off, const float* rec) {
  if (!p || np < 0 || (np > 0 && (!pf || !off))) return set_err(RCVD_ERR_INVALID, "bad constraint arrays");
  if (p->structure_ready) { int rc_ = save_state(p); if (rc_) return rc_; }
  p->pair_frames.assign(pf, pf + 2 * (size_t)np);
  if (np > 0) p->offsets.assign(off, off + np + 1); else p->offsets.assign(1, 0);
  for (int i = 0; i < np; ++i) {
    if (p->offsets[i + 1] < p->offsets[i]) return set_err(RCVD_ERR_INVALID, "offsets must be non-decreasing");
    if (pf[2 * i] < 0 || pf[2 * i] >= p->N || pf[2 * i + 1] < 0 || pf[2 * i + 1] >= p->N || pf[2 * i] == pf[2 * i + 1]) return set_err(RCVD_ERR_INVALID, "bad frame pair %d", i);
  }
  const int64_t C = p->offsets.back();
  if (C > 0 && !rec) return set_err(RCVD_ERR_INVALID, "null records");
  p->records_h.assign(rec, rec + (size_t)C * 6);
  p->structure_ready = false;
  return RCVD_OK;
}
RCVD_API int32_t rcvd_problem_set_triplets(rcvd_problem* p, int32_t nt, const int32_t* centers, const int64_t* off, const float* rec) {
  if (!p || nt < 0 || (nt > 0 && (!centers || !off))) return set_err(RCVD_ERR_INVALID, "bad triplet arrays");
  if (p->structure_ready) { int rc_ = save_state(p); if (rc_) return rc_; }
  p->trip_centers.assign(centers, centers + nt);
  if (nt > 0) p->trip_offsets.assign(off, off + nt + 1); else p->trip_offsets.assign(1, 0);
  for (int i = 0; i < nt; ++i) if (p->trip_offsets[i + 1] < p->trip_offsets[i] || centers[i] < 1 || centers[i] + 1 >= p->N) return set_err(RCVD_ERR_INVALID, "bad triplet group %d", i);
  const int64_t n = p->trip_offsets.back();
  if (n > 0 && !rec) return set_err(RCVD_ERR_INVALID, "null triplet records");
  p->trip_records.assign(rec, rec + (size_t)n * 10);
  p->structure_ready = false;
  return RCVD_OK;
}
// Global frame-pair graph for multi-GPU runs (every rank must build the same block structure).
RCVD_API int32_t rcvd_problem_set_structure(rcvd_problem* p, int32_t np, const int32_t* pf) {
  if (!p) return set_err(RCVD_ERR_INVALID, "null problem");
  p->struct_pairs.assign(pf, pf + 2 * (size_t)np);
  p->structure_ready = false;
  return RCVD_OK;
}
RCVD_API int32_t rcvd_nccl_unique_id(uint8_t out[128]) {
  if (!nccl::load()) return set_err(RCVD_ERR_NCCL, "libnccl.so.2 not found");
  nccl::UniqueId id; const int r = nccl::GetUniqueId(&id);
  if (r != 0) return set_err(RCVD_ERR_NCCL, "ncclGetUniqueId failed (%d)", r);
  memcpy(out, id.internal, 128); return RCVD_OK;
}
RCVD_API int32_t rcvd_problem_init_comm(rcvd_problem* p, int32_t nranks, int32_t rank, const uint8_t uid[128]) {
  if (!p || nranks < 1 || rank < 0 || rank >= nranks) return set_err(RCVD_ERR_INVALID, "bad rank/nranks");
  if (nranks == 1) { p->nranks = 1; p->rank = 0; return RCVD_OK; }
  if (!nccl::load()) return set_err(RCVD_ERR_NCCL, "libnccl.so.2 not found");
  SET_DEVICE(p->device);
  nccl::UniqueId id; memcpy(id.internal, uid, 128);
  const int r = nccl::CommInitRank(&p->comm, nranks, id, rank);
  if (r != 0) return set_err(RCVD_ERR_NCCL, "ncclCommInitRank failed: %s", nccl::GetErrorString ? nccl::GetErrorString(r) : "?");
  p->nranks = nranks; p->rank = rank; p->structure_ready = false;
  return RCVD_OK;
}
RCVD_API int32_t rcvd_problem_set_state(rcvd_problem* p, const double* x) {
  if (!p || !x) return set_err(RCVD_ERR_INVALID, "null argument");
  p->h_state.assign(x, x + (size_t)p->N * p->L.nf); p->state_dirty = true;
  return RCVD_OK;
}
RCVD_API int32_t rcvd_problem_get_state(rcvd_problem* p, double* x) {
  if (!p || !x) return set_err(RCVD_ERR_INVALID, "null argument");
  const size_t U = (size_t)p->N * p->L.nf;
  if (!p->structure_ready || p->state_dirty) { if (p->h_state.size() != U) p->h_state.assign(U, 0.0); memcpy(x, p->h_state.data(), U * sizeof(double)); return RCVD_OK; }
  SET_DEVICE(p->device);
  return download_frames(p, x, p->d_x, p->L.nf, p->L.nf, p->L.nf);
}
RCVD_API int32_t rcvd_evaluate(rcvd_problem* p, double* cost, double* gradient) {
  if (!p || !cost) return set_err(RCVD_ERR_INVALID, "null argument");
  SET_DEVICE(p->device);
  int rc = ensure_ready(p); if (rc) return rc;
  CK(cudaMemsetAsync(p->d_scal, 0, SC_N * sizeof(double), p->stream));
  rc = enqueue_evaluate(p, p->d_x, gradient != nullptr, false, p->d_g, SC_COST); if (rc) return rc;
  rc = read_scalars(p); if (rc) return rc;
  *cost = p->h_scal[SC_COST];
  if (gradient) {
    if ((rc = download_frames(p, gradient, p->d_g, p->L.nf, p->L.npad, p->L.nf))) return rc;
  }
  return RCVD_OK;
}
RCVD_API int32_t rcvd_normal_matrix_dense(rcvd_problem* p, double* Hout) {
  if (!p || !Hout) return set_err(RCVD_ERR_INVALID, "null argument");
  SET_DEVICE(p->device);
  int rc = ensure_ready(p); if (rc) return rc;
  p->force_full_H = true;                       // debug view: every rank assembles the whole matrix
  rc = enqueue_evaluate(p, p->d_x, true, true, p->d_g, SC_COST);
  p->force_full_H = false;
  if (rc) return rc;
  const size_t U = (size_t)p->N * p->L.nf;
  double* d_out = nullptr;
  CK(cudaMalloc((void**)&d_out, U * U * sizeof(double)));
  CK(cudaMemsetAsync(d_out, 0, U * U * sizeof(double), p->stream));
  k_h_to_dense<<<dim3(nblk((size_t)p->L.nf * p->L.nf), p->nHblocks), 256, 0, p->stream>>>(p->d_H, p->d_hblocks, p->nHblocks, d_out, p->N, p->L.nf, p->L.npad, p->d_uperm);
  cudaError_t e = cudaMemcpyAsync(Hout, d_out, U * U * sizeof(double), cudaMemcpyDeviceToHost, p->stream);
  cudaStreamSynchronize(p->stream); cudaFree(d_out);
  if (e != cudaSuccess) return set_err(RCVD_ERR_CUDA, "copy failed: %s", cudaGetErrorString(e));
  return RCVD_OK;
}
// Debug/test: solve (S H S + diag(D2)) y = b with H = J^T J at the current state.
// S, D2, b, y: N*stride host doubles.
RCVD_API int32_t rcvd_debug_linear_solve(rcvd_problem* p, const double* S, const double* D2, const double* b, double* y) {
  if (!p) return set_err(RCVD_ERR_INVALID, "null argument");
  SET_DEVICE(p->device);
  int rc = ensure_ready(p); if (rc) return rc;
  rc = enqueue_evaluate(p, p->d_x, true, true, p->d_g, SC_COST); if (rc) return rc;
  const int N = p->N, nf = p->L.nf, npad = p->L.npad; const size_t Upad = (size_t)N * npad;
  std::vector<double> hs(Upad, 1.0), hd(Upad, 1.0), hb(Upad, 0.0);
  for (int f = 0; f < N; ++f) for (int l = 0; l < nf; ++l) { const size_t u = (size_t)p->uperm[f] * nf + l; hs[(size_t)f * npad + l] = S[u]; hd[(size_t)f * npad + l] = D2[u]; hb[(size_t)f * npad + l] = b[u]; }
  CK(cudaMemcpyAsync(p->d_S, hs.data(), Upad * 8, cudaMemcpyHostToDevice, p->stream));
  CK(cudaMemcpyAsync(p->d_D2, hd.data(), Upad * 8, cudaMemcpyHostToDevice, p->stream));
  CK(cudaMemcpyAsync(p->d_gs, hb.data(), Upad * 8, cudaMemcpyHostToDevice, p->stream));
  CK(cudaMemsetAsync(p->d_fail, 0, sizeof(int), p->stream));
  rc = factor_solve(p); if (rc) return rc;
  std::vector<double> hy(Upad);
  CK(cudaMemcpyAsync(hy.data(), p->d_y, Upad * 8, cudaMemcpyDeviceToHost, p->stream));
  rc = read_scalars(p); if (rc) return rc;
  for (int f = 0; f < N; ++f) for (int l = 0; l < nf; ++l) y[(size_t)p->uperm[f] * nf + l] = hy[(size_t)f * npad + l];
  if (*p->h_fail) return set_err(RCVD_ERR_NUMERIC, "factorisation hit a non-positive pivot");
  return RCVD_OK;
}
RCVD_API int32_t rcvd_time_accumulate(rcvd_problem* p, int32_t iters, double* ms) {
  if (!p || iters <= 0) return set_err(RCVD_ERR_INVALID, "bad argument");
  SET_DEVICE(p->device);
  int rc = ensure_ready(p); if (rc) return rc;
  for (int i = 0; i < 2; ++i) if (!p->ev[i]) CK(cudaEventCreate(&p->ev[i]));
  if ((rc = enqueue_evaluate(p, p->d_x, true, true, p->d_g, SC_COST))) return rc;   // warm-up
  CK(cudaEventRecord(p->ev[0], p->stream));
  for (int i = 0; i < iters; ++i) if ((rc = enqueue_evaluate(p, p->d_x, true, true, p->d_g, SC_COST))) return rc;
  CK(cudaEventRecord(p->ev[1], p->stream));
  CK(cudaStreamSynchronize(p->stream));
  *ms = ev_ms(p->ev[0], p->ev[1]) / iters;
  return RCVD_OK;
}
RCVD_API int32_t rcvd_time_iteration(rcvd_problem* p, int32_t iters, double radius, double* ms_iter, double* ms_acc, double* ms_lin, double* ms_cost) {
  if (!p || iters <= 0) return set_err(RCVD_ERR_INVALID, "bad argument");
  SET_DEVICE(p->device);
  int rc = ensure_ready(p); if (rc) return rc;
  const int N = p->N, npad = p->L.npad; const size_t Upad = (size_t)N * npad; cudaStream_t st = p->stream;
  for (int i = 0; i < 8; ++i) if (!p->ev[i]) CK(cudaEventCreate(&p->ev[i]));
  double ta = 0, tl = 0, tc = 0, tt = 0;
  for (int it = -1; it < iters; ++it) {   // it == -1: warm-up (also instantiates the graph)
    CK(cudaMemsetAsync(p->d_scal, 0, SC_N * sizeof(double), st));
    CK(cudaMemsetAsync(p->d_fail, 0, sizeof(int), st));
    CK(cudaEventRecord(p->ev[0], st));
    if ((rc = enqueue_evaluate(p, p->d_x, true, true, p->d_g, SC_COST))) return rc;
    if (p->nranks <= 1) k_extract_diag<<<nblk(Upad), 256, 0, st>>>(p->d_H, p->d_diagH, N, npad);
    k_jacobi_scale<<<nblk(Upad), 256, 0, st>>>(p->d_diagH, p->d_S, (int)Upad, 1);
    CK(cudaEventRecord(p->ev[1], st));
    k_lm_prepare<<<nblk(Upad), 256, 0, st>>>(p->d_diagH, p->d_S, p->d_g, p->d_lmdiag, p->d_D2, p->d_gs, (int)Upad, 0, radius, 1e-6, 1e32);
    if ((rc = factor_solve(p))) return rc;
    if ((rc = enqueue_model_terms(p))) return rc;
    CK(cudaEventRecord(p->ev[2], st));
    if ((rc = enqueue_candidate(p, 1.0, p->d_g))) return rc;
    if ((rc = enqueue_evaluate(p, p->d_xc, false, false, nullptr, SC_CAND))) return rc;
    CK(cudaEventRecord(p->ev[3], st));
    if ((rc = read_scalars(p))) return rc;
    if (it >= 0) { ta += ev_ms(p->ev[0], p->ev[1]); tl += ev_ms(p->ev[1], p->ev[2]); tc += ev_ms(p->ev[2], p->ev[3]); tt += ev_ms(p->ev[0], p->ev[3]); }
  }
  *ms_iter = tt / iters; if (ms_acc) *ms_acc = ta / iters; if (ms_lin) *ms_lin = tl / iters; if (ms_cost) *ms_cost = tc / iters;
  return RCVD_OK;
}
// Bench hook: the arrays the last step of rcvd_time_iteration left on the device, in the caller's frame order (N x stride each).
RCVD_API int32_t rcvd_debug_iteration_outputs(rcvd_problem* p, double* gradient, double* step, double* candidate, double costs[2]) {
  if (!p || !gradient || !step || !candidate || !costs) return set_err(RCVD_ERR_INVALID, "null argument");
  if (!p->structure_ready) return set_err(RCVD_ERR_INVALID, "no iteration has run on this problem");
  SET_DEVICE(p->device);
  costs[0] = p->h_scal[SC_COST]; costs[1] = p->h_scal[SC_CAND];
  int rc = download_frames(p, gradient, p->d_g, p->L.nf, p->L.npad, p->L.nf); if (rc) return rc;
  if ((rc = download_frames(p, step, p->d_delta, p->L.nf, p->L.npad, p->L.nf))) return rc;
  return download_frames(p, candidate, p->d_xc, p->L.nf, p->L.nf, p->L.nf);
}
// Bench hook: one factorisation + solve, un-captured on a single stream with one CUDA event per launch; returns the
// summed device time per kernel class: out_ms[0..5] = load, potrf, trinv, trsm, update GEMM (k_gemm_nt), substitution;
// out_ms[6] = number of k_gemm_nt update launches, out_ms[7] = algorithmic flops of those GEMMs.
// reps < 0: keep the two-stream overlap (events on the main stream only: side-stream classes read ~0 and every wait for
// the side stream is charged to the next main-stream launch) -- shows where the chain is delayed by the overlapped work.
RCVD_API int32_t rcvd_debug_profile_linear(rcvd_problem* p, int32_t reps, double out_ms[8]) {
  const bool keep_overlap = reps < 0; if (reps < 0) reps = -reps;
  if (!p || !out_ms || reps == 0) return set_err(RCVD_ERR_INVALID, "bad argument");
  SET_DEVICE(p->device);
  int rc = ensure_ready(p); if (rc) return rc;
  const bool ov = p->overlap; if (!keep_overlap) p->overlap = false;
  for (int i = 0; i < 8; ++i) out_ms[i] = 0.0;
  std::vector<std::pair<int, cudaEvent_t>> evs;
  p->level_ms.assign(p->levels.size() * 6, 0.0);
  for (int r = -1; r < reps; ++r) {
    CK(cudaMemsetAsync(p->d_fail, 0, sizeof(int), p->stream));
    evs.clear(); p->prof = &evs;
    rc = enqueue_factor_solve(p);
    p->prof = nullptr;
    cudaStreamSynchronize(p->stream); cudaStreamSynchronize(p->side_stream);
    double ngemm = 0;
    for (size_t i = 1; i < evs.size(); ++i) {
      float ms = 0; cudaEventElapsedTime(&ms, evs[i - 1].second, evs[i].second);
      const int cls = evs[i].first < 0 ? -1 : (evs[i].first & 0xff), lvl = evs[i].first < 0 ? 0 : (evs[i].first >> 8);
      if (r >= 0 && cls >= 0 && cls < 6) out_ms[cls] += ms;
      if (cls == 4) ngemm += 1;
      if (r == reps - 1 && cls >= 0 && cls < 6 && p->level_ms.size() >= (size_t)(lvl + 1) * 6) p->level_ms[(size_t)lvl * 6 + cls] += ms;
    }
    for (auto& e : evs) cudaEventDestroy(e.second);
    out_ms[6] = ngemm;
    if (rc) break;
  }
  p->overlap = ov;
  for (int i = 0; i < 6; ++i) out_ms[i] /= reps;
  out_ms[7] = p->upd_flops;
  return rc;
}
// Bench hook: fp64 tensor-core (DMMA m8n8k4) peak of this device, measured live with a register-only loop on all SMs.
// MEASURED_PEAKS.json carries HBM and bf16 figures only; this is the denominator of the update-GEMM roofline.
__global__ void k_dmma_peak(double* out, int iters) {
  double c[8][2];
#pragma unroll
  for (int i = 0; i < 8; ++i) { c[i][0] = 0; c[i][1] = 0; }
  const double a = threadIdx.x * 1e-3, b = 1.0 + threadIdx.x * 1e-6;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < 8; ++i) dmma_8x8x4(c[i][0], c[i][1], a, b);
  }
  double s = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) s += c[i][0] + c[i][1];
  out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = s;
}
RCVD_API int32_t rcvd_debug_fp64_tensor_peak(int32_t device, double* tflops) {
  if (!tflops) return set_err(RCVD_ERR_INVALID, "null argument");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) return set_err(RCVD_ERR_NO_DEVICE, "no usable CUDA device");
  SET_DEVICE(device);
  cudaDeviceProp prop; CK(cudaGetDeviceProperties(&prop, device));
  const int threads = 512, blocks = prop.multiProcessorCount * 4, iters = 20000;
  double* out = nullptr; CK(cudaMalloc((void**)&out, (size_t)blocks * threads * sizeof(double)));
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  double best = 0;
  for (int rep = 0; rep < 4; ++rep) {
    cudaEventRecord(e0); k_dmma_peak<<<blocks, threads>>>(out, iters); cudaEventRecord(e1); cudaEventSynchronize(e1);
    float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
    const double tf = 2.0 * 256 * 8 * iters * (double)blocks * (threads / 32) / (ms * 1e-3) / 1e12;
    if (rep > 0 && tf > best) best = tf;
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(out);
  CK(cudaGetLastError());
  *tflops = best; return RCVD_OK;
}
// Test / bench hook: parity evidence at the size that is timed.  One LM trust-region step at the current state with the given radius
// (evaluate, Jacobi scaling, damped factorisation + substitution), then the residual of the linear system on the device:
//   out[0] = |(S H S + D2) y - S g| / |S g|   (k_spmv_sym over the assembled H, independent of the factorisation kernels)
//   out[1] = |S g|,  out[2] = cost,  out[3] = |g|_2,  out[4] = |y|_2,  out[5] = non-positive-pivot flag
__global__ void __launch_bounds__(256) k_lin_residual(const double* __restrict__ S, const double* __restrict__ HSy, const double* __restrict__ D2,
                                                       const double* __restrict__ y, const double* __restrict__ gs, const double* __restrict__ g,
                                                       int n, double* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  double r2 = 0.0, b2 = 0.0, g2 = 0.0, y2 = 0.0;
  if (i < n) { const double r = S[i] * HSy[i] + D2[i] * y[i] - gs[i]; r2 = r * r; b2 = gs[i] * gs[i]; g2 = g[i] * g[i]; y2 = y[i] * y[i]; }
  r2 = warp_sum(r2); b2 = warp_sum(b2); g2 = warp_sum(g2); y2 = warp_sum(y2);
  if ((threadIdx.x & 31) == 0) { red_add(out + 0, r2); red_add(out + 1, b2); red_add(out + 2, g2); red_add(out + 3, y2); }
}
RCVD_API int32_t rcvd_debug_linear_residual(rcvd_problem* p, double radius, double out[6]) {
  if (!p || !out || !(radius > 0.0)) return set_err(RCVD_ERR_INVALID, "bad argument");
  SET_DEVICE(p->device);
  int rc = ensure_ready(p); if (rc) return rc;
  const int N = p->N, npad = p->L.npad; const size_t Upad = (size_t)N * npad; cudaStream_t st = p->stream;
  CK(cudaMemsetAsync(p->d_scal, 0, SC_N * sizeof(double), st));
  CK(cudaMemsetAsync(p->d_fail, 0, sizeof(int), st));
  if ((rc = enqueue_evaluate(p, p->d_x, true, true, p->d_g, SC_COST))) return rc;
  if (p->nranks <= 1) k_extract_diag<<<nblk(Upad), 256, 0, st>>>(p->d_H, p->d_diagH, N, npad);
  k_jacobi_scale<<<nblk(Upad), 256, 0, st>>>(p->d_diagH, p->d_S, (int)Upad, 1);
  k_lm_prepare<<<nblk(Upad), 256, 0, st>>>(p->d_diagH, p->d_S, p->d_g, p->d_lmdiag, p->d_D2, p->d_gs, (int)Upad, 0, radius, 1e-6, 1e32);
  if ((rc = factor_solve(p))) return rc;
  if ((rc = enqueue_model_terms(p))) return rc;                      // leaves H (S y) in d_Hy
  if (p->dist && (rc = allreduce(p, p->d_Hy, Upad))) return rc;      // every rank multiplied only the H blocks it owns
  double* d_out = p->d_scal + 9;                                      // slots 9..12 are unused by the LM loop
  k_lin_residual<<<nblk(Upad), 256, 0, st>>>(p->d_S, p->d_Hy, p->d_D2, p->d_y, p->d_gs, p->d_g, (int)Upad, d_out);
  p->launches += 4;
  if ((rc = read_scalars(p))) return rc;
  const double r2 = p->h_scal[9], b2 = p->h_scal[10];
  out[0] = b2 > 0.0 ? std::sqrt(r2 / b2) : std::sqrt(r2); out[1] = std::sqrt(b2); out[2] = p->h_scal[SC_COST];
  out[3] = std::sqrt(p->h_scal[11]); out[4] = std::sqrt(p->h_scal[12]); out[5] = (double)*p->h_fail;
  return RCVD_OK;
}
// per-level view of the last rcvd_debug_profile_linear call: out[level][6] = ms of {load, potrf, trinv, trsm, update, substitution}; returns levels
RCVD_API int32_t rcvd_debug_level_profile(rcvd_problem* p, double* out, int32_t max_levels) {
  if (!p || !out) return -1;
  const int n = std::min<int>(max_levels, (int)(p->level_ms.size() / 6));
  for (int i = 0; i < n * 6; ++i) out[i] = p->level_ms[i];
  return n;
}
RCVD_API int64_t rcvd_launch_count(rcvd_problem* p) { return p ? p->launches : 0; }
// Test hook: 0 forces the generic accumulate kernel, 1 (default) allows the specialised one.
// Test / bench hook: elimination-order variant (-1 greedy minimum degree, >= 0 multiple elimination with that degree slack).
RCVD_API int32_t rcvd_debug_set_order_slack(rcvd_problem* p, int32_t slack) { if (!p) return RCVD_ERR_INVALID; p->order_slack = slack; p->structure_ready = false; return RCVD_OK; }
// Test / bench hook: 1 (default) = the substitutions of the narrow levels as one persistent dataflow kernel, 0 = level-scheduled GEMV launches throughout.
RCVD_API int32_t rcvd_debug_set_fused_substitution(rcvd_problem* p, int32_t on) { if (!p) return RCVD_ERR_INVALID; p->fused_subst = on; p->structure_ready = false; return RCVD_OK; }   // > 1: levels of at most that many tasks per phase go to the dataflow kernel
// Test / bench hook: 0 = single-stream factorisation graph, 1 (default) = overlap non-critical updates on a second stream.
RCVD_API int32_t rcvd_debug_set_overlap(rcvd_problem* p, int32_t on) { if (!p) return RCVD_ERR_INVALID; p->overlap = on != 0; if (p->solve_graph) { cudaGraphExecDestroy(p->solve_graph); p->solve_graph = nullptr; } return RCVD_OK; }
// Test / bench hook: 0 = explicit inverse + GEMM for the off-diagonal solves, 1 (default) = left-looking tensor-core TRSM.
RCVD_API int32_t rcvd_debug_set_trsm_ll(rcvd_problem* p, int32_t on) { if (!p) return RCVD_ERR_INVALID; p->allow_trsm_ll = (on & 1) != 0; p->trsm_deep = !(on & 2); p->structure_ready = false; return RCVD_OK; }   // bit 0: left-looking TRSM; bit 1: no deep panel prefetch on single-wave launches
// Test / bench hook: grid-size cap (CTAs) of one overlapped update launch on the side stream; 0 = unsliced.
RCVD_API int32_t rcvd_debug_set_side_slice(rcvd_problem* p, int32_t ctas) { if (!p) return RCVD_ERR_INVALID; p->side_slice = ctas; if (p->solve_graph) { cudaGraphExecDestroy(p->solve_graph); p->solve_graph = nullptr; } return RCVD_OK; }
// Test / bench hook: 0 = update GEMMs over the padded size, 1 (default) = trimmed to the unknowns rounded to 8.
RCVD_API int32_t rcvd_debug_set_trim_gemm(rcvd_problem* p, int32_t on) { if (!p) return RCVD_ERR_INVALID; p->trim_gemm = on != 0; if (p->solve_graph) { cudaGraphExecDestroy(p->solve_graph); p->solve_graph = nullptr; } return RCVD_OK; }
// Test / bench hook: 1 (default) = warp 0 of k_potrf_smem only runs the pivot-tile chain, 0 = it also takes trailing tiles.
RCVD_API int32_t rcvd_debug_set_potrf_chain_warp(rcvd_problem* p, int32_t on) { if (!p) return RCVD_ERR_INVALID; p->potrf_chain_warp = (on & 1) != 0; p->potrf_blocked = !(on & 2);   /* bit 1: round-1 shuffle Cholesky of the 16x16 pivot tile */ if (p->solve_graph) { cudaGraphExecDestroy(p->solve_graph); p->solve_graph = nullptr; } return RCVD_OK; }
// Test / bench hook: 1 (default) = persistent TMA-fed update kernel (k_update_tma), 0 = round-1 cp.async kernel (k_gemm_nt).
RCVD_API int32_t rcvd_debug_set_update_kernel(rcvd_problem* p, int32_t tma, int32_t side_items_per_cta) {
  if (!p) return RCVD_ERR_INVALID;
  p->gemm_tma = (tma & 1) != 0; p->upd_dbg = (tma >> 8) & 0xff; p->upd_team_items = (tma >> 16) ? (tma >> 16) - 1 : 1; p->upd_ipc = side_items_per_cta & 0xffff; p->upd_reserve = side_items_per_cta >> 16;   // second argument: items-per-CTA cap | reserved SMs << 16; bits 16+ of the first: (items per SM up to which the two-team shape is used) + 1   // bits 8+: timing experiments of k_update_tma (results invalid)
  if (p->solve_graph) { cudaGraphExecDestroy(p->solve_graph); p->solve_graph = nullptr; }
  if (p->gemm_tma && !p->tmap_ok) p->structure_ready = false;
  return RCVD_OK;
}
// Test / bench hook (nranks > 1): 1 (default) = distributed factorisation (owner-computes phase A, reduce-to-owner of H), 0 = round-1 scheme
// (all-reduce of H, factorisation replicated on every rank).  out (optional): {distributed active, first replicated level, levels}.
// Test / bench hook: 1 = the handle will only evaluate cost / gradient (rcvd_evaluate): no normal matrix, no factor storage is allocated
RCVD_API int32_t rcvd_debug_set_eval_only(rcvd_problem* p, int32_t on) { if (!p) return RCVD_ERR_INVALID; p->eval_only = on != 0; p->structure_ready = false; return RCVD_OK; }
RCVD_API int32_t rcvd_debug_set_distributed(rcvd_problem* p, int32_t on) { if (!p) return RCVD_ERR_INVALID; p->dist_enabled = on != 0; if (p->structure_ready) { int rc_ = save_state(p); if (rc_) return rc_; p->state_dirty = true; } p->structure_ready = false; return RCVD_OK; }
RCVD_API int32_t rcvd_distribution_info(rcvd_problem* p, int32_t out[4]) {
  if (!p || !out) return set_err(RCVD_ERR_INVALID, "null argument");
  SET_DEVICE(p->device);
  int rc = ensure_ready(p); if (rc) return rc;
  out[0] = p->dist ? 1 : 0; out[1] = p->LB; out[2] = (int)p->levels.size(); out[3] = p->dist ? p->fa_cnt[p->rank] + p->fb_cnt[p->rank] : p->N;
  return RCVD_OK;
}
// 0: generic kernel, 1 (default): specialised kernels (run path on a bilinear depth grid), 2: specialised kernel without the run path (round 1)
RCVD_API int32_t rcvd_debug_set_fast_path(rcvd_problem* p, int32_t on) {
  if (!p) return RCVD_ERR_INVALID;
  p->use_fast = on != 0;
  const bool runs = on != 2;
  if (runs != p->use_runs) { p->use_runs = runs; if (p->structure_ready) { int rc_ = save_state(p); if (rc_) return rc_; } p->structure_ready = false; }
  return RCVD_OK;
}
RCVD_API int32_t rcvd_solve(rcvd_problem* p, const rcvd_solve_options* opt, rcvd_solve_summary* summary) {
  if (!p || !summary) return set_err(RCVD_ERR_INVALID, "null argument");
  SET_DEVICE(p->device);
  rcvd_solve_options o; if (opt) o = *opt; else rcvd_default_solve_options(&o);
  return lm_solve(p, o, *summary);
}
// Structure statistics (for DESIGN.md / bench): frames, off-diagonal factor blocks, levels, H blocks, npad.
RCVD_API int32_t rcvd_structure_info(rcvd_problem* p, int32_t out[8]) {
  if (!p) return set_err(RCVD_ERR_INVALID, "null argument");
  SET_DEVICE(p->device);
  int rc = ensure_ready(p); if (rc) return rc;
  out[0] = p->N; out[1] = p->nLoff; out[2] = (int)p->levels.size(); out[3] = p->nHblocks; out[4] = p->L.npad; out[5] = p->L.nf; out[6] = p->num_tiles;
  int upd = 0; for (auto& l : p->levels) upd += l.nupd + l.nupd2; out[7] = upd;
  return RCVD_OK;
}

// ---- dense transform application (next-row kernels) ----
template <int MODE>
static int dense_run(const rcvd_config* cfg, int device, const double* params_in, int nparams, int param_off, const float* src, void* out, size_t out_bytes, int h, int w) {
  Layout L;
  if (!cfg || !make_layout(*cfg, L)) return set_err(RCVD_ERR_INVALID, "unsupported transform configuration");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) return set_err(RCVD_ERR_NO_DEVICE, "no usable CUDA device; this library has no CPU fallback");
  SET_DEVICE(device);
  std::vector<double> pv(L.nf, 0.0);
  for (int i = 0; i < nparams; ++i) pv[param_off + i] = params_in[i];
  double* d_p = nullptr; float* d_src = nullptr; void* d_out = nullptr;
  const size_t n = (size_t)w * h;
  // per-frame calls (DepthFrame::depth(), paramMap, warp for every frame of a video): stream-ordered pool allocations and one
  // synchronisation instead of three cudaMalloc/cudaFree pairs per call
  static thread_local cudaStream_t st = nullptr; static thread_local int st_dev = -1;
  if (!st || st_dev != device) {
    if (st) cudaStreamDestroy(st);
    CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking)); st_dev = device;
    cudaMemPool_t pool; unsigned long long keep = ~0ull;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
  }
  CK(cudaMallocAsync((void**)&d_p, pv.size() * 8, st)); CK(cudaMallocAsync(&d_out, out_bytes, st));
  CK(cudaMemcpyAsync(d_p, pv.data(), pv.size() * 8, cudaMemcpyHostToDevice, st));
  if (src) { CK(cudaMallocAsync((void**)&d_src, n * 4, st)); CK(cudaMemcpyAsync(d_src, src, n * 4, cudaMemcpyHostToDevice, st)); }
  k_dense<MODE><<<nblk(n), 256, 0, st>>>(*cfg, L, d_p, d_src, d_out, h, w);
  cudaError_t e = cudaMemcpyAsync(out, d_out, out_bytes, cudaMemcpyDeviceToHost, st);
  cudaFreeAsync(d_p, st); cudaFreeAsync(d_out, st); if (d_src) cudaFreeAsync(d_src, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return set_err(RCVD_ERR_CUDA, "dense kernel failed: %s", cudaGetErrorString(e));
  return RCVD_OK;
}
RCVD_API int32_t rcvd_depth_apply(const rcvd_config* cfg, int32_t device, const double* dp, const float* src, float* dst, int32_t h, int32_t w) {
  Layout L; if (!cfg || !make_layout(*cfg, L)) return set_err(RCVD_ERR_INVALID, "unsupported transform configuration");
  return dense_run<0>(cfg, device, dp, L.nd, L.offD, src, dst, (size_t)w * h * 4, h, w);
}
RCVD_API int32_t rcvd_depth_param_map(const rcvd_config* cfg, int32_t device, const double* dp, double* out, int32_t h, int32_t w) {
  Layout L; if (!cfg || !make_layout(*cfg, L)) return set_err(RCVD_ERR_INVALID, "unsupported transform configuration");
  if (cfg->depth_type != RCVD_DEPTH_GRID) return set_err(RCVD_ERR_INVALID, "Parameter map not implemented for this transform type.");
  return dense_run<1>(cfg, device, dp, L.nd, L.offD, nullptr, out, (size_t)w * h * L.k * 8, h, w);
}
RCVD_API int32_t rcvd_spatial_warp(const rcvd_config* cfg, int32_t device, const double* sp, float* out, int32_t h, int32_t w) {
  Layout L; if (!cfg || !make_layout(*cfg, L)) return set_err(RCVD_ERR_INVALID, "unsupported transform configuration");
  return dense_run<2>(cfg, device, sp, L.ns, L.offS, nullptr, out, (size_t)w * h * 8, h, w);
}

RCVD_API int32_t rcvd_trim_device_memory(int32_t device) {
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) return set_err(RCVD_ERR_NO_DEVICE, "no usable CUDA device");
  SET_DEVICE(device);
  CK(cudaDeviceSynchronize());
  cudaMemPool_t pool;
  CK(cudaDeviceGetDefaultMemPool(&pool, device));
  CK(cudaMemPoolTrimTo(pool, 0));
  unsigned long long none = 0;                       // rcvd_problem_create raises the threshold again for the next solve
  cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &none);
  return RCVD_OK;
}
// The device the host layer should work on: RCVD_DEVICE if set, else the caller's current CUDA device (so that a process launched
// per GPU -- torchrun LOCAL_RANK + torch.cuda.set_device -- lands on its own GPU); -1 without a usable device.
RCVD_API int32_t rcvd_current_device(void) {
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) { cudaGetLastError(); return -1; }
  if (const char* e = getenv("RCVD_DEVICE")) { const int d = atoi(e); return (d >= 0 && d < ndev) ? d : -1; }
  int d = 0;
  if (cudaGetDevice(&d) != cudaSuccess) { cudaGetLastError(); return -1; }
  return d;
}

// ---------------------------------------------------------------------------
// Flow-guided temporal depth filter (rcvd_filter.cuh)
// ---------------------------------------------------------------------------
RCVD_API int32_t rcvd_flow_guided_filter(const rcvd_filter_params* prm, int32_t device, const float* depth, const float* cams,
                                         const float* fwd_flow, const uint8_t* fwd_mask, const float* bwd_flow, const uint8_t* bwd_mask,
                                         const int32_t* far_pairs, const float* far_flow, const uint8_t* far_mask, float* out) {
  if (!prm || !depth || !cams || !out) return set_err(RCVD_ERR_INVALID, "null argument");
  const rcvd_filter_params& q = *prm;
  if (q.num_frames <= 0 || q.num_out <= 0 || q.first_out < 0 || q.first_out + q.num_out > q.num_frames || q.width <= 0 || q.height <= 0 ||
      q.depth_width <= 0 || q.depth_height <= 0 || q.frame_radius < 0 || q.spatial_radius < 0 || q.num_far < 0 || !(q.inv_aspect > 0.f))
    return set_err(RCVD_ERR_INVALID, "bad filter parameters");
  if (q.frame_radius > 0 && q.num_frames > 1 && (!fwd_flow || !fwd_mask || !bwd_flow || !bwd_mask)) return set_err(RCVD_ERR_INVALID, "flow stacks missing");
  if (q.num_far > 0 && (!far_pairs || !far_flow || !far_mask)) return set_err(RCVD_ERR_INVALID, "far-connection arrays missing");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev)
    return set_err(RCVD_ERR_NO_DEVICE, "no usable CUDA device (%s); this library has no CPU fallback", e != cudaSuccess ? cudaGetErrorString(e) : "device ordinal out of range");
  SET_DEVICE(device);
  const int F = q.num_frames; const size_t plane = (size_t)q.width * q.height, dplane = (size_t)q.depth_width * q.depth_height;
  // cameras: tan(fov / 2) in float on the host, like DepthVideo::project (lib/DepthVideo.cpp:640-641)
  std::vector<float> hc((size_t)F * 12, 0.f);
  for (int f = 0; f < F; ++f) {
    for (int i = 0; i < 7; ++i) hc[(size_t)f * 12 + i] = cams[(size_t)f * 9 + i];
    hc[(size_t)f * 12 + 7] = std::tan(cams[(size_t)f * 9 + 7] / 2.f);
    hc[(size_t)f * 12 + 8] = std::tan(cams[(size_t)f * 9 + 8] / 2.f);
  }
  // far connections grouped by source frame (stable: the caller's order within a frame is kept)
  std::vector<int> far_begin(F + 1, 0), order(q.num_far), pairs_sorted((size_t)2 * q.num_far);
  int maxfar = 0;
  for (int k = 0; k < q.num_far; ++k) {
    const int s = far_pairs[2 * k], d = far_pairs[2 * k + 1];
    if (s < 0 || s >= F || d < 0 || d >= F) return set_err(RCVD_ERR_INVALID, "far connection %d out of range", k);
    far_begin[s + 1]++;
  }
  for (int f = 0; f < F; ++f) { maxfar = std::max(maxfar, far_begin[f + 1]); far_begin[f + 1] += far_begin[f]; }
  { std::vector<int> cur(far_begin.begin(), far_begin.end() - 1); for (int k = 0; k < q.num_far; ++k) order[cur[far_pairs[2 * k]]++] = k; }
  cudaStream_t st; CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
  std::vector<void*> bufs; bool ok = true;
  // a failed allocation must be seen before anything is launched on null buffers (an illegal address is a sticky context error,
  // and PyTorch shares this context)
  auto dev = [&](size_t bytes) -> void* { void* ptr = nullptr; if (cudaMallocAsync(&ptr, std::max<size_t>(bytes, 16), st) != cudaSuccess) { ok = false; cudaGetLastError(); return nullptr; } bufs.push_back(ptr); return ptr; };
  auto up = [&](const void* src, size_t bytes) -> void* { void* d = dev(bytes); if (d && src && bytes) cudaMemcpyAsync(d, src, bytes, cudaMemcpyHostToDevice, st); return d; };
  FilterArgs a{};
  a.depth = (const float*)up(depth, (size_t)F * dplane * 4);
  a.cams = (const float*)up(hc.data(), hc.size() * 4);
  const bool chains = q.frame_radius > 0 && F > 1;
  a.fwd_flow = (const float*)up(chains ? fwd_flow : nullptr, chains ? (size_t)F * plane * 8 : 0); a.fwd_mask = (const uint8_t*)up(chains ? fwd_mask : nullptr, chains ? (size_t)F * plane : 0);
  a.bwd_flow = (const float*)up(chains ? bwd_flow : nullptr, chains ? (size_t)F * plane * 8 : 0); a.bwd_mask = (const uint8_t*)up(chains ? bwd_mask : nullptr, chains ? (size_t)F * plane : 0);
  if (q.num_far > 0) {
    float* ff = (float*)dev((size_t)q.num_far * plane * 8); uint8_t* fm = (uint8_t*)dev((size_t)q.num_far * plane);
    if (ff && fm)
      for (int k = 0; k < q.num_far; ++k) {   // sorted order on the device
        cudaMemcpyAsync(ff + (size_t)k * plane * 2, far_flow + (size_t)order[k] * plane * 2, plane * 8, cudaMemcpyHostToDevice, st);
        cudaMemcpyAsync(fm + (size_t)k * plane, far_mask + (size_t)order[k] * plane, plane, cudaMemcpyHostToDevice, st);
        pairs_sorted[2 * k] = far_pairs[2 * order[k]]; pairs_sorted[2 * k + 1] = far_pairs[2 * order[k] + 1];
      }
    a.far_flow = ff; a.far_mask = fm;
    a.far_pairs = (const int*)up(pairs_sorted.data(), pairs_sorted.size() * 4);
    a.far_begin = (const int*)up(far_begin.data(), far_begin.size() * 4);
  }
  a.out = (float*)dev((size_t)q.num_out * plane * 4);
  const int win = 2 * q.spatial_radius + 1;
  a.max_samples = win * win * (1 + 2 * q.frame_radius + maxfar);
  // the weighted median sorts a per-pixel sample row: the scratch is bounded to ~1 GiB by filtering the range in frame chunks
  const size_t per_frame_scratch = plane * (size_t)a.max_samples * sizeof(float2);
  const int chunk = q.median ? (int)std::max<size_t>(1, std::min<size_t>((size_t)q.num_out, ((size_t)1 << 30) / std::max<size_t>(per_frame_scratch, 1))) : q.num_out;
  if (q.median) a.scratch = (float2*)dev((size_t)chunk * per_frame_scratch);
  int rc = RCVD_OK;
  if (!ok) rc = set_err(RCVD_ERR_CUDA, "device allocation failed in rcvd_flow_guided_filter");
  else {
    cudaMemsetAsync(a.out, 0, (size_t)q.num_out * plane * 4, st);
    float* const out_dev = a.out;
    a.F = F; a.last_frame = q.first_out + q.num_out - 1;
    a.w = q.width; a.h = q.height; a.wd = q.depth_width; a.hd = q.depth_height;
    a.frame_radius = q.frame_radius; a.spatial_radius = q.spatial_radius; a.median = q.median; a.inv_aspect = q.inv_aspect;
    for (int c0 = 0; c0 < q.num_out; c0 += chunk) {
      a.first_out = q.first_out + c0; a.num_out = std::min(chunk, q.num_out - c0); a.out = out_dev + (size_t)c0 * plane;
      const dim3 grid((q.width + 31) / 32, (q.height + 3) / 4, a.num_out);
      if (q.median) k_flow_guided_filter<true><<<grid, 128, 0, st>>>(a); else k_flow_guided_filter<false><<<grid, 128, 0, st>>>(a);
      g_filter_launches++;
    }
    a.out = out_dev;
    e = cudaMemcpyAsync(out, a.out, (size_t)q.num_out * plane * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) rc = set_err(RCVD_ERR_CUDA, "flow-guided filter failed: %s", cudaGetErrorString(e));
  }
  for (void* b : bufs) cudaFreeAsync(b, st);
  cudaStreamSynchronize(st); cudaStreamDestroy(st);
  return rc;
}
RCVD_API int64_t rcvd_filter_launch_count() { return g_filter_launches; }

// ---------------------------------------------------------------------------
// Bilateral depth filter (rcvd_bilateral.cuh)
// ---------------------------------------------------------------------------
// 3-D float32 tensor map {d0, d1, d2} with byte strides s1 (dimension 1) and s2 (dimension 2), box {b0, b1, 1}, zero fill outside
static bool encode_f32_3d(CUtensorMap* m, void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t s1, uint64_t s2, uint32_t b0, uint32_t b1) {
  typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                               CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static EncodeFn fn = nullptr;
  if (!fn) {
    void* p = nullptr; cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || !p || q != cudaDriverEntryPointSuccess) { cudaGetLastError(); return false; }
    fn = (EncodeFn)p;
  }
  const cuuint64_t gdim[3] = {d0, d1, d2}, gstr[2] = {s1, s2};
  const cuuint32_t box[3] = {b0, b1, 1u}, estr[3] = {1u, 1u, 1u};
  return fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, base, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
            CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
template <bool MEDIAN, bool IN_PLACE>
static cudaError_t bilateral_prepare(size_t smem) { return cudaFuncSetAttribute(k_bilateral<MEDIAN, IN_PLACE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); }
template <bool MEDIAN, bool IN_PLACE>
static void bilateral_launch(dim3 grid, size_t smem, cudaStream_t st, const CUtensorMap& td, const CUtensorMap& tc, const BilateralArgs& a) {
  k_bilateral<MEDIAN, IN_PLACE><<<grid, kBilThreads, smem, st>>>(td, tc, a);
}

RCVD_API int32_t rcvd_bilateral_filter(const rcvd_bilateral_params* prm, int32_t device, const float* depth, const float* color, const int32_t* out_frames,
                                       const rcvd_config* xform_cfg, const double* xform_params, float* out) {
  if (!prm || !depth || !out_frames || !out) return set_err(RCVD_ERR_INVALID, "null argument");
  const rcvd_bilateral_params& q = *prm;
  if (q.num_frames <= 0 || q.num_out <= 0 || q.width <= 0 || q.height <= 0 || q.spatial_radius < 0 || q.frame_radius < 0)
    return set_err(RCVD_ERR_INVALID, "bad bilateral filter parameters");
  for (int k = 0; k < q.num_out; ++k)
    if (out_frames[k] < 0 || out_frames[k] >= q.num_frames || (k > 0 && out_frames[k] <= out_frames[k - 1]))
      return set_err(RCVD_ERR_INVALID, "output frames must be ascending local frame indices below num_frames");
  const bool use_c = q.color_sigma > 0.f;
  if (use_c && !color) return set_err(RCVD_ERR_INVALID, "colour frames missing (colorSigma > 0)");
  const bool in_place = q.in_place && q.frame_radius > 0;   // with frameRadius 0 no window reaches a filtered frame
  Layout L{};
  if (in_place && (!xform_cfg || !xform_params || !make_layout(*xform_cfg, L))) return set_err(RCVD_ERR_INVALID, "in-place filtering needs a supported depth transform and its parameters");
  const int r = q.spatial_radius, w = q.width, h = q.height, F = q.num_frames;
  // padded planes (rcvd_bilateral.cuh): halo boxes start at (tile_y, tile_x) of the padded plane; every extent <= 256 elements
  const int pad_l = (r + 3) / 4 * 4, box_w = kBilTW + 2 * pad_l, box_h = kBilTH + 2 * r, cbox_w = 3 * box_w;
  const uint32_t depth_bytes = (uint32_t)((box_w * box_h * 4 + 1023) / 1024 * 1024);
  const uint32_t stage_bytes = depth_bytes + (use_c ? (uint32_t)((cbox_w * box_h * 4 + 1023) / 1024 * 1024) : 0u);
  const size_t smem = 2 * (size_t)stage_bytes + 2 * sizeof(uint64_t);
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev)
    return set_err(RCVD_ERR_NO_DEVICE, "no usable CUDA device (%s); this library has no CPU fallback", e != cudaSuccess ? cudaGetErrorString(e) : "device ordinal out of range");
  SET_DEVICE(device);
  int smem_max = 0; CK(cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
  if (box_w > 256 || box_h > 256 || (use_c && cbox_w > 256) || smem > (size_t)smem_max)
    return set_err(RCVD_ERR_INVALID, "spatialRadius %d is too large: the %d x %d halo tile of one frame%s does not fit the TMA box / shared-memory limits", r,
                   box_w, box_h, use_c ? " with colour" : "");
  const int Wp = std::max((pad_l + w + r + 3) / 4 * 4, box_w), Hp = std::max(h + 2 * r, box_h);
  const size_t dplane = (size_t)Wp * Hp, cplane = 3 * dplane;
  const int P = F + (in_place ? q.num_out : 0);
  const int window = (int)std::min<int64_t>(2 * (int64_t)q.frame_radius + 1, F);
  const int max_samples = (2 * r + 1) * (2 * r + 1) * window;
  // the weighted median sorts a per-pixel sample row: the scratch is bounded to ~1 GiB by filtering frame chunks, and row bands of a
  // frame when one frame alone is larger
  const size_t row_scratch = (size_t)w * max_samples * sizeof(float2), limit = (size_t)1 << 30;
  int zmax = in_place ? 1 : std::min(q.num_out, 65535), band = h;
  if (q.median) {
    if (row_scratch * h <= limit) zmax = (int)std::min<size_t>((size_t)zmax, limit / (row_scratch * h));
    else { zmax = 1; band = (int)std::max<size_t>(1, limit / row_scratch); if (band >= kBilTH) band -= band % kBilTH; }
  }
  std::vector<int> retrans(F, -1);
  for (int k = 0; k < q.num_out; ++k) retrans[out_frames[k]] = k;
  std::vector<double> xp;
  if (in_place) {
    xp.assign((size_t)q.num_out * L.nf, 0.0);
    for (int k = 0; k < q.num_out; ++k) for (int i = 0; i < L.nd; ++i) xp[(size_t)k * L.nf + L.offD + i] = xform_params[(size_t)k * L.nd + i];
  }
  cudaStream_t st; CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
  std::vector<void*> bufs; bool ok = true;
  auto dev = [&](size_t bytes) -> void* { void* ptr = nullptr; if (cudaMallocAsync(&ptr, std::max<size_t>(bytes, 16), st) != cudaSuccess) { ok = false; cudaGetLastError(); return nullptr; } bufs.push_back(ptr); return ptr; };
  auto up = [&](const void* src, size_t bytes) -> void* { void* d = dev(bytes); if (d && bytes) cudaMemcpyAsync(d, src, bytes, cudaMemcpyHostToDevice, st); return d; };
  BilateralArgs a{};
  a.depth = (float*)dev((size_t)P * dplane * 4);
  if (a.depth) {
    cudaMemsetAsync(a.depth, 0, (size_t)P * dplane * 4, st);
    for (int f = 0; f < F; ++f)
      cudaMemcpy2DAsync(a.depth + f * dplane + (size_t)r * Wp + pad_l, (size_t)Wp * 4, depth + (size_t)f * h * w, (size_t)w * 4, (size_t)w * 4, h, cudaMemcpyHostToDevice, st);
  }
  if (use_c) {
    float* c = (float*)dev((size_t)F * cplane * 4);
    if (c) {
      cudaMemsetAsync(c, 0, (size_t)F * cplane * 4, st);
      for (int f = 0; f < F; ++f)
        cudaMemcpy2DAsync(c + f * cplane + 3 * ((size_t)r * Wp + pad_l), (size_t)Wp * 12, color + (size_t)f * h * w * 3, (size_t)w * 12, (size_t)w * 12, h, cudaMemcpyHostToDevice, st);
    }
    a.color = c;
  }
  a.out_frames = (const int*)up(out_frames, (size_t)q.num_out * 4);
  a.retrans = (const int*)up(retrans.data(), retrans.size() * 4);
  if (in_place) a.xparams = (const double*)up(xp.data(), xp.size() * 8);
  a.out = (float*)dev((size_t)q.num_out * h * w * 4);
  if (q.median) a.scratch = (float2*)dev((size_t)zmax * band * row_scratch);
  int rc = RCVD_OK;
  CUtensorMap tmd, tmc;
  if (!ok) rc = set_err(RCVD_ERR_CUDA, "device allocation failed in rcvd_bilateral_filter");
  else if (!encode_f32_3d(&tmd, a.depth, Wp, Hp, P, (uint64_t)Wp * 4, dplane * 4, box_w, box_h) ||
           (use_c && !encode_f32_3d(&tmc, (void*)a.color, 3 * (uint64_t)Wp, Hp, F, (uint64_t)Wp * 12, cplane * 4, cbox_w, box_h)))
    rc = set_err(RCVD_ERR_CUDA, "cuTensorMapEncodeTiled unavailable or failed: the TMA-fed bilateral filter cannot run");
  else {
    if (!use_c) tmc = tmd;   // not read
    if (xform_cfg && in_place) a.cfg = *xform_cfg;
    a.L = L; a.F = F; a.w = w; a.h = h; a.Wp = Wp; a.Hp = Hp; a.pad_l = pad_l;
    a.spatial_radius = r; a.frame_radius = q.frame_radius; a.max_samples = max_samples;
    a.box_w = box_w; a.box_h = box_h; a.stage_bytes = stage_bytes; a.depth_bytes = depth_bytes;
    a.depth_sigma2 = q.depth_sigma > 0.f ? q.depth_sigma * q.depth_sigma : 0.f;   // sqr(sigma) in float (:184-185)
    a.color_sigma2 = use_c ? q.color_sigma * q.color_sigma : 0.f;
    e = q.median ? (in_place ? bilateral_prepare<true, true>(smem) : bilateral_prepare<true, false>(smem))
                 : (in_place ? bilateral_prepare<false, true>(smem) : bilateral_prepare<false, false>(smem));
    // in place: one launch per frame in range order; each reads the re-transformed planes written by the launches before it
    for (int k0 = 0; e == cudaSuccess && k0 < q.num_out; k0 += zmax)
      for (int y0 = 0; y0 < h; y0 += band) {
        const int nz = std::min(zmax, q.num_out - k0), y1 = std::min(h, y0 + band);
        a.out_begin = k0; a.y_begin = y0; a.y_end = y1;
        const dim3 grid((w + kBilTW - 1) / kBilTW, (y1 - y0 + kBilTH - 1) / kBilTH, nz);
        if (q.median) { if (in_place) bilateral_launch<true, true>(grid, smem, st, tmd, tmc, a); else bilateral_launch<true, false>(grid, smem, st, tmd, tmc, a); }
        else { if (in_place) bilateral_launch<false, true>(grid, smem, st, tmd, tmc, a); else bilateral_launch<false, false>(grid, smem, st, tmd, tmc, a); }
        g_filter_launches++;
      }
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, a.out, (size_t)q.num_out * h * w * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) rc = set_err(RCVD_ERR_CUDA, "bilateral filter failed: %s", cudaGetErrorString(e));
  }
  for (void* b : bufs) cudaFreeAsync(b, st);
  cudaStreamSynchronize(st); cudaStreamDestroy(st);
  return rc;
}

// ---------------------------------------------------------------------------
// GPU flow-constraint builder (rcvd_builder.cuh)
// ---------------------------------------------------------------------------
static int64_t g_builder_launches = 0, g_builder_rounds = 0;
RCVD_API int64_t rcvd_builder_launch_count() { return g_builder_launches; }
RCVD_API int64_t rcvd_builder_last_rounds() { return g_builder_rounds; }
RCVD_API int32_t rcvd_build_constraints(const rcvd_builder_params* prm, int32_t device, const float* color_bgr, const float* dyn_dist,
                                        const int32_t* pair_frames, const float* pair_flow, const uint8_t* pair_mask,
                                        const int32_t* trip_frames, const float* trip_flow, const uint8_t* trip_mask,
                                        int64_t* pair_offsets, float* pair_out, int64_t pair_capacity,
                                        int64_t* trip_offsets, float* trip_out, int64_t trip_capacity) {
  if (!prm || !color_bgr) return set_err(RCVD_ERR_INVALID, "null argument");
  const rcvd_builder_params& q = *prm;
  const int P = q.num_pairs, T = q.num_triplets, F = q.num_frames, I = P + T;
  if (F <= 0 || q.width <= 0 || q.height <= 0 || P < 0 || T < 0 || q.match_separation < 0 || !(q.inv_aspect > 0.f)) return set_err(RCVD_ERR_INVALID, "bad builder parameters");
  if ((P > 0 && (!pair_frames || !pair_flow || !pair_mask || !pair_offsets)) || (T > 0 && (!trip_frames || !trip_flow || !trip_mask || !trip_offsets)))
    return set_err(RCVD_ERR_INVALID, "null argument");
  if (dyn_dist && (q.dyn_width <= 0 || q.dyn_height <= 0)) return set_err(RCVD_ERR_INVALID, "bad dynamic-distance size");
  for (int i = 0; i < P; ++i) if (pair_frames[2 * i] < 0 || pair_frames[2 * i] >= F || pair_frames[2 * i + 1] < 0 || pair_frames[2 * i + 1] >= F) return set_err(RCVD_ERR_INVALID, "pair %d out of range", i);
  for (int i = 0; i < T; ++i) if (trip_frames[i] < 1 || trip_frames[i] >= F) return set_err(RCVD_ERR_INVALID, "triplet %d out of range", i);
  if (pair_offsets) pair_offsets[0] = 0;
  if (trip_offsets) trip_offsets[0] = 0;
  if (I == 0) return RCVD_OK;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev)
    return set_err(RCVD_ERR_NO_DEVICE, "no usable CUDA device (%s); this library has no CPU fallback", e != cudaSuccess ? cudaGetErrorString(e) : "device ordinal out of range");
  SET_DEVICE(device);
  const size_t plane = (size_t)q.width * q.height, FP = plane * F;
  cudaStream_t st; CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
  std::vector<void*> bufs; bool ok = true;
  auto dev = [&](size_t bytes) -> void* { void* ptr = nullptr; if (cudaMallocAsync(&ptr, std::max<size_t>(bytes, 16), st) != cudaSuccess) { ok = false; return nullptr; } bufs.push_back(ptr); return ptr; };
  auto up = [&](const void* src, size_t bytes) -> void* { void* d = dev(bytes); if (d && src && bytes) cudaMemcpyAsync(d, src, bytes, cudaMemcpyHostToDevice, st); return d; };
  auto cleanup = [&]() { for (void* b : bufs) cudaFreeAsync(b, st); cudaStreamSynchronize(st); cudaStreamDestroy(st); };
  // ---- corner scores of every frame ----
  float* d_bgr = (float*)up(color_bgr, FP * 3 * sizeof(float));
  float* d_gray = (float*)dev(FP * 4), *d_pl = (float*)dev(FP * 12), *d_corner = (float*)dev(FP * 4); double* d_tmp = (double*)dev(FP * 24);
  BuilderArgs a{};
  a.dyn = dyn_dist ? (const float*)up(dyn_dist, (size_t)F * q.dyn_width * q.dyn_height * 4) : nullptr;
  a.pair_frames = (const int*)up(pair_frames, (size_t)P * 8); a.pair_flow = (const float*)up(pair_flow, (size_t)P * plane * 8); a.pair_mask = (const uint8_t*)up(pair_mask, (size_t)P * plane);
  a.trip_frames = (const int*)up(trip_frames, (size_t)T * 4); a.trip_flow = (const float*)up(trip_flow, (size_t)T * 2 * plane * 8); a.trip_mask = (const uint8_t*)up(trip_mask, (size_t)T * 2 * plane);
  a.prio = (float*)dev((size_t)I * plane * 4); a.state = (uint8_t*)dev((size_t)I * plane);
  unsigned long long* d_cnt = (unsigned long long*)dev((size_t)(2 * I + 2) * 8);   // [0] undecided, [1..I] counts / offsets, [I+1..2I] cursors
  if (!ok) { cleanup(); return set_err(RCVD_ERR_CUDA, "device allocation failed in rcvd_build_constraints"); }
  const int W = q.width, H = q.height;
  k_gray<<<(unsigned)((FP + 255) / 256), 256, 0, st>>>(d_bgr, d_gray, FP);
  k_sobel_products<<<(unsigned)((FP + 255) / 256), 256, 0, st>>>(d_gray, d_pl, F, H, W);
  k_box_h<<<(unsigned)((FP * 3 + 255) / 256), 256, 0, st>>>(d_pl, d_tmp, (size_t)3 * F * H, W);
  k_box_v_eig<<<(unsigned)(((size_t)F * W + 127) / 128), 128, 0, st>>>(d_tmp, d_corner, F, H, W);
  g_builder_launches += 4;
  a.corner = d_corner; a.P = P; a.T = T; a.h = H; a.w = W; a.dh = q.dyn_height; a.dw = q.dyn_width; a.sep = q.match_separation; a.min_dyn = q.min_dynamic_distance;
  // dynamic-mask scale (lib/FlowConstraints.cpp:415-417); without a dynamic mask the distance image has the colour size (:277-285)
  a.dsx = dyn_dist ? q.dyn_width / float(W) : 1.f; a.dsy = dyn_dist ? q.dyn_height / float(H) : 1.f;
  a.sx = 1.f / W; a.sy = q.inv_aspect / H;
  const unsigned gx = (unsigned)((plane + 255) / 256);
  if (P > 0) { k_pair_candidates<<<dim3(gx, P), 256, 0, st>>>(a); g_builder_launches++; }
  if (T > 0) { k_triplet_candidates<<<dim3(gx, T), 256, 0, st>>>(a); g_builder_launches++; }
  // ---- selection rounds until nothing is undecided ----
  int rounds = 0;
  for (;;) {
    cudaMemsetAsync(d_cnt, 0, 8, st);
    k_select_round<<<dim3(gx, I), 256, 0, st>>>(a, d_cnt); g_builder_launches++; ++rounds;
    unsigned long long und = 0;
    e = cudaMemcpyAsync(&und, d_cnt, 8, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) { cleanup(); return set_err(RCVD_ERR_CUDA, "constraint selection failed: %s", cudaGetErrorString(e)); }
    if (und == 0) break;
    if (rounds > 4 * (W + H) + 16) { cleanup(); return set_err(RCVD_ERR_CUDA, "constraint selection did not converge"); }
  }
  g_builder_rounds = rounds;
  // ---- counts, offsets, emission ----
  cudaMemsetAsync(d_cnt, 0, (size_t)(2 * I + 2) * 8, st);
  k_count_accepted<<<dim3(gx, I), 256, 0, st>>>(a, d_cnt + 1); g_builder_launches++;
  std::vector<unsigned long long> cnt(I), off(I + 1, 0);
  e = cudaMemcpyAsync(cnt.data(), d_cnt + 1, (size_t)I * 8, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) { cleanup(); return set_err(RCVD_ERR_CUDA, "constraint count read-back failed: %s", cudaGetErrorString(e)); }
  for (int i = 0; i < I; ++i) off[i + 1] = off[i] + cnt[i];
  const unsigned long long pair_total = off[P], total = off[I];
  for (int i = 0; i < P; ++i) pair_offsets[i + 1] = (int64_t)off[i + 1];
  for (int i = 0; i < T; ++i) trip_offsets[i + 1] = (int64_t)(off[P + i + 1] - pair_total);
  if ((int64_t)pair_total > pair_capacity || (int64_t)(total - pair_total) > trip_capacity || (pair_total > 0 && !pair_out) || (total > pair_total && !trip_out)) {
    cleanup(); return set_err(RCVD_ERR_INVALID, "output capacity too small: %llu pair and %llu triplet constraints", pair_total, total - pair_total);
  }
  int rc = RCVD_OK;
  if (total > 0) {
    unsigned long long* d_off = (unsigned long long*)up(off.data(), (size_t)(I + 1) * 8);
    int* d_idx = (int*)dev(total * 4); float* d_score = (float*)dev(total * 4);
    float* d_po = (float*)dev(std::max<size_t>(pair_total, 1) * 16); float* d_to = (float*)dev(std::max<size_t>(total - pair_total, 1) * 24);
    if (!ok) { cleanup(); return set_err(RCVD_ERR_CUDA, "device allocation failed in rcvd_build_constraints"); }
    k_emit<<<dim3(gx, I), 256, 0, st>>>(a, d_off, d_cnt + 1 + I, d_idx, d_score, d_po, d_to, pair_total); g_builder_launches++;
    std::vector<int> idx(total); std::vector<float> score(total), po(pair_total * 4), to((total - pair_total) * 6);
    cudaMemcpyAsync(idx.data(), d_idx, total * 4, cudaMemcpyDeviceToHost, st); cudaMemcpyAsync(score.data(), d_score, total * 4, cudaMemcpyDeviceToHost, st);
    if (pair_total) cudaMemcpyAsync(po.data(), d_po, pair_total * 16, cudaMemcpyDeviceToHost, st);
    if (total > pair_total) cudaMemcpyAsync(to.data(), d_to, (total - pair_total) * 24, cudaMemcpyDeviceToHost, st);
    e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) rc = set_err(RCVD_ERR_CUDA, "constraint emission failed: %s", cudaGetErrorString(e));
    else {
      // order each item's survivors by priority (host: a few hundred entries per item)
      std::vector<unsigned long long> perm;
      for (int i = 0; i < I; ++i) {
        const unsigned long long b = off[i], n = cnt[i];
        perm.resize(n); for (unsigned long long k = 0; k < n; ++k) perm[k] = b + k;
        std::sort(perm.begin(), perm.end(), [&](unsigned long long x, unsigned long long y) { return score[x] > score[y] || (score[x] == score[y] && idx[x] < idx[y]); });
        for (unsigned long long k = 0; k < n; ++k) {
          if (i < P) std::memcpy(pair_out + (b + k) * 4, po.data() + perm[k] * 4, 16);
          else std::memcpy(trip_out + (b - pair_total + k) * 6, to.data() + (perm[k] - pair_total) * 6, 24);
        }
      }
    }
  }
  cleanup();
  return rc;
}

// ---------------------------------------------------------------------------
// Dynamic-mask distance transform + static flags on the device (rcvd_builder.cuh)
// ---------------------------------------------------------------------------
static int64_t g_flag_launches = 0;
RCVD_API int64_t rcvd_static_flag_launch_count() { return g_flag_launches; }
// dist_out (optional): [F][h][w] float32 = cv::distanceTransform(mask >= 127 ? 255 : 0, DIST_L2, 5) of every frame (fixed-point chamfer).
// pair_static / trip_static (optional): one byte per constraint.
RCVD_API int32_t rcvd_static_flags(int32_t device, const uint8_t* masks, int32_t F, int32_t h, int32_t w, float distance,
                                   int32_t num_pairs, const int32_t* pair_frames, const int64_t* pair_offsets, const float* pair_locs, uint8_t* pair_static,
                                   int32_t num_triplets, const int32_t* trip_frames, const int64_t* trip_offsets, const float* trip_locs, uint8_t* trip_static,
                                   float* dist_out) {
  if (!masks || F <= 0 || h <= 0 || w <= 0 || num_pairs < 0 || num_triplets < 0) return set_err(RCVD_ERR_INVALID, "bad static-flag arguments");
  if ((num_pairs > 0 && (!pair_frames || !pair_offsets || !pair_static)) || (num_triplets > 0 && (!trip_frames || !trip_offsets || !trip_static))) return set_err(RCVD_ERR_INVALID, "null argument");
  for (int i = 0; i < num_pairs; ++i) if (pair_frames[2 * i] < 0 || pair_frames[2 * i] >= F || pair_frames[2 * i + 1] < 0 || pair_frames[2 * i + 1] >= F || pair_offsets[i + 1] < pair_offsets[i]) return set_err(RCVD_ERR_INVALID, "bad pair %d", i);
  for (int i = 0; i < num_triplets; ++i) if (trip_frames[i] < 1 || trip_frames[i] + 1 >= F || trip_offsets[i + 1] < trip_offsets[i]) return set_err(RCVD_ERR_INVALID, "bad triplet %d", i);
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev)
    return set_err(RCVD_ERR_NO_DEVICE, "no usable CUDA device (%s); this library has no CPU fallback", e != cudaSuccess ? cudaGetErrorString(e) : "device ordinal out of range");
  SET_DEVICE(device);
  const size_t plane = (size_t)w * h;
  cudaStream_t st; CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
  std::vector<void*> bufs; bool ok = true;
  auto dev = [&](size_t bytes) -> void* { void* ptr = nullptr; if (cudaMallocAsync(&ptr, std::max<size_t>(bytes, 16), st) != cudaSuccess) { ok = false; cudaGetLastError(); return nullptr; } bufs.push_back(ptr); return ptr; };
  auto up = [&](const void* src, size_t bytes) -> void* { void* d = dev(bytes); if (d && src && bytes) cudaMemcpyAsync(d, src, bytes, cudaMemcpyHostToDevice, st); return d; };
  auto cleanup = [&]() { for (void* b : bufs) cudaFreeAsync(b, st); cudaStreamSynchronize(st); cudaStreamDestroy(st); };
  const uint8_t* d_masks = (const uint8_t*)up(masks, (size_t)F * plane);
  unsigned* d_scratch = (unsigned*)dev((size_t)F * plane * 4); float* d_dist = (float*)dev((size_t)F * plane * 4);
  const int64_t np_total = num_pairs ? pair_offsets[num_pairs] : 0, nt_total = num_triplets ? trip_offsets[num_triplets] : 0;
  std::vector<int32_t> pf3((size_t)num_pairs * 3, -1), tf3((size_t)num_triplets * 3, -1);
  for (int i = 0; i < num_pairs; ++i) { pf3[3 * i] = pair_frames[2 * i]; pf3[3 * i + 1] = pair_frames[2 * i + 1]; }
  for (int i = 0; i < num_triplets; ++i) { tf3[3 * i] = trip_frames[i] - 1; tf3[3 * i + 1] = trip_frames[i]; tf3[3 * i + 2] = trip_frames[i] + 1; }
  int* d_pf = (int*)up(pf3.data(), pf3.size() * 4); int* d_tf = (int*)up(tf3.data(), tf3.size() * 4);
  long long* d_po = (long long*)up(pair_offsets, (size_t)(num_pairs + 1) * 8 * (num_pairs > 0)); long long* d_to = (long long*)up(trip_offsets, (size_t)(num_triplets + 1) * 8 * (num_triplets > 0));
  float* d_pl = (float*)up(pair_locs, (size_t)np_total * 16); float* d_tl = (float*)up(trip_locs, (size_t)nt_total * 24);
  uint8_t* d_ps = (uint8_t*)dev((size_t)np_total); uint8_t* d_ts = (uint8_t*)dev((size_t)nt_total);
  if (!ok) { cleanup(); return set_err(RCVD_ERR_CUDA, "device allocation failed in rcvd_static_flags"); }
  k_chamfer5<<<F, kChamThreads, 0, st>>>(d_masks, d_scratch, d_dist, h, w); g_flag_launches++;
  if (np_total > 0) { k_static_flags<<<dim3(8, num_pairs), 256, 0, st>>>(d_dist, h, w, distance, 2, d_pf, d_po, num_pairs, d_pl, d_ps); g_flag_launches++; }
  if (nt_total > 0) { k_static_flags<<<dim3(8, num_triplets), 256, 0, st>>>(d_dist, h, w, distance, 3, d_tf, d_to, num_triplets, d_tl, d_ts); g_flag_launches++; }
  if (np_total > 0) cudaMemcpyAsync(pair_static, d_ps, (size_t)np_total, cudaMemcpyDeviceToHost, st);
  if (nt_total > 0) cudaMemcpyAsync(trip_static, d_ts, (size_t)nt_total, cudaMemcpyDeviceToHost, st);
  if (dist_out) cudaMemcpyAsync(dist_out, d_dist, (size_t)F * plane * 4, cudaMemcpyDeviceToHost, st);
  e = cudaStreamSynchronize(st);
  if (e == cudaSuccess) e = cudaGetLastError();
  cleanup();
  if (e != cudaSuccess) return set_err(RCVD_ERR_CUDA, "static-flag kernels failed: %s", cudaGetErrorString(e));
  return RCVD_OK;
}
