// libsos_b200: C ABI over the sm_100a kernels (see include/sos_b200.h for the contract).
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <new>
#include <string>
#include <vector>

#include <nvtx3/nvToolsExt.h>  // header-only NVTX 3: ranges cost nothing unless a tool is attached

#include "common.cuh"
#include "first_order.cuh"
#include "gemm_f64.cuh"
#include "gemm_fold.cuh"
#include "gemm_lowrank.cuh"
#include "layer_shard.cuh"
#include "phase.cuh"
#include "quadrature.cuh"
#include "single_scatter.cuh"
#include "sweep.cuh"

namespace {

thread_local std::string g_last_cuda_error;

#define SOS_CUDA(call)                                                                          \
  do {                                                                                          \
    cudaError_t _e = (call);                                                                    \
    if (_e != cudaSuccess) {                                                                    \
      g_last_cuda_error = std::string(#call) + ": " + cudaGetErrorString(_e);                   \
      return SOS_ERR_CUDA;                                                                      \
    }                                                                                           \
  } while (0)

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

PFN_encodeTiled get_encode() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(p);
  }
  return fn;
}

// 2D row-major double tensor [rows][cols] with row stride ld (elements)
int encode_2d(CUtensorMap* map, const void* base, uint64_t cols, uint64_t rows, uint64_t ld, uint32_t box_cols,
              uint32_t box_rows, CUtensorMapSwizzle swz) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) {
    g_last_cuda_error = "cuTensorMapEncodeTiled entry point not available";
    return SOS_ERR_CUDA;
  }
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld * sizeof(double)};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    g_last_cuda_error = "cuTensorMapEncodeTiled failed with CUresult " + std::to_string(static_cast<int>(r));
    return SOS_ERR_CUDA;
  }
  return SOS_OK;
}

// 3D row-major double tensor [slabs][rows][cols] (row stride ld, slab stride rows*ld)
int encode_3d(CUtensorMap* map, const void* base, uint64_t cols, uint64_t rows, uint64_t slabs, uint64_t ld, uint32_t box_cols,
              uint32_t box_rows) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) {
    g_last_cuda_error = "cuTensorMapEncodeTiled entry point not available";
    return SOS_ERR_CUDA;
  }
  cuuint64_t dims[3] = {cols, rows, slabs};
  cuuint64_t strides[2] = {ld * sizeof(double), rows * ld * sizeof(double)};
  cuuint32_t box[3] = {box_cols, box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    g_last_cuda_error = "cuTensorMapEncodeTiled (3D) failed with CUresult " + std::to_string(static_cast<int>(r));
    return SOS_ERR_CUDA;
  }
  return SOS_OK;
}

}  // namespace

struct sos_plan {
  sos_grid grid;
  GridDev dev;
  int device = 0;  // ordinal the plan lives on: every entry point switches to it (DeviceGuard)
  int N;
  int n_sms;
  long long launches;
  // device allocations
  std::vector<void*> allocs;
  double* d_aggD = nullptr;
  double* d_aggU = nullptr;
  double* d_carryD = nullptr;
  double* d_carryU = nullptr;
  double* d_C = nullptr;     // [S][2][N] first-order coefficients
  double* d_Ctab = nullptr;  // sos_first_order_tab: the uploaded table, weights and indices the coefficients are assembled from
  double* d_sums = nullptr;  // [S][L][3]
  double* d_z = nullptr;     // [L]
  double* d_colint = nullptr;  // [N] column integrals of the device phase builder
  double* d_bs = nullptr;    // upward surface radiance of order 1: [S] over a diffuse Lambert ground, [S][M-1] over a Ross-Li one
  // Ross-Li / ocean ground (those surfaces only): the registered mode matrix pairs and the per-scenario data of
  // sosbrdf::BrdfDev; brdf_nk = matrices per set (Ross-Li 2, ocean 1, other surfaces 0)
  const double** d_brdf_R = nullptr;  // [MAX_SETS][2]
  char* d_brdf_scen = nullptr;        // [S][2] f | [S][2][M-1] beam | [S] set (int)
  int brdf_sets = 0, brdf_ldr = 0, brdf_nk = 0;
  bool brdf_scen_ready = false;
  int* h_poll = nullptr;     // pinned
  double* h_C[2] = {nullptr, nullptr};        // pinned staging of the first-order coefficients (sos_first_order never blocks)
  cudaEvent_t h_C_ev[2] = {nullptr, nullptr};
  int h_C_next = 0;
  std::vector<sos_scenario> scen_h;
  std::vector<double> mu_h;
  // GEMM
  int gemm_bm = 0;  // rows per tile
  int gemm_bn = 128;  // columns per tile (128, or 144 when that pads N less and the batch is large)
  int split_passes = 0;  // class-1 operand passes as separate tiles (small batches; see GemmParams)
  int split_general = 0; // ... as chosen at plan creation for the general kernel
  sosgemm::GroupTable groups;
  int* d_members = nullptr;      // scenario ids per group (static)
  int* d_active_list = nullptr;  // compacted per group (device-built)
  TilePlan* d_tile_plan = nullptr;
  int* d_work_counter = nullptr;
  int* d_order = nullptr;        // device-side order counter (sos_converge with order < 0)
  int nseg[2] = {0, 0};
  int lda = 0;
  sosgemm::GemmParams gp;
  std::map<const void*, CUtensorMap> map_cache;
  bool maps_A_ready = false;
  std::vector<const double*> A_ptrs;  // operands of sos_plan_set_phase (maps are re-encoded when the tile shape changes)
  // folded contraction (centrosymmetric operands, gemm_fold.cuh)
  bool fold = false;
  sosgemm::FoldParams fp;
  unsigned long long* d_fold_stats = nullptr;
  unsigned long long* d_lr_stats = nullptr;  // residual / max|A| / max|beta| of sos_build_lowrank_mu2
  std::vector<const double*> F_ptrs;
  // premixed aerosol operands (one per scenario) and the tile-plan tables that go with them
  int fold_segs = 8;       // 8-row segments per tile of the folded kernel: 8 (64-row tiles), or 7 when every dense tile is an aerosol layer of 7 segments
  int fold_ksplit = 1;     // 2: split k for launches with few tiles (single solves), see FoldParams
  bool fold_xform = true;  // transformer warps form (u, v) once per stage (SOS_FOLD_XFORM=0: every consumer warp does)
  bool premix = false;
  double* d_mix = nullptr;
  std::vector<int> members_h;  // host copy of d_members
  sosgemm::GroupTable groups_premix;   // fold-mode tables: class 2 = premixed aerosol rows, class 3 = low-rank operand rows
  int* d_members_premix = nullptr;
  // low-rank operands (gemm_lowrank.cuh): rank 0 = dense
  int lowrank_rank[SOS_MAX_PHASE] = {0};
  const double* lowrank_Ut[SOS_MAX_PHASE] = {nullptr};
  const double* lowrank_Vt[SOS_MAX_PHASE] = {nullptr};
  int lowrank_ldr = 0;
  int n_lowrank_groups = 0;
  int lowrank_rp = 4;
  // generated source inside sos_solve (sweep.cuh: SrcGen): the molecular rows never materialise J or I_n
  bool gen_ok = false;        // buffers exist (SOS_B200_GENSRC=0 disables)
  bool gen_disabled = false;  // a blend left the zone columns at run time: every row is read / stored from now on
  int gen_nslots = 0, gen_zlo = 0, gen_zu_end = 0;
  double* d_proj = nullptr;     // [S][L][nslots][2]
  double* d_cj[2] = {nullptr, nullptr};  // [S][L][2] source coefficients, ping-pong over the orders
  // CUDA graph of two consecutive orders (even + odd: the source coefficients ping-pong), replayed by sos_solve
  struct OrderGraph {
    const void* I; const void* In; const void* J; bool gen; cudaGraphExec_t exec; long long launches;
    sosgemm::GemmParams gp; sosgemm::FoldParams fp; int zlo, zu_end;   // what the captured launches baked in (see order_graph)
  };
  std::vector<OrderGraph> graphs;
  cudaStream_t cap_stream = nullptr;   // capture needs a non-legacy stream; replays go to the caller's stream
  cudaEvent_t graph_ev[4] = {nullptr, nullptr, nullptr, nullptr};
  // layer-block sharding over the GPUs of a node (layer_shard.cuh); n <= 1: off
  soslayer::LayerPeers layers;
  double* own_aggD = nullptr;   // the plan's own aggregate tables (d_aggD / d_aggU point into the mailbox while sharded)
  double* own_aggU = nullptr;
  int layer_seg_begin = 0, layer_seg_end = 0x7fffffff;  // segments of the rows whose J this rank needs (own rows + halos)
  // optional per-kernel-class timing with CUDA events (bench.py's roofline leg)
  bool profiling = false;
  std::vector<cudaEvent_t> ev_pool;
  size_t ev_used = 0;
  std::vector<std::pair<int, std::pair<cudaEvent_t, cudaEvent_t>>> ev_spans;  // (class, (start, stop))
};

namespace {

// makes the plan's device current for the duration of an entry point (callers may have another one current)
struct DeviceGuard {
  int prev = -1;
  bool switched = false;
  explicit DeviceGuard(int want) {
    if (cudaGetDevice(&prev) == cudaSuccess && prev != want) switched = cudaSetDevice(want) == cudaSuccess;
  }
  ~DeviceGuard() {
    if (switched) cudaSetDevice(prev);
  }
};
#define SOS_GUARD(p) DeviceGuard _guard((p)->device)

void pool_setup() {
  static bool done[64] = {false};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64 || done[dev]) return;
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
    unsigned long long keep = ~0ULL;  // keep freed blocks cached instead of returning them to the OS
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
  }
  done[dev] = true;
}

// pinned poll buffers are recycled across plans (cudaMallocHost is slow)
std::vector<int*>& pinned_free_list() {
  static std::vector<int*> v;
  return v;
}
constexpr int kPollSlots = 4096;

// ... and so are the staging buffers of the first-order coefficients, by size
std::vector<std::pair<size_t, double*>>& pinned_coef_free_list() {
  static std::vector<std::pair<size_t, double*>> v;
  return v;
}

template <typename T>
int dev_alloc(sos_plan* p, T** out, size_t count) {
  // stream-ordered pool allocation on the legacy default stream: plans are created and destroyed once
  // per batch in the end-to-end path, and cudaMalloc/cudaFree would each cost a device-wide sync
  void* ptr = nullptr;
  pool_setup();
  cudaError_t e = cudaMallocAsync(&ptr, std::max<size_t>(count, 1) * sizeof(T), nullptr);
  if (e != cudaSuccess) {
    g_last_cuda_error = std::string("cudaMallocAsync: ") + cudaGetErrorString(e);
    return SOS_ERR_NOMEM;
  }
  p->allocs.push_back(ptr);
  *out = static_cast<T*>(ptr);
  return SOS_OK;
}

template <typename T>
int dev_upload(sos_plan* p, const T** out, const T* host, size_t count) {
  T* d = nullptr;
  int r = dev_alloc(p, &d, count);
  if (r) return r;
  SOS_CUDA(cudaMemcpy(d, host, count * sizeof(T), cudaMemcpyHostToDevice));
  *out = d;
  return SOS_OK;
}

__global__ void plan_tiles_kernel(sosgemm::GroupTable gt, const int* members, const ScenState* state, int* active_list,
                                  TilePlan* plan, int nseg0, int nseg1, int segs_per_tile, int split_passes) {
  sosgemm::plan_tiles_block(gt, members, state, active_list, plan, nseg0, nseg1, segs_per_tile, split_passes);
}

// End of one scattering order in ONE launch: convergence bookkeeping (SOS_Aer_main_specular.py:309) + the tile plan of the
// next contraction.  Layer-sharded plans first wait here for the peers' halo rows and ratios (layer_shard.cuh), take the two
// ratios that arrived over as their own and advance the exchange epochs.
__global__ void __launch_bounds__(1024)
order_end_kernel(const GridDev g, int order_arg, int* order_counter, sosgemm::GroupTable gt, const int* members, int* active_list,
                 TilePlan* plan, int nseg0, int nseg1, int segs_per_tile, int split_passes, const soslayer::LayerPeers lp) {
  if (lp.n > 1) {
    if (g.state[0].active) {   // (uniform: nobody has touched the state yet)
      const bool late = soslayer::exchange_halos(g, lp);
      if (threadIdx.x == 0) {
        if (late) {  // give up: every later kernel of the solve returns at once; the host sees "nothing active" and the status bit
          atomicOr(&g.state[0].status, SOS_STATUS_PEER_TIMEOUT | SOS_STATUS_NONFINITE);
          g.state[0].active = 0;
        } else {
          const double* ratios_in = lp.box[lp.rank].ratios;
          g.state[0].ratio_toa = *reinterpret_cast<const volatile double*>(ratios_in);
          g.state[0].ratio_surf = *reinterpret_cast<const volatile double*>(ratios_in + 1);
        }
      }
    }
    __syncthreads();
  }
  sossweep::converge_block(g, order_arg, order_counter);
  __syncthreads();
  sosgemm::plan_tiles_block(gt, members, g.state, active_list, plan, nseg0, nseg1, segs_per_tile, split_passes);
}

// zero the aerosol rows of J of every scenario (split class-1 tiles add their two partials into them)
__global__ void zero_rows_kernel(double* J, int ld, int L, int r0, int r1, int N) {
  const int s = blockIdx.z;
  const int t = r0 + blockIdx.y;
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < r1 && m < N) J[(static_cast<size_t>(s) * L + t) * ld + m] = 0.0;
}

// ... of the scenarios that are still iterating only, sixteen bytes per store (the per-order form used with split-k chosen on the device)
__global__ void __launch_bounds__(256) zero_active_rows_kernel(double* J, int ld, int L, int r0, const ScenState* state) {
  const int s = blockIdx.y;
  if (!state[s].active) return;
  double2* row = reinterpret_cast<double2*>(J + (static_cast<size_t>(s) * L + r0 + blockIdx.x) * ld);
  for (int i = threadIdx.x; i < ld / 2; i += 256) row[i] = make_double2(0.0, 0.0);
}

cudaEvent_t prof_event(sos_plan* p) {
  if (p->ev_used == p->ev_pool.size()) {
    cudaEvent_t e;
    cudaEventCreate(&e);
    p->ev_pool.push_back(e);
  }
  return p->ev_pool[p->ev_used++];
}

// NVTX range around a kernel class / a phase of the solve (visible in Nsight Systems / ncu --nvtx)
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

struct ProfSpan {
  sos_plan* p;
  int cls;
  cudaStream_t st;
  cudaEvent_t e0 = nullptr;
  ProfSpan(sos_plan* plan, int c, cudaStream_t s) : p(plan), cls(c), st(s) {
    if (p->profiling) { e0 = prof_event(p); cudaEventRecord(e0, st); }
  }
  ~ProfSpan() {
    if (p->profiling && e0) {
      cudaEvent_t e1 = prof_event(p);
      cudaEventRecord(e1, st);
      p->ev_spans.push_back({cls, {e0, e1}});
    }
  }
};

int launch_check(sos_plan* p, const char* what = "kernel") {
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) {
    // SOS_B200_SYNC_DEBUG=1: wait for every kernel so that an asynchronous fault is reported with the kernel's name
    static const bool sync_debug = [] { const char* v = std::getenv("SOS_B200_SYNC_DEBUG"); return v && v[0] == '1'; }();
    if (sync_debug) e = cudaDeviceSynchronize();
  }
  if (e != cudaSuccess) {
    g_last_cuda_error = std::string(what) + " launch: " + cudaGetErrorString(e);
    return SOS_ERR_CUDA;
  }
  p->launches++;
  return SOS_OK;
}

int plan_tiles(sos_plan* p, cudaStream_t st) {
  const bool pm = p->fold && p->d_members_premix != nullptr;  // fold-mode tables (build_fold_tables)
  plan_tiles_kernel<<<1, 256, 0, st>>>(pm ? p->groups_premix : p->groups, pm ? p->d_members_premix : p->d_members, p->dev.state,
                                       p->d_active_list, p->d_tile_plan, p->nseg[0], p->nseg[1], p->fold ? p->fold_segs : p->gemm_bm / sosgemm::SEG_ROWS,
                                       p->split_passes);
  return launch_check(p);
}

// instantiated order graphs bake in kernel arguments (operand pointers, zone columns, tile shapes): anything that changes
// the plan's tables drops them
void drop_graphs(sos_plan* p) {
  for (auto& g : p->graphs) cudaGraphExecDestroy(g.exec);
  p->graphs.clear();
}

// ---------------------------------------------------------------------------------------------
// generated source (sweep.cuh: SrcGen): plan-side buffers
// ---------------------------------------------------------------------------------------------
// Ross-Li ground: layout of the per-scenario buffer and the view the kernels take of it
size_t brdf_scen_bytes(int S, int M) {
  return static_cast<size_t>(S) * (2 + 2 * (M - 1)) * sizeof(double) + static_cast<size_t>(S) * sizeof(int);
}

sosbrdf::BrdfDev brdf_dev(const sos_plan* p) {
  sosbrdf::BrdfDev b;
  std::memset(&b, 0, sizeof(b));
  if (!p->d_brdf_R) return b;
  const int S = p->dev.S, M = p->dev.M;
  const double* f = reinterpret_cast<const double*>(p->d_brdf_scen);
  b.R = p->d_brdf_R;
  b.f = f;
  b.beam = f + 2 * static_cast<size_t>(S);
  b.set = reinterpret_cast<const int*>(f + static_cast<size_t>(S) * (2 + 2 * (M - 1)));
  b.ldr = p->brdf_ldr;
  return b;
}

// a Ross-Li plan needs its mode matrices and per-scenario data before any first order or sweep
bool brdf_missing(const sos_plan* p) { return p->d_brdf_R && !(p->brdf_sets > 0 && p->brdf_scen_ready); }

int env_int(const char* name, int dflt) {
  const char* e = std::getenv(name);
  return (e && *e) ? std::atoi(e) : dflt;
}

// first downward column of the zone: every column the reference treats specially next to mu = 0-, the extrapolation
// targets and their sources, over all scenarios of the batch
int gen_zone_lo(const GridDev& g, const sos_scenario* scen_h) {
  const int M = g.M;
  int wmax = 0;
  for (int s = 0; s < g.S; ++s)
    for (int k = 0; k < g.nreg; ++k) wmax = std::max(wmax, scen_h[s].extrap_width[k]);
  const int ns = (wmax <= 0) ? 0 : (wmax < 2 ? 2 : std::min(5, wmax));
  return std::max(0, std::min(g.first_small, M - wmax - ns));
}

constexpr int kGenUpZone = 128;  // upward columns next to mu = 0+ whose raw I_n is kept for the find-first blend

int gen_setup(sos_plan* p, const sos_scenario* scen_h) {
  const GridDev& g = p->dev;
  const int L = g.L, M = g.M, N = g.N, S = g.S;
  p->gen_ok = false;
  if (env_int("SOS_B200_GENSRC", 1) == 0) return SOS_OK;
  // one projection slot per warp of the apply pass: two columns per thread on grids with odd M (sweep_apply2_kernel)
  const int T = (M & 1) ? 2 * sossweep::APPLY2_THREADS : sossweep::LOCAL_THREADS;
  const int nslots = ((M - 1 + T - 1) / T + (N - M - 1 + T - 1) / T) * 4;
  int r;
  if ((r = dev_alloc(p, &p->d_proj, static_cast<size_t>(S) * L * nslots * 2))) return r;
  for (int i = 0; i < 2; ++i)
    if ((r = dev_alloc(p, &p->d_cj[i], static_cast<size_t>(S) * L * 2))) return r;
  SOS_CUDA(cudaMemset(p->d_proj, 0, sizeof(double) * S * L * nslots * 2));
  for (int i = 0; i < 2; ++i) SOS_CUDA(cudaMemset(p->d_cj[i], 0, sizeof(double) * S * L * 2));
  p->gen_nslots = nslots;
  p->gen_zu_end = std::min(M + 1 + kGenUpZone, N);
  p->gen_zlo = gen_zone_lo(g, scen_h);
  p->gen_ok = true;
  return SOS_OK;
}

// aerosol rows with a vanishing second coefficient: split the first one in two equal halves on the same operand
// (exact in binary floating point) so that every class-1 tile runs two passes
void patch_scenarios(const sos_grid& grid, std::vector<sos_scenario>& sc) {
  if (grid.n_regions != 3) return;
  for (auto& x : sc) {
    if (x.coef_mix_aer == 0.0) {
      x.phase_aer = x.phase_atm;
      x.coef_mix_atm *= 0.5;
      x.coef_mix_aer = x.coef_mix_atm;
    }
  }
}

// operand groups of the source contraction: class 1 (aerosol rows, two operands) first, then class 0
int build_groups(sos_plan* p, const std::vector<sos_scenario>& sc, std::vector<int>& flat) {
  const int S = static_cast<int>(sc.size());
  std::vector<std::vector<int>> members;
  std::memset(&p->groups, 0, sizeof(p->groups));
  auto add_groups = [&](int cls) -> int {
    std::map<std::pair<int, int>, int> index;
    for (int s = 0; s < S; ++s) {
      const std::pair<int, int> key = cls == 1 ? std::make_pair(sc[s].phase_atm, sc[s].phase_aer) : std::make_pair(sc[s].phase_atm, -1);
      auto it = index.find(key);
      if (it == index.end()) {
        if (p->groups.n_groups >= SOS_MAX_GROUPS) return SOS_ERR_UNSUPPORTED;
        const int g = p->groups.n_groups++;
        p->groups.cls[g] = cls;
        p->groups.phaseA[g] = key.first;
        p->groups.phaseB[g] = cls == 1 ? key.second : key.first;
        members.emplace_back();
        it = index.emplace(key, g).first;
      }
      members[it->second].push_back(s);
    }
    return SOS_OK;
  };
  int r;
  if (p->grid.n_regions == 3 && (r = add_groups(1))) return r;
  if ((r = add_groups(0))) return r;
  flat.clear();
  for (int g = 0; g < p->groups.n_groups; ++g) {
    p->groups.member_off[g] = static_cast<int>(flat.size());
    flat.insert(flat.end(), members[g].begin(), members[g].end());
  }
  p->groups.member_off[p->groups.n_groups] = static_cast<int>(flat.size());
  return SOS_OK;
}

int validate_scenarios(const sos_grid& grid, const sos_scenario* scen_h) {
  const int M = grid.nb_angles;
  int widx[4], wns[4], woff[4];
  sos_extrap_layout(M, widx, wns, woff);
  for (int s = 0; s < grid.n_scenarios; ++s) {
    for (int k = 0; k < grid.n_regions; ++k) {
      const int w = scen_h[s].extrap_width[k];
      if (w != widx[0] && w != widx[1] && w != widx[2] && w != widx[3]) return SOS_ERR_INVALID;
      if (w + 5 > M - 1) return SOS_ERR_INVALID;
    }
    if (scen_h[s].phase_atm < 0 || scen_h[s].phase_atm >= SOS_MAX_PHASE || scen_h[s].phase_aer < 0 || scen_h[s].phase_aer >= SOS_MAX_PHASE)
      return SOS_ERR_INVALID;
  }
  return SOS_OK;
}

}  // namespace

extern "C" {

static bool gen_applies(const sos_plan* p);
static bool gen_usable(const sos_plan* p);

int sos_abi_version(void) { return SOS_ABI_VERSION; }

const char* sos_strerror(int err) {
  switch (err) {
    case SOS_OK: return "ok";
    case SOS_ERR_INVALID: return "invalid argument";
    case SOS_ERR_CUDA: return "CUDA call failed";
    case SOS_ERR_NOMEM: return "out of device memory";
    case SOS_ERR_UNSUPPORTED: return "unsupported device or configuration";
    case SOS_ERR_STATE: return "call order violated";
    case SOS_ERR_RETRY: return "solve must be repeated: the plan switched to its general kernels";
    default: return "unknown error";
  }
}

const char* sos_last_cuda_error(void) { return g_last_cuda_error.c_str(); }

int sos_extrap_layout(int nb_angles, int* idx, int* ns, int* off) {
  const double f[4] = {0.005, 0.02, 0.04, 0.06};
  int total = 0;
  for (int c = 0; c < 4; ++c) {
    const int w = static_cast<int>(f[c] * nb_angles);
    idx[c] = w;
    ns[c] = (w <= 0) ? 0 : (w < 2 ? 2 : std::min(5, w));
    off[c] = total;
    total += idx[c] * ns[c];
  }
  return total;
}

int sos_plan_create(sos_plan** out, const sos_grid* grid, const double* mu_h, const double* tau_h,
                    const sos_scenario* scen_h, const double* extrap_W_h, int extrap_W_len) {
  if (!out || !grid || !mu_h || !tau_h || !scen_h) return SOS_ERR_INVALID;
  const int L = grid->nb_layers, M = grid->nb_angles, S = grid->n_scenarios, N = 2 * M;
  if (L < 2 || M < 4 || S < 1) return SOS_ERR_INVALID;
  if (grid->n_regions != 1 && grid->n_regions != 3) return SOS_ERR_INVALID;
  if (grid->ld < N || (grid->ld & 1)) return SOS_ERR_INVALID;
  if (grid->region_start[0] != 0 || grid->region_start[grid->n_regions] != L) return SOS_ERR_INVALID;
  for (int k = 0; k < grid->n_regions; ++k)
    if (grid->region_start[k + 1] <= grid->region_start[k]) return SOS_ERR_INVALID;
  if (grid->n_regions == 3 && (grid->region_start[1] < 2 || grid->region_start[2] < grid->region_start[1] + 1))
    return SOS_ERR_INVALID;
  if (grid->surface < 0 || grid->surface > 6) return SOS_ERR_INVALID;
  if ((grid->surface == SOS_SURFACE_LAMBERT_DIFFUSE || grid->surface == SOS_SURFACE_ROSSLI || grid->surface == SOS_SURFACE_OCEAN) &&
      grid->n_regions != 3)
    return SOS_ERR_UNSUPPORTED;

  int dev = 0;
  SOS_CUDA(cudaGetDevice(&dev));
  // (cudaGetDeviceProperties costs milliseconds; two attribute queries do)
  int cc_major = 0, cc_minor = 0, n_sms = 0;
  SOS_CUDA(cudaDeviceGetAttribute(&cc_major, cudaDevAttrComputeCapabilityMajor, dev));
  SOS_CUDA(cudaDeviceGetAttribute(&cc_minor, cudaDevAttrComputeCapabilityMinor, dev));
  SOS_CUDA(cudaDeviceGetAttribute(&n_sms, cudaDevAttrMultiProcessorCount, dev));
  if (cc_major != 10) {
    g_last_cuda_error = "libsos_b200 is built for sm_100a only; device is sm_" + std::to_string(cc_major) +
                        std::to_string(cc_minor);
    return SOS_ERR_UNSUPPORTED;
  }

  sos_plan* p = new (std::nothrow) sos_plan();
  if (!p) return SOS_ERR_NOMEM;
  p->grid = *grid;
  p->device = dev;
  p->N = N;
  p->n_sms = n_sms;
  p->launches = 0;
  p->scen_h.assign(scen_h, scen_h + S);
  p->mu_h.assign(mu_h, mu_h + N);
  std::memset(&p->gp, 0, sizeof(p->gp));
  std::memset(&p->fp, 0, sizeof(p->fp));

  int widx[4], wns[4], woff[4];
  const int wlen = sos_extrap_layout(M, widx, wns, woff);
  if (wlen != extrap_W_len || (wlen > 0 && !extrap_W_h)) { delete p; return SOS_ERR_INVALID; }
  for (int s = 0; s < S; ++s) {
    for (int k = 0; k < grid->n_regions; ++k) {
      const int w = scen_h[s].extrap_width[k];
      if (w != widx[0] && w != widx[1] && w != widx[2] && w != widx[3]) { delete p; return SOS_ERR_INVALID; }
      if (w + 5 > M - 1) { delete p; return SOS_ERR_INVALID; }
    }
    if (scen_h[s].phase_atm < 0 || scen_h[s].phase_atm >= SOS_MAX_PHASE || scen_h[s].phase_aer < 0 ||
        scen_h[s].phase_aer >= SOS_MAX_PHASE) { delete p; return SOS_ERR_INVALID; }
  }

  // ---- chunks: never straddle a region ----
  int chunk = grid->chunk_rows;
  if (chunk <= 0) chunk = env_int("SOS_B200_CHUNK_ROWS", 0);  // (experiments; 0 = choose)
  if (chunk <= 0) {
    // enough (scenario x chunk x column) threads to fill the chip
    const long long want = 4LL * p->n_sms * 2048;
    long long c = static_cast<long long>(S) * L * N / want;
    // measured in round 1 (sweep over chunk_rows with tools/bench_kernels.py): 48-row chunks are the sweet spot for small batches -- shorter chunks
    // lengthen the serial carry chain more than they help the two scan passes
    chunk = static_cast<int>(std::max<long long>(48, std::min<long long>(128, c)));
    if (grid->n_regions == 1 && grid->surface == SOS_SURFACE_NONE) {
      // the carry chain is a two-level scan per column (sweep_carry_cols_kernel): short chunks cost nothing there, and one grid
      // alone (or a layer block of it) is latency bound in the scan passes -- 24-row chunks (10 000 x 1024: the same 49 ms on one
      // GPU as with 48, 12 us less per order on a layer block of 1 250 rows)
      chunk = static_cast<int>(std::max<long long>(24, std::min<long long>(128, c)));
      chunk = std::max(chunk, (L + 1023) / 1024);
    } else {
      chunk = std::max(chunk, (L + 47) / 48);  // keep the serial carry chain short
    }
  }
  std::vector<int> cstart, cregion, rowchunk(L);
  for (int k = 0; k < grid->n_regions; ++k) {
    const int r0 = grid->region_start[k], r1 = grid->region_start[k + 1];
    const int len = r1 - r0;
    const int nck = (len + chunk - 1) / chunk;
    for (int i = 0; i < nck; ++i) {
      // balanced split, chunk lengths in whole groups of four rows (the scan passes run four rows per step: only the
      // chunk that ends its region is left with a remainder for the row-by-row tail)
      const int a = r0 + static_cast<int>(static_cast<long long>(len) * i / nck) / 4 * 4;
      cstart.push_back(a);
      cregion.push_back(k);
    }
  }
  cstart.push_back(L);
  const int nch = static_cast<int>(cregion.size());
  cregion.push_back(grid->n_regions);  // sentinel: chunk_region[nchunks] differs from the last region
  for (int c = 0; c < nch; ++c)
    for (int t = cstart[c]; t < cstart[c + 1]; ++t) rowchunk[t] = c;

  // ---- mu-grid constants ----
  std::vector<double> w(N, 0.0);
  for (int k = 0; k + 1 < N; ++k) {
    const double d = mu_h[k + 1] - mu_h[k];
    w[k] += d / 2;
    w[k + 1] += d / 2;
  }
  int first_small = M - 1;
  for (int m = 0; m < M - 1; ++m)
    if (std::fabs(mu_h[m]) < SOS_MU_THRESHOLD) { first_small = m; break; }
  // the standard/small split must be a prefix/suffix split (|mu| decreasing on the downward half)
  for (int m = first_small; m < M - 1; ++m)
    if (!(std::fabs(mu_h[m]) < SOS_MU_THRESHOLD)) { delete p; return SOS_ERR_INVALID; }

  GridDev& d = p->dev;
  std::memset(&d, 0, sizeof(d));
  d.L = L; d.M = M; d.N = N; d.S = S; d.ld = grid->ld;
  d.nreg = grid->n_regions;
  for (int k = 0; k < 4; ++k) d.rstart[k] = grid->region_start[k];
  d.surface = grid->surface;
  d.nchunks = nch;
  d.first_small = first_small;
  d.col0 = 0;
  d.col1 = N;
  d.row0 = 0;
  d.row1 = L;
  d.c_lo = 0;
  d.c_hi = nch;
  std::memset(&p->layers, 0, sizeof(p->layers));
  for (int c = 0; c < 4; ++c) { d.widx[c] = widx[c]; d.wns[c] = wns[c]; d.woff[c] = woff[c]; }

  int r = SOS_OK;
#define TRY(x) do { r = (x); if (r) { sos_plan_destroy(p); return r; } } while (0)
  TRY(dev_upload(p, &d.chunk_start, cstart.data(), cstart.size()));
  TRY(dev_upload(p, &d.chunk_region, cregion.data(), cregion.size()));
  TRY(dev_upload(p, &d.row_chunk, rowchunk.data(), rowchunk.size()));
  TRY(dev_upload(p, &d.mu, mu_h, static_cast<size_t>(N)));
  TRY(dev_upload(p, &d.wmu, w.data(), static_cast<size_t>(N)));
  TRY(dev_upload(p, &d.tau, tau_h, static_cast<size_t>(S) * L));
  TRY(dev_upload(p, &d.scen, scen_h, static_cast<size_t>(S)));
  {
    std::vector<double> Wtmp(std::max(wlen, 1), 0.0);
    if (wlen > 0) std::memcpy(Wtmp.data(), extrap_W_h, sizeof(double) * wlen);
    TRY(dev_upload(p, &d.W, Wtmp.data(), Wtmp.size()));
  }
  {
    std::vector<ScenState> st(S);
    for (int s = 0; s < S; ++s) { st[s].ratio_toa = 1; st[s].ratio_surf = 1; st[s].n_orders = 1; st[s].active = 1; st[s].status = 0; st[s].pad = 0; }
    const ScenState* tmp = nullptr;
    TRY(dev_upload(p, &tmp, st.data(), st.size()));
    d.state = const_cast<ScenState*>(tmp);
  }
  TRY(dev_alloc(p, &d.n_active, 1));
  TRY(dev_alloc(p, &d.active_flat, static_cast<size_t>(S)));
  {
    std::vector<int> ids(S);
    for (int s = 0; s < S; ++s) ids[s] = s;
    if (cudaMemcpy(d.active_flat, ids.data(), sizeof(int) * S, cudaMemcpyHostToDevice) != cudaSuccess) { sos_plan_destroy(p); return SOS_ERR_CUDA; }
  }
  {
    cudaError_t e = cudaMemcpy(d.n_active, &S, sizeof(int), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { sos_plan_destroy(p); return SOS_ERR_CUDA; }
  }
  const size_t nagg = static_cast<size_t>(S) * nch * N;
  TRY(dev_alloc(p, &p->d_aggD, nagg));
  TRY(dev_alloc(p, &p->d_aggU, nagg));
  p->own_aggD = p->d_aggD;
  p->own_aggU = p->d_aggU;
  TRY(dev_alloc(p, &p->d_carryD, nagg));
  TRY(dev_alloc(p, &p->d_carryU, nagg));
  TRY(dev_alloc(p, &p->d_C, static_cast<size_t>(S) * 2 * N));
  TRY(dev_alloc(p, &p->d_sums, static_cast<size_t>(S) * L * 3));
  TRY(dev_alloc(p, &p->d_z, static_cast<size_t>(L)));
  TRY(dev_alloc(p, &p->d_colint, static_cast<size_t>(N)));
  if (grid->surface == SOS_SURFACE_LAMBERT_DIFFUSE) TRY(dev_alloc(p, &p->d_bs, static_cast<size_t>(S)));
  if (grid->surface == SOS_SURFACE_ROSSLI || grid->surface == SOS_SURFACE_OCEAN) {
    p->brdf_nk = (grid->surface == SOS_SURFACE_ROSSLI) ? 2 : 1;
    TRY(dev_alloc(p, &p->d_bs, static_cast<size_t>(S) * (M - 1)));
    TRY(dev_alloc(p, &p->d_brdf_R, static_cast<size_t>(2) * sosbrdf::MAX_SETS));
    TRY(dev_alloc(p, &p->d_brdf_scen, brdf_scen_bytes(S, M)));
  }
  {
    cudaError_t e = cudaMemset(p->d_carryD, 0, nagg * sizeof(double));
    if (e == cudaSuccess) e = cudaMemset(p->d_carryU, 0, nagg * sizeof(double));
    if (e == cudaSuccess) {
      auto& fl = pinned_free_list();
      if (!fl.empty()) { p->h_poll = fl.back(); fl.pop_back(); }
      else e = cudaMallocHost(reinterpret_cast<void**>(&p->h_poll), (kPollSlots + 1) * sizeof(int));  // (+1: the order graph's slot)
    }
    if (e != cudaSuccess) { g_last_cuda_error = cudaGetErrorString(e); sos_plan_destroy(p); return SOS_ERR_CUDA; }
  }

  // ---- source contraction: operand groups, 8-row segments, device tile plan ----
  {
    std::vector<sos_scenario> patched(scen_h, scen_h + S);
    patch_scenarios(*grid, patched);
    if (grid->n_regions == 3) {
      if (cudaMemcpy(const_cast<sos_scenario*>(d.scen), patched.data(), sizeof(sos_scenario) * S, cudaMemcpyHostToDevice) != cudaSuccess) {
        g_last_cuda_error = "cudaMemcpy(scenarios) failed";
        sos_plan_destroy(p);
        return SOS_ERR_CUDA;
      }
      p->scen_h = patched;
    }
    std::vector<int> flat;
    TRY(build_groups(p, patched, flat));
    // segments: regions cut into 8-row pieces; class 1 = aerosol region, class 0 = the rest
    std::vector<int> srow[2], sval[2];
    for (int k = 0; k < grid->n_regions; ++k) {
      const int cls = (grid->n_regions == 3 && k == 1) ? 1 : 0;
      for (int r = grid->region_start[k]; r < grid->region_start[k + 1]; r += sosgemm::SEG_ROWS) {
        srow[cls].push_back(r);
        sval[cls].push_back(std::min(sosgemm::SEG_ROWS, grid->region_start[k + 1] - r));
      }
    }
    for (int c = 0; c < 2; ++c) {
      if (srow[c].empty()) { srow[c].push_back(0); sval[c].push_back(0); p->nseg[c] = 0; }
      else p->nseg[c] = static_cast<int>(srow[c].size());
      TRY(dev_upload(p, &p->gp.seg_row[c], srow[c].data(), srow[c].size()));
      TRY(dev_upload(p, &p->gp.seg_valid[c], sval[c].data(), sval[c].size()));
      p->gp.nseg[c] = std::max(p->nseg[c], 1);
    }
    const int* tmpi = nullptr;
    TRY(dev_upload(p, &tmpi, flat.data(), flat.size()));
    p->d_members = const_cast<int*>(tmpi);
    p->members_h = flat;
    TRY(dev_alloc(p, &p->d_active_list, flat.size()));
    TRY(dev_alloc(p, &p->d_tile_plan, 1));
    TRY(dev_alloc(p, &p->d_work_counter, 1));
    TRY(dev_alloc(p, &p->d_order, 1));
    TRY(dev_alloc(p, &p->d_fold_stats, 2));
    TRY(dev_alloc(p, &p->d_lr_stats, 3));
    {
      const int one = 1;
      if (cudaMemcpy(p->d_order, &one, sizeof(int), cudaMemcpyHostToDevice) != cudaSuccess) {
        g_last_cuda_error = "cudaMemcpy(order counter) failed";
        sos_plan_destroy(p);
        return SOS_ERR_CUDA;
      }
    }
    p->gemm_bm = sosgemm::Cfg<2, 4, 4, 4>::BM;
    {
      // 128 x 144 tiles (12 consumer warps of 32 x 48) when 144 pads N less than 128 (N = 1002: 1008 vs 1024
      // issued columns) and the batch still gives every SM several tiles
      const long long pad128 = (N + 127) / 128 * 128, pad144 = (N + 143) / 144 * 144;
      const long long segs_all = static_cast<long long>(S) * (p->nseg[0] + p->nseg[1]);
      const long long tiles144 = (segs_all + 15) / 16 * ((N + 143) / 144);
      if (pad144 < pad128 && tiles144 >= 8LL * p->n_sms) {
        p->gemm_bm = sosgemm::Cfg<4, 3, 4, 6>::BM;
        p->gemm_bn = sosgemm::Cfg<4, 3, 4, 6>::BN;
      }
    }
    {
      // few tiles: the two-pass aerosol tiles are the critical path of the launch -> split them
      const long long segs = static_cast<long long>(S) * (p->nseg[0] + p->nseg[1]);
      const long long tiles = (segs + 7) / 8 * ((N + 127) / 128);  // (small batches always use 64 x 128 tiles)
      p->split_passes = (grid->n_regions == 3 && tiles < 2LL * p->n_sms) ? 1 : 0;
      p->split_general = p->split_passes;
    }
  }
#undef TRY
  // opt in to the large dynamic shared memory of the kernels used
  cudaFuncSetAttribute(sosgemm::jn_gemm_dmma_kernel<2, 4, 4, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, sosgemm::Cfg<2, 4, 4, 4>::SMEM);
  cudaFuncSetAttribute(sosgemm::jn_gemm_dmma_kernel<4, 3, 4, 6>, cudaFuncAttributeMaxDynamicSharedMemorySize, sosgemm::Cfg<4, 3, 4, 6>::SMEM);
  {
    int r2 = plan_tiles(p, nullptr);  // all scenarios active
    if (r2) { sos_plan_destroy(p); return r2; }
    cudaDeviceSynchronize();
  }
  if (p->d_bs && (M + 32) * sizeof(double) > 48 * 1024) {
    cudaFuncSetAttribute(sosfirst::first_order_surface_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (M + 32) * sizeof(double));
    cudaFuncSetAttribute(sosfirst::first_order_surface_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (M + 32) * sizeof(double));
    cudaFuncSetAttribute(sosfirst::first_order_surface_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (M + 32) * sizeof(double));
  }
  if ((N + 32 + 2 * (nch + 1)) * sizeof(double) > 48 * 1024) {
    cudaFuncSetAttribute(sossweep::sweep_carry_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (N + 32 + 2 * (nch + 1)) * sizeof(double));
    cudaFuncSetAttribute(sossweep::sweep_carry_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (N + 32 + 2 * (nch + 1)) * sizeof(double));
    cudaFuncSetAttribute(sossweep::sweep_carry_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (N + 32 + 2 * (nch + 1)) * sizeof(double));
  }
  {
    int r3 = gen_setup(p, p->scen_h.data());
    if (r3) { sos_plan_destroy(p); return r3; }
  }
  *out = p;
  return SOS_OK;
}

static int refresh_fold_plan(sos_plan* p);
static int premix_folded(sos_plan* p);

int sos_plan_update(sos_plan* p, const double* tau_h, const sos_scenario* scen_h, void* stream) {
  if (!p || !tau_h || !scen_h) return SOS_ERR_INVALID;
  SOS_GUARD(p);
  const GridDev& g = p->dev;
  const int S = g.S, L = g.L;
  if (g.col0 != 0 || g.col1 != g.N) return SOS_ERR_UNSUPPORTED;   // column-sharded plans are created per block
  if (p->layers.n > 1) return SOS_ERR_UNSUPPORTED;                 // layer blocks and their halos were laid out for the old tau: set the layers again afterwards
  int r = validate_scenarios(p->grid, scen_h);
  if (r) return r;
  const int n_phase = static_cast<int>(p->A_ptrs.size());
  for (int s = 0; s < S; ++s)
    if (p->maps_A_ready && (scen_h[s].phase_atm >= n_phase || scen_h[s].phase_aer >= n_phase)) return SOS_ERR_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  SOS_CUDA(cudaStreamSynchronize(st));  // nothing of the previous batch may still be reading the tables rewritten below
  std::vector<sos_scenario> patched(scen_h, scen_h + S);
  patch_scenarios(p->grid, patched);
  p->scen_h = patched;
  SOS_CUDA(cudaMemcpyAsync(const_cast<double*>(g.tau), tau_h, sizeof(double) * S * L, cudaMemcpyHostToDevice, st));
  SOS_CUDA(cudaMemcpyAsync(const_cast<sos_scenario*>(g.scen), patched.data(), sizeof(sos_scenario) * S, cudaMemcpyHostToDevice, st));
  std::vector<int> flat;
  if ((r = build_groups(p, patched, flat))) return r;
  if (flat.size() != p->members_h.size()) return SOS_ERR_STATE;
  p->members_h = flat;
  SOS_CUDA(cudaMemcpyAsync(p->d_members, flat.data(), flat.size() * sizeof(int), cudaMemcpyHostToDevice, st));
  std::vector<ScenState> state(S);
  for (int s = 0; s < S; ++s) { state[s].ratio_toa = 1; state[s].ratio_surf = 1; state[s].n_orders = 1; state[s].active = 1; state[s].status = 0; state[s].pad = 0; }
  SOS_CUDA(cudaMemcpyAsync(g.state, state.data(), sizeof(ScenState) * S, cudaMemcpyHostToDevice, st));
  if (p->gen_ok) {
    p->gen_zlo = gen_zone_lo(g, patched.data());
    p->gen_disabled = false;  // a new batch gets the generated source again
  }
  SOS_CUDA(cudaStreamSynchronize(st));  // the host vectors above go out of scope
  sossweep::count_active_kernel<<<1, 256, 0, st>>>(p->dev);
  if ((r = launch_check(p, "count_active_kernel"))) return r;
  if (p->fold) {
    if (p->premix && (r = premix_folded(p))) return r;
    return refresh_fold_plan(p);
  }
  r = plan_tiles(p, st);
  if (r) return r;
  SOS_CUDA(cudaStreamSynchronize(st));
  return SOS_OK;
}

int sos_plan_destroy(sos_plan* p) {
  if (!p) return SOS_OK;
  SOS_GUARD(p);  // the sync and the stream-ordered frees below must run on the plan's own device
  for (cudaEvent_t e : p->ev_pool) cudaEventDestroy(e);
  cudaDeviceSynchronize();  // nothing of this plan may still be running on any stream
  drop_graphs(p);
  for (int k = 0; k < 2; ++k) {
    if (p->h_C[k]) {
      auto& fl = pinned_coef_free_list();
      if (fl.size() < 8) fl.push_back({sizeof(double) * p->dev.S * 2 * p->dev.N, p->h_C[k]});
      else cudaFreeHost(p->h_C[k]);
    }
    if (p->h_C_ev[k]) cudaEventDestroy(p->h_C_ev[k]);
  }
  for (cudaEvent_t& e : p->graph_ev) if (e) cudaEventDestroy(e);
  if (p->cap_stream) cudaStreamDestroy(p->cap_stream);
  for (void* a : p->allocs) cudaFreeAsync(a, nullptr);
  if (p->h_poll) pinned_free_list().push_back(p->h_poll);
  delete p;
  return SOS_OK;
}

long long sos_launch_count(const sos_plan* p) { return p ? p->launches : 0; }

int sos_plan_query(const sos_plan* p, int what) {
  if (!p) return SOS_ERR_INVALID;
  switch (what) {
    case SOS_QUERY_FUSED_ORDER: return gen_usable(p) ? 1 : 0;
    case SOS_QUERY_GENERATED_SOURCE: return (gen_usable(p) && gen_applies(p)) ? 1 : 0;
    case SOS_QUERY_FOLDED: return p->fold ? 1 : 0;
    case SOS_QUERY_DEVICE: return p->device;
    default: return SOS_ERR_INVALID;
  }
}

int sos_plan_set_columns(sos_plan* p, int col0, int col1) {
  if (!p) return SOS_ERR_INVALID;
  SOS_GUARD(p);
  drop_graphs(p);
  GridDev& g = p->dev;
  if (col0 < 0 || col1 > g.N || col0 >= col1) return SOS_ERR_INVALID;
  if (col0 == 0 && col1 == g.N) { g.col0 = 0; g.col1 = g.N; return SOS_OK; }
  // mu-block sharding: only grids without a surface coupling (the coupling mixes mirror columns)
  if (g.surface != SOS_SURFACE_NONE || g.nreg != 1) return SOS_ERR_UNSUPPORTED;
  if (p->gemm_bn != 128) return SOS_ERR_UNSUPPORTED;  // sharded plans are single-scenario: always 128-column tiles
  if ((col0 % 128) != 0 || (col1 != g.N && (col1 % 128) != 0)) return SOS_ERR_INVALID;
  // the mu -> 0 zones must not straddle a block boundary
  int wmax = 0;
  for (const sos_scenario& sc : p->scen_h) wmax = std::max(wmax, sc.extrap_width[0]);
  const int zlo = std::min(g.first_small, g.M - wmax - 5);
  const bool cuts_down = (col0 > zlo && col0 < g.M) || (col1 > zlo && col1 < g.M);
  const bool cuts_up = (col0 == g.M + 1) || (col1 == g.M + 1);
  if (cuts_down || cuts_up) return SOS_ERR_UNSUPPORTED;
  g.col0 = col0;
  g.col1 = col1;
  return SOS_OK;
}

int sos_layer_mailbox_bytes(const sos_plan* p, size_t* bytes) {
  if (!p || !bytes) return SOS_ERR_INVALID;
  *bytes = soslayer::mailbox_layout(nullptr, p->dev.nchunks, p->dev.N, nullptr);
  return SOS_OK;
}

int sos_plan_set_layers(sos_plan* p, int rank, int n_ranks, void* const* mailbox_peers_d, double* const* In_peers_d, int* row0_out,
                        int* row1_out) {
  if (!p) return SOS_ERR_INVALID;
  SOS_GUARD(p);
  drop_graphs(p);
  GridDev& g = p->dev;
  if (n_ranks <= 1) {  // back to the whole grid
    std::memset(&p->layers, 0, sizeof(p->layers));
    p->d_aggD = p->own_aggD;
    p->d_aggU = p->own_aggU;
    g.row0 = 0; g.row1 = g.L; g.c_lo = 0; g.c_hi = g.nchunks;
    p->layer_seg_begin = 0; p->layer_seg_end = 0x7fffffff;
    if (row0_out) *row0_out = 0;
    if (row1_out) *row1_out = g.L;
    return SOS_OK;
  }
  if (!mailbox_peers_d || !In_peers_d || rank < 0 || rank >= n_ranks || n_ranks > SOS_MAX_PEERS) return SOS_ERR_INVALID;
  // one scenario, one region, no surface coupling (the single-layer operator of SOS_Aer_I1_In.py:77-130), all columns
  if (g.S != 1 || g.nreg != 1 || g.surface != SOS_SURFACE_NONE || g.col0 != 0 || g.col1 != g.N) return SOS_ERR_UNSUPPORTED;
  if (g.nchunks < n_ranks || (g.N + soslayer::COL_GROUP - 1) / soslayer::COL_GROUP > soslayer::MAX_GROUPS) return SOS_ERR_UNSUPPORTED;
  for (int r = 0; r < n_ranks; ++r)
    if (!mailbox_peers_d[r] || !In_peers_d[r] || (reinterpret_cast<uintptr_t>(mailbox_peers_d[r]) & 127)) return SOS_ERR_INVALID;
  std::vector<int> cstart(g.nchunks + 1);
  std::vector<double> tau(g.L);
  SOS_CUDA(cudaMemcpy(cstart.data(), g.chunk_start, sizeof(int) * (g.nchunks + 1), cudaMemcpyDeviceToHost));
  SOS_CUDA(cudaMemcpy(tau.data(), g.tau, sizeof(double) * g.L, cudaMemcpyDeviceToHost));
  auto first_chunk = [&](int r) { return static_cast<int>(static_cast<long long>(g.nchunks) * r / n_ranks); };
  // rows above `a` whose J the sweeps of the block starting at `a` read: the previous row (first trapezoid of the downward
  // recurrence, Taylor slope of the |mu| < 0.001 columns) and the window tau' >= tau - 5 |mu|, |mu| < 0.01, of
  // SOS_Aer_In_limit.py:96-107
  auto halo_above = [&](int a) {
    if (a == 0) return 0;
    int h = 1;
    while (a - h > 0 && tau[a - h] >= tau[a] - 5.0 * SOS_MU_THRESHOLD) ++h;
    return std::min(a, h + 1);
  };
  soslayer::LayerPeers& lp = p->layers;
  std::memset(&lp, 0, sizeof(lp));
  lp.rank = rank;
  lp.n = n_ranks;
  // (SOS_B200_PEER_TIMEOUT_MS=0: never wait -- one rank profiled alone, its results are meaningless)
  lp.timeout_ns = static_cast<unsigned long long>(std::max(0, env_int("SOS_B200_PEER_TIMEOUT_MS", 4000))) * 1000000ull;
  for (int r = 0; r < n_ranks; ++r) {
    soslayer::mailbox_layout(mailbox_peers_d[r], g.nchunks, g.N, &lp.box[r]);
    lp.In[r] = In_peers_d[r];
  }
  g.c_lo = first_chunk(rank);
  g.c_hi = first_chunk(rank + 1);
  g.row0 = cstart[g.c_lo];
  g.row1 = cstart[g.c_hi];
  lp.halo_above = halo_above(g.row0);
  lp.next_halo_above = rank + 1 < n_ranks ? halo_above(g.row1) : 0;
  // the chunk-local pass writes, and the carry chain reads, the aggregate tables inside the mailbox (peers write theirs there)
  p->d_aggD = lp.box[rank].aggD;
  p->d_aggU = lp.box[rank].aggU;
  // J is needed on the rows [row0 - halo, row1] (the upward recurrence reads one row below the block); whole 64-row tiles
  const int tile_segs = p->gemm_bm / sosgemm::SEG_ROWS;
  p->layer_seg_begin = (g.row0 - lp.halo_above) / sosgemm::SEG_ROWS / tile_segs * tile_segs;
  p->layer_seg_end = (std::min(g.L, g.row1 + 1) + sosgemm::SEG_ROWS - 1) / sosgemm::SEG_ROWS;
  if (row0_out) *row0_out = g.row0;
  if (row1_out) *row1_out = g.row1;
  return SOS_OK;
}

int sos_state_ratios(sos_plan* p, double* buf_d, int set, void* stream) {
  if (!p || !buf_d) return SOS_ERR_INVALID;
  SOS_GUARD(p);
  sossweep::ratios_kernel<<<(p->dev.S + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(p->dev, buf_d, set);
  return launch_check(p);
}

int sos_set_profiling(sos_plan* p, int enabled) {
  if (!p) return SOS_ERR_INVALID;
  SOS_GUARD(p);
  drop_graphs(p);
  p->profiling = enabled != 0;
  return SOS_OK;
}

int sos_get_profile(sos_plan* p, double* ms, long long* spans, void* stream) {
  if (!p || !ms || !spans) return SOS_ERR_INVALID;
  SOS_GUARD(p);
  SOS_CUDA(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
  for (int i = 0; i < SOS_PROFILE_CLASSES; ++i) { ms[i] = 0.0; spans[i] = 0; }
  for (auto& sp : p->ev_spans) {
    float t = 0.f;
    SOS_CUDA(cudaEventElapsedTime(&t, sp.second.first, sp.second.second));
    if (sp.first < 0 || sp.first >= SOS_PROFILE_CLASSES) continue;
    ms[sp.first] += t;
    spans[sp.first] += 1;
  }
  p->ev_spans.clear();
  p->ev_used = 0;
  return SOS_OK;
}

int sos_build_contraction(sos_plan* p, const double* P_d, int ldp, double* A_d, int lda, void* stream) {
  if (!p || !P_d || !A_d || ldp < p->N || lda < p->N) return SOS_ERR_INVALID;
  SOS_GUARD(p);
  const int N = p->N;
  dim3 grid((N + 31) / 32, (N + 31) / 32);
  sosquad::build_contraction_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(P_d, ldp, A_d, lda, N, p->dev.wmu);
  return launch_check(p);
}

int sos_build_phase(sos_plan* p, int family, double g, double mu0, const double* phi_h, const double* cphi_h,
                    const double* tab_x_d, const double* tab_y_d, int tab_n, double* P_d, int ldp, double* P0_d,
                    void* stream) {
  if (!p || !phi_h || !cphi_h || (!P_d && !P0_d)) return SOS_ERR_INVALID;
  SOS_GUARD(p);
  if (family < 0 || family > 2 || (family == 2 && (!tab_x_d || !tab_y_d || tab_n < 2))) return SOS_ERR_INVALID;
  if (P_d && ldp < p->N) return SOS_ERR_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  sosphase::PhaseArgs a;
  a.family = family; a.g = g; a.tab_x = tab_x_d; a.tab_y = tab_y_d; a.tab_n = tab_n;
  for (int k = 0; k < sosphase::NPHI; ++k) { a.phi[k] = phi_h[k]; a.cphi[k] = cphi_h[k]; }
  const int N = p->N;
  if (P_d) {
    dim3 grid((N + 31) / 32, (N + 7) / 8);
    sosphase::phase_raw_kernel<<<grid, 256, 0, st>>>(a, p->dev.mu, N, P_d, ldp);
    int r = launch_check(p);
    if (r) return r;
    double* colint = p->d_colint;
    sosphase::phase_colint_kernel<<<(N + 127) / 128, 128, 0, st>>>(p->dev.mu, N, P_d, ldp, colint);
    r = launch_check(p);
    if (r) return r;
    sosphase::phase_normalise_kernel<<<grid, 256, 0, st>>>(N, P_d, ldp, colint);
    r = launch_check(p);
    if (r) return r;
  }
  if (P0_d) {
    sosphase::phase_p0_kernel<<<1, 256, 0, st>>>(a, p->dev.mu, N, mu0, P0_d);
    return launch_check(p);
  }
  return SOS_OK;
}

int sos_build_phase_modes(sos_plan* p, int family, double g, double mu0, int n_phi, const double* phi_h, const double* cphi_h,
                          int n_modes, const double* tab_x_d, const double* tab_y_d, int tab_n, double* P_d, int ldp,
                          size_t mode_stride, double* P0_d, void* stream) {
  if (!p || !phi_h || !cphi_h || (!P_d && !P0_d)) return SOS_ERR_INVALID;
  SOS_GUARD(p);
  if (family < 0 || family > 2 || (family == 2 && (!tab_x_d || !tab_y_d || tab_n < 2))) return SOS_ERR_INVALID;
  if (n_phi < 2 || n_phi > sosphase::MAX_NPHI || n_modes < 1 || n_modes > sosphase::MAX_MODES) return SOS_ERR_INVALID;
  const int N = p->N;
  if (P_d && (ldp < N || (n_modes > 1 && mode_stride < static_cast<size_t>(N) * ldp))) return SOS_ERR_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // node table [phi | cos(0 - phi) | trapezoid weight * cos(m phi)] computed here from what the host passed
  std::vector<double> tab(static_cast<size_t>(n_phi) * (2 + n_modes), 0.0);
  double* phi = tab.data();
  double* cphi = phi + n_phi;
  double* wcos = cphi + n_phi;
  for (int k = 0; k < n_phi; ++k) {
    phi[k] = phi_h[k];
    cphi[k] = cphi_h[k];
    const double tw = 0.5 * ((k + 1 < n_phi ? phi_h[k + 1] : phi_h[k]) - (k > 0 ? phi_h[k - 1] : phi_h[k]));
    for (int m = 1; m < n_modes; ++m) wcos[static_cast<size_t>(k) * n_modes + m] = tw * cphi_h[static_cast<size_t>(1 + m) * n_phi + k];
  }
  double* tab_d = nullptr;
  SOS_CUDA(cudaMallocAsync(&tab_d, tab.size() * sizeof(double), st));
  SOS_CUDA(cudaMemcpyAsync(tab_d, tab.data(), tab.size() * sizeof(double), cudaMemcpyHostToDevice, st));
  sosphase::ModeArgs a;
  std::memset(&a, 0, sizeof(a));
  a.pa.family = family; a.pa.g = g; a.pa.tab_x = tab_x_d; a.pa.tab_y = tab_y_d; a.pa.tab_n = tab_n;
  a.n_phi = n_phi; a.n_modes = n_modes;
  a.phi = tab_d; a.cphi = tab_d + n_phi; a.wcos = tab_d + 2 * n_phi;
  const size_t smem = static_cast<size_t>(n_modes - 1) * sosphase::MODE_THREADS * sizeof(double);
  int r = SOS_OK;
  if (P_d) {
    cudaFuncSetAttribute(sosphase::phase_modes_raw_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    const long long n_el = static_cast<long long>(N) * N;
    sosphase::phase_modes_raw_kernel<false><<<static_cast<unsigned>((n_el + sosphase::MODE_THREADS - 1) / sosphase::MODE_THREADS),
                                             sosphase::MODE_THREADS, smem, st>>>(a, p->dev.mu, N, mu0, P_d, ldp, mode_stride);
    r = launch_check(p, "phase_modes_raw_kernel");
    if (!r) {
      // every mode is normalised by the column integrals of mode 0 (the same kernels as sos_build_phase)
      sosphase::phase_colint_kernel<<<(N + 127) / 128, 128, 0, st>>>(p->dev.mu, N, P_d, ldp, p->d_colint);
      r = launch_check(p);
    }
    const dim3 grid((N + 31) / 32, (N + 7) / 8);
    for (int m = 0; m < n_modes && !r; ++m) {
      sosphase::phase_normalise_kernel<<<grid, 256, 0, st>>>(N, P_d + m * mode_stride, ldp, p->d_colint);
      r = launch_check(p);
    }
  }
  if (P0_d && !r) {
    cudaFuncSetAttribute(sosphase::phase_modes_raw_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    sosphase::phase_modes_raw_kernel<true><<<(N + sosphase::MODE_THREADS - 1) / sosphase::MODE_THREADS, sosphase::MODE_THREADS, smem,
                                            st>>>(a, p->dev.mu, N, mu0, P0_d, N, 0);
    r = launch_check(p, "phase_modes_raw_kernel");
    if (!r) {
      sosphase::phase_p0_modes_norm_kernel<<<1, 256, 0, st>>>(p->dev.mu, N, n_modes, P0_d);
      r = launch_check(p);
    }
  }
  SOS_CUDA(cudaFreeAsync(tab_d, st));
  return r;
}

int sos_azimuth_synthesis(sos_plan* p, const double* I_d, const int* geo_h, const double* w_h, int n_geo, const int* rows_h,
                          int n_rows, int n_az, double* out_d, int accumulate, void* stream) {
  if (!p || !I_d || !geo_h || !w_h || !rows_h || !out_d || n_geo < 1 || n_rows < 1 || n_az < 1) return SOS_ERR_INVALID;
  SOS_GUARD(p);
  const GridDev& g = p->dev;
  const int S = g.S;
  for (int r = 0; r < n_rows; ++r)
    if (rows_h[r] < 0 || rows_h[r] >= g.L) return SOS_ERR_INVALID;
  // members of every present geometry, ascending; one int table [geo | mem_off | members | rows] + the weights
  std::vector<std::vector<int>> by_geo(n_geo);
  for (int s = 0; s < S; ++s) {
    if (geo_h[s] < -1 || geo_h[s] >= n_geo) return SOS_ERR_INVALID;
    if (geo_h[s] >= 0) by_geo[geo_h[s]].push_back(s);
  }
  std::vector<int> geo, off(1, 0), members;
  for (int k = 0; k < n_geo; ++k) {
    if (by_geo[k].empty()) continue;
    geo.push_back(k);
    members.insert(members.end(), by_geo[k].begin(), by_geo[k].end());
    off.push_back(static_cast<int>(members.size()));
  }
  const int n_present = static_cast<int>(geo.size());
  if (n_present == 0) return SOS_OK;
  if (static_cast<long long>(n_present) * n_rows > 65535) return SOS_ERR_UNSUPPORTED;
  const size_t n_w = static_cast<size_t>(S) * n_az;
  std::vector<int> itab;
  itab.reserve(geo.size() + off.size() + members.size() + n_rows);
  itab.insert(itab.end(), geo.begin(), geo.end());
  itab.insert(itab.end(), off.begin(), off.end());
  itab.insert(itab.end(), members.begin(), members.end());
  itab.insert(itab.end(), rows_h, rows_h + n_rows);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  char* buf = nullptr;
  const size_t wbytes = n_w * sizeof(double);
  SOS_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&buf), wbytes + itab.size() * sizeof(int), st));
  SOS_CUDA(cudaMemcpyAsync(buf, w_h, wbytes, cudaMemcpyHostToDevice, st));
  SOS_CUDA(cudaMemcpyAsync(buf + wbytes, itab.data(), itab.size() * sizeof(int), cudaMemcpyHostToDevice, st));
  const int* it = reinterpret_cast<const int*>(buf + wbytes);
  sosquad::SynthTables t;
  t.w = reinterpret_cast<const double*>(buf);
  t.geo = it;
  t.mem_off = t.geo + geo.size();
  t.members = t.mem_off + off.size();
  t.rows = t.members + members.size();
  const dim3 grid((g.N + sosquad::AZ_THREADS - 1) / sosquad::AZ_THREADS, n_present * n_rows,
                  (n_az + sosquad::AZ_CHUNK - 1) / sosquad::AZ_CHUNK);
  if (grid.z > 65535) { cudaFreeAsync(buf, st); return SOS_ERR_UNSUPPORTED; }
  sosquad::azimuth_synthesis_kernel<<<grid, sosquad::AZ_THREADS, 0, st>>>(I_d, g.L, g.ld, g.N, t, n_rows, n_az, out_d, accumulate ? 1 : 0);
  const int r = launch_check(p, "azimuth_synthesis_kernel");
  SOS_CUDA(cudaFreeAsync(buf, st));
  return r;
}

static int encode_A_maps(sos_plan* p) {
  const int bn = p->gemm_bn + 8;  // rows are loaded 8 columns wider than the tile (bank layout)
  for (size_t i = 0; i < p->A_ptrs.size(); ++i) {
    int r = encode_2d(&p->gp.map_A[i], p->A_ptrs[i], p->N, p->N, p->lda, bn, sosgemm::BK, CU_TENSOR_MAP_SWIZZLE_NONE);
    if (r) return r;
  }
  return SOS_OK;
}

int sos_plan_set_phase(sos_plan* p, const double* const* A_d, int n, int lda) {
  if (!p || !A_d || n < 1 || n > SOS_MAX_PHASE || lda < p->N || (lda & 1)) return SOS_ERR_INVALID;
  SOS_GUARD(p);
  drop_graphs(p);
  for (const sos_scenario& sc : p->scen_h)
    if (sc.phase_atm >= n || sc.phase_aer >= n) return SOS_ERR_INVALID;
  for (int i = 0; i < n; ++i)
    if (!A_d[i] || (reinterpret_cast<uintptr_t>(A_d[i]) & 15)) return SOS_ERR_INVALID;
  p->A_ptrs.assign(A_d, A_d + n);
  p->lda = lda;
  const bool was_premix = p->fold;
  p->fold = false;  // new operands: the folded set and the low-rank factors (if any) must be given again
  for (int i = 0; i < SOS_MAX_PHASE; ++i) p->lowrank_rank[i] = 0;
  p->split_passes = p->split_general;
  int r = encode_A_maps(p);
  if (r) return r;
  p->maps_A_ready = true;
  if (was_premix) {  // the device tile plan was laid out for per-scenario aerosol tiles
    r = plan_tiles(p, nullptr);
    if (r) return r;
    SOS_CUDA(cudaDeviceSynchronize());
  }
  return SOS_OK;
}

int sos_build_brdf_modes(sos_plan* p, int n_nodes, const double* phi_h, const double* cos_h, int n_modes, double mu_min,
                         double* Rvol_d, double* Rgeo_d, int ldr, size_t mode_stride, void* stream) {
  if (!p || !phi_h || !cos_h || !Rvol_d || !Rgeo_d) return SOS_ERR_INVALID;
  SOS_GUARD(p);
  const int M = p->dev.M;
  if (n_nodes < 2 || n_nodes > sosbrdf::MAX_NODES || n_modes < 1 || n_modes > sosbrdf::MAX_MODES) return SOS_ERR_INVALID;
  if (!(mu_min > 0.0 && mu_min < 1.0) || M < 2 || ldr < M - 1 || (n_modes > 1 && mode_stride < static_cast<size_t>(M) * ldr))
    return SOS_ERR_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // node table [cos(phi_k - pi) | trapezoid weight * cos(m phi_k) / pi] computed here from what the host passed
  const double PI = 3.14159265358979323846;
  std::vector<double> tab(static_cast<size_t>(n_nodes) * (1 + n_modes), 0.0);
  double* cpsi = tab.data();
  double* wcos = cpsi + n_nodes;
  for (int k = 0; k < n_nodes; ++k) {
    cpsi[k] = cos_h[k];
    const double tw = 0.5 * ((k + 1 < n_nodes ? phi_h[k + 1] : phi_h[k]) - (k > 0 ? phi_h[k - 1] : phi_h[k]));
    for (int m = 0; m < n_modes; ++m) wcos[static_cast<size_t>(k) * n_modes + m] = tw * cos_h[static_cast<size_t>(1 + m) * n_nodes + k] / PI;
  }
  double* tab_d = nullptr;
  SOS_CUDA(cudaMallocAsync(&tab_d, tab.size() * sizeof(double), st));
  SOS_CUDA(cudaMemcpyAsync(tab_d, tab.data(), tab.size() * sizeof(double), cudaMemcpyHostToDevice, st));
  const size_t smem = static_cast<size_t>(2 * n_modes) * sosbrdf::BUILD_THREADS * sizeof(double);
  cudaFuncSetAttribute(sosbrdf::brdf_modes_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
  const long long n_el = static_cast<long long>(M) * (M - 1);
  sosbrdf::brdf_modes_kernel<<<static_cast<unsigned>((n_el + sosbrdf::BUILD_THREADS - 1) / sosbrdf::BUILD_THREADS), sosbrdf::BUILD_THREADS,
                               smem, st>>>(p->dev.mu, M, mu_min, tab_d, tab_d + n_nodes, n_nodes, n_modes, Rvol_d, Rgeo_d, ldr, mode_stride);
  const int r = launch_check(p, "brdf_modes_kernel");
  SOS_CUDA(cudaFreeAsync(tab_d, st));
  return r;
}

int sos_build_glint_modes(sos_plan* p, int n_nodes, const double* phi_h, const double* cos_h, int n_modes, double sigma2,
                          double n_ref, double* R_d, int ldr, size_t mode_stride, void* stream) {
  if (!p || !phi_h || !cos_h || !R_d) return SOS_ERR_INVALID;
  SOS_GUARD(p);
  const int M = p->dev.M;
  if (n_nodes < 2 || n_nodes > sosbrdf::MAX_NODES || n_modes < 1 || n_modes > sosbrdf::MAX_MODES) return SOS_ERR_INVALID;
  if (!(sigma2 > 0.0 && std::isfinite(sigma2)) || !(n_ref > 1.0 && std::isfinite(n_ref))) return SOS_ERR_INVALID;
  if (M < 2 || ldr < M - 1 || (n_modes > 1 && mode_stride < static_cast<size_t>(M) * ldr)) return SOS_ERR_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // node table [cos(phi_k) | trapezoid weight * cos(m phi_k) / pi], as for sos_build_brdf_modes
  const double PI = 3.14159265358979323846;
  std::vector<double> tab(static_cast<size_t>(n_nodes) * (1 + n_modes), 0.0);
  double* cphi = tab.data();
  double* wcos = cphi + n_nodes;
  for (int k = 0; k < n_nodes; ++k) {
    cphi[k] = cos_h[k];
    const double tw = 0.5 * ((k + 1 < n_nodes ? phi_h[k + 1] : phi_h[k]) - (k > 0 ? phi_h[k - 1] : phi_h[k]));
    for (int m = 0; m < n_modes; ++m) wcos[static_cast<size_t>(k) * n_modes + m] = tw * cos_h[static_cast<size_t>(1 + m) * n_nodes + k] / PI;
  }
  double* tab_d = nullptr;
  SOS_CUDA(cudaMallocAsync(&tab_d, tab.size() * sizeof(double), st));
  SOS_CUDA(cudaMemcpyAsync(tab_d, tab.data(), tab.size() * sizeof(double), cudaMemcpyHostToDevice, st));
  const size_t smem = static_cast<size_t>(n_modes) * sosbrdf::BUILD_THREADS * sizeof(double);
  cudaFuncSetAttribute(sosglint::glint_modes_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
  const long long n_el = static_cast<long long>(M) * (M - 1);
  sosglint::glint_modes_kernel<<<static_cast<unsigned>((n_el + sosbrdf::BUILD_THREADS - 1) / sosbrdf::BUILD_THREADS), sosbrdf::BUILD_THREADS,
                                 smem, st>>>(p->dev.mu, M, sigma2, n_ref, tab_d, tab_d + n_nodes, n_nodes, n_modes, R_d, ldr, mode_stride);
  const int r = launch_check(p, "glint_modes_kernel");
  SOS_CUDA(cudaFreeAsync(tab_d, st));
  return r;
}

int sos_glint_correction(sos_plan* p, int n, const int* geo_h, const double* par_h, const double* tau_h, int n_rows,
                         const double* beam_h, int n_modes, const double* phi_h, int n_az, int n_geo, double* out_d,
                         void* stream) {
  if (!p || !geo_h || !par_h || !tau_h || !beam_h || !phi_h || !out_d || n < 1 || n_rows < 1 || n_az < 1 || n_geo < 1)
    return SOS_ERR_INVALID;
  SOS_GUARD(p);
  const int M = p->dev.M, N = p->dev.N;
  if (n_modes < 1 || n_modes > sosbrdf::MAX_MODES || M < 2) return SOS_ERR_INVALID;
  for (int k = 0; k < n; ++k) {
    const double* q = par_h + 4 * static_cast<size_t>(k);
    if (geo_h[k] < 0 || geo_h[k] >= n_geo) return SOS_ERR_INVALID;
    if (!(q[0] > 0.0 && q[0] <= 1.0) || !std::isfinite(q[1]) || !(q[2] > 0.0 && std::isfinite(q[2])) ||
        !(q[3] > 1.0 && std::isfinite(q[3])))
      return SOS_ERR_INVALID;
  }
  // one table: par [n][4] | tau [n][n_rows] | beam [n][K][M-1] | w [n_az][K] | cos(phi) [n_az] | geo [n] (int)
  const size_t n_par = 4 * static_cast<size_t>(n), n_tau = static_cast<size_t>(n) * n_rows,
               n_beam = static_cast<size_t>(n) * n_modes * (M - 1), n_w = static_cast<size_t>(n_az) * n_modes;
  std::vector<double> tab(n_par + n_tau + n_beam + n_w + n_az);
  std::copy(par_h, par_h + n_par, tab.begin());
  std::copy(tau_h, tau_h + n_tau, tab.begin() + n_par);
  std::copy(beam_h, beam_h + n_beam, tab.begin() + n_par + n_tau);
  double* w = tab.data() + n_par + n_tau + n_beam;
  double* cphi = w + n_w;
  for (int q = 0; q < n_az; ++q) {
    cphi[q] = std::cos(phi_h[q]);
    for (int m = 0; m < n_modes; ++m) w[static_cast<size_t>(q) * n_modes + m] = m == 0 ? 1.0 : 2.0 * std::cos(m * phi_h[q]);
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  char* buf = nullptr;
  const size_t dbytes = tab.size() * sizeof(double);
  SOS_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&buf), dbytes + n * sizeof(int), st));
  SOS_CUDA(cudaMemcpyAsync(buf, tab.data(), dbytes, cudaMemcpyHostToDevice, st));
  SOS_CUDA(cudaMemcpyAsync(buf + dbytes, geo_h, n * sizeof(int), cudaMemcpyHostToDevice, st));
  const double* d = reinterpret_cast<const double*>(buf);
  sosquad::GlintCorrection t;
  t.par = d;
  t.tau = d + n_par;
  t.beam = t.tau + n_tau;
  t.w = t.beam + n_beam;
  t.cphi = t.w + n_w;
  t.geo = reinterpret_cast<const int*>(buf + dbytes);
  const long long n_el = static_cast<long long>(n) * n_rows * n_az * (M - 1);
  sosquad::glint_correction_kernel<<<static_cast<unsigned>((n_el + 127) / 128), 128, 0, st>>>(p->dev.mu, M, N, t, n, n_modes,
                                                                                           n_rows, n_az, out_d);
  const int r = launch_check(p, "glint_correction_kernel");
  SOS_CUDA(cudaFreeAsync(buf, st));
  return r;
}

int sos_single_scatter_correction(sos_plan* p, int n, const sos_ss_entry* ent_h, const double* P0m_h, int n_vec, int n_modes,
                                  const double* tab_h, int n_tab, const int* rows_h, int n_rows, const double* phi_h, int n_az,
                                  int n_geo, double* out_d, void* stream) {
  if (!p || !ent_h || !P0m_h || !rows_h || !phi_h || !out_d || n < 1 || n_vec < 1 || n_rows < 1 || n_az < 1 || n_geo < 1 ||
      n_tab < 0 || (n_tab > 0 && !tab_h))
    return SOS_ERR_INVALID;
  SOS_GUARD(p);
  const GridDev& g = p->dev;
  if (g.nreg != 3) return SOS_ERR_UNSUPPORTED;
  if (n_modes < 1 || n_modes > sosphase::MAX_MODES) return SOS_ERR_INVALID;
  for (int r = 0; r < n_rows; ++r)
    if (rows_h[r] < 0 || rows_h[r] >= g.L) return SOS_ERR_INVALID;
  for (int k = 0; k < n; ++k) {
    const sos_ss_entry& e = ent_h[k];
    if (e.scenario < 0 || e.scenario >= g.S || e.geo < 0 || e.geo >= n_geo) return SOS_ERR_INVALID;
    for (int j = 0; j < 4; ++j)
      if (!std::isfinite(e.w[j])) return SOS_ERR_INVALID;
    for (int j = 0; j < 2; ++j) {
      if (e.family[j] < -1 || e.family[j] > 2) return SOS_ERR_INVALID;
      if (e.family[j] < 0) continue;
      if (e.series[j] < 0 || e.series[j] >= n_vec || !(e.norm[j] > 0.0 && std::isfinite(e.norm[j])) || !std::isfinite(e.g[j]))
        return SOS_ERR_INVALID;
      if (e.family[j] == 2 && (e.tab_n[j] < 2 || e.tab_off[j] < 0 || static_cast<long long>(e.tab_off[j]) + 2LL * e.tab_n[j] > n_tab))
        return SOS_ERR_INVALID;
    }
  }
  static_assert(sizeof(sos_ss_entry) == sizeof(sosss::Entry), "sos_ss_entry and sosss::Entry must match");
  // one table: P0m [n_vec][K][N] | tab [n_tab] | wcos [n_az][K] | cos(phi) [n_az] | entries | rows (int)
  const int N = g.N;
  const size_t n_p0 = static_cast<size_t>(n_vec) * n_modes * N, n_w = static_cast<size_t>(n_az) * n_modes;
  std::vector<double> tab(n_p0 + n_tab + n_w + n_az);
  std::copy(P0m_h, P0m_h + n_p0, tab.begin());
  if (n_tab) std::copy(tab_h, tab_h + n_tab, tab.begin() + n_p0);
  double* w = tab.data() + n_p0 + n_tab;
  double* cphi = w + n_w;
  for (int q = 0; q < n_az; ++q) {
    cphi[q] = std::cos(phi_h[q]);
    for (int m = 0; m < n_modes; ++m) w[static_cast<size_t>(q) * n_modes + m] = m == 0 ? 1.0 : 2.0 * std::cos(m * phi_h[q]);
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  char* buf = nullptr;
  const size_t dbytes = tab.size() * sizeof(double), ebytes = static_cast<size_t>(n) * sizeof(sos_ss_entry);
  SOS_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&buf), dbytes + ebytes + n_rows * sizeof(int), st));
  SOS_CUDA(cudaMemcpyAsync(buf, tab.data(), dbytes, cudaMemcpyHostToDevice, st));
  SOS_CUDA(cudaMemcpyAsync(buf + dbytes, ent_h, ebytes, cudaMemcpyHostToDevice, st));
  SOS_CUDA(cudaMemcpyAsync(buf + dbytes + ebytes, rows_h, n_rows * sizeof(int), cudaMemcpyHostToDevice, st));
  const double* d = reinterpret_cast<const double*>(buf);
  sosss::Tables t;
  t.P0m = d;
  t.tab = d + n_p0;
  t.wcos = t.tab + n_tab;
  t.cphi = t.wcos + n_w;
  t.ent = reinterpret_cast<const sosss::Entry*>(buf + dbytes);
  t.rows = reinterpret_cast<const int*>(buf + dbytes + ebytes);
  const long long n_el = static_cast<long long>(n) * n_az * N;
  sosss::single_scatter_kernel<<<static_cast<unsigned>((n_el + sosss::THREADS - 1) / sosss::THREADS), sosss::THREADS, 0, st>>>(
      g, t, n, n_modes, n_rows, n_az, out_d);
  const int r = launch_check(p, "single_scatter_kernel");
  SOS_CUDA(cudaFreeAsync(buf, st));
  return r;
}

int sos_plan_set_brdf(sos_plan* p, const double* const* Rvol_d, const double* const* Rgeo_d, int n_sets, int ldr) {
  if (!p || !Rvol_d) return SOS_ERR_INVALID;
  SOS_GUARD(p);
  if (!p->d_brdf_R) return SOS_ERR_UNSUPPORTED;
  // one matrix per set (ocean) exactly when the second array is absent
  if ((p->brdf_nk == 1) != (Rgeo_d == nullptr)) return SOS_ERR_INVALID;
  if (n_sets < 1 || n_sets > sosbrdf::MAX_SETS || ldr < p->dev.M - 1) return SOS_ERR_INVALID;
  std::vector<const double*> ptrs(2 * static_cast<size_t>(n_sets), nullptr);
  for (int j = 0; j < n_sets; ++j) {
    if (!Rvol_d[j] || (Rgeo_d && !Rgeo_d[j])) return SOS_ERR_INVALID;
    ptrs[2 * j] = Rvol_d[j];
    if (Rgeo_d) ptrs[2 * j + 1] = Rgeo_d[j];
  }
  drop_graphs(p);
  SOS_CUDA(cudaMemcpy(p->d_brdf_R, ptrs.data(), ptrs.size() * sizeof(const double*), cudaMemcpyHostToDevice));
  p->brdf_sets = n_sets;
  p->brdf_ldr = ldr;
  p->brdf_scen_ready = false;   // the set indices refer to the previous registration
  return SOS_OK;
}

int sos_plan_set_brdf_scenarios(sos_plan* p, const int* set_h, const double* f_h, const double* beam_h, void* stream) {
  if (!p || !set_h || !f_h || !beam_h) return SOS_ERR_INVALID;
  SOS_GUARD(p);
  if (!p->d_brdf_R) return SOS_ERR_UNSUPPORTED;
  if (p->brdf_sets < 1) return SOS_ERR_STATE;
  const int S = p->dev.S, M = p->dev.M;
  const bool one = p->brdf_nk == 1;   // ocean: (f_glint, 0), the second beam vector is not read
  for (int s = 0; s < S; ++s) {
    if (set_h[s] < 0 || set_h[s] >= p->brdf_sets) return SOS_ERR_INVALID;
    if (!(f_h[2 * s] >= 0.0 && f_h[2 * s + 1] >= 0.0) || !std::isfinite(f_h[2 * s]) || !std::isfinite(f_h[2 * s + 1])) return SOS_ERR_INVALID;
    if (one && f_h[2 * s + 1] != 0.0) return SOS_ERR_INVALID;
  }
  const size_t nf = 2 * static_cast<size_t>(S), nb = nf * (M - 1);
  for (size_t k = 0; k < nb; ++k)
    if (!(one && (k / (M - 1)) % 2 == 1) && !std::isfinite(beam_h[k])) return SOS_ERR_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  double* d = reinterpret_cast<double*>(p->d_brdf_scen);
  SOS_CUDA(cudaMemcpyAsync(d, f_h, nf * sizeof(double), cudaMemcpyHostToDevice, st));
  SOS_CUDA(cudaMemcpyAsync(d + nf, beam_h, nb * sizeof(double), cudaMemcpyHostToDevice, st));
  SOS_CUDA(cudaMemcpyAsync(d + nf + nb, set_h, S * sizeof(int), cudaMemcpyHostToDevice, st));
  SOS_CUDA(cudaStreamSynchronize(st));   // (the host arrays may be pageable and are the caller's after this call)
  p->brdf_scen_ready = true;
  return SOS_OK;
}

int sos_fold_layout(int nb_angles, int* rows, int* ld) {
  const int Mh = (nb_angles + 15) / 16 * 16;
  if (rows) *rows = Mh;       // k rows, padded to the k-step
  if (ld) *ld = 2 * Mh;       // [B+ | B-], each Mh columns wide
  return 2 * Mh * Mh;
}

int sos_build_folded(sos_plan* p, const double* A_d, int lda, double* F_d, int ldf, double* defect_out, void* stream) {
  if (!p || !A_d || !F_d || !defect_out || lda < p->N) return SOS_ERR_INVALID;
  SOS_GUARD(p);
  int rows = 0, ld = 0;
  sos_fold_layout(p->dev.M, &rows, &ld);
  if (ldf != ld) return SOS_ERR_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  SOS_CUDA(cudaMemsetAsync(p->d_fold_stats, 0, 2 * sizeof(unsigned long long), st));
  dim3 grid((rows + 127) / 128, rows);
  sosgemm::build_folded_kernel<<<grid, 128, 0, st>>>(A_d, lda, p->N, F_d, ldf, rows, rows, p->d_fold_stats);
  int r = launch_check(p);
  if (r) return r;
  unsigned long long bits[2] = {0, 0};
  SOS_CUDA(cudaMemcpyAsync(bits, p->d_fold_stats, sizeof(bits), cudaMemcpyDeviceToHost, st));
  SOS_CUDA(cudaStreamSynchronize(st));
  double defect, amax;
  std::memcpy(&defect, &bits[0], 8);
  std::memcpy(&amax, &bits[1], 8);
  *defect_out = amax > 0.0 ? defect / amax : 0.0;
  return SOS_OK;
}

// Fold-mode tile-plan tables: aerosol rows = one class-2 group (premixed operand per scenario) or the class-1 groups of
// the general plan; every class-0 group whose operand is low rank becomes class 3 (no dense tiles, jn_lowrank_kernel).
static int build_fold_tables(sos_plan* p) {
  const int S = p->dev.S;
  sosgemm::GroupTable& gt = p->groups_premix;
  std::memset(&gt, 0, sizeof(gt));
  std::vector<int> flat;
  const std::vector<int>& members_h = p->members_h;
  auto copy_group = [&](int g, int cls) {
    const int ng = gt.n_groups++;
    gt.cls[ng] = cls; gt.phaseA[ng] = p->groups.phaseA[g]; gt.phaseB[ng] = p->groups.phaseB[g];
    gt.member_off[ng] = static_cast<int>(flat.size());
    flat.insert(flat.end(), members_h.begin() + p->groups.member_off[g], members_h.begin() + p->groups.member_off[g + 1]);
  };
  if (p->premix) {
    gt.cls[0] = 2; gt.phaseA[0] = 0; gt.phaseB[0] = 0; gt.member_off[0] = 0;
    for (int sidx = 0; sidx < S; ++sidx) flat.push_back(sidx);
    gt.n_groups = 1;
  } else {
    for (int g = 0; g < p->groups.n_groups; ++g)
      if (p->groups.cls[g] == 1) copy_group(g, 1);
  }
  p->n_lowrank_groups = 0;
  p->lowrank_rp = 4;
  for (int g = 0; g < p->groups.n_groups; ++g) {
    if (p->groups.cls[g] != 0) continue;
    const int r = p->lowrank_rank[p->groups.phaseA[g]];
    copy_group(g, r > 0 ? 3 : 0);
    if (r > 0) { p->n_lowrank_groups++; if (r > 4) p->lowrank_rp = 16; }
  }
  gt.member_off[gt.n_groups] = static_cast<int>(flat.size());
  if (flat.size() != members_h.size()) return SOS_ERR_STATE;  // (both hold every scenario once per row class)
  if (!p->d_members_premix) {
    int r = dev_alloc(p, &p->d_members_premix, flat.size());
    if (r) return r;
  }
  SOS_CUDA(cudaMemcpy(p->d_members_premix, flat.data(), flat.size() * sizeof(int), cudaMemcpyHostToDevice));
  return SOS_OK;
}

// dense (DMMA) row tiles of an all-active launch in fold mode, for the small-launch heuristics
static long long fold_dense_row_tiles(const sos_plan* p) {
  struct FC { int SEGS; } fc{p->fold_segs};
  long long rows = 0;
  for (int g = 0; g < p->groups_premix.n_groups; ++g) {
    const long long members = p->groups_premix.member_off[g + 1] - p->groups_premix.member_off[g];
    const int cls = p->groups_premix.cls[g];
    if (cls == 3) continue;
    if (cls == 2) rows += members * ((p->nseg[1] + fc.SEGS - 1) / fc.SEGS);
    else rows += (members * (cls == 1 ? p->nseg[1] : p->nseg[0]) + fc.SEGS - 1) / fc.SEGS;
  }
  return rows;
}

static int refresh_fold_plan(sos_plan* p) {
  using FC = sosgemm::FoldCfg;
  int r = build_fold_tables(p);
  if (r) return r;
  {
    // every dense tile is the aerosol layer of one scenario (premixed operand; the other rows are low rank): a layer of 7 segments
    // (54 rows on the default grid) fills a 56-row tile exactly
    bool only_aerosol = p->premix && p->fold_xform && p->groups_premix.n_groups > 0;
    for (int g = 0; g < p->groups_premix.n_groups; ++g)
      if (p->groups_premix.cls[g] != 2 && p->groups_premix.cls[g] != 3) only_aerosol = false;
    const int segs = (only_aerosol && p->nseg[1] % 7 == 0 && env_int("SOS_FOLD_ROWS56", 1) != 0) ? 7 : 8;
    if (segs != p->fold_segs) drop_graphs(p);  // (captured order graphs hold the kernel of the other tile shape)
    p->fold_segs = segs;
  }
  const long long tiles = fold_dense_row_tiles(p) * ((p->dev.M + FC::BN - 1) / FC::BN);
  p->split_passes = (!p->premix && p->grid.n_regions == 3 && tiles < 2LL * p->n_sms) ? 1 : 0;
  {
    // single solves: fewer tiles than half the SMs and long k loops -> two tiles per output tile
    const char* e = std::getenv("SOS_FOLD_KSPLIT");
    const bool allow = !(e && e[0] == '0');
    // (never together with split operand passes: four atomic partials per element would not be order independent)
    p->fold_ksplit = (allow && !p->split_passes && 2 * tiles <= p->n_sms && p->dev.M >= 64) ? 2 : 1;
  }
  r = plan_tiles(p, nullptr);
  if (r) return r;
  SOS_CUDA(cudaDeviceSynchronize());
  return SOS_OK;
}

int sos_lowrank_layout(int nb_angles, int* rows, int* ldr) {
  if (rows) *rows = 4;                                // rank <= 2 here; jn_lowrank_kernel<4> takes 4 factor rows
  if (ldr) *ldr = (2 * nb_angles + 15) / 16 * 16;
  return 4 * ((2 * nb_angles + 15) / 16 * 16);
}

int sos_build_lowrank_mu2(sos_plan* p, const double* A_d, int lda, double* Ut_d, double* Vt_d, int ldr, double* residual_out,
                          int* rank_out, void* stream) {
  if (!p || !A_d || !Ut_d || !Vt_d || !residual_out || !rank_out || lda < p->N || ldr < p->N) return SOS_ERR_INVALID;
  SOS_GUARD(p);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int N = p->N, M = p->dev.M;
  SOS_CUDA(cudaMemsetAsync(p->d_lr_stats, 0, 3 * sizeof(unsigned long long), st));
  sosgemm::lowrank_mu2_fit_kernel<<<(ldr + 127) / 128, 128, 0, st>>>(A_d, lda, N, M, p->dev.mu, Ut_d, Vt_d, ldr, 4);
  int r = launch_check(p);
  if (r) return r;
  dim3 grid(static_cast<unsigned>(std::min(8, (N + 255) / 256)), N);
  sosgemm::lowrank_mu2_residual_kernel<<<grid, 256, 0, st>>>(A_d, lda, N, Ut_d, Vt_d, ldr, p->d_lr_stats);
  r = launch_check(p);
  if (r) return r;
  unsigned long long bits[3] = {0, 0, 0};
  SOS_CUDA(cudaMemcpyAsync(bits, p->d_lr_stats, sizeof(bits), cudaMemcpyDeviceToHost, st));
  SOS_CUDA(cudaStreamSynchronize(st));
  double res, amax, bmax;
  std::memcpy(&res, &bits[0], 8);
  std::memcpy(&amax, &bits[1], 8);
  std::memcpy(&bmax, &bits[2], 8);
  *residual_out = amax > 0.0 ? res / amax : (res > 0.0 ? INFINITY : 0.0);
  *rank_out = (bmax <= 1e-15 * amax) ? 1 : 2;   // isotropic operand: beta vanishes
  return SOS_OK;
}

int sos_plan_set_lowrank(sos_plan* p, const double* const* Ut_d, const double* const* Vt_d, const int* rank, int n, int ldr) {
  if (!p) return SOS_ERR_INVALID;
  SOS_GUARD(p);
  drop_graphs(p);
  if (n == 0) {
    for (int i = 0; i < SOS_MAX_PHASE; ++i) p->lowrank_rank[i] = 0;
  } else {
    if (!Ut_d || !Vt_d || !rank || !p->maps_A_ready || n != static_cast<int>(p->A_ptrs.size()) || ldr < p->N) return SOS_ERR_INVALID;
    for (int i = 0; i < n; ++i) {
      if (rank[i] < 0 || rank[i] > 16) return SOS_ERR_INVALID;
      if (rank[i] > 0 && (!Ut_d[i] || !Vt_d[i])) return SOS_ERR_INVALID;
    }
    for (int i = 0; i < SOS_MAX_PHASE; ++i) {
      p->lowrank_rank[i] = i < n ? rank[i] : 0;
      p->lowrank_Ut[i] = i < n ? Ut_d[i] : nullptr;
      p->lowrank_Vt[i] = i < n ? Vt_d[i] : nullptr;
    }
    p->lowrank_ldr = ldr;
  }
  return p->fold ? refresh_fold_plan(p) : SOS_OK;
}

// (re)build the per-scenario premixed aerosol operands from the registered folded operands and the current coefficients
static int premix_folded(sos_plan* p) {
  int rows = 0, ld = 0;
  sos_fold_layout(p->dev.M, &rows, &ld);
  const size_t per = static_cast<size_t>(rows) * ld;
  const int S = p->dev.S, n = static_cast<int>(p->F_ptrs.size());
  sosgemm::MixSources src;
  for (int i = 0; i < SOS_MAX_PHASE; ++i) src.F[i] = i < n ? p->F_ptrs[i] : nullptr;
  dim3 grid(static_cast<unsigned>(std::min<size_t>((per + 255) / 256, 64)), S);
  sosgemm::mix_folded_kernel<<<grid, 256, 0, nullptr>>>(src, p->dev.scen, p->d_mix, per);
  return launch_check(p, "mix_folded_kernel");
}

int sos_plan_set_folded(sos_plan* p, const double* const* F_d, int n, int ldf) {
  if (!p) return SOS_ERR_INVALID;
  SOS_GUARD(p);
  drop_graphs(p);
  if (n == 0 || !F_d) {
    const bool replan = p->fold;
    p->fold = false;
    p->split_passes = p->split_general;
    if (replan) {
      int r = plan_tiles(p, nullptr);
      if (r) return r;
      SOS_CUDA(cudaDeviceSynchronize());
    }
    return SOS_OK;
  }
  if (!p->maps_A_ready) return SOS_ERR_STATE;
  if (n != static_cast<int>(p->A_ptrs.size())) return SOS_ERR_INVALID;
  int rows = 0, ld = 0;
  sos_fold_layout(p->dev.M, &rows, &ld);
  if (ldf != ld) return SOS_ERR_INVALID;
  using FC = sosgemm::FoldCfg;
  for (int i = 0; i < n; ++i) {
    if (!F_d[i] || (reinterpret_cast<uintptr_t>(F_d[i]) & 15)) return SOS_ERR_INVALID;
    int r = encode_2d(&p->fp.map_F[i], F_d[i], ld, rows, ldf, FC::BN_PAD, sosgemm::BK, CU_TENSOR_MAP_SWIZZLE_NONE);
    if (r) return r;
  }
  // the folded kernel and the general fallback (column-sharded or peer launches) share the tile shape:
  // 64-row tiles, 128-column general tiles
  const bool reshape = p->gemm_bm != FC::BM || p->gemm_bn != 128;
  p->gemm_bm = FC::BM;
  p->gemm_bn = 128;
  if (reshape) { int r = encode_A_maps(p); if (r) return r; }
  p->F_ptrs.assign(F_d, F_d + n);
  { const char* e = std::getenv("SOS_FOLD_XFORM"); p->fold_xform = !(e && e[0] == '0'); }
  // aerosol rows: premix c1 F[atm] + c2 F[aer] per scenario so that their tiles need one operand pass instead of two
  // (S operands of rows*ldf doubles; above 2 GB the two-pass tiles stay)
  p->premix = false;
  {
    const char* env = std::getenv("SOS_FOLD_PREMIX");  // read per call: tests switch it inside one process
    const bool allow = !(env && env[0] == '0');
    const size_t per = static_cast<size_t>(rows) * ldf;
    const int S = p->dev.S;
    if (allow && p->grid.n_regions == 3 && per * S * sizeof(double) <= (2ull << 30)) {
      if (!p->d_mix) { int r = dev_alloc(p, &p->d_mix, per * S); if (r) return r; }
      int r = premix_folded(p);
      if (r) return r;
      r = encode_3d(&p->fp.map_mix, p->d_mix, ld, rows, S, ldf, FC::BN_PAD, sosgemm::BK);
      if (r) return r;
      p->premix = true;
    }
  }
  p->fold = true;
  int r = refresh_fold_plan(p);
  if (r) return r;
  cudaFuncSetAttribute(sosgemm::jn_gemm_fold_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, FC::SMEM);
  cudaFuncSetAttribute(sosgemm::jn_gemm_fold_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, FC::SMEM);
  cudaFuncSetAttribute(sosgemm::jn_gemm_fold_kernel<true, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, sosgemm::FoldCfgT<3>::SMEM);
  cudaFuncSetAttribute(sosgemm::jn_gemm_fold_kernel<true, 7, 1, 8, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, sosgemm::FoldCfgT<7, 1, 8, 2>::SMEM);
  return SOS_OK;
}

int sos_first_order(sos_plan* p, const double* C_h, double* I1_d, void* stream) {
  return sos_first_order2(p, C_h, I1_d, nullptr, stream);
}

// The caller's host arrays (possibly pageable) are copied into one of two pinned staging buffers owned by the plan, so the
// H2D copy is truly asynchronous and the first-order entry points return without waiting for the stream.  Returns the buffer.
static int first_order_stage(sos_plan* p, double** buf, cudaEvent_t* ev) {
  const GridDev& g = p->dev;
  const size_t bytes = sizeof(double) * g.S * 2 * g.N;
  const int k = p->h_C_next;
  p->h_C_next ^= 1;
  if (!p->h_C[k]) {
    auto& fl = pinned_coef_free_list();
    for (size_t i = 0; i < fl.size() && !p->h_C[k]; ++i)
      if (fl[i].first == bytes) { p->h_C[k] = fl[i].second; fl.erase(fl.begin() + i); }
    if (!p->h_C[k]) SOS_CUDA(cudaMallocHost(reinterpret_cast<void**>(&p->h_C[k]), bytes));
    SOS_CUDA(cudaEventCreateWithFlags(&p->h_C_ev[k], cudaEventDisableTiming));
  } else {
    SOS_CUDA(cudaEventSynchronize(p->h_C_ev[k]));  // the copy issued two calls ago has left this buffer
  }
  *buf = p->h_C[k];
  *ev = p->h_C_ev[k];
  return SOS_OK;
}

static int first_order_launch(sos_plan* p, double* I1_d, double* I1_copy_d, cudaStream_t st) {
  const GridDev& g = p->dev;
  if (brdf_missing(p)) return SOS_ERR_STATE;
  const int rows_per_block = std::min(64, std::max(8, env_int("SOS_B200_FO_ROWS", 64)));  // (the kernel stages 64 rows at most)
  dim3 grid((g.N + 127) / 128, (g.L + rows_per_block - 1) / rows_per_block, g.S);
  if (p->d_bs) {
    // diffuse Lambert / Ross-Li / ocean ground: the upward radiance of order 1 at the surface row, read by the upward columns
    const size_t smem = (g.M + 32) * sizeof(double);
    if (p->brdf_nk == 2)
      sosfirst::first_order_surface_kernel<2><<<g.S, 128, smem, st>>>(g, p->d_C, p->d_bs, brdf_dev(p));
    else if (p->brdf_nk == 1)
      sosfirst::first_order_surface_kernel<1><<<g.S, 128, smem, st>>>(g, p->d_C, p->d_bs, brdf_dev(p));
    else
      sosfirst::first_order_surface_kernel<0><<<g.S, 128, smem, st>>>(g, p->d_C, p->d_bs, brdf_dev(p));
    int r = launch_check(p, "first_order_surface_kernel");
    if (r) return r;
  }
  if (g.nreg == 3 && p->d_brdf_R)
    sosfirst::first_order_regions_kernel<true><<<grid, 128, 0, st>>>(g, p->d_C, I1_d, I1_copy_d, rows_per_block, p->d_bs);
  else if (g.nreg == 3)
    sosfirst::first_order_regions_kernel<false><<<grid, 128, 0, st>>>(g, p->d_C, I1_d, I1_copy_d, rows_per_block, p->d_bs);
  else
    sosfirst::first_order_single_kernel<<<grid, 128, 0, st>>>(g, p->d_C, I1_d, I1_copy_d, rows_per_block);
  return launch_check(p);
}

int sos_first_order2(sos_plan* p, const double* C_h, double* I1_d, double* I1_copy_d, void* stream) {
  if (!p || !C_h || !I1_d || I1_copy_d == I1_d) return SOS_ERR_INVALID;
  SOS_GUARD(p);
  NvtxRange nvtx("sos:first_order");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const GridDev& g = p->dev;
  const size_t bytes = sizeof(double) * g.S * 2 * g.N;
  double* buf;
  cudaEvent_t ev;
  int r = first_order_stage(p, &buf, &ev);
  if (r) return r;
  std::memcpy(buf, C_h, bytes);
  SOS_CUDA(cudaMemcpyAsync(p->d_C, buf, bytes, cudaMemcpyHostToDevice, st));
  SOS_CUDA(cudaEventRecord(ev, st));
  return first_order_launch(p, I1_d, I1_copy_d, st);
}

// C[s][0][m] = P0[ia][m] * w0,  C[s][1][m] = (P0[ia][m] * w0) * w1 + (P0[ie][m] * w2) * w3 -- every product and the sum rounded
// separately (no contraction into FMAs): the same bits as the host arithmetic the reference does on its P0 vectors
__global__ void __launch_bounds__(256)
first_order_coef_kernel(const double* __restrict__ tab, const double* __restrict__ w, const int* __restrict__ idx, double* __restrict__ C, int N) {
  const int s = blockIdx.y, m = blockIdx.x * 256 + threadIdx.x;
  if (m >= N) return;
  const int ia = idx[2 * s], ie = idx[2 * s + 1];
  const double c0 = __dmul_rn(tab[static_cast<size_t>(ia) * N + m], w[4 * s]);
  const double e = __dmul_rn(__dmul_rn(tab[static_cast<size_t>(ie) * N + m], w[4 * s + 2]), w[4 * s + 3]);
  C[(static_cast<size_t>(s) * 2) * N + m] = c0;
  C[(static_cast<size_t>(s) * 2 + 1) * N + m] = __dadd_rn(__dmul_rn(c0, w[4 * s + 1]), e);
}

int sos_first_order_tab(sos_plan* p, const double* P0tab_h, int n_tab, const int* idx_h, const double* w_h, double* I1_d,
                        double* I1_copy_d, void* stream) {
  if (!p || !P0tab_h || !idx_h || !w_h || !I1_d || I1_copy_d == I1_d || n_tab < 1) return SOS_ERR_INVALID;
  SOS_GUARD(p);
  NvtxRange nvtx("sos:first_order");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const GridDev& g = p->dev;
  const size_t S = g.S, N = g.N;
  // staging layout (doubles): [n_tab][N] table | [S][4] weights | [S][2] indices (ints); it must fit the [S][2][N] staging buffer
  const size_t tab_d = static_cast<size_t>(n_tab) * N, all_d = tab_d + 4 * S + S;
  if (all_d > S * 2 * N) return SOS_ERR_UNSUPPORTED;
  for (size_t i = 0; i < 2 * S; ++i)
    if (idx_h[i] < 0 || idx_h[i] >= n_tab) return SOS_ERR_INVALID;
  if (!p->d_Ctab) {
    int r = dev_alloc(p, &p->d_Ctab, S * 2 * N);
    if (r) return r;
    SOS_CUDA(cudaStreamSynchronize(nullptr));  // (the pool allocates on the legacy default stream; once per plan)
  }
  double* buf;
  cudaEvent_t ev;
  int r = first_order_stage(p, &buf, &ev);
  if (r) return r;
  std::memcpy(buf, P0tab_h, sizeof(double) * tab_d);
  std::memcpy(buf + tab_d, w_h, sizeof(double) * 4 * S);
  std::memcpy(buf + tab_d + 4 * S, idx_h, sizeof(int) * 2 * S);
  SOS_CUDA(cudaMemcpyAsync(p->d_Ctab, buf, sizeof(double) * all_d, cudaMemcpyHostToDevice, st));
  SOS_CUDA(cudaEventRecord(ev, st));
  dim3 cg(static_cast<unsigned>((N + 255) / 256), static_cast<unsigned>(S));
  first_order_coef_kernel<<<cg, 256, 0, st>>>(p->d_Ctab, p->d_Ctab + tab_d, reinterpret_cast<const int*>(p->d_Ctab + tab_d + 4 * S), p->d_C,
                                              static_cast<int>(N));
  r = launch_check(p, "first_order_coef_kernel");
  if (r) return r;
  return first_order_launch(p, I1_d, I1_copy_d, st);
}

static int source_impl(sos_plan* p, const double* In1_d, double* J_d, int seg_begin, int seg_end, void* stream,
                       const double* const* peers = nullptr, int n_peers = 0, const int* peer_col = nullptr, bool skip_lowrank = false);

int sos_source(sos_plan* p, const double* In1_d, double* J_d, void* stream) {
  return source_impl(p, In1_d, J_d, 0, 0x7fffffff, stream);
}

int sos_source_rows(sos_plan* p, const double* In1_d, double* J_d, int row0, int row1, void* stream) {
  if (!p) return SOS_ERR_INVALID;
  SOS_GUARD(p);
  // row-chunked contraction: single scenario, single region (the mu-sharded large grid), 64-row granularity
  if (p->dev.S != 1 || p->dev.nreg != 1) return SOS_ERR_UNSUPPORTED;
  if (row0 < 0 || row1 > p->dev.L || row0 >= row1 || (row0 % p->gemm_bm) != 0) return SOS_ERR_INVALID;
  const int seg0 = row0 / sosgemm::SEG_ROWS;
  const int seg1 = (row1 + sosgemm::SEG_ROWS - 1) / sosgemm::SEG_ROWS;
  return source_impl(p, In1_d, J_d, seg0, seg1, stream);
}

int sos_source_peers(sos_plan* p, const double* const* In1_peers_d, int n_peers, const int* peer_col, double* J_d, void* stream) {
  if (!p || !In1_peers_d || !peer_col || n_peers < 1 || n_peers > SOS_MAX_PEERS) return SOS_ERR_INVALID;
  SOS_GUARD(p);
  if (peer_col[0] != 0 || peer_col[n_peers] != p->dev.N) return SOS_ERR_INVALID;
  for (int r = 0; r < n_peers; ++r)
    if (!In1_peers_d[r] || peer_col[r + 1] <= peer_col[r] || (peer_col[r] % sosgemm::BK) != 0) return SOS_ERR_INVALID;
  return source_impl(p, In1_peers_d[0], J_d, 0, 0x7fffffff, stream, In1_peers_d, n_peers, peer_col);
}

// ---- CUDA IPC helpers: buffers that peer ranks (one process per GPU) map into their address space ----
int sos_ipc_alloc(size_t bytes, void** ptr_d, unsigned char* handle64) {
  if (!ptr_d || !handle64 || bytes == 0) return SOS_ERR_INVALID;
  SOS_CUDA(cudaMalloc(ptr_d, bytes));
  SOS_CUDA(cudaMemset(*ptr_d, 0, bytes));
  cudaIpcMemHandle_t h;
  SOS_CUDA(cudaIpcGetMemHandle(&h, *ptr_d));
  static_assert(sizeof(h) == 64, "IPC handle size");
  std::memcpy(handle64, &h, 64);
  return SOS_OK;
}
int sos_ipc_open(const unsigned char* handle64, void** ptr_d) {
  if (!ptr_d || !handle64) return SOS_ERR_INVALID;
  cudaIpcMemHandle_t h;
  std::memcpy(&h, handle64, 64);
  SOS_CUDA(cudaIpcOpenMemHandle(ptr_d, h, cudaIpcMemLazyEnablePeerAccess));
  return SOS_OK;
}
int sos_ipc_close(void* ptr_d) {
  if (!ptr_d) return SOS_OK;
  SOS_CUDA(cudaIpcCloseMemHandle(ptr_d));
  return SOS_OK;
}
int sos_ipc_free(void* ptr_d) {
  if (!ptr_d) return SOS_OK;
  SOS_CUDA(cudaFree(ptr_d));
  return SOS_OK;
}
int sos_copy_d2d(void* dst_d, const void* src_d, size_t bytes, void* stream) {
  if (!dst_d || !src_d) return SOS_ERR_INVALID;
  SOS_CUDA(cudaMemcpyAsync(dst_d, src_d, bytes, cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream)));
  return SOS_OK;
}

static int source_impl(sos_plan* p, const double* In1_d, double* J_d, int seg_begin, int seg_end, void* stream,
                       const double* const* peers, int n_peers, const int* peer_col, bool skip_lowrank) {
  NvtxRange nvtx("sos:source_contraction");
  if (!p || !In1_d || !J_d) return SOS_ERR_INVALID;
  SOS_GUARD(p);
  if (!p->maps_A_ready) return SOS_ERR_STATE;
  if ((reinterpret_cast<uintptr_t>(In1_d) & 15) || (reinterpret_cast<uintptr_t>(J_d) & 15)) return SOS_ERR_INVALID;
  const GridDev& g = p->dev;
  auto it = p->map_cache.find(In1_d);
  if (it == p->map_cache.end()) {
    CUtensorMap m;
    int r = encode_2d(&m, In1_d, g.N, static_cast<uint64_t>(g.S) * g.L, g.ld, sosgemm::BK, sosgemm::SEG_ROWS,
                      CU_TENSOR_MAP_SWIZZLE_128B);
    if (r) return r;
    if (p->map_cache.size() > 64) p->map_cache.clear();
    it = p->map_cache.emplace(In1_d, m).first;
  }
  p->gp.map_I = it->second;
  p->gp.n_peers = 0;
  if (peers) {
    for (int r = 0; r < n_peers; ++r) {
      auto ip = p->map_cache.find(peers[r]);
      if (ip == p->map_cache.end()) {
        CUtensorMap m;
        int rr = encode_2d(&m, peers[r], g.N, static_cast<uint64_t>(g.S) * g.L, g.ld, sosgemm::BK, sosgemm::SEG_ROWS,
                           CU_TENSOR_MAP_SWIZZLE_128B);
        if (rr) return rr;
        ip = p->map_cache.emplace(peers[r], m).first;
      }
      p->gp.map_peer[r] = ip->second;
      p->gp.peer_col[r] = peer_col[r];
    }
    p->gp.peer_col[n_peers] = peer_col[n_peers];
    p->gp.n_peers = n_peers;
  }
  p->gp.plan = p->d_tile_plan;
  p->gp.work_counter = p->d_work_counter;
  p->gp.active_list = p->d_active_list;
  p->gp.ct0 = g.col0 / p->gemm_bn;
  p->gp.n_col_tiles = (g.col1 + p->gemm_bn - 1) / p->gemm_bn - p->gp.ct0;
  p->gp.split_passes = p->split_passes;
  p->gp.seg_begin = seg_begin;
  p->gp.seg_end = seg_end;
  p->gp.L = g.L;
  p->gp.N = g.N;
  p->gp.ld = g.ld;
  p->gp.J = J_d;
  p->gp.scen = g.scen;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  SOS_CUDA(cudaMemsetAsync(p->d_work_counter, 0, sizeof(int), st));
  const bool full_columns = g.col0 == 0 && g.col1 == g.N;
  const bool layered = p->layers.n > 1;
  if (layered && seg_begin == 0 && seg_end == 0x7fffffff) { seg_begin = p->layer_seg_begin; seg_end = p->layer_seg_end; p->gp.seg_begin = seg_begin; p->gp.seg_end = seg_end; }
  const bool use_fold = p->fold && full_columns && !peers && (layered || (seg_begin == 0 && seg_end == 0x7fffffff));
  // inside sos_solve with a generated source only the aerosol rows have dense tiles: the kernel then decides per launch,
  // from the device-built tile plan, whether to split k (few scenarios still iterating) -- their J rows start from zero
  const bool dyn_ksplit = use_fold && skip_lowrank && p->fold_ksplit == 1 && !p->split_passes && g.nreg == 3 && g.M >= 64 &&
                          env_int("SOS_B200_DYN_KSPLIT", 1) != 0;
  if (use_fold && p->fold_ksplit > 1) {
    // split-k tiles add two partials per element into a zeroed J
    SOS_CUDA(cudaMemsetAsync(J_d, 0, static_cast<size_t>(g.S) * g.L * g.ld * sizeof(double), st));
  } else if (dyn_ksplit) {
    zero_active_rows_kernel<<<dim3(g.rstart[2] - g.rstart[1], g.S), 256, 0, st>>>(J_d, g.ld, g.L, g.rstart[1], g.state);
    int rz = launch_check(p, "zero_active_rows_kernel");
    if (rz) return rz;
  } else if (p->split_passes) {
    const int r0 = g.rstart[1], r1 = g.rstart[2];
    dim3 zgrid((g.N + 255) / 256, r1 - r0, g.S);
    zero_rows_kernel<<<zgrid, 256, 0, st>>>(J_d, g.ld, g.L, r0, r1, g.N);
    int rz = launch_check(p);
    if (rz) return rz;
  }
  ProfSpan span(p, 0, st);
  if (use_fold) {
    // centrosymmetric operands: half the DMMA work (gemm_fold.cuh)
    using FC = sosgemm::FoldCfg;
    sosgemm::FoldParams& f = p->fp;
    f.map_I = p->gp.map_I;
    f.plan = p->d_tile_plan;
    f.work_counter = p->d_work_counter;
    f.active_list = p->d_active_list;
    for (int c = 0; c < 2; ++c) { f.seg_row[c] = p->gp.seg_row[c]; f.seg_valid[c] = p->gp.seg_valid[c]; f.nseg[c] = p->gp.nseg[c]; }
    f.n_col_tiles = (g.M + FC::BN - 1) / FC::BN;
    f.split_passes = p->split_passes;
    f.ksplit = dyn_ksplit ? 0 : p->fold_ksplit;
    f.seg_begin = seg_begin;
    f.seg_end = seg_end;
    // One grid (a single scenario, one region: one operand group): the kernel lays its tiles out itself over the segment range,
    // so the tile height is free.  A tile is ~70 us of DMMA work per SM at M = 512 and a launch is whole tiles per SM: take the
    // 48-row shape when (waves x rows per tile) is smaller -- 10 000 rows: 6 x 48 instead of 5 x 64; a layer block of 1 269: 1 x 48.
    bool rows48 = false;
    const bool restricted_launch = f.seg_begin > 0 || f.seg_end != 0x7fffffff;
    if (p->fold_segs != 8 && restricted_launch) return SOS_ERR_UNSUPPORTED;  // (the device tile plan counts 56-row tiles)
    if (g.S == 1 && g.nreg == 1 && p->fold_xform && f.ksplit == 1 && env_int("SOS_FOLD_ROWS48", 1) != 0) {
      if (f.seg_end == 0x7fffffff) { f.seg_begin = 0; f.seg_end = p->nseg[0]; }
      const long long segs = std::min(f.seg_end, p->nseg[0]) - f.seg_begin;
      auto cost = [&](int segs_per_tile) {
        const long long tiles = (segs + segs_per_tile - 1) / segs_per_tile * f.n_col_tiles;
        return (tiles + p->n_sms - 1) / p->n_sms * segs_per_tile;
      };
      rows48 = cost(6) < cost(8);
    }
    f.L = g.L; f.N = g.N; f.M = g.M; f.Mh = (g.M + 15) / 16 * 16; f.ld = g.ld;
    f.J = J_d;
    f.scen = g.scen;
    if (p->n_lowrank_groups > 0 && !skip_lowrank) {  // (skipped inside sos_solve when the strip kernel rebuilds J for those rows)
      // rows whose operand is low rank (Rayleigh / isotropic): two skinny products, HBM bound (gemm_lowrank.cuh)
      sosgemm::LowRankParams lr;
      lr.I = In1_d; lr.J = J_d;
      for (int i = 0; i < SOS_MAX_PHASE; ++i) { lr.Ut[i] = p->lowrank_Ut[i]; lr.Vt[i] = p->lowrank_Vt[i]; }
      lr.plan = p->d_tile_plan; lr.active_list = p->d_active_list;
      lr.seg_row0 = p->gp.seg_row[0]; lr.seg_valid0 = p->gp.seg_valid[0]; lr.nseg0 = p->nseg[0];
      lr.L = g.L; lr.N = g.N; lr.ld = g.ld; lr.ldr = p->lowrank_ldr;
      lr.scen = g.scen;
      const long long units = static_cast<long long>(g.S) * p->nseg[0] * (sosgemm::SEG_ROWS / sosgemm::LR_ROWS);
      const int blocks = static_cast<int>(std::min<long long>((units + 7) / 8, 8LL * p->n_sms));
      if (p->lowrank_rp <= 4) sosgemm::jn_lowrank_kernel<4><<<blocks, sosgemm::LR_THREADS, 0, st>>>(lr);
      else sosgemm::jn_lowrank_kernel<16><<<blocks, sosgemm::LR_THREADS, 0, st>>>(lr);
      int rl = launch_check(p);
      if (rl) return rl;
    }
    ProfSpan dense_span(p, 3, st);
    if (rows48) sosgemm::jn_gemm_fold_kernel<true, 3><<<p->n_sms, sosgemm::FoldCfgT<3>::THREADS, sosgemm::FoldCfgT<3>::SMEM, st>>>(f);
    else if (p->fold_segs == 7 && !restricted_launch)
      sosgemm::jn_gemm_fold_kernel<true, 7, 1, 8, 2><<<p->n_sms, sosgemm::FoldCfgT<7, 1, 8, 2>::THREADS, sosgemm::FoldCfgT<7, 1, 8, 2>::SMEM, st>>>(f);
    else if (p->fold_xform) sosgemm::jn_gemm_fold_kernel<true><<<p->n_sms, FC::THREADS, FC::SMEM, st>>>(f);
    else sosgemm::jn_gemm_fold_kernel<false><<<p->n_sms, FC::THREADS, FC::SMEM, st>>>(f);
    return launch_check(p, "jn_gemm_fold_kernel");
  }
  if (p->fold && (p->premix || p->n_lowrank_groups)) return SOS_ERR_UNSUPPORTED;  // the device tile plan has fold-only group classes
  // 64 x 128 tiles with 8 consumer warps of 32 x 32 (profiles/r01_gemm_variants.md), or 128 x 144 with 12 warps of 32 x 48
  if (p->gemm_bn == 144)
    sosgemm::jn_gemm_dmma_kernel<4, 3, 4, 6><<<p->n_sms, sosgemm::Cfg<4, 3, 4, 6>::THREADS, sosgemm::Cfg<4, 3, 4, 6>::SMEM, st>>>(p->gp);
  else
    sosgemm::jn_gemm_dmma_kernel<2, 4, 4, 4><<<p->n_sms, sosgemm::Cfg<2, 4, 4, 4>::THREADS, sosgemm::Cfg<2, 4, 4, 4>::SMEM, st>>>(p->gp);
  return launch_check(p);
}

// SrcGen of order n (n < 0: every J row is read from memory, every I_n row stored)
static sossweep::SrcGen source_gen(const sos_plan* p, int n) {
  sossweep::SrcGen sg;
  std::memset(&sg, 0, sizeof(sg));
  sg.zu_end = p->dev.N;
  if (n < 0) return sg;
  sg.cj = p->d_cj[n & 1];
  sg.cj_out = p->d_cj[(n + 1) & 1];
  sg.Lp = p->dev.L;
  sg.proj = p->d_proj;
  sg.nslots = p->gen_nslots;
  sg.zlo = p->gen_zlo;
  sg.zu_end = p->gen_zu_end;
  sg.zu_proj = std::min(p->dev.M + 1 + sossweep::ZONE_UP, p->dev.N);
  sg.store_all = env_int("SOS_B200_GENSRC_STORE_ALL", 0);
  sg.ldr = p->lowrank_ldr;
  for (int i = 0; i < SOS_MAX_PHASE; ++i) {
    sg.rank[i] = p->lowrank_rank[i];
    sg.Ut[i] = p->lowrank_Ut[i];
  }
  return sg;
}

// convergence bookkeeping of the order just accumulated + tile plan of the next contraction (one launch)
static int order_end(sos_plan* p, int order_arg, cudaStream_t st) {
  const bool pm = p->fold && p->d_members_premix != nullptr;  // fold-mode tables (build_fold_tables)
  // (sharded plans: the CTA also copies the halo rows to the neighbours -- more threads, more loads in flight)
  order_end_kernel<<<1, p->layers.n > 1 ? 1024 : 256, 0, st>>>(p->dev, order_arg, p->d_order, pm ? p->groups_premix : p->groups,
                                                               pm ? p->d_members_premix : p->d_members, p->d_active_list, p->d_tile_plan, p->nseg[0], p->nseg[1],
                                                               p->fold ? p->fold_segs : p->gemm_bm / sosgemm::SEG_ROWS, p->split_passes, p->layers);
  return launch_check(p, "order_end_kernel");
}

static int sweeps_impl(sos_plan* p, const double* J_d, double* In_d, double* I_d, double* saved_d, cudaStream_t st, int gen_order = -1,
                       bool in_order_loop = false) {
  const GridDev& g = p->dev;
  const sossweep::SrcGen sg = source_gen(p, gen_order);
  NvtxRange nvtx("sos:layer_sweeps");
  ProfSpan span(p, 1, st);
  const int T = sossweep::LOCAL_THREADS;
  dim3 cgrid((g.M - 1 + T - 1) / T + (g.N - g.M - 1 + T - 1) / T, g.c_hi - g.c_lo, g.S);
  const bool layered = p->layers.n > 1;
  if (brdf_missing(p)) return SOS_ERR_STATE;
  if (layered && !in_order_loop) return SOS_ERR_UNSUPPORTED;  // sharded plans run whole orders only (sos_solve): the exchange ends in order_end_kernel
  if (layered && In_d != p->layers.In[p->layers.rank]) return SOS_ERR_INVALID;  // the neighbours write their halo rows into the registered field
  {
    sossweep::sweep_local_kernel<<<cgrid, T, 0, st>>>(g, sg, J_d, p->d_aggD, p->d_aggU);
    int r = launch_check(p, "sweep_local_kernel");
    if (r) return r;
  }
  if (g.nreg == 1 && g.surface == SOS_SURFACE_NONE) {
    // nothing couples the columns: a two-level scan per column, 16 columns per CTA (sharded plans exchange their chunk
    // aggregates with the peers inside this kernel)
    const int T3 = sossweep::CARRY_COLS;
    const size_t smem = 2 * static_cast<size_t>(g.nchunks + 1) * sizeof(double);
    if (smem > 30 * 1024) return SOS_ERR_UNSUPPORTED;
    sossweep::sweep_carry_cols_kernel<<<dim3((g.N + T3 - 1) / T3, g.S), T3 * sossweep::CARRY_GROUPS, smem, st>>>(g, p->d_aggD, p->d_aggU, p->d_carryD,
                                                                                                           p->d_carryU, p->layers);
    int r = launch_check(p, "sweep_carry_cols_kernel");
    if (r) return r;
  } else {
    const size_t smem = (g.N + 32 + 2 * (g.nchunks + 1)) * sizeof(double);
    if (p->brdf_nk == 2)
      sossweep::sweep_carry_kernel<2><<<g.S, sossweep::CARRY_THREADS, smem, st>>>(g, sg, J_d, p->d_aggD, p->d_aggU, p->d_carryD,
                                                                                  p->d_carryU, brdf_dev(p));
    else if (p->brdf_nk == 1)
      sossweep::sweep_carry_kernel<1><<<g.S, sossweep::CARRY_THREADS, smem, st>>>(g, sg, J_d, p->d_aggD, p->d_aggU, p->d_carryD,
                                                                                  p->d_carryU, brdf_dev(p));
    else
      sossweep::sweep_carry_kernel<0><<<g.S, sossweep::CARRY_THREADS, smem, st>>>(g, sg, J_d, p->d_aggD, p->d_aggU, p->d_carryD,
                                                                                  p->d_carryU, sosbrdf::BrdfDev{});
    int r = launch_check(p, "sweep_carry_kernel");
    if (r) return r;
  }
  {
    ProfSpan apply_span(p, 2, st);
    if ((g.M & 1) && g.col0 == 0 && g.col1 == g.N && I_d) {
      // odd M: every column pair is 16-byte aligned and inside one half -> two columns per thread
      const int T2 = 2 * sossweep::APPLY2_THREADS;
      dim3 grid2((g.M - 1 + T2 - 1) / T2 + (g.N - g.M - 1 + T2 - 1) / T2, g.c_hi - g.c_lo, g.S);
      sossweep::sweep_apply2_kernel<<<grid2, sossweep::APPLY2_THREADS, 0, st>>>(g, sg, J_d, In_d, p->d_carryD, p->d_carryU, I_d, saved_d);
    } else {
      sossweep::sweep_apply_kernel<<<cgrid, T, 0, st>>>(g, sg, J_d, In_d, p->d_carryD, p->d_carryU, I_d, saved_d);
    }
    int r = launch_check(p, "sweep_apply_kernel");
    if (r) return r;
  }
  {
    // per-warp buffer of the downward values next to mu = 0-: the widest extrapolation class (0.06 M) + 5
    // sources, or all non-standard columns, whichever is more (with a generated source: the plan-wide zone)
    const int down = std::max(g.M - g.first_small, g.widx[3] + 6) + 1;
    int zone_buf = std::min(g.M, down);
    if (gen_order >= 0) zone_buf = std::max(zone_buf, g.M - p->gen_zlo);
    const size_t smem = static_cast<size_t>(zone_buf + sossweep::ZONE_UP + 4) * sossweep::ZONE_ROWS * sizeof(double);
    if (smem > 48 * 1024) {
      if (smem > 200 * 1024) return SOS_ERR_UNSUPPORTED;
      cudaFuncSetAttribute(sossweep::sweep_zone_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    }
    dim3 grid((g.row1 - g.row0 + sossweep::ZONE_ROWS - 1) / sossweep::ZONE_ROWS, g.S);
    sossweep::sweep_zone_kernel<<<grid, 32 * sossweep::ZONE_ROWS, smem, st>>>(g, sg, J_d, In_d, I_d, saved_d, zone_buf);
    int r = launch_check(p, "sweep_zone_kernel");
    if (r) return r;
  }
  return SOS_OK;  // (sharded plans: halo rows and ratios travel in order_end_kernel)
}

int sos_sweeps(sos_plan* p, const double* J_d, double* In_d, double* I_d, void* stream) {
  if (!p || !J_d || !In_d) return SOS_ERR_INVALID;
  SOS_GUARD(p);
  return sweeps_impl(p, J_d, In_d, I_d, nullptr, static_cast<cudaStream_t>(stream));
}

int sos_converge(sos_plan* p, int order, void* stream) {
  if (!p) return SOS_ERR_INVALID;
  SOS_GUARD(p);
  sossweep::converge_kernel<<<1, 256, 0, static_cast<cudaStream_t>(stream)>>>(p->dev, order, p->d_order);
  int r = launch_check(p);
  if (r) return r;
  return plan_tiles(p, static_cast<cudaStream_t>(stream));
}

int sos_reset(sos_plan* p, const double* I1_d, void* stream) {
  if (!p || !I1_d) return SOS_ERR_INVALID;
  SOS_GUARD(p);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  sossweep::reset_kernel<<<p->dev.S, 256, 0, st>>>(p->dev, I1_d, p->d_order);
  int r = launch_check(p);
  if (r) return r;
  sossweep::count_active_kernel<<<1, 256, 0, st>>>(p->dev);
  r = launch_check(p);
  if (r) return r;
  return plan_tiles(p, st);
}

int sos_get_results(sos_plan* p, sos_result* results_h, void* stream) {
  if (!p || !results_h) return SOS_ERR_INVALID;
  SOS_GUARD(p);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  std::vector<ScenState> tmp(p->dev.S);
  SOS_CUDA(cudaMemcpyAsync(tmp.data(), p->dev.state, sizeof(ScenState) * p->dev.S, cudaMemcpyDeviceToHost, st));
  SOS_CUDA(cudaStreamSynchronize(st));
  for (int s = 0; s < p->dev.S; ++s) {
    results_h[s].ratio_toa = tmp[s].ratio_toa;
    results_h[s].ratio_surf = tmp[s].ratio_surf;
    results_h[s].n_orders = tmp[s].n_orders;
    results_h[s].active = tmp[s].active;
    results_h[s].status = tmp[s].status;
    results_h[s].reserved = 0;
  }
  return SOS_OK;
}

// can this solve run on the fused strip kernel, and with generated J?
static bool gen_usable(const sos_plan* p) {
  const GridDev& g = p->dev;
  return p->gen_ok && !p->gen_disabled && g.col0 == 0 && g.col1 == g.N;
}
static bool gen_applies(const sos_plan* p) {
  // the molecular rows leave the contraction only in fold mode (class-3 groups of the tile plan) and only with the
  // closed-form rank <= 2 factors; otherwise every J row is read from memory
  if (!p->fold || p->n_lowrank_groups == 0) return false;
  for (int i = 0; i < SOS_MAX_PHASE; ++i)
    if (p->lowrank_rank[i] > 2) return false;
  return true;
}

// one scattering order: source (dense rows) -> sweeps -> convergence bookkeeping -> tile plan of the next contraction
static int order_body(sos_plan* p, double* I_d, double* In_d, double* J_d, double* saved, int n, bool gen, cudaStream_t st,
                      bool device_order) {
  int rc = source_impl(p, In_d, J_d, 0, 0x7fffffff, st, nullptr, 0, nullptr, gen);
  if (rc) return rc;
  rc = sweeps_impl(p, J_d, In_d, I_d, saved, st, gen ? n : -1, true);
  if (rc) return rc;
  // (inside a graph the order number comes from the device-side counter: replays cannot change kernel arguments)
  return order_end(p, device_order ? -1 : n, st);
}

// The order loop is launch-latency bound for small batches (a single default-grid solve: ~45 us of kernels per order
// behind ~10 launches) and keeps one host thread per GPU busy for large ones.  Two consecutive orders (even + odd: the
// source coefficients ping-pong between two buffers) are captured once per (plan, field buffers) into a CUDA graph and
// replayed; every kernel takes what changes from device memory (active list, tile plan, order counter) and exits at once
// when nothing is active, so replays past convergence cost only their launch.  Returns nullptr when the order body
// cannot be captured (the caller then launches kernel by kernel).
static sos_plan::OrderGraph* order_graph(sos_plan* p, double* I_d, double* In_d, double* J_d, bool gen) {
  for (auto& g : p->graphs) {
    if (g.I == I_d && g.In == In_d && g.J == J_d && g.gen == gen) {
      if (std::memcmp(&g.gp, &p->gp, sizeof(p->gp)) == 0 && std::memcmp(&g.fp, &p->fp, sizeof(p->fp)) == 0 && g.zlo == p->gen_zlo &&
          g.zu_end == p->gen_zu_end)
        return &g;
      drop_graphs(p);   // the plan's tables have changed since the capture
      break;
    }
  }
  if (!p->cap_stream && cudaStreamCreateWithFlags(&p->cap_stream, cudaStreamNonBlocking) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  for (auto& e : p->graph_ev)
    if (!e && cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  const long long l0 = p->launches;
  if (cudaStreamBeginCapture(p->cap_stream, cudaStreamCaptureModeRelaxed) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  int rc = order_body(p, I_d, In_d, J_d, nullptr, 2, gen, p->cap_stream, true);
  if (!rc) rc = order_body(p, I_d, In_d, J_d, nullptr, 3, gen, p->cap_stream, true);
  if (!rc && cudaMemcpyAsync(p->h_poll + kPollSlots, p->dev.n_active, sizeof(int), cudaMemcpyDeviceToHost, p->cap_stream) != cudaSuccess) rc = SOS_ERR_CUDA;
  cudaGraph_t graph = nullptr;
  const cudaError_t ee = cudaStreamEndCapture(p->cap_stream, &graph);
  const long long per_replay = p->launches - l0;
  p->launches = l0;
  if (rc || ee != cudaSuccess || !graph) {
    if (graph) cudaGraphDestroy(graph);
    cudaGetLastError();
    return nullptr;
  }
  sos_plan::OrderGraph og;
  og.I = I_d; og.In = In_d; og.J = J_d; og.gen = gen; og.launches = per_replay;
  std::memcpy(&og.gp, &p->gp, sizeof(p->gp));
  std::memcpy(&og.fp, &p->fp, sizeof(p->fp));
  og.zlo = p->gen_zlo; og.zu_end = p->gen_zu_end;
  if (cudaGraphInstantiate(&og.exec, graph, 0) != cudaSuccess) { cudaGraphDestroy(graph); cudaGetLastError(); return nullptr; }
  cudaGraphDestroy(graph);
  if (p->graphs.size() >= 4) drop_graphs(p);
  p->graphs.push_back(og);
  return &p->graphs.back();
}

int sos_solve(sos_plan* p, double* I_d, double* In_d, double* J_d, double* orders_d, int max_saved, int max_orders,
              int poll_every, sos_result* results_h, void* stream) {
  if (!p || !I_d || !In_d || !J_d) return SOS_ERR_INVALID;
  SOS_GUARD(p);
  NvtxRange nvtx("sos:solve");
  if (!p->maps_A_ready || brdf_missing(p)) return SOS_ERR_STATE;
  if (poll_every < 1) poll_every = 1;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const GridDev& g = p->dev;
  int r = sos_reset(p, I_d, stream);
  if (r) return r;
  const size_t field = static_cast<size_t>(g.S) * g.L * g.ld;
  const bool gen = gen_usable(p) && gen_applies(p) && p->layers.n <= 1;
  if (p->layers.n > 1 && orders_d) return SOS_ERR_UNSUPPORTED;
  if (gen) {
    // projections of the first order onto the molecular factors: what order 2 rebuilds its J from
    dim3 pg((g.L + 7) / 8, g.S);
    sossweep::project_rows_kernel<<<pg, 256, 0, st>>>(g, source_gen(p, 2), In_d, p->d_cj[0]);
    r = launch_check(p, "project_rows_kernel");
    if (r) return r;
  }
  // The host never blocks inside the loop: after every order the device-side "still active" counter
  // is copied to a pinned slot; the host looks at the newest slot that has already landed.  Kernels
  // of converged scenarios exit immediately, so the few orders enqueued past convergence cost only
  // their launch latency.
  const int nslots = kPollSlots;
  volatile int* poll = p->h_poll;
  for (int i = 0; i < nslots; ++i) poll[i] = -1;
  int rc = SOS_OK;
  int issued = 0;
  bool done = false;
  int next_check = 0;  // slot index next to be examined
  int n = 2;
  // ---- graph replays, two orders each (not while saving per-order fields, timing kernel classes or debugging launches) ----
  const bool graphs_on = env_int("SOS_B200_GRAPH", 1) != 0 && env_int("SOS_B200_SYNC_DEBUG", 0) == 0;
  if (graphs_on && !orders_d && !p->profiling && max_orders >= 3) {
    sos_plan::OrderGraph* og = order_graph(p, I_d, In_d, J_d, gen);
    if (og) {
      volatile int* gslot = p->h_poll + kPollSlots;
      *gslot = -1;
      int k = 0;
      while (!done && n + 1 <= max_orders) {
        if (k >= 3) cudaEventSynchronize(p->graph_ev[(k - 3) & 3]);   // run-ahead: at most three replays (six orders)
        if (*gslot == 0) { done = true; break; }
        if (cudaGraphLaunch(og->exec, st) != cudaSuccess) { g_last_cuda_error = "cudaGraphLaunch failed"; return SOS_ERR_CUDA; }
        cudaEventRecord(p->graph_ev[k & 3], st);
        p->launches += og->launches;
        ++k;
        n += 2;
      }
      if (!done && n <= max_orders) {   // an odd remainder up to max_orders: know first whether it is needed at all
        cudaStreamSynchronize(st);
        if (*gslot == 0) done = true;
      }
    }
  }
  for (; n <= max_orders && !done; ++n) {
    double* saved = (orders_d && n - 2 < max_saved) ? orders_d + static_cast<size_t>(n - 2) * field : nullptr;
    rc = order_body(p, I_d, In_d, J_d, saved, n, gen, st, false);
    if (rc) break;
    const int slot = issued % nslots;
    if (issued >= nslots) poll[slot] = -1;  // that copy finished long ago (run-ahead is bounded below)
    cudaError_t e = cudaMemcpyAsync(const_cast<int*>(&poll[slot]), g.n_active, sizeof(int), cudaMemcpyDeviceToHost, st);
    if (e != cudaSuccess) { g_last_cuda_error = cudaGetErrorString(e); rc = SOS_ERR_CUDA; break; }
    ++issued;
    if (issued % poll_every == 0) {
      // non-blocking look at the slots that have landed so far
      while (next_check < issued && poll[next_check % nslots] >= 0) {
        if (poll[next_check % nslots] == 0) done = true;
        ++next_check;
      }
      // bound the run-ahead so a long tail of no-op orders cannot pile up
      if (!done && issued - next_check >= 8) {
        cudaStreamSynchronize(st);
      }
    }
  }
  if (rc) return rc;
  if (gen) {
    // a blend that left the columns whose raw I_n is kept cannot be finished: switch this plan to stored sources
    // and ask the caller to run the solve again (I_d / In_d have been consumed)
    std::vector<sos_result> tmp(g.S);
    rc = sos_get_results(p, tmp.data(), stream);
    if (rc) return rc;
    for (int s = 0; s < g.S; ++s)
      if (tmp[s].status & SOS_STATUS_STRIP_FALLBACK) { p->gen_disabled = true; return SOS_ERR_RETRY; }
  }
  if (results_h) {
    rc = sos_get_results(p, results_h, stream);
    if (rc) return rc;
    // the loop stopped at max_orders with these scenarios still above threshold: say so (the reference's while would go on)
    for (int s = 0; s < g.S; ++s)
      if (results_h[s].active) results_h[s].status |= SOS_STATUS_MAX_ORDERS;
  }
  return SOS_OK;
}

int sos_quadratures(sos_plan* p, const double* I_d, double direct_scale, const double* z_h, double* flux_up_d,
                    double* flux_down_d, double* net_flux_d, double* diffusivity_d, double* heating_d, void* stream) {
  if (!p || !I_d) return SOS_ERR_INVALID;
  SOS_GUARD(p);
  NvtxRange nvtx("sos:quadratures");
  if (heating_d && (!z_h || p->dev.nreg != 3)) return SOS_ERR_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const GridDev& g = p->dev;
  if (z_h) {
    SOS_CUDA(cudaMemcpyAsync(p->d_z, z_h, sizeof(double) * g.L, cudaMemcpyHostToDevice, st));
    SOS_CUDA(cudaStreamSynchronize(st));
  }
  {
    dim3 grid(g.L, g.S);
    sosquad::row_sums_kernel<<<grid, 256, 0, st>>>(g, I_d, p->d_sums);
    int r = launch_check(p);
    if (r) return r;
  }
  {
    dim3 grid((g.L + 127) / 128, g.S);
    sosquad::quadrature_outputs_kernel<<<grid, 128, 0, st>>>(g, p->d_sums, p->d_z, direct_scale, flux_up_d, flux_down_d,
                                                            net_flux_d, diffusivity_d, heating_d);
    return launch_check(p);
  }
}

// ---------------------------------------------------------------------------------------------
// FP64 throughput probes (roofline denominators; MEASURED_PEAKS.json has no FP64 entry)
// ---------------------------------------------------------------------------------------------
namespace {
__global__ void __launch_bounds__(256) probe_dfma(double* out, int iters, double a, double b) {
  double acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = threadIdx.x * 1e-3 + i;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int r = 0; r < 8; ++r)
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[i] = fma(acc[i], a, b);
  }
  double s = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) s += acc[i];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
__global__ void __launch_bounds__(256) probe_dmma(double* out, int iters, double a, double b) {
  double c[8][2];
#pragma unroll
  for (int i = 0; i < 8; ++i) { c[i][0] = threadIdx.x * 1e-3; c[i][1] = i; }
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int i = 0; i < 8; ++i)
        asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                     : "+d"(c[i][0]), "+d"(c[i][1]) : "d"(a), "d"(b));
  }
  double s = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) s += c[i][0] + c[i][1];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
}  // namespace

int sos_fp64_peak(int kind, int repeats, double* tflops) {
  if (!tflops || repeats < 1) return SOS_ERR_INVALID;
  int dev = 0;
  SOS_CUDA(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  SOS_CUDA(cudaGetDeviceProperties(&prop, dev));
  const int grid = prop.multiProcessorCount * 2, iters = 2048;
  double* out = nullptr;
  SOS_CUDA(cudaMalloc(&out, sizeof(double) * 256 * grid));
  cudaEvent_t e0, e1;
  SOS_CUDA(cudaEventCreate(&e0));
  SOS_CUDA(cudaEventCreate(&e1));
  double best = 0;
  for (int r = 0; r < repeats + 2; ++r) {
    SOS_CUDA(cudaEventRecord(e0));
    if (kind == 0) probe_dfma<<<grid, 256>>>(out, iters, 1.0000001, 1e-9);
    else probe_dmma<<<grid, 256>>>(out, iters, 1.0000001, 1e-9);
    SOS_CUDA(cudaEventRecord(e1));
    SOS_CUDA(cudaEventSynchronize(e1));
    float ms = 0;
    SOS_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    const double fl = (kind == 0) ? 2.0 * 64 * iters * 256.0 * grid : 512.0 * 32 * iters * 8.0 * grid;
    if (r >= 2) best = std::max(best, fl / ms * 1e-9);
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(out);
  *tflops = best;
  return SOS_OK;
}

}  // extern "C"
