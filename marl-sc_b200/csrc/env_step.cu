// env_step.cu - C-ABI entry points of K1 (fused environment step / reset) and the dispatch onto the
// per-team-width kernel instantiations (env_kernels.cuh, env_inst_g*.cu).
#include <cuda_runtime.h>

#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <new>
#include <string>

#include "env_compact.cuh"
#include "env_split.cuh"

namespace marlsc {

// K1d of the split step (env_split.cuh): cost -> reward per agent or team (multi_env.py:316-327), truncation flag.
__global__ void __launch_bounds__(256)
env_reward_kernel(const __grid_constant__ DevSpec sp, int64_t num_envs, const double* __restrict__ cost_alloc,
                  const double* __restrict__ cost_rows, float* __restrict__ rewards, uint8_t* __restrict__ truncated, int t) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= num_envs) return;
  const int W = sp.W;
  if (sp.scope == MARLSC_SCOPE_TEAM) {
    double rew = 0.0;
    for (int w = 0; w < W; ++w) rew += -((cost_rows[e * W + w] + cost_alloc[e * W + w]) * sp.scale);
    for (int w = 0; w < W; ++w) rewards[e * W + w] = (float)rew;
  } else {
    for (int w = 0; w < W; ++w) rewards[e * W + w] = (float)(-((cost_rows[e * W + w] + cost_alloc[e * W + w]) * sp.scale));
  }
  if (truncated) truncated[e] = (uint8_t)(t + 1 >= sp.episode_length);
}

thread_local std::string g_last_error;
std::atomic<long long> g_launches{0};

int set_error(int code, const std::string& msg) {
  g_last_error = msg;
  return code;
}

}  // namespace marlsc

using namespace marlsc;

struct marlsc_env {
  DevSpec ds;
  HostTables tb;
  int device = 0;
  int team = 1;        // lanes per environment in use
  int team_auto = 1;
  int tiny_fallback = 0;   // team_auto is 8 for a tiny SKU count: launches outside the split step run thread-per-environment
  int team_explicit = 0;   // marlsc_env_set_team_size chose the width: no automatic fallback
  int spl = 1;         // SKUs per lane of the instantiation in use
  void* d_blob = nullptr;  // one allocation holding every device table
  int max_smem_optin = 0;
  int force_generic = 0;   // tests: always run the generic instantiation
  int force_fused = 0;     // tests / comparisons: lean launches stay in the fused kernel
  double* d_work = nullptr;    // split step: [2, work_envs, W] cost partials
  int64_t work_envs = 0;
  int timing = 0;              // marlsc_env_set_timing: events around the launches of a step
  int timed_launches = 0;      // launches the last timed step made (4 split, 1 fused)
  cudaEvent_t marks[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
  int layout = MARLSC_LAYOUT_WIDE;     // state layout this handle works on (marlsc_env_layout)
  int line_stride = 128;               // rounds per environment of the library-owned line buffer (dense orders on a compact handle)
  uint16_t* d_lines = nullptr;         // [line_envs * line_stride, 32]
  int32_t* d_line_counts = nullptr;    // [line_envs]
  int64_t line_envs = 0;
  int32_t* h_overflow = nullptr;       // mapped host flag the conversion kernel sets when a stream does not fit
  int32_t* d_overflow = nullptr;       // its device alias
  cudaStream_t copy_stream = nullptr;        // marlsc_env_rollout_host: H2D copies of the next step
  cudaEvent_t ready[2] = {nullptr, nullptr};  // staging set filled
  cudaEvent_t done[2] = {nullptr, nullptr};   // staging set consumed by its step kernel
  int metrics_on = 0;                         // marlsc_env_set_metrics: episode accumulators registered
  marlsc_episode_metrics_t metrics = {};
};

namespace {

// SKUs-per-lane values instantiated for each team width (env_inst_g*.cu)
int pick_spl(int G, int S) {
  static const int k1[] = {1, 2, 4, 8, 0}, k2[] = {1, 2, 4, 0}, k4[] = {1, 2, 4, 0}, k8[] = {1, 4, 0},
                   k16[] = {1, 4, 8, 0}, k32[] = {1, 4, 8, 16, 0}, k64[] = {2, 4, 8, 0};
  const int* tbl = G == 1 ? k1 : G == 2 ? k2 : G == 4 ? k4 : G == 8 ? k8 : G == 16 ? k16 : G == 32 ? k32 : G == 64 ? k64 : nullptr;
  if (!tbl) return 0;
  const int need = skus_per_lane(S, G);
  for (; *tbl; ++tbl)
    if (*tbl >= need) return *tbl;
  return 0;
}

// Capabilities (env_core.cuh C_*) a launch needs; the lean kernel is used when they all fit kCapsLean.
uint32_t required_caps(const DevSpec& ds, const HostTables& tb, const marlsc_step_io_t* io) {
  uint32_t c = 0;
  const uint32_t F = ds.feat;
  if (ds.lead_mode == MARLSC_LEAD_STOCHASTIC) c |= C_STOCH;
  if (ds.norm == MARLSC_NORM_RATIO) c |= C_RATIO;
  if (ds.norm == MARLSC_NORM_MEANSTD) c |= C_MEANSTD;
  if (ds.need_ship) c |= C_SHIP;
  if (ds.need_fcst) c |= C_FCST;
  if (F & (MARLSC_F_DAYS_OF_SUPPLY | MARLSC_F_NET_INV_POSITION | MARLSC_F_DEMAND_VARIABILITY | MARLSC_F_DEMAND_HISTORY)) c |= C_XFEAT;
  if (F & (MARLSC_F_PIPELINE_AGG | MARLSC_F_DEMAND_HOME_AGG | MARLSC_F_ROLLING_MEAN_AGG)) c |= C_AGGX;
  if (ds.action_type != MARLSC_ACTION_DIRECT) c |= C_ACTX;
  if (!ds.unit_weights) c |= C_WEIGHT;
  for (uint8_t v : tb.prio_static) if (!v) c |= C_DYNPRIO;
  if (!tb.region_map.empty()) c |= C_REGMAP;
  if (ds.id_off) c |= C_IDHOT;
  if (ds.W > 32) c |= C_BIGW;
  if (ds.dh_mode == 2) c |= C_DHSMEM;
  if (ds.lost_type == MARLSC_LOST_COST) c |= C_LOSTCOST;
  if (ds.has_fixed) c |= C_FIXED;
  if (ds.max_splits < ds.W - 1) c |= C_SPLITLIM;
  if (io) {
    if (io->order_qty_bytes == 2) c |= C_QTY16;
    if (io->cost_breakdown || io->d_ordered || io->d_ship || io->d_ship_count || io->d_unfulfilled || io->d_lost_orders ||
        io->d_lost_sales) c |= C_DIAG;
  }
  return c;
}

int set_team(marlsc_env* env, int G) {
  const int spl = pick_spl(G, env->ds.S);
  if (!spl)
    return set_error(MARLSC_EUNSUPPORTED, "team size " + std::to_string(G) + " cannot hold " + std::to_string(env->ds.S) +
                                              " SKUs (at most 16 per lane, 512 SKUs in total); use a wider team");
  if (G > 32 && !pick_spl(32, env->ds.S))
    return set_error(MARLSC_EUNSUPPORTED, "a two-warp team needs the 32-lane instantiation as its generic fallback");
  env->team = G;
  env->spl = spl;
  return MARLSC_OK;
}

#define MARLSC_DISPATCH_G(team, FN, ...)                                                   \
  switch (team) {                                                                          \
    case 1: return FN##1(__VA_ARGS__);                                                     \
    case 2: return FN##2(__VA_ARGS__);                                                     \
    case 4: return FN##4(__VA_ARGS__);                                                     \
    case 8: return FN##8(__VA_ARGS__);                                                     \
    case 16: return FN##16(__VA_ARGS__);                                                   \
    case 32: return FN##32(__VA_ARGS__);                                                   \
    case 64: return FN##64(__VA_ARGS__);                                                   \
    default: return set_error(MARLSC_EINVAL, "team size must be a power of two in [1,64]"); \
  }

// Split-step workspace (cost partials between K1b/K1c and K1d), grown on demand. Growing synchronises the
// device, so reset sizes it up front.
int ensure_work(marlsc_env* env, int64_t num_envs) {
  if (env->work_envs >= num_envs) return MARLSC_OK;
  if (env->d_work) {
    MARLSC_CUDA(cudaDeviceSynchronize());
    MARLSC_CUDA(cudaFree(env->d_work));
    env->d_work = nullptr;
    env->work_envs = 0;
  }
  MARLSC_CUDA(cudaMalloc(reinterpret_cast<void**>(&env->d_work), sizeof(double) * 2 * (size_t)num_envs * env->ds.W));
  env->work_envs = num_envs;
  return MARLSC_OK;
}

// The split step covers what the lean instantiation covers, for teams of at least 8 lanes (and the SKUs-per-lane
// values the automatic team choice produces).
constexpr int64_t kTinySplitMaxEnvs = 4096;

bool split_ok(const marlsc_env* env) {
  if (env->force_fused) return false;
  const int g = env->team, k = env->spl;   // instantiated pairs, see MARLSC_DEFINE_SPLIT in env_inst_g*.cu
  return ((g == 8 || g == 16) && (k == 1 || k == 4)) || (g == 32 && (k == 1 || k == 4 || k == 8 || k == 16)) || g == 64;
}

// Configurations the compact layout and its fused kernel cover (include/marlsc_b200.h, MARLSC_LAYOUT_COMPACT).
bool compact_eligible(const DevSpec& ds, const HostTables& tb) {
  const uint32_t caps = required_caps(ds, tb, nullptr) & ~C_REGMAP;    // the region map is applied when lines are built
  if (caps & ~kCapsLean) return false;
  if (ds.dh_mode == 2) return false;                                    // home-demand block without a history plane
  if (ds.S <= 32 || ds.S > kCompactMaxS || (ds.S & 3)) return false;      // rows are read as 32-bit words of four cells
  if (ds.W > kCompactMaxW || ds.R > kCompactMaxR || ds.L > kCompactMaxL || !ds.perm5) return false;
  for (double v : tb.action_max) if (!(v >= 0.0 && v <= 255.0) || v != (double)(int)v) return false;
  return true;
}

// Line buffer for dense orders given to a compact handle, grown on demand (growing synchronises the device).
int ensure_lines(marlsc_env* env, int64_t num_envs) {
  if (!env->h_overflow) {
    MARLSC_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&env->h_overflow), sizeof(int32_t), cudaHostAllocMapped));
    *env->h_overflow = 0;
    MARLSC_CUDA(cudaHostGetDevicePointer(reinterpret_cast<void**>(&env->d_overflow), env->h_overflow, 0));
  }
  if (env->line_envs >= num_envs) return MARLSC_OK;
  if (env->d_lines) {
    MARLSC_CUDA(cudaDeviceSynchronize());
    MARLSC_CUDA(cudaFree(env->d_lines));
    MARLSC_CUDA(cudaFree(env->d_line_counts));
    env->d_lines = nullptr;
    env->d_line_counts = nullptr;
    env->line_envs = 0;
  }
  MARLSC_CUDA(cudaMalloc(reinterpret_cast<void**>(&env->d_lines), sizeof(uint16_t) * 32 * (size_t)num_envs * env->line_stride));
  MARLSC_CUDA(cudaMalloc(reinterpret_cast<void**>(&env->d_line_counts), sizeof(int32_t) * (size_t)num_envs));
  env->line_envs = num_envs;
  return MARLSC_OK;
}

int check_state(const marlsc_env* env, const marlsc_env_state_t* st) {
  if (!env || !st) return set_error(MARLSC_EINVAL, "null handle or state");
  if (st->layout != env->layout)
    return set_error(MARLSC_EINVAL, std::string("state.layout does not match the handle's layout (") +
                                        (env->layout == MARLSC_LAYOUT_COMPACT ? "COMPACT" : "WIDE") + ", see marlsc_env_layout)");
  if (env->h_overflow && *env->h_overflow)
    return set_error(MARLSC_EINVAL, "an earlier step's orders did not fit the line buffer (a stream needed more than line_stride "
                                    "rounds): raise it with marlsc_env_set_line_stride");
  if (st->num_envs < 1) return set_error(MARLSC_EINVAL, "num_envs must be positive");
  if (st->num_envs > (int64_t)0x7fffffff) return set_error(MARLSC_EINVAL, "num_envs too large");
  if (!st->inventory || !st->ring_qty) return set_error(MARLSC_EINVAL, "state.inventory / state.ring_qty are NULL");
  if (env->ds.lead_mode == MARLSC_LEAD_STOCHASTIC && !st->ring_lead)
    return set_error(MARLSC_EINVAL, "state.ring_lead is required with a stochastic lead-time sampler");
  if (env->ds.need_hist && !st->demand_hist) return set_error(MARLSC_EINVAL, "state.demand_hist is required by this configuration");
  if (env->ds.need_fcst && !st->forecast) return set_error(MARLSC_EINVAL, "state.forecast is required by this configuration");
  return MARLSC_OK;
}

template <typename T>
size_t blob_add(size_t& off, const std::vector<T>& v) {
  off = (off + 15) & ~size_t(15);
  const size_t at = off;
  off += v.size() * sizeof(T);
  return at;
}

}  // namespace

extern "C" {

int marlsc_env_create(const marlsc_env_spec_t* spec, int device, marlsc_env_t** out) {
  if (!spec || !out) return set_error(MARLSC_EINVAL, "null spec or out");
  marlsc_env* env = new (std::nothrow) marlsc_env();
  if (!env) return set_error(MARLSC_ENOMEM, "out of host memory");
  const std::string err = build_devspec(*spec, env->ds, env->tb);
  if (!err.empty()) {
    delete env;
    return set_error(MARLSC_EINVAL, err);
  }
  env->device = device;
  env->team_auto = auto_team_size(env->ds.S);
  // Tiny SKU counts: small batches (up to 4,096 environments) take the split step with 8-lane teams, which spreads an
  // environment over more lanes while most SMs would otherwise idle; larger batches, and launches the split step does
  // not cover (diagnostic outputs, generic capabilities, the fused-kernel switch), go thread-per-environment, see
  // marlsc_env_step.
  if (env->team_auto == 1 && (required_caps(env->ds, env->tb, nullptr) & ~kCapsLean) == 0 && pick_spl(8, env->ds.S) == 1) {
    env->team_auto = 8;
    env->tiny_fallback = 1;
  }
  if (set_team(env, env->team_auto) != MARLSC_OK) {
    const std::string msg = g_last_error;
    delete env;
    return set_error(MARLSC_EUNSUPPORTED, msg);
  }
  cudaError_t ce = cudaSetDevice(device);
  if (ce == cudaSuccess) ce = cudaDeviceGetAttribute(&env->max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
  if (ce != cudaSuccess) {
    delete env;
    return set_error(MARLSC_ECUDA, std::string("no usable CUDA device: ") + cudaGetErrorString(ce));
  }
  // pack every table into one device allocation
  const HostTables& t = env->tb;
  size_t off = 0;
  const size_t o_amax = blob_add(off, t.action_max), o_of = blob_add(off, t.out_fixed), o_ov = blob_add(off, t.out_var),
               o_if = blob_add(off, t.in_fixed), o_iv = blob_add(off, t.in_var), o_hr = blob_add(off, t.hold_rate),
               o_pr = blob_add(off, t.pen_rate), o_sw = blob_add(off, t.skw), o_le = blob_add(off, t.lead_exp),
               o_hm = blob_add(off, t.home), o_cl = blob_add(off, t.closest), o_rm = blob_add(off, t.region_map),
               o_pp = blob_add(off, t.prio), o_ps = blob_add(off, t.prio_static), o_om = blob_add(off, t.obs_mean),
               o_os = blob_add(off, t.obs_std), o_hk = blob_add(off, t.home_mask), o_l8 = blob_add(off, t.lead_u8),
               o_pm = blob_add(off, t.prio_perm), o_p5 = blob_add(off, t.perm5), o_p16 = blob_add(off, t.prio16),
               o_hw = blob_add(off, t.home_wh);
  std::vector<unsigned char> host(off + 16, 0);
  auto put = [&](size_t at, const void* src, size_t n) { if (n) std::memcpy(host.data() + at, src, n); };
  put(o_amax, t.action_max.data(), t.action_max.size() * 8); put(o_of, t.out_fixed.data(), t.out_fixed.size() * 8);
  put(o_ov, t.out_var.data(), t.out_var.size() * 8); put(o_if, t.in_fixed.data(), t.in_fixed.size() * 8);
  put(o_iv, t.in_var.data(), t.in_var.size() * 8); put(o_hr, t.hold_rate.data(), t.hold_rate.size() * 8);
  put(o_pr, t.pen_rate.data(), t.pen_rate.size() * 8); put(o_sw, t.skw.data(), t.skw.size() * 8);
  put(o_le, t.lead_exp.data(), t.lead_exp.size() * 4); put(o_hm, t.home.data(), t.home.size() * 4);
  put(o_cl, t.closest.data(), t.closest.size() * 4); put(o_rm, t.region_map.data(), t.region_map.size() * 4);
  put(o_pp, t.prio.data(), t.prio.size()); put(o_ps, t.prio_static.data(), t.prio_static.size());
  put(o_om, t.obs_mean.data(), t.obs_mean.size() * 4); put(o_os, t.obs_std.data(), t.obs_std.size() * 4);
  put(o_hk, t.home_mask.data(), t.home_mask.size() * 4); put(o_l8, t.lead_u8.data(), t.lead_u8.size());
  put(o_pm, t.prio_perm.data(), t.prio_perm.size() * 2);
  put(o_p5, t.perm5.data(), t.perm5.size() * 2); put(o_p16, t.prio16.data(), t.prio16.size()); put(o_hw, t.home_wh.data(), t.home_wh.size());
  ce = cudaMalloc(&env->d_blob, host.size());
  if (ce == cudaSuccess) ce = cudaMemcpy(env->d_blob, host.data(), host.size(), cudaMemcpyHostToDevice);
  if (ce != cudaSuccess) {
    if (env->d_blob) cudaFree(env->d_blob);
    delete env;
    return set_error(MARLSC_ECUDA, std::string("uploading tables: ") + cudaGetErrorString(ce));
  }
  unsigned char* b = static_cast<unsigned char*>(env->d_blob);
  auto D = [&](size_t at) { return reinterpret_cast<const double*>(b + at); };
  auto I = [&](size_t at) { return reinterpret_cast<const int32_t*>(b + at); };
  bind_tables(env->ds, D(o_amax), D(o_of), D(o_ov), D(o_if), D(o_iv), D(o_hr), D(o_pr), D(o_sw), I(o_le), I(o_hm),
              I(o_cl), t.region_map.empty() ? nullptr : I(o_rm), b + o_pp, b + o_ps,
              t.home_mask.empty() ? nullptr : reinterpret_cast<const uint32_t*>(b + o_hk), b + o_l8,
              t.obs_mean.empty() ? nullptr : reinterpret_cast<const float*>(b + o_om),
              t.obs_std.empty() ? nullptr : reinterpret_cast<const float*>(b + o_os));
  env->ds.prio_perm = t.prio_perm.empty() ? nullptr : reinterpret_cast<const uint16_t*>(b + o_pm);
  env->ds.perm5 = t.perm5.empty() ? nullptr : reinterpret_cast<const uint16_t*>(b + o_p5);
  env->ds.prio16 = t.prio16.empty() ? nullptr : b + o_p16;
  env->ds.home_wh = b + o_hw;
  env->ds.compact_ok = compact_eligible(env->ds, env->tb) ? 1 : 0;
  // cp.async.bulk.prefetch.L2 wants 16-byte aligned addresses and sizes: true for every environment's block when the
  // smallest one (W*S bytes of uint8 quantities) is a multiple of 16 (MARLSC_NO_PREFETCH=1 switches them off for A/B runs)
  env->ds.compact_prefetch = ((env->ds.W * env->ds.S) % 16 == 0 && !std::getenv("MARLSC_NO_PREFETCH")) ? 1 : 0;
  env->ds.feature_bulk = ((env->ds.W * env->ds.S) % 8 == 0 && std::getenv("MARLSC_FEATURE_BULK")) ? 1 : 0;   // opt-in: measured slower
  env->layout = env->ds.compact_ok ? MARLSC_LAYOUT_COMPACT : MARLSC_LAYOUT_WIDE;
  *out = env;
  return MARLSC_OK;
}

void marlsc_env_destroy(marlsc_env_t* env) {
  if (!env) return;
  if (env->copy_stream) cudaStreamDestroy(env->copy_stream);
  for (int i = 0; i < 2; ++i) {
    if (env->ready[i]) cudaEventDestroy(env->ready[i]);
    if (env->done[i]) cudaEventDestroy(env->done[i]);
  }
  if (env->d_blob) cudaFree(env->d_blob);
  if (env->d_work) cudaFree(env->d_work);
  if (env->d_lines) cudaFree(env->d_lines);
  if (env->d_line_counts) cudaFree(env->d_line_counts);
  if (env->h_overflow) cudaFreeHost(env->h_overflow);
  for (cudaEvent_t ev : env->marks)
    if (ev) cudaEventDestroy(ev);
  delete env;
}

int32_t marlsc_env_obs_dim(const marlsc_env_t* env) { return env ? env->ds.obs_dim : 0; }
int32_t marlsc_env_needs_history(const marlsc_env_t* env) { return env ? env->ds.need_hist : 0; }
int32_t marlsc_env_needs_forecast(const marlsc_env_t* env) { return env ? env->ds.need_fcst : 0; }
int32_t marlsc_env_team_size(const marlsc_env_t* env) { return env ? env->team : 0; }
int32_t marlsc_env_layout(const marlsc_env_t* env) { return env ? env->layout : 0; }

int marlsc_env_set_layout(marlsc_env_t* env, int32_t layout) {
  if (!env) return set_error(MARLSC_EINVAL, "null handle");
  if (layout != MARLSC_LAYOUT_WIDE && layout != MARLSC_LAYOUT_COMPACT) return set_error(MARLSC_EINVAL, "unknown layout");
  if (layout == MARLSC_LAYOUT_COMPACT && !env->ds.compact_ok)
    return set_error(MARLSC_EUNSUPPORTED, "this configuration does not qualify for the compact layout (see MARLSC_LAYOUT_COMPACT in marlsc_b200.h)");
  env->layout = layout;
  return MARLSC_OK;
}

int marlsc_env_set_line_stride(marlsc_env_t* env, int32_t rounds) {
  if (!env) return set_error(MARLSC_EINVAL, "null handle");
  if (rounds < 2 || rounds > 4096 || (rounds & 1)) return set_error(MARLSC_EINVAL, "line stride must be even and in [2, 4096]");
  if (env->d_lines) {
    MARLSC_CUDA(cudaSetDevice(env->device));
    MARLSC_CUDA(cudaDeviceSynchronize());
    MARLSC_CUDA(cudaFree(env->d_lines));
    MARLSC_CUDA(cudaFree(env->d_line_counts));
    env->d_lines = nullptr;
    env->d_line_counts = nullptr;
    env->line_envs = 0;
  }
  if (env->h_overflow) *env->h_overflow = 0;
  env->line_stride = rounds;
  return MARLSC_OK;
}

int marlsc_env_set_team_size(marlsc_env_t* env, int32_t tpe) {
  if (!env) return set_error(MARLSC_EINVAL, "null handle");
  if (env->layout == MARLSC_LAYOUT_COMPACT && tpe != 0)
    return set_error(MARLSC_EINVAL, "the compact layout runs one warp per environment; force MARLSC_LAYOUT_WIDE to choose a team size");
  if (tpe == 0) {
    env->team_explicit = 0;
    return set_team(env, env->team_auto);
  }
  if (tpe < 1 || tpe > 64 || (tpe & (tpe - 1))) return set_error(MARLSC_EINVAL, "team size must be a power of two in [1,64]");
  const int rc = set_team(env, tpe);
  if (rc == MARLSC_OK) env->team_explicit = 1;
  return rc;
}

int marlsc_env_set_generic(marlsc_env_t* env, int32_t on) {
  if (!env) return set_error(MARLSC_EINVAL, "null handle");
  if (on && env->layout == MARLSC_LAYOUT_COMPACT) return set_error(MARLSC_EINVAL, "force MARLSC_LAYOUT_WIDE first: the compact layout has one kernel");
  env->force_generic = on ? 1 : 0;
  return MARLSC_OK;
}

int marlsc_env_set_fused(marlsc_env_t* env, int32_t on) {
  if (!env) return set_error(MARLSC_EINVAL, "null handle");
  if (on && env->metrics_on && env->layout == MARLSC_LAYOUT_COMPACT)
    return set_error(MARLSC_EUNSUPPORTED, "the compact fused step kernel does not accumulate episode metrics (marlsc_env_set_metrics)");
  env->force_fused = on ? 1 : 0;                       // compact layout: the single fused kernel instead of the split step
  return MARLSC_OK;
}

int marlsc_env_set_metrics(marlsc_env_t* env, const marlsc_episode_metrics_t* m) {
  if (!env) return set_error(MARLSC_EINVAL, "null handle");
  if (!m) {
    env->metrics_on = 0;
    env->metrics = marlsc_episode_metrics_t{};
    return MARLSC_OK;
  }
  if (!m->holding_cost || !m->penalty_cost || !m->outbound_cost || !m->inbound_cost || !m->ordered_units || !m->shipped_units ||
      !m->episode_return || !m->demand_units || !m->lost_units)
    return set_error(MARLSC_EINVAL, "every marlsc_episode_metrics pointer is required");
  if (env->force_fused && env->layout == MARLSC_LAYOUT_COMPACT)
    return set_error(MARLSC_EUNSUPPORTED, "the compact fused step kernel does not accumulate episode metrics (marlsc_env_set_fused)");
  env->metrics = *m;
  env->metrics_on = 1;
  return MARLSC_OK;
}

int marlsc_env_set_timing(marlsc_env_t* env, int32_t on) {
  if (!env) return set_error(MARLSC_EINVAL, "null handle");
  MARLSC_CUDA(cudaSetDevice(env->device));
  if (on)
    for (cudaEvent_t& ev : env->marks)
      if (!ev) MARLSC_CUDA(cudaEventCreate(&ev));
  env->timing = on ? 1 : 0;
  env->timed_launches = 0;
  return MARLSC_OK;
}

int marlsc_env_last_timing(marlsc_env_t* env, float* ms, int32_t capacity) {
  if (!env || !ms) return set_error(MARLSC_EINVAL, "null handle or output");
  const int n = env->timed_launches;
  if (!env->timing || n == 0) return set_error(MARLSC_EINVAL, "no timed step: call marlsc_env_set_timing(env, 1) and step first");
  if (capacity < n) return set_error(MARLSC_EINVAL, "ms[] too small");
  MARLSC_CUDA(cudaEventSynchronize(env->marks[n]));
  for (int i = 0; i < n; ++i) MARLSC_CUDA(cudaEventElapsedTime(&ms[i], env->marks[i], env->marks[i + 1]));
  return n;
}

int marlsc_env_reset(marlsc_env_t* env, const marlsc_env_state_t* state, const int32_t* init_inventory, int32_t per_env,
                     float* obs, void* stream) {
  int rc = check_state(env, state);
  if (rc) return rc;
  if (!init_inventory || !obs) return set_error(MARLSC_EINVAL, "init_inventory and obs must not be NULL");
  MARLSC_CUDA(cudaSetDevice(env->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (env->metrics_on) {                               // a new episode: its accumulators start from zero
    const marlsc_episode_metrics_t& m = env->metrics;
    const size_t rows = sizeof(double) * (size_t)state->num_envs * env->ds.W, envs = sizeof(double) * (size_t)state->num_envs;
    for (double* p : {m.holding_cost, m.penalty_cost, m.outbound_cost, m.inbound_cost, m.ordered_units, m.shipped_units, m.episode_return})
      MARLSC_CUDA(cudaMemsetAsync(p, 0, rows, s));
    MARLSC_CUDA(cudaMemsetAsync(m.demand_units, 0, envs, s));
    MARLSC_CUDA(cudaMemsetAsync(m.lost_units, 0, envs, s));
  }
  if (env->layout == MARLSC_LAYOUT_COMPACT) {
    const LaunchArgs lc{env->ds, *state, env->max_smem_optin, true};
    return launch_reset_compact(lc, init_inventory, per_env, obs, s);
  }
  if (split_ok(env)) {
    rc = ensure_work(env, state->num_envs);
    if (rc) return rc;
  }
  const LaunchArgs la{env->ds, *state, env->max_smem_optin, false};
  // the state layout does not depend on the team width: two-warp teams reset through the 32-lane kernel
  const int team = env->team > 32 ? 32 : env->team;
  const int spl = env->team > 32 ? pick_spl(32, env->ds.S) : env->spl;
  MARLSC_DISPATCH_G(team, launch_reset_g, spl, la, init_inventory, per_env, obs, s)
}

}  // extern "C"

namespace {

// marlsc_env_step without the episode-metrics epilogue
int step_impl(marlsc_env_t* env, const marlsc_env_state_t* state, const marlsc_step_io_t* io, int32_t t, void* stream) {
  int rc = check_state(env, state);
  if (rc) return rc;
  if (!io) return set_error(MARLSC_EINVAL, "null io");
  if ((!io->actions && !io->action_qty && !io->base_stock_level) || !io->rewards || !io->obs)
    return set_error(MARLSC_EINVAL, "io.actions (or io.action_qty / io.base_stock_level), io.rewards and io.obs must not be NULL");
  if (io->base_stock_level && !io->actions && !io->action_qty && (env->layout != MARLSC_LAYOUT_COMPACT || env->force_fused))
    return set_error(MARLSC_EINVAL, "io.base_stock_level needs a handle with the COMPACT layout running the split step");
  if (io->lines) {
    if (env->layout != MARLSC_LAYOUT_COMPACT) return set_error(MARLSC_EINVAL, "io.lines needs a handle with the COMPACT layout");
    if (!io->line_offsets && !io->line_counts) return set_error(MARLSC_EINVAL, "io.lines needs io.line_offsets or io.line_counts");
    if (io->line_counts && (io->line_stride < 2 || (io->line_stride & 1))) return set_error(MARLSC_EINVAL, "line_stride must be positive and even with line_counts");
  } else if (!io->order_offsets && !io->order_counts) {
    return set_error(MARLSC_EINVAL, "one of io.lines / io.order_offsets / io.order_counts must not be NULL");
  }
  if (io->action_qty && env->layout != MARLSC_LAYOUT_COMPACT) return set_error(MARLSC_EINVAL, "io.action_qty needs a handle with the COMPACT layout");
  if (io->order_counts && io->order_stride < 1) return set_error(MARLSC_EINVAL, "order_stride must be positive with order_counts");
  if (io->order_qty_bytes != 1 && io->order_qty_bytes != 2) return set_error(MARLSC_EINVAL, "order_qty_bytes must be 1 or 2");
  if (env->ds.lead_mode == MARLSC_LEAD_STOCHASTIC && !io->actual_lead)
    return set_error(MARLSC_EINVAL, "io.actual_lead is required with a stochastic lead-time sampler");
  if (io->d_lost_sales && !io->d_unfulfilled) return set_error(MARLSC_EINVAL, "d_lost_sales needs d_unfulfilled");
  if (t < 0) return set_error(MARLSC_EINVAL, "timestep must be >= 0");
  MARLSC_CUDA(cudaSetDevice(env->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (env->layout == MARLSC_LAYOUT_COMPACT) {
    if (io->order_qty_bytes == 2 && !io->lines) return set_error(MARLSC_EUNSUPPORTED, "two-byte order quantities need MARLSC_LAYOUT_WIDE");
    if (io->cost_breakdown || io->d_ordered || io->d_ship || io->d_ship_count || io->d_unfulfilled || io->d_lost_orders || io->d_lost_sales)
      return set_error(MARLSC_EUNSUPPORTED, "the diagnostic outputs need MARLSC_LAYOUT_WIDE (marlsc_env_set_layout before the first reset)");
    const LaunchArgs lc{env->ds, *state, env->max_smem_optin, true};
    marlsc_step_io_t ioc = *io;
    if (env->timing) MARLSC_CUDA(cudaEventRecord(env->marks[0], s));
    int n_marks = 1;
    if (!io->lines) {                                  // dense orders: build the lines in the library's buffer first
      rc = ensure_lines(env, state->num_envs);
      if (rc) return rc;
      rc = launch_lines_from_orders(env->ds, state->num_envs, *io, env->line_stride, env->d_lines, env->d_line_counts, env->d_overflow, s);
      if (rc) return rc;
      ioc.lines = env->d_lines;
      ioc.line_offsets = nullptr;
      ioc.line_counts = env->d_line_counts;
      ioc.line_stride = env->line_stride;
      if (env->timing) MARLSC_CUDA(cudaEventRecord(env->marks[n_marks], s));
      ++n_marks;
    }
    if (!env->force_fused && state->num_envs * (int64_t)env->ds.W < (int64_t)0xffffffffLL) {
      // the step as row / environment kernels (K1a' place, K1b' allocate, K1c' features, K1d rewards)
      rc = ensure_work(env, state->num_envs);
      if (rc) return rc;
      const SplitWork wk{env->d_work, env->d_work + (size_t)env->work_envs * env->ds.W,
                         (env->timing && io->lines) ? env->marks : nullptr, env->metrics_on ? &env->metrics : nullptr};
      env->timed_launches = (env->timing && io->lines) ? 4 : 0;
      return launch_split_compact(lc, ioc, wk, t, s);
    }
    if (env->metrics_on)
      return set_error(MARLSC_EUNSUPPORTED, "episode metrics need the compact split step (not the fused kernel, fewer than 2^32 rows)");
    rc = launch_step_compact(lc, ioc, t, s);
    if (rc) return rc;
    if (env->timing) MARLSC_CUDA(cudaEventRecord(env->marks[n_marks], s));
    env->timed_launches = env->timing ? n_marks : 0;
    return MARLSC_OK;
  }
  const bool lean = !env->force_generic && (required_caps(env->ds, env->tb, io) & ~kCapsLean) == 0;
  const LaunchArgs la{env->ds, *state, env->max_smem_optin, lean};
  // the row kernels of the split step index (environment, warehouse) rows with 32 bits
  // automatic 8-lane teams of a tiny SKU count: the split step only wins while the batch leaves most SMs idle (3 x 2
  // network, 4,096 environments: 40 against 48 us, 27 against 42 us inside a CUDA graph); beyond that the
  // thread-per-environment kernel's single launch is faster (8,192: 49 against 52 us; 16,384: 52 against 69 us)
  const bool tiny = env->tiny_fallback && !env->team_explicit;
  const bool tiny_split = !tiny || state->num_envs <= kTinySplitMaxEnvs;
  if (lean && tiny_split && split_ok(env) && state->num_envs * (int64_t)env->ds.W < (int64_t)0xffffffffLL) {
    rc = ensure_work(env, state->num_envs);
    if (rc) return rc;
    const SplitWork wk{env->d_work, env->d_work + (size_t)env->work_envs * env->ds.W, env->timing ? env->marks : nullptr};
    env->timed_launches = env->timing ? 4 : 0;
    switch (env->team) {
      case 8: return launch_split_g8(env->spl, la, *io, wk, t, s);
      case 16: return launch_split_g16(env->spl, la, *io, wk, t, s);
      case 32: return launch_split_g32(env->spl, la, *io, wk, t, s);
      case 64: return launch_split_g64(env->spl, la, *io, wk, t, s);
      default: break;
    }
  }
  // two-warp teams exist for the lean instantiation only; generic launches fall back to 32 lanes
  const bool narrow = env->team > 32 && !lean;
  const int team = narrow ? 32 : (tiny ? 1 : env->team);
  const int spl = narrow ? pick_spl(32, env->ds.S) : (tiny ? pick_spl(1, env->ds.S) : env->spl);
  if (env->timing) {
    MARLSC_CUDA(cudaEventRecord(env->marks[0], s));
    rc = [&]() -> int { MARLSC_DISPATCH_G(team, launch_step_g, spl, la, *io, t, s) }();
    if (rc) return rc;
    MARLSC_CUDA(cudaEventRecord(env->marks[1], s));
    env->timed_launches = 1;
    return MARLSC_OK;
  }
  MARLSC_DISPATCH_G(team, launch_step_g, spl, la, *io, t, s)
}

}  // namespace

extern "C" {

int marlsc_env_step(marlsc_env_t* env, const marlsc_env_state_t* state, const marlsc_step_io_t* io, int32_t t, void* stream) {
  const bool metrics = env && env->metrics_on && io;
  if (metrics && env->layout == MARLSC_LAYOUT_WIDE && (!io->cost_breakdown || !io->d_ordered || !io->d_ship || !io->d_unfulfilled))
    return set_error(MARLSC_EINVAL, "episode metrics on a WIDE handle need io.cost_breakdown, d_ordered, d_ship and d_unfulfilled");
  const int rc = step_impl(env, state, io, t, stream);
  if (rc || !metrics) return rc;
  // after the step's last launch, on its stream
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (env->layout == MARLSC_LAYOUT_COMPACT) return launch_metrics_returns(env->metrics, io->rewards, state->num_envs, env->ds.W, s);
  return launch_metrics_fold(env->metrics, *io, state->num_envs, env->ds.W, env->ds.R, env->ds.S, s);
}

}  // extern "C" (host-buffer entry points follow their staging helper)

namespace {

// Host -> device copies of one step's inputs into a staging set (on stream cp); returns the io the step should use.
int stage_host_step(marlsc_env* env, const marlsc_env_state_t* state, const marlsc_step_io_t& dv, const marlsc_host_step_t& h,
                    cudaStream_t cp, marlsc_step_io_t* io_out) {
  const int64_t E = state->num_envs, WS = (int64_t)env->ds.W * env->ds.S;
  if (!h.rewards || (!h.actions && !h.action_qty)) return set_error(MARLSC_EINVAL, "host step with NULL rewards or without actions");
  marlsc_step_io_t io = dv;
  if (h.action_qty) {
    if (!dv.action_qty) return set_error(MARLSC_EINVAL, "host.action_qty needs a staging set with an action_qty buffer");
    MARLSC_CUDA(cudaMemcpyAsync(const_cast<uint8_t*>(dv.action_qty), h.action_qty, (size_t)E * WS, cudaMemcpyHostToDevice, cp));
    io.actions = nullptr;
  } else {
    if (!dv.actions) return set_error(MARLSC_EINVAL, "host.actions needs a staging set with an actions buffer");
    MARLSC_CUDA(cudaMemcpyAsync(const_cast<float*>(dv.actions), h.actions, sizeof(float) * E * WS, cudaMemcpyHostToDevice, cp));
    io.action_qty = nullptr;
  }
  if (h.lines) {
    if (!dv.lines || !dv.line_offsets || !h.line_offsets) return set_error(MARLSC_EINVAL, "host.lines needs host.line_offsets and staging lines / line_offsets buffers");
    MARLSC_CUDA(cudaMemcpyAsync(const_cast<int32_t*>(dv.line_offsets), h.line_offsets, sizeof(int32_t) * (E + 1), cudaMemcpyHostToDevice, cp));
    if (h.n_rounds > 0)
      MARLSC_CUDA(cudaMemcpyAsync(const_cast<uint16_t*>(dv.lines), h.lines, (size_t)h.n_rounds * 64, cudaMemcpyHostToDevice, cp));
    io.line_counts = nullptr;
  } else {
    if (!h.order_offsets) return set_error(MARLSC_EINVAL, "host step without order_offsets or lines");
    if (h.n_orders > 0 && (!h.order_region || !h.order_qty)) return set_error(MARLSC_EINVAL, "host order arrays are NULL");
    MARLSC_CUDA(cudaMemcpyAsync(const_cast<int32_t*>(dv.order_offsets), h.order_offsets, sizeof(int32_t) * (E + 1), cudaMemcpyHostToDevice, cp));
    if (h.n_orders > 0) {
      MARLSC_CUDA(cudaMemcpyAsync(const_cast<int16_t*>(dv.order_region), h.order_region, sizeof(int16_t) * h.n_orders, cudaMemcpyHostToDevice, cp));
      MARLSC_CUDA(cudaMemcpyAsync(const_cast<void*>(dv.order_qty), h.order_qty, (size_t)h.n_orders * env->ds.S * dv.order_qty_bytes, cudaMemcpyHostToDevice, cp));
    }
    io.lines = nullptr;
    io.order_counts = nullptr;
  }
  if (env->ds.lead_mode == MARLSC_LEAD_STOCHASTIC) {
    if (!h.actual_lead) return set_error(MARLSC_EINVAL, "host.actual_lead is required with a stochastic lead-time sampler");
    MARLSC_CUDA(cudaMemcpyAsync(const_cast<uint8_t*>(dv.actual_lead), h.actual_lead, (size_t)E * WS, cudaMemcpyHostToDevice, cp));
  }
  *io_out = io;
  return MARLSC_OK;
}

}  // namespace

extern "C" {

int marlsc_env_step_host(marlsc_env_t* env, const marlsc_env_state_t* state, const marlsc_step_io_t* dev,
                         const marlsc_host_step_t* host, int32_t t, void* stream) {
  int rc = check_state(env, state);
  if (rc) return rc;
  if (!dev || !host) return set_error(MARLSC_EINVAL, "null staging or host descriptor");
  MARLSC_CUDA(cudaSetDevice(env->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int64_t E = state->num_envs;
  marlsc_step_io_t io;
  rc = stage_host_step(env, state, *dev, *host, s, &io);
  if (rc) return rc;
  rc = marlsc_env_step(env, state, &io, t, stream);
  if (rc) return rc;
  MARLSC_CUDA(cudaMemcpyAsync(host->rewards, io.rewards, sizeof(float) * E * env->ds.W, cudaMemcpyDeviceToHost, s));
  if (host->obs) MARLSC_CUDA(cudaMemcpyAsync(host->obs, io.obs, sizeof(float) * E * env->ds.W * env->ds.obs_dim, cudaMemcpyDeviceToHost, s));
  MARLSC_CUDA(cudaStreamSynchronize(s));
  return MARLSC_OK;
}

int marlsc_env_rollout_host(marlsc_env_t* env, const marlsc_env_state_t* state, const marlsc_step_io_t staging[2],
                            const marlsc_host_step_t* host, int32_t n_steps, int32_t t0, float* rewards_dev, void* stream) {
  int rc = check_state(env, state);
  if (rc) return rc;
  if (!staging || !host || !rewards_dev) return set_error(MARLSC_EINVAL, "null staging, host descriptors or rewards_dev");
  if (n_steps < 1 || t0 < 0) return set_error(MARLSC_EINVAL, "n_steps must be positive and t0 >= 0");
  if (env->metrics_on && env->layout == MARLSC_LAYOUT_WIDE)
    return set_error(MARLSC_EUNSUPPORTED, "episode metrics on a WIDE handle fold the diagnostic outputs, which the caller zeroes "
                                          "before every step: use marlsc_env_step");
  MARLSC_CUDA(cudaSetDevice(env->device));
  if (!env->copy_stream) {
    MARLSC_CUDA(cudaStreamCreateWithFlags(&env->copy_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
      MARLSC_CUDA(cudaEventCreateWithFlags(&env->ready[i], cudaEventDisableTiming));
      MARLSC_CUDA(cudaEventCreateWithFlags(&env->done[i], cudaEventDisableTiming));
    }
  }
  cudaStream_t cs = static_cast<cudaStream_t>(stream), cp = env->copy_stream;
  const int64_t E = state->num_envs, W = env->ds.W;
  // the copy stream must not run ahead of work already queued on the caller's stream
  MARLSC_CUDA(cudaEventRecord(env->done[0], cs));
  MARLSC_CUDA(cudaEventRecord(env->done[1], cs));
  for (int i = 0; i < n_steps; ++i) {
    const int b = i & 1;
    const marlsc_host_step_t& h = host[i];
    MARLSC_CUDA(cudaStreamWaitEvent(cp, env->done[b], 0));      // staging set b is free again
    marlsc_step_io_t io;
    rc = stage_host_step(env, state, staging[b], h, cp, &io);
    if (rc) return rc;
    MARLSC_CUDA(cudaEventRecord(env->ready[b], cp));
    MARLSC_CUDA(cudaStreamWaitEvent(cs, env->ready[b], 0));
    io.rewards = rewards_dev + (int64_t)i * E * W;
    rc = marlsc_env_step(env, state, &io, t0 + i, stream);
    if (rc) return rc;
    MARLSC_CUDA(cudaEventRecord(env->done[b], cs));
    MARLSC_CUDA(cudaMemcpyAsync(h.rewards, io.rewards, sizeof(float) * E * W, cudaMemcpyDeviceToHost, cs));
    if (h.obs) MARLSC_CUDA(cudaMemcpyAsync(h.obs, io.obs, sizeof(float) * E * W * env->ds.obs_dim, cudaMemcpyDeviceToHost, cs));
  }
  MARLSC_CUDA(cudaStreamSynchronize(cs));
  return MARLSC_OK;
}

}  // extern "C"

extern "C" {

int marlsc_policy_base_stock(marlsc_env_t* env, const marlsc_env_state_t* state, const float* level, int32_t t,
                             float* actions, void* stream) {
  int rc = check_state(env, state);
  if (rc) return rc;
  if (!level || !actions) return set_error(MARLSC_EINVAL, "level and actions must not be NULL");
  if (env->ds.action_type != MARLSC_ACTION_DIRECT) return set_error(MARLSC_EINVAL, "the base-stock heuristic assumes the direct action space");
  if (t < 0) return set_error(MARLSC_EINVAL, "timestep must be >= 0");
  MARLSC_CUDA(cudaSetDevice(env->device));
  if (env->layout == MARLSC_LAYOUT_COMPACT) return launch_base_stock_compact(env->ds, *state, level, 0, t, actions, static_cast<cudaStream_t>(stream));
  return launch_base_stock(env->ds, *state, level, 0, t, actions, static_cast<cudaStream_t>(stream));
}

int marlsc_policy_base_stock_per_env(marlsc_env_t* env, const marlsc_env_state_t* state, const float* level, int32_t t,
                                     float* actions, void* stream) {
  int rc = check_state(env, state);
  if (rc) return rc;
  if (!level || !actions) return set_error(MARLSC_EINVAL, "level and actions must not be NULL");
  if (env->ds.action_type != MARLSC_ACTION_DIRECT) return set_error(MARLSC_EINVAL, "the base-stock heuristic assumes the direct action space");
  if (t < 0) return set_error(MARLSC_EINVAL, "timestep must be >= 0");
  MARLSC_CUDA(cudaSetDevice(env->device));
  if (env->layout == MARLSC_LAYOUT_COMPACT) return launch_base_stock_compact(env->ds, *state, level, 1, t, actions, static_cast<cudaStream_t>(stream));
  return launch_base_stock(env->ds, *state, level, 1, t, actions, static_cast<cudaStream_t>(stream));
}

int marlsc_lines_from_orders(marlsc_env_t* env, int64_t num_envs, const marlsc_step_io_t* orders, int32_t line_stride,
                             uint16_t* lines, int32_t* line_counts, int32_t* overflow_flag, void* stream) {
  if (!env || !orders || !lines || !line_counts || !overflow_flag) return set_error(MARLSC_EINVAL, "null argument");
  if (!env->ds.compact_ok) return set_error(MARLSC_EUNSUPPORTED, "lines exist for configurations that qualify for the compact layout");
  if (num_envs < 1 || line_stride < 2 || (line_stride & 1)) return set_error(MARLSC_EINVAL, "num_envs must be positive and line_stride positive and even");
  if (!orders->order_offsets && !orders->order_counts) return set_error(MARLSC_EINVAL, "orders need order_offsets or order_counts");
  if (orders->order_qty_bytes != 1) return set_error(MARLSC_EUNSUPPORTED, "lines carry one-byte quantities");
  MARLSC_CUDA(cudaSetDevice(env->device));
  return launch_lines_from_orders(env->ds, num_envs, *orders, line_stride, lines, line_counts, overflow_flag, static_cast<cudaStream_t>(stream));
}

const char* marlsc_last_error(void) { return g_last_error.c_str(); }
int32_t marlsc_abi_version(void) { return MARLSC_ABI_VERSION; }
int64_t marlsc_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

}  // extern "C"
