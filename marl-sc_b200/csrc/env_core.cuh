// env_core.cuh - per-environment step logic of the fused env-step kernel (K1).
//
// One "team" of G lanes (G = 1..32, an aligned slice of one warp) advances one environment by one
// timestep. Lane l owns SKUs s = l + G*j, j < SPL (compile-time), so per-order remainders and the
// per-cell feature values live in registers; the environment's on-hand stock and the per-step
// accumulators live in the team's shared-memory scratch; the small lookup tables every environment
// needs (warehouse priority per region, home-warehouse masks, expected lead times, per-SKU rates) are
// staged once per CTA in shared memory. Global memory is touched once per array element, coalesced
// over SKUs, with the loads of a batch of cells issued before any of them is consumed.
//
// The same source compiles
//   * for sm_100a (env_step.cu), and
//   * as plain C++ with G == 1 (tests/emu/emu.cpp, -DMARLSC_HOST_EMU) so the step logic can be
//     checked against the oracle in a container without a GPU. The emulation is test-only.
//
// Reference semantics restated here (paths under the reference repo):
//   step order ................. src/environment/envs/multi_env.py:253-366
//   action rescale ............. multi_env.py:795-848
//   orders / arrivals .......... multi_env.py:850-919
//   greedy allocation .......... src/environment/components/demand_allocator.py:150-208
//   feature buffers ............ multi_env.py:747-793
//   lost sales ................. src/environment/components/lost_sales_handler.py:71-210
//   cost reward ................ src/environment/components/reward_calculator.py:127-188
//   observation ................ multi_env.py:577-745, 941-968
#pragma once
#include <stdint.h>
#include "../../include/marlsc_b200.h"

#ifdef MARLSC_HOST_EMU
#include <cmath>
#include <cstring>
#define MDEV static inline
#define MARLSC_RESTRICT
#define MARLSC_UNROLL
#else
#define MDEV __device__ __forceinline__
#define MARLSC_RESTRICT __restrict__
#define MARLSC_UNROLL _Pragma("unroll")
#endif

namespace marlsc {

constexpr int kWindow = MARLSC_ROLLING_WINDOW;
constexpr int kPipeBatch = 5;   // pipeline slots loaded together per cell
#ifndef MARLSC_LANE_CHAINS
#define MARLSC_LANE_CHAINS 1        // independent allocation chains a lane interleaves (1 or 2)
#endif
#ifndef MARLSC_FORCE_LANE_ALLOC
#define MARLSC_FORCE_LANE_ALLOC 0   // the host emulation sets this to run the wide-team allocation with G == 1
#endif

// Capabilities compiled into a kernel instantiation. The lean instantiation (kCapsLean) covers the
// common configurations - fixed lead times, direct actions, unit SKU weights, static warehouse
// priority, the inventory / pipeline / home-demand / rolling-mean feature blocks, normalisation off
// or fixed mean-std, no diagnostics - and is several times smaller than the generic one (kCapsAll),
// which handles everything. Host code picks per launch (env_step.cu: required_caps()).
enum : uint32_t {
  C_STOCH = 1u << 0,     // stochastic lead times (ring_lead, per-plane scans)
  C_RATIO = 1u << 1,     // ratio normalisation
  C_MEANSTD = 1u << 2,   // fixed mean/std normalisation
  C_SHIP = 1u << 3,      // shipped-home / shipped-away / stockout features
  C_FCST = 1u << 4,      // EMA forecast state
  C_XFEAT = 1u << 5,     // days of supply, net inventory position, demand variability, demand history
  C_ACTX = 1u << 6,      // demand_centered / base_stock action spaces
  C_WEIGHT = 1u << 7,    // non-unit SKU weights
  C_DIAG = 1u << 8,      // diagnostic outputs (cost breakdown, per-step dumps)
  C_DYNPRIO = 1u << 9,   // weight-dependent warehouse priority
  C_REGMAP = 1u << 10,   // raw -> included region map
  C_QTY16 = 1u << 11,    // two-byte order quantities
  C_IDHOT = 1u << 12,    // one-hot warehouse id prefix
  C_AGGX = 1u << 13,     // pipeline / home-demand / rolling-mean aggregates
  C_BIGW = 1u << 14,     // more than 32 warehouses (no home bitmask)
  C_DHSMEM = 1u << 15,   // home demand needed without a history plane (kept in shared memory)
  C_LOSTCOST = 1u << 16, // softmax ("cost") lost-sales handler
  C_FIXED = 1u << 17,    // non-zero outbound fixed costs (per-(warehouse, region) shipment counts)
  C_SPLITLIM = 1u << 18, // max_splits < W-1: the split limit can bind, shipping warehouses are counted per order
};
constexpr uint32_t kCapsAll = 0xffffffffu;
constexpr uint32_t kCapsLean = C_MEANSTD | C_IDHOT;
// Wide teams whose configuration couples the SKUs of an order through nothing but the inventory
// (no binding split limit, no per-shipment fixed cost, static warehouse priority, no diagnostics) run
// the allocation as independent per-lane chains, see step_env phase 2.
template <int G, uint32_t CAPS>
struct LaneAlloc {
  static constexpr bool value = (G >= 8 || MARLSC_FORCE_LANE_ALLOC) &&
                                !(CAPS & (C_SPLITLIM | C_FIXED | C_DIAG | C_DYNPRIO | C_QTY16 | C_BIGW));
};

// Device-side view of a marlsc_env_spec_t: device table pointers, observation block offsets and
// the shared-memory layouts. Passed by value to the kernels.
struct DevSpec {
  int W, S, R, Rraw, L, D, episode_length;
  int action_type, lead_mode, lost_type, scope, max_splits, norm, id_off, obs_dim;
  uint32_t feat;
  int need_hist, need_fcst, need_ship, unit_weights;
  int dh_mode;     // home-demand accumulator: 0 not needed, 1 the history plane of step t (global, L1 resident), 2 shared memory
  int has_fixed;   // some outbound fixed cost is non-zero (shipment counts matter)
  double scale, alpha;
  const double* action_max;
  const double* out_fixed;
  const double* out_var;
  const double* in_fixed;
  const double* in_var;
  const double* hold_rate;
  const double* pen_rate;
  const double* skw;
  const int32_t* lead_exp;
  const int32_t* home;
  const int32_t* closest;
  const int32_t* region_map;
  const uint8_t* prio;         // [R,W] warehouses in ascending (cost, index) order, valid where prio_static[r]
  const uint8_t* prio_static;  // [R] 1 when the order does not depend on the order's weight
  const uint32_t* home_mask;   // [R] bit w set when region r is warehouse w's home region (W <= 32), else null
  const uint8_t* lead_u8;      // [W*S] expected lead times as bytes
  const uint16_t* prio_perm;   // [R,perm_chunks,16] availability bits -> priority-order bits (W <= 16), else null
  int perm_chunks;
  int pen_uniform;             // every SKU has the same lost-sales penalty rate
  // compact layout (env_compact.cu): five warehouse bits per lookup, priority rows padded to 16, home warehouse per region
  const uint16_t* perm5;       // [R,perm5_chunks,32] availability bits -> priority-order bits (W <= 16), else null
  const uint8_t* prio16;       // [R,16] warehouses in priority order
  const uint8_t* home_wh;      // [R] the warehouse whose home region r is; 255 none, 254 several (see home_mask)
  int perm5_chunks;
  int compact_ok;              // the configuration fits the compact state layout
  int row_rates_uniform;       // holding / weight / inbound rates do not vary over the SKUs of a warehouse
  const float* obs_mean;
  const float* obs_std;        // holds 1/std (precomputed on the host in float32)
  // observation block offsets inside one warehouse's vector (before the id prefix); -1 = block disabled
  int off_inv, off_pipe, off_dh, off_sh, off_sa, off_so, off_rm, off_fc, off_dos, off_nip, off_dv, off_hist;
  // per-CTA shared tables (byte offsets from the start of dynamic shared memory)
  int t_skw, t_pen, t_hold, t_prio, t_pstat, t_hmask, t_lead, t_bytes;
  // per-team scratch: a double area and a 32-bit word area
  int och;                                   // orders staged per chunk (one-byte rows)
  int d_lostW, d_lostP, d_ctot, d_shipw, d_words;
  int w_inv, w_dh, w_sh, w_st, w_shipq, w_cnt, w_lostN, w_prio, w_sreg, w_sqty, w_words;
};

// Lookup tables shared by every environment of a CTA (shared memory on the device).
struct Tables {
  const double* skw;
  const double* pen;
  const double* hold;
  const uint8_t* prio;
  const uint8_t* pstat;
  const uint32_t* hmask;   // null when W > 32
  const uint8_t* lead;
};

struct Scratch {
  double* d;
  int32_t* w;
};

// ------------------------------------------------------------------------------------------------
// Team: G lanes (an aligned slice of a warp, or G/32 whole warps) working on one environment.
// ------------------------------------------------------------------------------------------------
template <int G>
struct Team {
  int gl;    // lane inside the team
#ifndef MARLSC_HOST_EMU
  // G <= 32: an aligned slice of one warp, synchronised with warp-level primitives.
  // G  > 32: G/32 whole warps; team-wide steps go through a named barrier (id 1 + team index in the CTA)
  //          and a few doubles of static shared memory (xs) for the cross-warp sums.
  unsigned gmask;
  unsigned live;   // lanes of this warp whose team has an environment (teams narrower than a warp, see converge())
  int bar;
  double* xs;
  __device__ __forceinline__ void init(double* xchg = nullptr, unsigned live_lanes = 0xffffffffu) {
    live = live_lanes;
    gl = threadIdx.x % G;
    const int wl = threadIdx.x & 31;
    gmask = (G >= 32) ? 0xffffffffu : (((1u << (G & 31)) - 1u) << (wl & ~(G - 1)));
    bar = 1 + threadIdx.x / G;
    xs = G > 32 ? xchg + (threadIdx.x / G) * (G / 32) : nullptr;
  }
  __device__ __forceinline__ void sync() const {
    if (G > 32) asm volatile("bar.sync %0, %1;" ::"r"(bar), "n"(G) : "memory");
    else if (G > 1) __syncwarp(gmask);
  }
  // Teams narrower than a warp: the teams of a warp run data-dependent loops of different lengths, and nothing brings
  // them back together afterwards - measured on the thread-per-environment kernel, 2.1 of 32 lanes were active per
  // instruction in the straight-line code after the allocation. converge() is a team sync that also reconverges the warp;
  // it may only stand where every live lane of the warp passes (the top level of the step).
  __device__ __forceinline__ void converge() const {
    if (G >= 32) sync();
    else __syncwarp(live);
  }
  // vote over every live lane of the warp (teams narrower than a warp running a loop in lockstep), else over the team
  __device__ __forceinline__ bool lock_any(bool p) const {
    if (G >= 32) return warp_any(p);
    return __ballot_sync(live, p) != 0u;
  }
  // the largest v over the teams of this warp (v itself for whole-warp teams): trip counts for loops that converge()
  __device__ __forceinline__ int warp_max(int v) const {
    if (G >= 32) return v;
    return __reduce_max_sync(live, v);
  }
  __device__ __forceinline__ bool any(bool p) const {
    if (G == 1) return p;
    if (G > 32) {
      int r;
      asm volatile("{ .reg .pred q, o; setp.ne.s32 q, %1, 0; bar.red.or.pred o, %2, %3, q; selp.s32 %0, 1, 0, o; }"
                   : "=r"(r) : "r"((int)p), "r"(bar), "n"(G) : "memory");
      return r != 0;
    }
    return __ballot_sync(gmask, p) != 0u;
  }
  // vote among the lanes of this team that share a warp (all of them for G <= 32)
  __device__ __forceinline__ bool warp_any(bool p) const {
    if (G == 1) return p;
    return __ballot_sync(gmask, p) != 0u;
  }
  // lanes of the team for which p holds, as a bit mask relative to the team's first lane (G <= 32 only)
  __device__ __forceinline__ unsigned ballot(bool p) const {
    static_assert(G <= 32, "ballot needs a team inside one warp");
    if (G == 1) return p ? 1u : 0u;
    const unsigned b = __ballot_sync(gmask, p) & gmask;
    return G == 32 ? b : (b >> ((threadIdx.x & 31) & ~(G - 1)));
  }
  template <typename T>
  __device__ __forceinline__ T sum_t(T v) const {
#pragma unroll
    for (int o = (G > 32 ? 32 : G) / 2; o > 0; o >>= 1) v += __shfl_xor_sync(gmask, v, o);
    if (G > 32) {
      if ((threadIdx.x & 31) == 0) xs[gl >> 5] = (double)v;      // int / float / double all fit a double exactly
      sync();
      double r = 0.0;
#pragma unroll
      for (int i = 0; i < G / 32; ++i) r += xs[i];
      sync();
      v = (T)r;
    }
    return v;
  }
  __device__ __forceinline__ int sum(int v) const {
    if (G == 32) return __reduce_add_sync(0xffffffffu, v);   // one REDUX instead of five shuffle rounds
    return sum_t(v);
  }
  __device__ __forceinline__ float sum(float v) const { return sum_t(v); }
  __device__ __forceinline__ double sum(double v) const { return sum_t(v); }
#else
  void init(double* = nullptr, unsigned = 0) { gl = 0; }
  void sync() const {}
  void converge() const {}
  int warp_max(int v) const { return v; }
  bool lock_any(bool p) const { return p; }
  bool any(bool p) const { return p; }
  bool warp_any(bool p) const { return p; }
  unsigned ballot(bool p) const { return p ? 1u : 0u; }
  int sum(int v) const { return v; }
  float sum(float v) const { return v; }
  double sum(double v) const { return v; }
#endif
};

// ---- arithmetic that must round exactly like NumPy (no fused multiply-add) -----------------------
#ifndef MARLSC_HOST_EMU
MDEV float f_add(float a, float b) { return __fadd_rn(a, b); }
MDEV float f_sub(float a, float b) { return __fsub_rn(a, b); }
MDEV float f_mul(float a, float b) { return __fmul_rn(a, b); }
MDEV float f_div(float a, float b) { return __fdiv_rn(a, b); }
MDEV float f_sqrt(float a) { return __fsqrt_rn(a); }
MDEV double d_add(double a, double b) { return __dadd_rn(a, b); }
MDEV double d_mul(double a, double b) { return __dmul_rn(a, b); }
MDEV double d_rint(double a) { return rint(a); }
MDEV int lowest_bit(uint32_t m) { return __ffs((int)m) - 1; }
MDEV void smem_add(int32_t* addr, int v) { atomicAdd(addr, v); }
// fire-and-forget add to a global cell (RED); read the cell back with load_cg() after a team sync
MDEV void global_add(int32_t* addr, int v) { asm volatile("red.global.add.s32 [%0], %1;" ::"l"(addr), "r"(v) : "memory"); }
MDEV int load_cg(const int32_t* addr) { return __ldcg(addr); }
MDEV void smem_add(double* addr, double v) { atomicAdd(addr, v); }
#else
MDEV float f_add(float a, float b) { volatile float r = a + b; return r; }
MDEV float f_sub(float a, float b) { volatile float r = a - b; return r; }
MDEV float f_mul(float a, float b) { volatile float r = a * b; return r; }
MDEV float f_div(float a, float b) { volatile float r = a / b; return r; }
MDEV float f_sqrt(float a) { return std::sqrt(a); }
MDEV double d_add(double a, double b) { volatile double r = a + b; return r; }
MDEV double d_mul(double a, double b) { volatile double r = a * b; return r; }
MDEV double d_rint(double a) { return std::nearbyint(a); }
MDEV int lowest_bit(uint32_t m) { return __builtin_ctz(m); }
MDEV void smem_add(int32_t* addr, int v) { *addr += v; }
MDEV void global_add(int32_t* addr, int v) { *addr += v; }
MDEV int load_cg(const int32_t* addr) { return *addr; }
MDEV void smem_add(double* addr, double v) { *addr += v; }
#endif
// Keep a derived pointer in registers: without this the compiler re-derives per-environment bases
// from the kernel parameters (constant-bank load + 64-bit adds) at every access.
template <typename T>
MDEV T* pinned(T* p) {
#ifndef MARLSC_HOST_EMU
  asm volatile("" : "+l"(p));
#endif
  return p;
}
MDEV int imin(int a, int b) { return a < b ? a : b; }
MDEV int imax(int a, int b) { return a > b ? a : b; }
MDEV int pmod(int a, int m) { int r = a % m; return r < 0 ? r + m : r; }

// Write one observation element (index j inside the un-prefixed local vector) with the fixed
// mean/std normalisation of multi_env.py:700-702 applied when enabled.
// ``out`` points at the first element after the optional one-hot id prefix.
template <uint32_t CAPS>
MDEV void emit(const DevSpec& sp, float* MARLSC_RESTRICT out, unsigned j, float x) {
  // (x - mean) * (1/std): within 2 ulp of the reference's division, far inside the 1e-5 parity tolerance
  if ((CAPS & C_MEANSTD) && sp.norm == MARLSC_NORM_MEANSTD) x = f_mul(f_sub(x, sp.obs_mean[j]), sp.obs_std[j]);
  out[j] = x;
}

// Per-environment global pointers.
struct EnvPtrs {
  int32_t* inv;        // [W,S]
  int32_t* ring_q;     // [D,W,S]
  uint8_t* ring_l;     // [D,W,S] or null
  int32_t* hist;       // [5,W,S] or null
  float* fcst;         // [W,S] or null
};

MDEV EnvPtrs env_ptrs(const DevSpec& sp, const marlsc_env_state_t& st, int64_t e) {
  const int64_t ws = (int64_t)sp.W * sp.S;
  EnvPtrs p;
  p.inv = pinned(static_cast<int32_t*>(st.inventory) + e * ws);
  p.ring_q = pinned(static_cast<int32_t*>(st.ring_qty) + e * ws * sp.D);
  p.ring_l = st.ring_lead ? pinned(st.ring_lead + e * ws * sp.D) : nullptr;
  p.hist = st.demand_hist ? pinned(static_cast<int32_t*>(st.demand_hist) + e * ws * kWindow) : nullptr;
  p.fcst = st.forecast ? pinned(st.forecast + e * ws) : nullptr;
  return p;
}

// ---- stochastic lead times: generic (slow) in-transit bookkeeping --------------------------------
// Quantity in expected-arrival slot k (0-based) for cell i at the end of step t (multi_env.py:941-968).
// The order placed at step t itself is already in the ring.
MDEV int pipeline_value_stoch(const DevSpec& sp, const EnvPtrs& p, int t, int i, int le, int k) {
  const int WS = sp.W * sp.S;
  int v = 0;
  for (int d = 0; d < sp.D; ++d) {
    const int tau = t - pmod(t - d, sp.D);  // youngest placement step <= t that maps to plane d
    if (tau < 0) continue;
    const int q = p.ring_q[d * WS + i];
    if (q <= 0 || tau + (int)p.ring_l[d * WS + i] <= t) continue;  // nothing placed, or delivered
    const int slot = tau + le - t;
    if (slot > sp.L) continue;
    const int kk = slot <= 1 ? 0 : slot - 1;  // late orders pile into slot 0
    if (kk == k) v += q;
  }
  return v;
}

// Units on their way to cell i at the start of step t, before this step's arrivals are taken out
// (what the base_stock action space subtracts, multi_env.py:841-845).
MDEV int pending_before(const DevSpec& sp, const EnvPtrs& p, int t, int i, int le) {
  const int WS = sp.W * sp.S;
  int v = 0;
  if (sp.lead_mode == MARLSC_LEAD_FIXED) {
    for (int a = 1; a <= le; ++a) {
      const int tau = t - a;
      if (tau < 0) break;
      v += p.ring_q[(tau % sp.D) * WS + i];
    }
    return v;
  }
  for (int d = 0; d < sp.D; ++d) {
    const int tau = (t - 1) - pmod(t - 1 - d, sp.D);
    if (tau < 0) continue;
    const int q = p.ring_q[d * WS + i];
    if (q > 0 && tau + (int)p.ring_l[d * WS + i] >= t) v += q;
  }
  return v;
}

// Units arriving at cell i at step t under stochastic lead times (actual_arrival == t, multi_env.py:910-919).
MDEV int arrivals_stoch(const DevSpec& sp, const EnvPtrs& p, int t, int i) {
  const int WS = sp.W * sp.S;
  int v = 0;
  for (int d = 0; d < sp.D; ++d) {
    const int tau = (t - 1) - pmod(t - 1 - d, sp.D);
    if (tau < 0) continue;
    const int q = p.ring_q[d * WS + i];
    if (q > 0 && tau + (int)p.ring_l[d * WS + i] == t) v += q;
  }
  return v;
}

// Action in [-1,1] -> integer order quantity with the reference's mixed fp32/fp64 arithmetic and
// round-half-even (multi_env.py:824-846).
template <uint32_t CAPS>
MDEV int rescale_action(const DevSpec& sp, float a, double mx, int prev_home_demand, int pending) {
  if (!(CAPS & C_ACTX) || sp.action_type == MARLSC_ACTION_DIRECT) {
    const float u = f_mul(f_add(a, 1.0f), 0.5f);   // == (a + 1) / 2 exactly
    double q = d_rint(d_mul((double)u, mx));
    if (q < 0.0) q = 0.0;
    if (q > mx) q = mx;
    return (int)q;
  }
  if (sp.action_type == MARLSC_ACTION_DEMAND_CENTERED) {
    const long long adj = (long long)d_rint(d_mul(mx, (double)a));
    const long long q = adj + (long long)prev_home_demand;
    return q < 0 ? 0 : (int)q;
  }
  const float u = f_mul(f_add(a, 1.0f), 0.5f);   // == (a + 1) / 2 exactly
  const double target = d_mul((double)u, mx);
  const double x = d_add(d_add(target, -(double)prev_home_demand), -(double)pending);
  const double q = d_rint(x);
  return q < 0.0 ? 0 : (int)q;
}

// Share of region r's lost volume attributed to warehouse w (lost_sales_handler.py:71-210).
// ``shipped_r`` >= 0: units shipped to region r from all warehouses, when the caller has it at hand.
template <uint32_t CAPS>
MDEV double lost_weight(const DevSpec& sp, const int32_t* s_shipq, const int32_t* s_lostN, const double* s_lostW,
                        int w, int r, int shipped_r = -1) {
  const int W = sp.W, R = sp.R;
  if (sp.lost_type == MARLSC_LOST_CLOSEST) return sp.closest[r] == w ? 1.0 : 0.0;
  if (sp.lost_type == MARLSC_LOST_SHIPMENT) {
    int tot = shipped_r;
    if (tot < 0) {
      tot = 0;
      for (int ww = 0; ww < W; ++ww) tot += s_shipq[ww * R + r];
    }
    if (tot > 0) return (double)s_shipq[w * R + r] / (double)tot;
    return sp.closest[r] == w ? 1.0 : 0.0;
  }
  if (!(CAPS & C_LOSTCOST)) return 0.0;
  const double n = (double)s_lostN[r], lwt = s_lostW[r];
  double zmax = -1e300;
  for (int ww = 0; ww < W; ++ww) {
    const double z = -(sp.out_fixed[ww * R + r] * n + sp.out_var[ww * R + r] * lwt) / sp.alpha;
    if (z > zmax) zmax = z;
  }
  double zsum = 0.0, mine = 0.0;
  for (int ww = 0; ww < W; ++ww) {
    const double z = -(sp.out_fixed[ww * R + r] * n + sp.out_var[ww * R + r] * lwt) / sp.alpha;
    const double ez = exp(z - zmax);
    zsum += ez;
    if (ww == w) mine = ez;
  }
  return mine / zsum;
}

// ------------------------------------------------------------------------------------------------
// Pipeline block of warehouse w's observation row (multi_env.py:603-633, 941-968). It depends only on the
// in-transit ring (including the order just placed at step t), not on this step's demand, so it is
// emitted in phase 1 right after the ring row was read for arrivals: every ring sector is then touched
// once per step instead of twice with the allocation phase in between (L2 cannot hold the in-flight
// working set of all resident environments, so the second touch used to go back to DRAM).
// ------------------------------------------------------------------------------------------------
template <int G, int SPL, uint32_t CAPS>
MDEV void write_obs_pipeline(const DevSpec& sp, const Tables& tb, const Team<G>& tm, const EnvPtrs& p,
                             float* MARLSC_RESTRICT obs_w, int w, int t) {
  const int S = sp.S, L = sp.L, D = sp.D, WS = sp.W * sp.S;
  const int base = w * S;
  const bool ratio = (CAPS & C_RATIO) && sp.norm == MARLSC_NORM_RATIO;
  const uint32_t F = sp.feat & (MARLSC_F_PIPELINE | ((CAPS & C_AGGX) ? MARLSC_F_PIPELINE_AGG : 0u));
  const bool fixed_lead = !(CAPS & C_STOCH) || sp.lead_mode == MARLSC_LEAD_FIXED;
  float* MARLSC_RESTRICT const out = pinned(obs_w + ((CAPS & C_IDHOT) ? sp.id_off : 0));
  // pipeline, slot-major (L,S) ravel. Fixed leads: the order placed at tau sits in slot
  //    tau + le - t, so slot k reads ring plane (t + k + 1 - le) mod D for k < le and is 0 otherwise
  //    (planes of placement steps < 0 have not been written since reset and read 0).
  if (sp.off_pipe >= 0) {
    const bool need_total = ratio || (F & MARLSC_F_PIPELINE_AGG);
    const int tm1 = (t + 1) % D;
    const int32_t* const ring = p.ring_q;      // pinned per-env base; cells are addressed by 32-bit offsets
    const unsigned WSu = (unsigned)WS, Su = (unsigned)S;
    float* MARLSC_RESTRICT const pout = pinned(out + sp.off_pipe);
    const bool ms = (CAPS & C_MEANSTD) && sp.norm == MARLSC_NORM_MEANSTD;
    float den = 1.0f;
    int total = 0;
    if (fixed_lead && !need_total) {
      // common case: every cell of the row in flight at once, kPipeBatch slots per round
      int le[SPL], row0[SPL];
      MARLSC_UNROLL
      for (int j = 0; j < SPL; ++j) {
        const int s = tm.gl + G * j;
        le[j] = s < S ? (int)tb.lead[base + s] : 0;
        row0[j] = tm1 - le[j];                 // ring plane of slot 0
        row0[j] += row0[j] < 0 ? D : 0;
      }
#ifndef MARLSC_HOST_EMU
#pragma unroll 1
#endif
      for (int k0 = 0; k0 < L; k0 += kPipeBatch) {
        int v[SPL][kPipeBatch];
        MARLSC_UNROLL
        for (int j = 0; j < SPL; ++j) {
          const unsigned cell = (unsigned)(base + tm.gl + G * j);
          MARLSC_UNROLL
          for (int kk = 0; kk < kPipeBatch; ++kk) {
            const int k = k0 + kk;
            v[j][kk] = 0;
            if (k < le[j]) {
              int row = row0[j] + k;
              row -= row >= D ? D : 0;
              v[j][kk] = ring[(unsigned)row * WSu + cell];
            }
          }
        }
        MARLSC_UNROLL
        for (int j = 0; j < SPL; ++j) {
          const int s = tm.gl + G * j;
          if (s < S) {
            MARLSC_UNROLL
            for (int kk = 0; kk < kPipeBatch; ++kk) {
              const int k = k0 + kk;
              if (k < L) {
                float x = (float)v[j][kk];
                const unsigned idx = (unsigned)k * Su + (unsigned)s;
                if (ms) x = f_mul(f_sub(x, sp.obs_mean[sp.off_pipe + idx]), sp.obs_std[sp.off_pipe + idx]);
                pout[idx] = x;
              }
            }
          }
        }
      }
    } else
    for (int pass = need_total ? 0 : 1; pass < 2; ++pass) {
      // pass 0 only sums (ratio denominator / aggregate), pass 1 writes
#ifndef MARLSC_HOST_EMU
#pragma unroll 1
#endif
      for (int j = 0; j < SPL; ++j) {
        const int s = tm.gl + G * j;
        if (s >= S) break;
        const unsigned cell = (unsigned)(base + s);
        const int le = (int)tb.lead[cell];
        int row0 = tm1 - le;                   // ring plane of slot 0
        row0 += row0 < 0 ? D : 0;
        for (int k0 = 0; k0 < L; k0 += kPipeBatch) {
          int v[kPipeBatch];
          MARLSC_UNROLL
          for (int kk = 0; kk < kPipeBatch; ++kk) {       // loads of the batch first
            const int k = k0 + kk;
            int val = 0;
            if (fixed_lead) {
              if (k < le) {
                int row = row0 + k;
                row -= row >= D ? D : 0;
                val = ring[(unsigned)row * WSu + cell];
              }
            } else if ((CAPS & C_STOCH) && k < L) {
              val = pipeline_value_stoch(sp, p, t, (int)cell, le, k);
            }
            v[kk] = val;
          }
          MARLSC_UNROLL
          for (int kk = 0; kk < kPipeBatch; ++kk) {
            const int k = k0 + kk;
            if (k < L) {
              if (pass == 0) {
                total += v[kk];
              } else {
                float x = (float)v[kk];
                if (ratio) x = f_div(x, den);
                const unsigned idx = (unsigned)k * Su + (unsigned)s;
                if (ms) x = f_mul(f_sub(x, sp.obs_mean[sp.off_pipe + idx]), sp.obs_std[sp.off_pipe + idx]);
                pout[idx] = x;
              }
            }
          }
        }
      }
      if (pass == 0) {
        total = tm.sum(total);
        den = (float)((double)total + 1e-8);
      }
    }
    if ((F & MARLSC_F_PIPELINE_AGG) && tm.gl == 0) emit<CAPS>(sp, out, sp.off_pipe + L * S, (float)total);
  }

}

// ------------------------------------------------------------------------------------------------
// Observation row of warehouse w (multi_env.py:577-710) from per-lane register values.
//   vI/vdh/vsh/vst: on-hand, home demand, shipped home, shipped total (ints); vrm/vfc: rolling mean,
//   forecast. hist_n = valid history entries including the current step (0 right after reset).
// ------------------------------------------------------------------------------------------------
template <int G, int SPL, uint32_t CAPS>
MDEV void write_obs_row(const DevSpec& sp, const Tables& tb, const Team<G>& tm, const EnvPtrs& p,
                        float* MARLSC_RESTRICT obs_w, int w, int t, int hist_n, const int (&vI)[SPL],
                        const int (&vdh)[SPL], const int (&vsh)[SPL], const int (&vst)[SPL], const float (&vrm)[SPL],
                        const float (&vfc)[SPL]) {
  const int S = sp.S, W = sp.W, L = sp.L, D = sp.D, WS = sp.W * sp.S;
  const int base = w * S;
  const bool ratio = (CAPS & C_RATIO) && sp.norm == MARLSC_NORM_RATIO;
  // feature bits this instantiation can emit
  constexpr uint32_t kFeatMask =
      MARLSC_F_INVENTORY | MARLSC_F_INVENTORY_AGG | MARLSC_F_PIPELINE | MARLSC_F_DEMAND_HOME | MARLSC_F_ROLLING_MEAN |
      ((CAPS & C_AGGX) ? (MARLSC_F_PIPELINE_AGG | MARLSC_F_DEMAND_HOME_AGG | MARLSC_F_ROLLING_MEAN_AGG) : 0u) |
      ((CAPS & C_SHIP) ? (MARLSC_F_SHIPPED_HOME | MARLSC_F_SHIPPED_AWAY | MARLSC_F_SHIPPED_AWAY_AGG | MARLSC_F_STOCKOUT) : 0u) |
      ((CAPS & C_FCST) ? (MARLSC_F_FORECAST | MARLSC_F_FORECAST_AGG) : 0u) |
      ((CAPS & C_XFEAT) ? (MARLSC_F_DAYS_OF_SUPPLY | MARLSC_F_NET_INV_POSITION | MARLSC_F_DEMAND_VARIABILITY |
                           MARLSC_F_DEMAND_HISTORY) : 0u);
  const uint32_t F = sp.feat & kFeatMask;
  const bool fixed_lead = !(CAPS & C_STOCH) || sp.lead_mode == MARLSC_LEAD_FIXED;
  const bool need_ship = (CAPS & C_SHIP) && sp.need_ship;
  const int off_dh = (F & MARLSC_F_DEMAND_HOME) ? sp.off_dh : -1;
  const int off_sh = (F & MARLSC_F_SHIPPED_HOME) ? sp.off_sh : -1;
  const int off_sa = (F & MARLSC_F_SHIPPED_AWAY) ? sp.off_sa : -1;
  const int off_so = (F & MARLSC_F_STOCKOUT) ? sp.off_so : -1;
  const int off_rm = (F & MARLSC_F_ROLLING_MEAN) ? sp.off_rm : -1;
  const int off_fc = (F & MARLSC_F_FORECAST) ? sp.off_fc : -1;
  const int off_dos = (F & MARLSC_F_DAYS_OF_SUPPLY) ? sp.off_dos : -1;
  const int off_nip = (F & MARLSC_F_NET_INV_POSITION) ? sp.off_nip : -1;
  const int off_dv = (F & MARLSC_F_DEMAND_VARIABILITY) ? sp.off_dv : -1;
  const int off_hist = (F & MARLSC_F_DEMAND_HISTORY) ? sp.off_hist : -1;

  if ((CAPS & C_IDHOT) && sp.id_off) {
    for (int j = tm.gl; j < W; j += G) obs_w[j] = (j == w) ? 1.0f : 0.0f;
  }
  float* MARLSC_RESTRICT const out = pinned(obs_w + ((CAPS & C_IDHOT) ? sp.id_off : 0));

  // team totals (ratio denominators and aggregates)
  int sumI = 0, sumDh = 0, sumSh = 0, sumSt = 0;
  float sumRm = 0.f, sumFc = 0.f;
  MARLSC_UNROLL
  for (int j = 0; j < SPL; ++j) {
    sumI += vI[j];
    sumDh += vdh[j];
    sumSh += vsh[j];
    sumSt += vst[j];
    sumRm += vrm[j];
    sumFc += vfc[j];
  }
  if (ratio || (F & MARLSC_F_INVENTORY_AGG)) sumI = tm.sum(sumI);
  if (ratio || (F & MARLSC_F_DEMAND_HOME_AGG)) sumDh = tm.sum(sumDh);
  if (need_ship && (ratio || (F & MARLSC_F_SHIPPED_AWAY_AGG))) {
    sumSh = tm.sum(sumSh);
    sumSt = tm.sum(sumSt);
  }
  if (off_rm >= 0 && (ratio || (F & MARLSC_F_ROLLING_MEAN_AGG))) sumRm = tm.sum(sumRm);
  if (off_fc >= 0 && (ratio || (F & MARLSC_F_FORECAST_AGG))) sumFc = tm.sum(sumFc);
  const float dhDen = f_add((float)sumDh, 1e-8f);  // float32 total + eps (multi_env.py:614,737)

  // 1. inventory
  if (sp.off_inv >= 0) {
    MARLSC_UNROLL
    for (int j = 0; j < SPL; ++j) {
      const int s = tm.gl + G * j;
      if (s < S) emit<CAPS>(sp, out, sp.off_inv + s, ratio ? (float)((double)vI[j] / ((double)sumI + 1e-8)) : (float)vI[j]);
    }
    if ((F & MARLSC_F_INVENTORY_AGG) && tm.gl == 0) emit<CAPS>(sp, out, sp.off_inv + S, (float)sumI);
  }

  // 2. pipeline block: written by write_obs_pipeline() where the ring row is first touched (phase 1)

  MARLSC_UNROLL
  for (int j = 0; j < SPL; ++j) {
    const int s = tm.gl + G * j;
    if (s >= S) continue;
    // 3. incoming home-region demand
    if (off_dh >= 0) emit<CAPS>(sp, out, off_dh + s, ratio ? f_div((float)vdh[j], dhDen) : (float)vdh[j]);
    // 4. units shipped to the home region (float64 in the reference)
    if (off_sh >= 0) emit<CAPS>(sp, out, off_sh + s, ratio ? (float)((double)vsh[j] / (double)dhDen) : (float)vsh[j]);
    // 5. units shipped to other regions
    if (off_sa >= 0) {
      const int v = vst[j] - vsh[j];
      emit<CAPS>(sp, out, off_sa + s, ratio ? (float)((double)v / ((double)sumSt + 1e-8)) : (float)v);
    }
    // 6. stockout = max(home demand - shipped home, 0)
    if (off_so >= 0) {
      const float v = (float)imax(vdh[j] - vsh[j], 0);
      emit<CAPS>(sp, out, off_so + s, ratio ? f_div(v, dhDen) : v);
    }
    // 7. rolling mean of home demand
    if (off_rm >= 0) emit<CAPS>(sp, out, off_rm + s, ratio ? f_div(vrm[j], f_add(sumRm, 1e-8f)) : vrm[j]);
    // 8. EMA forecast
    if (off_fc >= 0) emit<CAPS>(sp, out, off_fc + s, ratio ? f_div(vfc[j], f_add(sumFc, 1e-8f)) : vfc[j]);
    // 9. days of supply
    if (off_dos >= 0)
      emit<CAPS>(sp, out, off_dos + s, (float)((double)vI[j] / (double)(vrm[j] > 1.0f ? vrm[j] : 1.0f)));
    // 10. net inventory position = on hand + in transit - forecast * expected lead
    if (off_nip >= 0) {
      const int le = (int)tb.lead[base + s];
      float ptot = 0.f;                         // units in transit to this cell, summed slot by slot in float32
      for (int k = 0; k < L; ++k) {
        int val = 0;
        if (fixed_lead) {
          if (k < le) val = p.ring_q[pmod(t + k + 1 - le, D) * WS + base + s];
        } else if (CAPS & C_STOCH) {
          val = pipeline_value_stoch(sp, p, t, base + s, le, k);
        }
        ptot += (float)val;
      }
      const double v = ((double)vI[j] + (double)ptot) - (double)vfc[j] * (double)le;
      emit<CAPS>(sp, out, off_nip + s, (float)v);
    }
    // 11. demand variability: population std over the history window, float32 like np.std
    if (off_dv >= 0) {
      float v = 0.f;
      if (hist_n > 1) {
        float h[kWindow];
        float sum = 0.f;
        for (int a = 0; a < hist_n; ++a) {  // oldest .. newest, the deque order of the reference
          const int back = hist_n - 1 - a;
          h[a] = back == 0 ? (float)vdh[j] : (float)p.hist[pmod(t - back, kWindow) * WS + base + s];
          sum = f_add(sum, h[a]);
        }
        const float mean = f_div(sum, (float)hist_n);
        float acc = 0.f;
        for (int a = 0; a < hist_n; ++a) {
          const float dlt = f_sub(h[a], mean);
          acc = f_add(acc, f_mul(dlt, dlt));
        }
        v = f_sqrt(f_div(acc, (float)hist_n));
      }
      emit<CAPS>(sp, out, off_dv + s, v);
    }
    // 12. demand history, most recent first, zero padded
    if (off_hist >= 0) {
      for (int a = 0; a < kWindow; ++a) {
        float v = 0.f;
        if (a < hist_n) v = a == 0 ? (float)vdh[j] : (float)p.hist[pmod(t - a, kWindow) * WS + base + s];
        emit<CAPS>(sp, out, off_hist + a * S + s, v);
      }
    }
  }
  if (tm.gl == 0) {
    if (off_dh >= 0 && (F & MARLSC_F_DEMAND_HOME_AGG)) emit<CAPS>(sp, out, off_dh + S, (float)sumDh);
    if (off_sa >= 0 && (F & MARLSC_F_SHIPPED_AWAY_AGG))
      emit<CAPS>(sp, out, off_sa + S, (float)((double)(sumSt - sumSh) / ((double)sumSt + 1e-8)));
    if (off_rm >= 0 && (F & MARLSC_F_ROLLING_MEAN_AGG)) emit<CAPS>(sp, out, off_rm + S, sumRm);
    if (off_fc >= 0 && (F & MARLSC_F_FORECAST_AGG)) emit<CAPS>(sp, out, off_fc + S, sumFc);
  }
}

// ------------------------------------------------------------------------------------------------
// Phase 2 of a step: sequential greedy allocation of environment e's orders against the stock in the
// team's shared-memory scratch (demand_allocator.py:150-208). Shared by the fused step kernel and the
// allocation kernel of the split step (env_split.cuh). Expects s_inv filled, the shipped / lost
// accumulators zeroed and the team synchronised; leaves the team unsynchronised.
// ------------------------------------------------------------------------------------------------
template <int G, int SPL, uint32_t CAPS>
MDEV void allocate_orders(const DevSpec& sp, const Tables& tb, const Team<G>& tm, const Scratch& sc, const EnvPtrs& p,
                          const marlsc_step_io_t& io, int64_t e, int32_t* dh_acc, int dh_mode) {
  const int W = sp.W, S = sp.S, R = sp.R;
  int32_t* s_inv = sc.w + sp.w_inv;
  int32_t* s_sh = sc.w + sp.w_sh;
  int32_t* s_st = sc.w + sp.w_st;
  int32_t* s_shipq = sc.w + sp.w_shipq;
  int32_t* s_cnt = sc.w + sp.w_cnt;
  int32_t* s_lostN = sc.w + sp.w_lostN;
  uint8_t* s_prio = reinterpret_cast<uint8_t*>(sc.w + sp.w_prio);
  int16_t* s_sreg = reinterpret_cast<int16_t*>(sc.w + sp.w_sreg);
  uint8_t* s_sqty = reinterpret_cast<uint8_t*>(sc.w + sp.w_sqty);
  double* s_lostW = sc.d + sp.d_lostW;
  double* s_lostP = sc.d + sp.d_lostP;
  double* s_shipw = sc.d + sp.d_shipw;
  const bool need_ship = (CAPS & C_SHIP) && sp.need_ship;
  const bool unit_w = !(CAPS & C_WEIGHT) || sp.unit_weights;
  const bool has_fixed = (CAPS & C_FIXED) && sp.has_fixed;
  constexpr bool kDiag = (CAPS & C_DIAG) != 0;
  (void)p; (void)s_cnt; (void)s_prio; (void)s_sh; (void)s_st; (void)s_shipw; (void)has_fixed; (void)kDiag;

  // CSR (offsets) or padded layout (row e * stride, count[e]); the latter is what the device sampler writes
  const long long o_begin = io.order_counts ? e * (long long)io.order_stride : (long long)io.order_offsets[e];
  const int n_orders = io.order_counts ? io.order_counts[e] : io.order_offsets[e + 1] - (int)o_begin;
  const int qb = (CAPS & C_QTY16) ? io.order_qty_bytes : 1;
  const int row_bytes = S * qb;
  const int och = qb == 1 ? sp.och : sp.och / 2;   // the staging area is sized for och one-byte rows
  // Staging of a chunk: regions (mapped onto included regions) and quantity rows, as aligned words. When a
  // lane's share of a chunk fits kPre registers the words of the NEXT chunk are requested before the current
  // chunk is allocated and written to shared memory afterwards, so the allocation hides their latency.
  constexpr int kPre = 12;
  const bool prefetch = LaneAlloc<G, CAPS>::value && ((och * row_bytes + 6 + 3) >> 2) <= kPre * G && och <= G;
  uint32_t pre[kPre];
  int pre_r = 0, pre_shift = 0;
  MARLSC_UNROLL
  for (int k = 0; k < kPre; ++k) pre[k] = 0;
  auto request = [&](int c0) {
    const int cn = imin(och, n_orders - c0);
    if (tm.gl < cn) pre_r = io.order_region[o_begin + c0 + tm.gl];
    const uint8_t* src = reinterpret_cast<const uint8_t*>(io.order_qty) + (int64_t)(o_begin + c0) * row_bytes;
    pre_shift = (int)(reinterpret_cast<uintptr_t>(src) & 3u);
    const uint32_t* src_w = reinterpret_cast<const uint32_t*>(src - pre_shift);
    const int nw = (pre_shift + cn * row_bytes + 3) >> 2;
    MARLSC_UNROLL
    for (int k = 0; k < kPre; ++k)
      if (tm.gl + G * k < nw) pre[k] = src_w[tm.gl + G * k];
  };
  if (prefetch && n_orders > 0) request(0);
  // teams narrower than a warp that allocate order by order stay in lockstep with the other teams of their warp
  // (see one_order below): every team takes the chunk trips of the longest order list, with empty chunks at the end
  constexpr bool kLockstep = G < 32 && !LaneAlloc<G, CAPS>::value;
  const int n_trips = G < 32 ? tm.warp_max(n_orders) : n_orders;
  for (int c0 = 0; c0 < n_trips; c0 += och) {
    const int cn = imax(0, imin(och, n_orders - c0));
    int shift = 0;
    if (prefetch) {
      if (tm.gl < cn) {
        int r = pre_r;
        if ((CAPS & C_REGMAP) && sp.region_map) r = sp.region_map[r];
        s_sreg[tm.gl] = (int16_t)r;
      }
      shift = pre_shift;
      uint32_t* dst_w = reinterpret_cast<uint32_t*>(s_sqty);
      const int nw = (shift + cn * row_bytes + 3) >> 2;
      MARLSC_UNROLL
      for (int k = 0; k < kPre; ++k)
        if (tm.gl + G * k < nw) dst_w[tm.gl + G * k] = pre[k];
    } else if (cn > 0) {
      for (int j = tm.gl; j < cn; j += G) {
        int r = io.order_region[o_begin + c0 + j];
        if ((CAPS & C_REGMAP) && sp.region_map) r = sp.region_map[r];
        s_sreg[j] = (int16_t)r;
      }
      const uint8_t* src = reinterpret_cast<const uint8_t*>(io.order_qty) + (int64_t)(o_begin + c0) * row_bytes;
      shift = (int)(reinterpret_cast<uintptr_t>(src) & 3u);
      const uint32_t* src_w = reinterpret_cast<const uint32_t*>(src - shift);
      uint32_t* dst_w = reinterpret_cast<uint32_t*>(s_sqty);
      const int nw = (shift + cn * row_bytes + 3) >> 2;
      int k = tm.gl;
      for (; k + 3 * G < nw; k += 4 * G) {          // four words per lane in flight
        const uint32_t a0 = src_w[k], a1 = src_w[k + G], a2 = src_w[k + 2 * G], a3 = src_w[k + 3 * G];
        dst_w[k] = a0;
        dst_w[k + G] = a1;
        dst_w[k + 2 * G] = a2;
        dst_w[k + 3 * G] = a3;
      }
      for (; k < nw; k += G) dst_w[k] = src_w[k];
    }
    tm.sync();
    if (prefetch && c0 + och < n_orders) request(c0 + och);   // in flight while this chunk is allocated
    if constexpr (LaneAlloc<G, CAPS>::value) {
      // Wide teams, SKUs coupled only through the inventory: the greedy allocation of one SKU never looks
      // at another SKU, so every lane runs the chains of the SKUs it owns (s = lane + G*j, as everywhere else)
      // on its own. A pass covers up to kPassOrders staged orders: the lane first notes which of its cells
      // are non-zero, then works through those lines in order - take the next line, walk it down the
      // region's warehouse priority list (four warehouses per trip) until it is filled or lost. A lane runs
      // TWO such chains side by side, over its even and its odd SKU slots, so that every trip carries two
      // independent dependency chains and the longest lane finishes in about half the trips. Orders stay in
      // sequence per SKU, which is all the sequential semantics of demand_allocator.py:150-208 asks for
      // when no split limit binds; the lanes only meet again at the end of the pass.
      constexpr int NC = MARLSC_LANE_CHAINS < SPL ? MARLSC_LANE_CHAINS : SPL;   // chains per lane
      constexpr int NS = (SPL + NC - 1) / NC;                         // SKU slots per chain
      constexpr int NA = NS < 32 ? NS : 32;                           // ... per pass (mask bits per order, a power of two)
      constexpr int kPassOrders = 64 / NA;
      const uint8_t* rows = s_sqty + shift;
      const int Wp = (W + 3) & ~3;
      // teams narrower than a warp run their passes in lockstep with the other teams of the warp: the same number of
      // passes (empty ones for the shorter order lists) and one exit vote for all of them, so that the chains of
      // four or two teams advance in the same instructions instead of one team after the other
      const int cn_pass = G < 32 ? tm.warp_max(cn) : cn;
      for (int j0 = 0; j0 < cn_pass; j0 += kPassOrders)
      for (int q0 = 0; q0 < NS; q0 += NA) {                           // one trip unless a lane owns > 32 * NC SKUs
        const int pn = imax(0, imin(kPassOrders, cn - j0));
        uint32_t m[2][2] = {{0u, 0u}, {0u, 0u}};                      // [chain][low / high word], order-major bits
        for (int jj = 0; jj < pn; ++jj) {
          const uint8_t* row = rows + (j0 + jj) * row_bytes;
          uint32_t nb[2] = {0u, 0u};                                  // this order's non-zero cells per chain
          MARLSC_UNROLL
          for (int jq = 0; jq < NA * NC; ++jq) {
            const int j = q0 * NC + jq;
            const int s = tm.gl + G * j;
            if (j < SPL && s < S && row[s] != 0) nb[jq % NC] |= 1u << (jq / NC);
          }
          const int at = jj * NA;                                     // NA divides 32: an order never straddles the words
          MARLSC_UNROLL
          for (int c = 0; c < NC; ++c) {
            if (at < 32) m[c][0] |= nb[c] << at; else m[c][1] |= nb[c] << (at - 32);
          }
        }
        int rem[2] = {0, 0}, v[2] = {0, 0}, r[2] = {0, 0}, sku[2] = {0, 0}, oj[2] = {0, 0};
        while (true) {
          MARLSC_UNROLL
          for (int c = 0; c < NC; ++c) {
            if (rem[c] == 0 && (m[c][0] | m[c][1]) != 0) {            // next line of this chain
              int bit;
              if (m[c][0]) {
                bit = lowest_bit(m[c][0]);
                m[c][0] &= m[c][0] - 1;
              } else {
                bit = 32 + lowest_bit(m[c][1]);
                m[c][1] &= m[c][1] - 1;
              }
              oj[c] = j0 + bit / NA;
              sku[c] = tm.gl + G * (NC * (q0 + bit % NA) + c);
              rem[c] = rows[oj[c] * row_bytes + sku[c]];
              r[c] = s_sreg[oj[c]] & 0x7fff;
              v[c] = 0;
              // home-region demand of this step (multi_env.py:763-768); the cell belongs to this lane
              if (dh_mode) {
                uint32_t hm = tb.hmask[r[c]];
                while (hm) {
                  const int w = lowest_bit(hm);
                  hm &= hm - 1;
                  if (dh_mode == 1) global_add(&dh_acc[w * S + sku[c]], rem[c]);   // nobody waits for the sum
                  else dh_acc[w * S + sku[c]] += rem[c];
                }
              }
            }
          }
          MARLSC_UNROLL
          for (int c = 0; c < NC; ++c) {
            if (rem[c] > 0) {                                         // four warehouses down the priority list
              // the stock cells of the line's SKU belong to this lane: the four reads go out together, the
              // takes follow in priority order (rows of the priority table are padded to whole words)
              const uint32_t pw = *reinterpret_cast<const uint32_t*>(tb.prio + r[c] * Wp + v[c]);
              int a[4], wk[4];
              MARLSC_UNROLL
              for (int k = 0; k < 4; ++k) {
                wk[k] = (int)((pw >> (8 * k)) & 0xffu);
                a[k] = v[c] + k < W ? s_inv[wk[k] * S + sku[c]] : 0;
              }
              MARLSC_UNROLL
              for (int k = 0; k < 4; ++k) {
                const int f = imin(rem[c], a[k]);
                if (f > 0) {
                  const int w = wk[k];
                  s_inv[w * S + sku[c]] = a[k] - f;
                  smem_add(&s_shipq[w * R + r[c]], f);
                  if (!unit_w) smem_add(&s_shipw[w * R + r[c]], (double)f * tb.skw[sku[c]]);
                  if (need_ship) {
                    s_st[w * S + sku[c]] += f;
                    if (sp.home[w] == r[c]) s_sh[w * S + sku[c]] += f;
                  }
                }
                rem[c] -= f;
              }
              v[c] += 4;
              if (rem[c] > 0 && v[c] >= W) {
                // no warehouse can supply the rest: lost (demand_allocator.py:205-208)
                smem_add(&s_lostW[r[c]], (double)rem[c] * tb.skw[sku[c]]);
                smem_add(&s_lostP[r[c]], (double)rem[c] * tb.pen[sku[c]]);
                s_sreg[oj[c]] = (int16_t)(r[c] | 0x8000);            // the order counts as lost once, below
                rem[c] = 0;
              }
            }
          }
          // the team's warps run their chains apart
          if (!tm.lock_any((rem[0] | rem[1]) > 0 || (m[0][0] | m[0][1] | m[1][0] | m[1][1]) != 0)) break;
        }
      }
      tm.sync();
#pragma unroll 1
      for (int j = tm.gl; j < cn; j += G)
        if (s_sreg[j] & 0x8000) smem_add(&s_lostN[s_sreg[j] & 0x7fff], 1);
    } else {
      // One order, every SKU of it walked down the region's warehouse list together. Teams narrower than a warp take
      // the same number of trips (the longest order list among the teams of the warp) and meet after every order:
      // the walks are data-dependent, and teams that are never brought back together run one after the other.
      const auto one_order = [&](const int j) {
        const int r = s_sreg[j];
        const uint8_t* row = s_sqty + shift + j * row_bytes;
        int rem[SPL];
        int dsum = 0;
        MARLSC_UNROLL
        for (int jj = 0; jj < SPL; ++jj) {
          const int s = tm.gl + G * jj;
          int d = 0;
          if (s < S) d = qb == 1 ? (int)row[s] : (int)reinterpret_cast<const uint16_t*>(row)[s];
          rem[jj] = d;
          dsum += d;
        }
        if (!tm.any(dsum > 0)) return;                           // all-zero order: nothing can ship or be lost
        // home-region demand of this step (multi_env.py:763-768)
        if (!dh_mode) {
        } else if (!(CAPS & C_BIGW) || tb.hmask) {
          uint32_t hm = tb.hmask[r];
          while (hm) {
            const int w = lowest_bit(hm);
            hm &= hm - 1;
            MARLSC_UNROLL
            for (int jj = 0; jj < SPL; ++jj) {
              const int s = tm.gl + G * jj;
              if (s < S && rem[jj] > 0) {
                // narrow teams: a fire-and-forget reduction instead of a load the next order would wait behind (the
                // plane lives in L2; the cell belongs to this lane, phase 3 reads it back with ld.cg)
                if (G < 32 && dh_mode == 1) global_add(&dh_acc[w * S + s], rem[jj]);
                else dh_acc[w * S + s] += rem[jj];
              }
            }
          }
        } else {
          for (int w = 0; w < W; ++w)
            if (sp.home[w] == r) {
              MARLSC_UNROLL
              for (int jj = 0; jj < SPL; ++jj) {
                const int s = tm.gl + G * jj;
                if (s < S && rem[jj] > 0) dh_acc[w * S + s] += rem[jj];
              }
            }
        }
        const uint8_t* prio;
        if (!(CAPS & C_DYNPRIO) || tb.pstat[r]) {
          prio = tb.prio + r * ((W + 3) & ~3);
        } else {
          // warehouse order depends on the order's weight: key = fixed + variable * weight in float64,
          // stable ascending (demand_allocator.py:168-173; ties to the lowest index, SURVEY 7.2-1)
          double wt = 0.0;
          MARLSC_UNROLL
          for (int jj = 0; jj < SPL; ++jj) {
            const int s = tm.gl + G * jj;
            if (s < S) wt += (double)rem[jj] * tb.skw[s];
          }
          const double wtot = tm.sum(wt);
          if (tm.gl == 0) {
            for (int w = 0; w < W; ++w) {
              const double key = d_add(sp.out_fixed[w * R + r], d_mul(sp.out_var[w * R + r], wtot));
              int pos = w;
              while (pos > 0) {
                const int pw = s_prio[pos - 1];
                const double pk = d_add(sp.out_fixed[pw * R + r], d_mul(sp.out_var[pw * R + r], wtot));
                if (pk <= key) break;
                s_prio[pos] = (uint8_t)pw;
                --pos;
              }
              s_prio[pos] = (uint8_t)w;
            }
          }
          tm.sync();
          prio = s_prio;
        }
        // the order's priority list, four warehouses per register (W <= 16 in the packed form)
        uint32_t pk[4] = {0u, 0u, 0u, 0u};
        const bool packed = W <= 16;
        if (packed) {
          MARLSC_UNROLL
          for (int q4 = 0; q4 < 4; ++q4)
            if (q4 * 4 < W) pk[q4] = reinterpret_cast<const uint32_t*>(prio)[q4];   // rows are 4-byte aligned, see spec_build.h
        }
        int used = 0;
        bool left = true;
        constexpr bool kCount = (CAPS & (C_SPLITLIM | C_FIXED | C_DIAG)) != 0;   // else: no per-order bookkeeping
        for (int v = 0; v < W; ++v) {
          if ((CAPS & C_SPLITLIM) && used >= sp.max_splits + 1) break;
          int w;
          if (packed) {
            const uint32_t word = (v & 8) ? ((v & 4) ? pk[3] : pk[2]) : ((v & 4) ? pk[1] : pk[0]);
            w = (int)((word >> ((v & 3) * 8)) & 0xffu);
          } else {
            w = prio[v];
          }
          int32_t* inv_w = s_inv + w * S;
          const bool is_home = need_ship && (sp.home[w] == r);
          int fsum = 0, rsum = 0;
          double wsum = 0.0;
          MARLSC_UNROLL
          for (int jj = 0; jj < SPL; ++jj) {
            const int s = tm.gl + G * jj;            // rem[jj] > 0 implies s < S (rows beyond S were loaded as 0)
            const int a = rem[jj] > 0 ? inv_w[s] : 0;
            const int f = imin(rem[jj], a);
            if (f > 0) inv_w[s] = a - f;
            rem[jj] -= f;
            fsum += f;
            rsum += rem[jj];
            if ((CAPS & (C_WEIGHT | C_SHIP | C_DIAG)) && f > 0) {
              if (!unit_w) wsum += (double)f * tb.skw[s];
              if (need_ship) {
                s_st[w * S + s] += f;
                if (is_home) s_sh[w * S + s] += f;
              }
              if (kDiag && io.d_ship) io.d_ship[((e * W + w) * R + r) * S + s] += f;
            }
          }
          // Only two votes sit on the order's critical path; the shipped totals go to shared memory
          // with (warp-aggregated) atomic adds that nobody waits for.
          if (fsum > 0) {
            smem_add(&s_shipq[w * R + r], fsum);
            if (!unit_w) smem_add(&s_shipw[w * R + r], wsum);
          }
          if (kCount) {
            const unsigned shipped = tm.ballot(fsum > 0);
            if (shipped == 0u) continue;                         // this warehouse had nothing the order needs
            if ((has_fixed || kDiag) && tm.gl == lowest_bit(shipped)) {
              if (has_fixed) s_cnt[w * R + r] += 1;
              if (kDiag && io.d_ship_count) io.d_ship_count[(e * W + w) * R + r] += 1;
            }
            ++used;
          }
          left = tm.any(rsum > 0);
          if (!left) break;
        }
        // whatever is left is lost (demand_allocator.py:205-208)
        if (left) {
          double lw = 0.0, lp = 0.0;
          MARLSC_UNROLL
          for (int jj = 0; jj < SPL; ++jj) {
            const int s = tm.gl + G * jj;
            if (s < S && rem[jj] > 0) {
              lw += (double)rem[jj] * tb.skw[s];
              lp += (double)rem[jj] * tb.pen[s];
              if (kDiag && io.d_unfulfilled) io.d_unfulfilled[(e * R + r) * S + s] += rem[jj];
            }
          }
          lw = tm.sum(lw);
          lp = tm.sum(lp);
          if (tm.gl == 0) {
            s_lostN[r] += 1;
            s_lostW[r] += lw;
            s_lostP[r] += lp;
            if (kDiag && io.d_lost_orders) io.d_lost_orders[e * R + r] += 1;
          }
        }
      };
      const int cn_trips = kLockstep ? tm.warp_max(cn) : cn;
      for (int j = 0; j < cn_trips; ++j) {
        if (!kLockstep || j < cn) one_order(j);
        if (kLockstep) tm.converge();
      }
    }
    tm.sync();
  }
}

// ------------------------------------------------------------------------------------------------
// One environment, one step.
// ------------------------------------------------------------------------------------------------
template <int G, int SPL, uint32_t CAPS>
MDEV void step_env(const DevSpec& sp, const Tables& tb, const Team<G>& tm, const Scratch& sc,
                   const marlsc_env_state_t& st, const marlsc_step_io_t& io, int64_t e, int t) {
  const int W = sp.W, S = sp.S, R = sp.R, D = sp.D, WS = W * S;
  const EnvPtrs p = env_ptrs(sp, st, e);

  int32_t* s_inv = sc.w + sp.w_inv;
  int32_t* s_dh = sc.w + sp.w_dh;
  int32_t* s_sh = sc.w + sp.w_sh;
  int32_t* s_st = sc.w + sp.w_st;
  int32_t* s_shipq = sc.w + sp.w_shipq;
  int32_t* s_cnt = sc.w + sp.w_cnt;
  int32_t* s_lostN = sc.w + sp.w_lostN;
  double* s_lostW = sc.d + sp.d_lostW;
  double* s_lostP = sc.d + sp.d_lostP;
  double* s_ctot = sc.d + sp.d_ctot;
  double* s_shipw = sc.d + sp.d_shipw;

  const float* act = pinned(io.actions + e * WS);
  const bool fixed_lead = !(CAPS & C_STOCH) || sp.lead_mode == MARLSC_LEAD_FIXED;
  const bool need_ship = (CAPS & C_SHIP) && sp.need_ship;
  const bool need_fcst = (CAPS & C_FCST) && sp.need_fcst;
  const bool unit_w = !(CAPS & C_WEIGHT) || sp.unit_weights;
  const bool direct = !(CAPS & C_ACTX) || sp.action_type == MARLSC_ACTION_DIRECT;
  constexpr bool kDiag = (CAPS & C_DIAG) != 0;
  const uint8_t* lead_new = fixed_lead ? nullptr : io.actual_lead + e * WS;
  const int slot_new = t % D;
  int32_t* ring_new = pinned(p.ring_q + slot_new * WS);
  // accumulator of this step's home-region demand per (warehouse, SKU)
  const int dh_mode = (CAPS & C_DHSMEM) ? sp.dh_mode : (sp.dh_mode == 1 ? 1 : 0);
  int32_t* const dh_acc = dh_mode == 1 ? pinned(p.hist + (t % kWindow) * WS) : s_dh;
  const bool has_fixed = (CAPS & C_FIXED) && sp.has_fixed;

  // ---- phase 1: orders in, arrivals in (multi_env.py:287-292) ------------------------------------
  for (int w = 0; w < W; ++w) {
    const int base = w * S;
    float a_in[SPL];
    int inv_in[SPL], arr_in[SPL], le[SPL];
    MARLSC_UNROLL
    for (int j = 0; j < SPL; ++j) {                 // issue every load of this row first
      const int s = tm.gl + G * j;
      a_in[j] = 0.f;
      inv_in[j] = arr_in[j] = le[j] = 0;
      if (s < S) {
        const int i = base + s;
        le[j] = tb.lead[i];
        a_in[j] = act[i];
        inv_in[j] = p.inv[i];
        if (fixed_lead) {
          int row = slot_new - le[j];               // plane of the order placed at t - le
          if (row < 0) row += D;
          arr_in[j] = p.ring_q[row * WS + i];        // t < le: plane not written since reset, reads 0
        }
      }
    }
    MARLSC_UNROLL
    for (int j = 0; j < SPL; ++j) {
      const int s = tm.gl + G * j;
      if (s < S) {
        const int i = base + s;
        int prev_dem = 0, pend = 0;
        if (!direct) {
          if (t > 0) prev_dem = p.hist[pmod(t - 1, kWindow) * WS + i];
          if (sp.action_type == MARLSC_ACTION_BASE_STOCK) pend = pending_before(sp, p, t, i, le[j]);
        }
        if ((CAPS & C_STOCH) && !fixed_lead) arr_in[j] = arrivals_stoch(sp, p, t, i);   // reads the ring before the slot is reused
        const int q = rescale_action<CAPS>(sp, a_in[j], sp.action_max[s], prev_dem, pend);
        s_inv[i] = inv_in[j] + arr_in[j];
        ring_new[i] = q;
        if (lead_new) p.ring_l[slot_new * WS + i] = lead_new[i];
        if (dh_mode) dh_acc[i] = 0;
        if (need_ship) {
          s_sh[i] = 0;
          s_st[i] = 0;
        }
        if (kDiag && io.d_ordered) io.d_ordered[e * WS + i] = q;
      }
    }
    tm.sync();   // stochastic lead times / small teams: cells of this row were written by other lanes
    write_obs_pipeline<G, SPL, CAPS>(sp, tb, tm, p, io.obs + (e * W + w) * (int64_t)sp.obs_dim, w, t);
  }
  for (int i = tm.gl; i < W * R; i += G) {
    s_shipq[i] = 0;
    if (has_fixed) s_cnt[i] = 0;
    if (!unit_w) s_shipw[i] = 0.0;
  }
  for (int i = tm.gl; i < R; i += G) {
    s_lostN[i] = 0;
    s_lostW[i] = 0.0;
    s_lostP[i] = 0.0;
  }
  tm.converge();

  // ---- phase 2: sequential greedy allocation of this step's orders (demand_allocator.py:150-208)
  allocate_orders<G, SPL, CAPS>(sp, tb, tm, sc, p, io, e, dh_acc, dh_mode);
  tm.converge();

  // ---- phase 3: per warehouse - state write-back, feature buffers, costs, observation row ----------
  const int hist_n = imin(t + 1, kWindow);
  int hoff[kWindow - 1];                              // history planes of steps t-1 .. t-4
  MARLSC_UNROLL
  for (int back = 1; back < kWindow; ++back) hoff[back - 1] = pmod(t - back, kWindow) * WS;
  for (int w = 0; w < W; ++w) {
    const int base = w * S;
    int vI[SPL], vdh[SPL], vsh[SPL], vst[SPL], vq[SPL];
    float vrm[SPL], vfc[SPL];
    int hsum[SPL];
    MARLSC_UNROLL
    for (int j = 0; j < SPL; ++j) {                 // loads first
      const int s = tm.gl + G * j;
      vI[j] = vdh[j] = vsh[j] = vst[j] = vq[j] = hsum[j] = 0;
      vrm[j] = vfc[j] = 0.f;
      if (s < S) {
        const int i = base + s;
        vI[j] = s_inv[i];
        if (dh_mode) vdh[j] = ((LaneAlloc<G, CAPS>::value || G < 32) && dh_mode == 1) ? load_cg(&dh_acc[i]) : dh_acc[i];
        vq[j] = ring_new[i];
        if (need_ship) {
          vsh[j] = s_sh[i];
          vst[j] = s_st[i];
        }
        if (sp.need_hist) {
          MARLSC_UNROLL
          for (int back = 1; back < kWindow; ++back)
            if (back < hist_n) hsum[j] += p.hist[hoff[back - 1] + i];
        }
        if (need_fcst) vfc[j] = p.fcst[i];
      }
    }
    double hold = 0.0, inb = 0.0;
    MARLSC_UNROLL
    for (int j = 0; j < SPL; ++j) {
      const int s = tm.gl + G * j;
      if (s < S) {
        const int i = base + s;
        p.inv[i] = vI[j];                                      // multi_env.py:307 (never negative)
        hold += (double)vI[j] * tb.hold[s];
        if (vq[j] > 0) inb += sp.in_fixed[i] + ((double)vq[j] * tb.skw[s]) * sp.in_var[i];
        if (sp.need_hist) {
          // integer-valued float32 sum over the window is exact in any order (multi_env.py:785-787)
          vrm[j] = f_div((float)(hsum[j] + vdh[j]), (float)hist_n);
          if (dh_mode != 1) p.hist[(t % kWindow) * WS + i] = vdh[j];   // mode 1 accumulated in place
        }
        if (need_fcst) {
          vfc[j] = f_add(f_mul(0.3f, (float)vdh[j]), f_mul(0.7f, vfc[j]));   // multi_env.py:790-793
          p.fcst[i] = vfc[j];
        }
      }
    }
    if (kDiag) {
      hold = tm.sum(hold);
      inb = tm.sum(inb);
    }

    // outbound cost and penalty: lanes over regions
    double outc = 0.0, pen = 0.0;
    for (int r0 = 0; r0 < R; r0 += G) {
      const int r = r0 + tm.gl;
      if (r < R) {
        const int sq = s_shipq[w * R + r];
        if (sq > 0) {
          const double shw = unit_w ? (double)sq : s_shipw[w * R + r];
          outc += shw * sp.out_var[w * R + r];
          if (has_fixed) outc += (double)s_cnt[w * R + r] * sp.out_fixed[w * R + r];
        }
        if (s_lostN[r] > 0) pen += lost_weight<CAPS>(sp, s_shipq, s_lostN, s_lostW, w, r) * s_lostP[r];
      }
    }
    if (kDiag) {
      outc = tm.sum(outc);
      pen = tm.sum(pen);
    } else {
      hold = tm.sum((hold + inb) + (outc + pen));              // one reduction for the whole cost
      inb = outc = pen = 0.0;
    }
    if (tm.gl == 0) {
      s_ctot[w] = hold + pen + outc + inb;
      if (kDiag && io.cost_breakdown) {
        float* cb = io.cost_breakdown + (e * W + w) * 4;
        cb[0] = (float)hold;
        cb[1] = (float)pen;
        cb[2] = (float)outc;
        cb[3] = (float)inb;
      }
    }
    write_obs_row<G, SPL, CAPS>(sp, tb, tm, p, io.obs + (e * W + w) * (int64_t)sp.obs_dim, w, t, hist_n, vI, vdh, vsh, vst,
                          vrm, vfc);
  }
  tm.converge();

  // ---- phase 4: rewards (multi_env.py:316-327) ------------------------------------------------------
  for (int w = tm.gl; w < W; w += G) {
    double rew;
    if (sp.scope == MARLSC_SCOPE_TEAM) {
      rew = 0.0;
      for (int ww = 0; ww < W; ++ww) rew += -(s_ctot[ww] * sp.scale);
    } else {
      rew = -(s_ctot[w] * sp.scale);
    }
    io.rewards[e * W + w] = (float)rew;
  }
  if (io.truncated && tm.gl == 0) io.truncated[e] = (uint8_t)(t + 1 >= sp.episode_length);

  // optional: lost sales per (warehouse, SKU) from the dumped unfulfilled matrix (diagnostics only)
  if (kDiag && io.d_lost_sales && io.d_unfulfilled) {
    tm.sync();
    for (int i = tm.gl; i < WS; i += G) {
      const int w = i / S, s = i - w * S;
      double acc = 0.0;
      for (int r = 0; r < R; ++r) {
        const int u = io.d_unfulfilled[(e * R + r) * S + s];
        if (u != 0) acc += lost_weight<CAPS>(sp, s_shipq, s_lostN, s_lostW, w, r) * (double)u;
      }
      io.d_lost_sales[e * WS + i] = (float)acc;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Reset of one environment (multi_env.py:233-246): clear pipeline and feature state, load the start
// inventory, emit the first observation (all demand-derived features are zero).
// ------------------------------------------------------------------------------------------------
template <int G, int SPL, uint32_t CAPS>
MDEV void reset_env(const DevSpec& sp, const Tables& tb, const Team<G>& tm, const marlsc_env_state_t& st,
                    const int32_t* MARLSC_RESTRICT init_inventory, int per_env, float* MARLSC_RESTRICT obs,
                    int64_t e) {
  const int W = sp.W, S = sp.S, WS = W * S;
  const EnvPtrs p = env_ptrs(sp, st, e);
  const int32_t* init = init_inventory + (per_env ? e * WS : 0);
  for (int i = tm.gl; i < WS; i += G) {
    p.inv[i] = init[i];
    if (p.fcst) p.fcst[i] = 0.f;
    for (int d = 0; d < sp.D; ++d) {
      p.ring_q[d * WS + i] = 0;
      if (p.ring_l) p.ring_l[d * WS + i] = 0;
    }
    if (p.hist)
      for (int h = 0; h < kWindow; ++h) p.hist[h * WS + i] = 0;
  }
  tm.sync();
  for (int w = 0; w < W; ++w) {
    int vI[SPL], vz[SPL];
    float vf[SPL];
    MARLSC_UNROLL
    for (int j = 0; j < SPL; ++j) {
      const int s = tm.gl + G * j;
      vI[j] = s < S ? init[w * S + s] : 0;
      vz[j] = 0;
      vf[j] = 0.f;
    }
    write_obs_pipeline<G, SPL, CAPS>(sp, tb, tm, p, obs + (e * W + w) * (int64_t)sp.obs_dim, w, 0);
    write_obs_row<G, SPL, CAPS>(sp, tb, tm, p, obs + (e * W + w) * (int64_t)sp.obs_dim, w, 0, 0, vI, vz, vz, vz, vf, vf);
  }
}

}  // namespace marlsc
