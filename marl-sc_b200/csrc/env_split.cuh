// env_split.cuh - the step of the common configurations as a sequence of four kernels (K1a..K1d).
//
// The fused kernel (env_kernels.cuh) keeps one environment's stock, shipped totals and order staging in
// shared memory for the whole step, which caps it at 24 warps per SM although only the allocation needs
// that scratch. For configurations the lean capability set covers (fixed lead times, direct actions, static
// warehouse priority, unit SKU weights, inventory / pipeline / home-demand / rolling-mean blocks, no
// diagnostics) the step is split along its data dependencies instead:
//
//   K1a place   - one team per (environment, warehouse) row, no shared memory: action -> order quantity
//                 into the ring (multi_env.py:819-903), arrivals added to the inventory in place
//                 (multi_env.py:905-919), this step's home-demand plane cleared, pipeline block of the
//                 observation row written (multi_env.py:603-633, 941-968). Pure streaming.
//   K1b allocate- one team per environment with the shared-memory scratch: inventory in, greedy allocation
//                 (allocate_orders), inventory out, outbound + lost-sales cost of every warehouse.
//   K1c features- one team per row, no shared memory: holding and inbound cost, rolling mean, the remaining
//                 blocks of the observation row (multi_env.py:577-710, 747-793). Pure streaming.
//   K1d rewards - one thread per environment: cost -> reward per agent or team (multi_env.py:316-327),
//                 truncation flag.
//
// Results are the fused kernel's up to the order of float64 additions in the cost sums.
#pragma once
#include "env_kernels.cuh"

#ifndef MARLSC_ROW_MIN_BLOCKS
#define MARLSC_ROW_MIN_BLOCKS 1   // resident CTAs per SM the row kernels (K1a, K1c) are compiled for
#endif

namespace marlsc {

struct SplitWork {
  double* cost_alloc;   // [E,W] outbound + penalty cost (K1b)
  double* cost_rows;    // [E,W] holding + inbound cost (K1c)
  cudaEvent_t* marks;   // five events around the four launches when timing is on (marlsc_env_set_timing), else null
  const marlsc_episode_metrics_t* metrics = nullptr;   // compact split step: episode accumulators (marlsc_env_set_metrics), or null
};

// Lookup tables straight from global memory (a few KB, read-only, L1 resident) for the kernels without scratch.
MDEV Tables global_tables(const DevSpec& sp) {
  Tables tb;
  tb.skw = sp.skw;
  tb.pen = sp.pen_rate;
  tb.hold = sp.hold_rate;
  tb.prio = sp.prio;
  tb.pstat = sp.prio_static;
  tb.hmask = sp.home_mask;
  tb.lead = sp.lead_u8;
  return tb;
}

// ---- K1a ------------------------------------------------------------------------------------------
template <int G, int SPL>
__global__ void __launch_bounds__(128, MARLSC_ROW_MIN_BLOCKS)
env_place_kernel(const __grid_constant__ DevSpec sp, const __grid_constant__ marlsc_env_state_t st,
                 const __grid_constant__ marlsc_step_io_t io, int t) {
  constexpr uint32_t CAPS = kCapsLean;
  const int W = sp.W, S = sp.S, D = sp.D, WS = W * S;
  const unsigned row = blockIdx.x * (128u / G) + threadIdx.x / G;     // rows fit 32 bits (split_ok, env_step.cu)
  if (row >= (unsigned)st.num_envs * (unsigned)W) return;
  Team<G> tm;
  tm.init();
  const unsigned eu = row / (unsigned)W;
  const int64_t e = eu;
  const int w = (int)(row - eu * (unsigned)W);
  const Tables tb = global_tables(sp);
  const EnvPtrs p = env_ptrs(sp, st, e);
  const float* act = pinned(io.actions + e * WS);
  const int slot_new = t % D;
  int32_t* ring_new = pinned(p.ring_q + slot_new * WS);
  int32_t* dh_plane = sp.dh_mode == 1 ? p.hist + (t % kWindow) * WS : nullptr;
  const int base = w * S;
  float a_in[SPL];
  int inv_in[SPL], arr_in[SPL];
  MARLSC_UNROLL
  for (int j = 0; j < SPL; ++j) {                   // every load of the row first
    const int s = tm.gl + G * j;
    a_in[j] = 0.f;
    inv_in[j] = arr_in[j] = 0;
    if (s < S) {
      const int i = base + s;
      int src = slot_new - (int)tb.lead[i];         // plane of the order placed at t - lead
      if (src < 0) src += D;
      a_in[j] = act[i];
      arr_in[j] = p.ring_q[src * WS + i];           // t < lead: plane not written since reset, reads 0
      inv_in[j] = p.inv[i];
    }
  }
  MARLSC_UNROLL
  for (int j = 0; j < SPL; ++j) {
    const int s = tm.gl + G * j;
    if (s < S) {
      const int i = base + s;
      ring_new[i] = rescale_action<CAPS>(sp, a_in[j], sp.action_max[s], 0, 0);
      if (arr_in[j] != 0) p.inv[i] = inv_in[j] + arr_in[j];
      if (dh_plane) dh_plane[i] = 0;
    }
  }
  // the cells of a lane's pipeline slots are its own: no team synchronisation needed before reading them back
  write_obs_pipeline<G, SPL, CAPS>(sp, tb, tm, p, io.obs + row * (int64_t)sp.obs_dim, w, t);
}

// ---- K1b ------------------------------------------------------------------------------------------
// The allocation needs three of the lookup tables at shared-memory latency (warehouse priority per region,
// static-priority flags, home-warehouse masks); the per-SKU rates are only touched when a line is lost and
// stay in global memory. One round of loads per thread instead of one dependent round per table.
__device__ __forceinline__ Tables stage_alloc_tables(const DevSpec& sp, unsigned char* smem) {
  const int n_prio = (sp.R * ((sp.W + 3) & ~3)) >> 2, n_stat = (sp.R + 3) >> 2, n_mask = sp.home_mask ? sp.R : 0;
  const int n = n_prio + n_stat + n_mask;
  for (int i0 = threadIdx.x; i0 < n; i0 += 2 * blockDim.x) {
    uint32_t v[2];
    uint32_t* dst[2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int i = i0 + k * blockDim.x;
      v[k] = 0;
      dst[k] = nullptr;
      if (i < n_prio) {
        v[k] = reinterpret_cast<const uint32_t*>(sp.prio)[i];
        dst[k] = reinterpret_cast<uint32_t*>(smem + sp.t_prio) + i;
      } else if (i < n_prio + n_stat) {
        v[k] = reinterpret_cast<const uint32_t*>(sp.prio_static)[i - n_prio];
        dst[k] = reinterpret_cast<uint32_t*>(smem + sp.t_pstat) + (i - n_prio);
      } else if (i < n) {
        v[k] = sp.home_mask[i - n_prio - n_stat];
        dst[k] = reinterpret_cast<uint32_t*>(smem + sp.t_hmask) + (i - n_prio - n_stat);
      }
    }
#pragma unroll
    for (int k = 0; k < 2; ++k)
      if (dst[k]) *dst[k] = v[k];
  }
  Tables tb = global_tables(sp);
  tb.prio = smem + sp.t_prio;
  tb.pstat = smem + sp.t_pstat;
  tb.hmask = sp.home_mask ? reinterpret_cast<const uint32_t*>(smem + sp.t_hmask) : nullptr;
  return tb;
}

template <int G, int SPL>
__global__ void __launch_bounds__(Block<G>::threads, G >= 32 ? (G > 32 ? 4 : 6) : 1)
env_alloc_kernel(const __grid_constant__ DevSpec sp, const __grid_constant__ marlsc_env_state_t st,
                 const __grid_constant__ marlsc_step_io_t io, double* __restrict__ cost_alloc, int t) {
  constexpr uint32_t CAPS = kCapsLean;
  extern __shared__ __align__(16) unsigned char smem[];
  __shared__ double xchg[Block<G>::threads / 32];
  constexpr int TEAMS = Block<G>::teams;
  const Tables tb = stage_alloc_tables(sp, smem);
  __syncthreads();
  const int team = threadIdx.x / G;
  const int64_t e = (int64_t)blockIdx.x * TEAMS + team;
  const unsigned live = __ballot_sync(0xffffffffu, e < st.num_envs);
  if (e >= st.num_envs) return;
  Team<G> tm;
  tm.init(xchg, live);
  Scratch sc;
  unsigned char* sbase = smem + sp.t_bytes;
  sc.d = reinterpret_cast<double*>(sbase) + (size_t)team * sp.d_words;
  sc.w = reinterpret_cast<int32_t*>(sbase + (size_t)TEAMS * sp.d_words * sizeof(double)) + (size_t)team * sp.w_words;

  const int W = sp.W, S = sp.S, R = sp.R, WS = W * S;
  const EnvPtrs p = env_ptrs(sp, st, e);
  int32_t* s_inv = sc.w + sp.w_inv;
  int32_t* s_shipq = sc.w + sp.w_shipq;
  int32_t* s_lostN = sc.w + sp.w_lostN;
  double* s_lostW = sc.d + sp.d_lostW;
  double* s_lostP = sc.d + sp.d_lostP;
  for (int i0 = 0; i0 < WS; i0 += 8 * G) {           // inventory in, eight cells per lane in flight
    int v[8];
    MARLSC_UNROLL
    for (int k = 0; k < 8; ++k) {
      const int i = i0 + tm.gl + G * k;
      v[k] = i < WS ? p.inv[i] : 0;
    }
    MARLSC_UNROLL
    for (int k = 0; k < 8; ++k) {
      const int i = i0 + tm.gl + G * k;
      if (i < WS) s_inv[i] = v[k];
    }
  }
  for (int i = tm.gl; i < W * R; i += G) s_shipq[i] = 0;
  for (int i = tm.gl; i < R; i += G) {
    s_lostN[i] = 0;
    s_lostW[i] = 0.0;
    s_lostP[i] = 0.0;
  }
  tm.sync();

  const int dh_mode = sp.dh_mode == 1 ? 1 : 0;
  int32_t* const dh_acc = dh_mode ? pinned(p.hist + (t % kWindow) * WS) : nullptr;
  allocate_orders<G, SPL, CAPS>(sp, tb, tm, sc, p, io, e, dh_acc, dh_mode);
  tm.converge();                                                // the teams of a warp meet again here

  for (int i = tm.gl; i < WS; i += G) p.inv[i] = s_inv[i];      // multi_env.py:307 (never negative)
  tm.sync();
  // Outbound cost and lost-sales penalty of every warehouse (reward_calculator.py:150-175). Lanes take regions;
  // a lane's partial sums per warehouse go to a [W][G + 1] tile laid over the stock scratch (written back above),
  // then lane w adds up row w. Needs (W * (G + 1)) doubles <= W * S words, i.e. 2 * (G + 1) <= S.
  const bool tiled = 2 * (G + 1) <= S && W <= G;
  double* tile = reinterpret_cast<double*>(reinterpret_cast<uintptr_t>(s_inv + 1) & ~uintptr_t(7));
  if (tiled) {
    for (int w = 0; w < W; ++w) tile[w * (G + 1) + tm.gl] = 0.0;
    for (int r = tm.gl; r < R; r += G) {
      const bool lost = s_lostN[r] > 0;
      const double lp = lost ? s_lostP[r] : 0.0;
      int shipped_r = 0;
      if (lost)
        for (int w = 0; w < W; ++w) shipped_r += s_shipq[w * R + r];
      for (int w = 0; w < W; ++w) {
        const int sq = s_shipq[w * R + r];
        double c = 0.0;
        if (sq > 0) c = (double)sq * sp.out_var[w * R + r];
        if (lost) c += lost_weight<CAPS>(sp, s_shipq, s_lostN, s_lostW, w, r, shipped_r) * lp;
        if (sq > 0 || lost) tile[w * (G + 1) + tm.gl] += c;
      }
    }
    tm.sync();
    if (tm.gl < W) {
      double c = 0.0;
      for (int l = 0; l < G; ++l) c += tile[tm.gl * (G + 1) + l];
      cost_alloc[e * W + tm.gl] = c;
    }
  } else {
    for (int w = 0; w < W; ++w) {
      double c = 0.0;
      for (int r = tm.gl; r < R; r += G) {
        const int sq = s_shipq[w * R + r];
        if (sq > 0) c += (double)sq * sp.out_var[w * R + r];
        if (s_lostN[r] > 0) c += lost_weight<CAPS>(sp, s_shipq, s_lostN, s_lostW, w, r) * s_lostP[r];
      }
      c = tm.sum(c);
      if (tm.gl == 0) cost_alloc[e * W + w] = c;
    }
  }
}

// ---- K1c ------------------------------------------------------------------------------------------
template <int G, int SPL>
__global__ void __launch_bounds__(128, MARLSC_ROW_MIN_BLOCKS)
env_feature_kernel(const __grid_constant__ DevSpec sp, const __grid_constant__ marlsc_env_state_t st,
                   const __grid_constant__ marlsc_step_io_t io, double* __restrict__ cost_rows, int t) {
  constexpr uint32_t CAPS = kCapsLean;
  const int W = sp.W, S = sp.S, D = sp.D, WS = W * S;
  const unsigned row = blockIdx.x * (128u / G) + threadIdx.x / G;     // rows fit 32 bits (split_ok, env_step.cu)
  if (row >= (unsigned)st.num_envs * (unsigned)W) return;
  Team<G> tm;
  tm.init();
  const unsigned eu = row / (unsigned)W;
  const int64_t e = eu;
  const int w = (int)(row - eu * (unsigned)W);
  const Tables tb = global_tables(sp);
  const EnvPtrs p = env_ptrs(sp, st, e);
  const int32_t* ring_new = pinned(p.ring_q + (t % D) * WS);
  const int hist_n = imin(t + 1, kWindow);
  const int base = w * S;
  // Every load of the row is issued before any of them is consumed: one pointer per plane (this lane's first cell),
  // the lane's other cells at constant offsets, predicates instead of branches. (Summing the window inside the
  // load loop made each cell wait for its own loads - 7 in flight per lane instead of 28.)
  const bool need_hist = sp.need_hist != 0;
  const int32_t* const inv_l = p.inv + base + tm.gl;
  const int32_t* const ring_l = ring_new + base + tm.gl;
  const int32_t* hist_l[kWindow];                   // plane of step t, then the older planes, newest first
  MARLSC_UNROLL
  for (int back = 0; back < kWindow; ++back)
    hist_l[back] = need_hist ? p.hist + pmod(t - back, kWindow) * WS + base + tm.gl : nullptr;
  bool own[SPL];
  MARLSC_UNROLL
  for (int j = 0; j < SPL; ++j) own[j] = tm.gl + G * j < S;
  int vI[SPL], vdh[SPL], vz[SPL], vq[SPL], hsum[SPL], hv[SPL][kWindow - 1];
  float vrm[SPL], vf[SPL];
  MARLSC_UNROLL
  for (int j = 0; j < SPL; ++j) {
    vz[j] = 0;
    vrm[j] = vf[j] = 0.f;
    vI[j] = own[j] ? inv_l[G * j] : 0;
    vq[j] = own[j] ? ring_l[G * j] : 0;
    vdh[j] = own[j] && need_hist ? load_cg(hist_l[0] + G * j) : 0;   // accumulated by K1b with fire-and-forget adds
    MARLSC_UNROLL
    for (int back = 1; back < kWindow; ++back)
      hv[j][back - 1] = own[j] && need_hist && back < hist_n ? hist_l[back][G * j] : 0;
  }
  MARLSC_UNROLL
  for (int j = 0; j < SPL; ++j) {
    hsum[j] = 0;
    MARLSC_UNROLL
    for (int back = 1; back < kWindow; ++back) hsum[j] += hv[j][back - 1];
  }
  double cost = 0.0;
  const bool by_row = sp.row_rates_uniform != 0;      // rates constant over the row: integer sums, three products
  int nI = 0, nQ = 0, nPos = 0;
  MARLSC_UNROLL
  for (int j = 0; j < SPL; ++j) {
    const int s = tm.gl + G * j;
    if (s < S) {
      const int i = base + s;
      if (by_row) {
        nI += vI[j];
        nQ += vq[j];
        nPos += vq[j] > 0 ? 1 : 0;
      } else {
        cost += (double)vI[j] * tb.hold[s];                                                     // holding
        if (vq[j] > 0) cost += sp.in_fixed[i] + ((double)vq[j] * tb.skw[s]) * sp.in_var[i];    // inbound
      }
      // integer-valued float32 sum over the window is exact in any order (multi_env.py:785-787)
      if (sp.need_hist) vrm[j] = f_div((float)(hsum[j] + vdh[j]), (float)hist_n);
    }
  }
  if (by_row) {
    nI = tm.sum(nI);
    nQ = tm.sum(nQ);
    nPos = tm.sum(nPos);
    cost = (double)nI * tb.hold[0] + ((double)nPos * sp.in_fixed[base] + ((double)nQ * tb.skw[0]) * sp.in_var[base]);
  } else {
    cost = tm.sum(cost);
  }
  if (tm.gl == 0) cost_rows[row] = cost;
  write_obs_row<G, SPL, CAPS>(sp, tb, tm, p, io.obs + row * (int64_t)sp.obs_dim, w, t, hist_n, vI, vdh, vz, vz, vrm, vf);
}

// ---- K1d ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
env_reward_kernel(const __grid_constant__ DevSpec sp, int64_t num_envs, const double* __restrict__ cost_alloc,
                  const double* __restrict__ cost_rows, float* __restrict__ rewards, uint8_t* __restrict__ truncated, int t);

// K1b for one-warp teams (env_alloc.cu): 1 = launched, 0 = not applicable (the caller launches env_alloc_kernel), < 0 = error
int launch_alloc_warp(int spl, const LaunchArgs& a, const marlsc_step_io_t& io, double* cost_alloc, int t, cudaStream_t s,
                      bool prepare_only = false);

// One launcher per (G, SPL); defined through MARLSC_DEFINE_SPLIT in the per-width translation units.
template <int G, int SPL>
int launch_split_t(const LaunchArgs& a, const marlsc_step_io_t& io, const SplitWork& wk, int t, cudaStream_t s) {
  constexpr int GR = G > 32 ? 32 : G;               // the row kernels never need more than a warp per row
  constexpr int SPLR = G > 32 ? SPL * (G / 32) : SPL;
  const int64_t rows = a.st.num_envs * a.ds.W;
  const unsigned grid_rows = (unsigned)((rows + 128 / GR - 1) / (128 / GR));
  // every check and attribute call of the allocation launch first: a failure must not leave the state half-stepped
  bool warp_chains = false;
  if constexpr (G == 32) {
    const int rc = launch_alloc_warp(SPL, a, io, wk.cost_alloc, t, s, true);
    if (rc < 0) return rc;
    warp_chains = rc == 1;
  }
  const size_t smem = step_smem_bytes(a.ds, G);
  if (!warp_chains) {
    if ((int)smem > a.max_smem_optin)
      return set_error(MARLSC_EUNSUPPORTED, "shared-memory scratch of " + std::to_string(smem) + " bytes per CTA does not fit; use a wider team");
    static std::atomic<size_t> configured[kMaxDevices];   // per device: the attributes belong to the device's context
    static std::atomic<bool> carveout[kMaxDevices];
    int dev = 0;
    MARLSC_CUDA(cudaGetDevice(&dev));
    const int di = dev < kMaxDevices ? dev : kMaxDevices - 1;
    if (dev >= kMaxDevices || !carveout[di].load()) {
      MARLSC_CUDA(cudaFuncSetAttribute((const void*)env_alloc_kernel<G, SPL>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                       (int)cudaSharedmemCarveoutMaxShared));
      carveout[di].store(true);
    }
    if (smem > 48 * 1024 && (dev >= kMaxDevices || smem > configured[di].load())) {
      MARLSC_CUDA(cudaFuncSetAttribute((const void*)env_alloc_kernel<G, SPL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      configured[di].store(smem);
    }
  }
  if (wk.marks) MARLSC_CUDA(cudaEventRecord(wk.marks[0], s));
  env_place_kernel<GR, SPLR><<<grid_rows, 128, 0, s>>>(a.ds, a.st, io, t);
  MARLSC_CUDA(cudaGetLastError());
  if (wk.marks) MARLSC_CUDA(cudaEventRecord(wk.marks[1], s));
  if (warp_chains) {
    const int rc = launch_alloc_warp(SPL, a, io, wk.cost_alloc, t, s);
    if (rc < 0) return rc;
  } else {
    const unsigned grid_envs = (unsigned)((a.st.num_envs + Block<G>::teams - 1) / Block<G>::teams);
    env_alloc_kernel<G, SPL><<<grid_envs, Block<G>::threads, smem, s>>>(a.ds, a.st, io, wk.cost_alloc, t);
    MARLSC_CUDA(cudaGetLastError());
  }
  if (wk.marks) MARLSC_CUDA(cudaEventRecord(wk.marks[2], s));

  env_feature_kernel<GR, SPLR><<<grid_rows, 128, 0, s>>>(a.ds, a.st, io, wk.cost_rows, t);
  MARLSC_CUDA(cudaGetLastError());
  if (wk.marks) MARLSC_CUDA(cudaEventRecord(wk.marks[3], s));

  env_reward_kernel<<<(unsigned)((a.st.num_envs + 255) / 256), 256, 0, s>>>(a.ds, a.st.num_envs, wk.cost_alloc, wk.cost_rows,
                                                                           io.rewards, io.truncated, t);
  MARLSC_CUDA(cudaGetLastError());
  if (wk.marks) MARLSC_CUDA(cudaEventRecord(wk.marks[4], s));
  g_launches.fetch_add(4, std::memory_order_relaxed);
  return MARLSC_OK;
}

#define MARLSC_DECLARE_SPLIT(G) \
  int launch_split_g##G(int spl, const LaunchArgs& a, const marlsc_step_io_t& io, const SplitWork& wk, int t, cudaStream_t s);
MARLSC_DECLARE_SPLIT(8)
MARLSC_DECLARE_SPLIT(16)
MARLSC_DECLARE_SPLIT(32)
MARLSC_DECLARE_SPLIT(64)

#define MARLSC_SPLIT_CASE(G, SPL) case SPL: return launch_split_t<G, SPL>(a, io, wk, t, s);
#define MARLSC_DEFINE_SPLIT(G, CASES)                                                                          \
  namespace marlsc {                                                                                           \
  int launch_split_g##G(int spl, const LaunchArgs& a, const marlsc_step_io_t& io, const SplitWork& wk, int t,  \
                        cudaStream_t s) {                                                                      \
    switch (spl) { CASES default: break; }                                                                     \
    return set_error(MARLSC_EUNSUPPORTED, "no split-step kernels instantiated for this team size / SKU count"); \
  }                                                                                                            \
  }

}  // namespace marlsc
