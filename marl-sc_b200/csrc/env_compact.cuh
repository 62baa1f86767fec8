// env_compact.cuh - the environment step of the common configurations as ONE fused kernel over the compact state
// layout (MARLSC_LAYOUT_COMPACT): a warp advances one environment by one timestep.
//
// What changed against the split step (env_split.cuh) and why (ncu, profiles/r1_k1_split_65536envs.summary.txt: the three
// kernels issued 27 k warp instructions per env-step - 70 % of the row kernels' were address arithmetic of the per-cell
// ring gather - and moved 154 KB per env-step, 44 KB of it the int32 ring):
//
//   * state in the width the values need - on-hand stock and home-demand history uint16, in-transit ring uint8 - and the
//     ring indexed by ARRIVAL time: an order placed at t with (fixed) lead l goes to plane (t + l) % L of its warehouse
//     row, ring[e][w][d][s]. Arrivals of step t are plane t % L for every cell and pipeline slot k of the observation
//     (multi_env.py:941-968) is plane (t + 1 + k) % L for every cell: both are plain row copies, no per-cell plane
//     arithmetic. The only scattered access left is the single byte a new order writes.
//   * demand as sparse "lines" (marlsc_step_io.lines): the non-zero (order, SKU) cells, pre-sorted into 32 streams by
//     SKU % 32. Lane l walks stream l - no pass over 80 %-zero dense rows, no shuffles, 2 bytes per line instead of
//     S + 2 bytes per order.
//   * the lane that owns SKU s owns every cell (w, s): stock [W,S] lives in shared memory for the step, a SKU's
//     availability over the warehouses in two registers, and a trip of the allocation loop is one shipment from the
//     cheapest warehouse that has the SKU (same chains as env_alloc.cuh; demand_allocator.py:150-208).
//   * rewards come out of the same kernel: no cost workspaces, no reward launch, inventory and the home-demand plane
//     cross HBM once.
//
// Semantics are the reference's (multi_env.py:253-366), results equal the wide kernels' (integers exact; float64 cost
// sums in a different order).
#pragma once
#include "env_kernels.cuh"

namespace marlsc {

constexpr int kCompactWarps = 8;          // environments per CTA
constexpr int kCompactMaxS = 128;         // four SKU slots per lane
constexpr int kCompactMaxR = 64;          // region id field of a line
constexpr int kCompactMaxW = 16;          // availability masks
constexpr int kCompactMaxL = 16;

// shared memory of the step kernel: [perm5 | prio16 | home_wh | warp 0 | warp 1 | ...], byte offsets
struct CompactSmem {
  int t_perm, t_prio, t_home, t_bytes;          // per CTA
  int inv, shipq, lostU, lostP, avail, ring, warp_bytes;     // per warp, from the warp's base
};
__host__ __device__ inline CompactSmem compact_smem(int W, int S, int R, int nch, int pen_uniform) {
  CompactSmem l;
  int o = 0;
  l.t_perm = o; o += (R * nch * 32 * 2 + 15) & ~15;
  l.t_prio = o; o += R * 16;
  l.t_home = o; o += (R + 15) & ~15;
  l.t_bytes = o;
  o = 0;
  l.lostP = o; o += pen_uniform ? 0 : R * 8;
  l.inv = o; o += (W * S * 2 + 15) & ~15;
  l.shipq = o; o += W * R * 4;
  l.lostU = o; o += R * 4;
  l.avail = o;                                      // (unused: availability masks live in registers)
  l.ring = o;                                       // (unused: the line words in flight live in registers)
  l.warp_bytes = (o + 15) & ~15;
  return l;
}

// entry of a line stream: quantity (1..255) | region << 8 | SKU slot << 14; 0 pads a stream to the environment's round count.
// Entries 0 and 1 of a lane (its first 32-bit word) are the lane's SKU map: byte k = the SKU slot k stands for, 255 = none.
__host__ __device__ inline uint16_t line_entry(int qty, int region, int slot) { return (uint16_t)(qty | (region << 8) | (slot << 14)); }

// the map word of lane l when SKUs are dealt round-robin (SKU s on lane s % 32, slot s / 32)
__host__ __device__ inline uint32_t identity_map_word(int lane, int S) {
  uint32_t m = 0u;
  for (int k = 0; k < 4; ++k) m |= (uint32_t)(lane + 32 * k < S ? lane + 32 * k : 255) << (8 * k);
  return m;
}

int launch_step_compact(const LaunchArgs& a, const marlsc_step_io_t& io, int t, cudaStream_t s);
struct SplitWork;
int launch_split_compact(const LaunchArgs& a, const marlsc_step_io_t& io, const SplitWork& wk, int t, cudaStream_t s);
int launch_reset_compact(const LaunchArgs& a, const int32_t* init, int per_env, float* obs, cudaStream_t s);
int launch_base_stock_compact(const DevSpec& ds, const marlsc_env_state_t& st, const float* level, int level_per_env, int t,
                              float* actions, cudaStream_t s);
int launch_lines_from_orders(const DevSpec& ds, int64_t num_envs, const marlsc_step_io_t& io, int32_t line_stride, uint16_t* lines,
                             int32_t* line_counts, int32_t* overflow, cudaStream_t s);

// Episode metrics (csrc/metrics.cu): after a COMPACT split step, add the step's rewards to episode_return; after a WIDE
// step, fold its diagnostic outputs (cost_breakdown, d_ordered, d_ship, d_unfulfilled) and rewards into every accumulator.
int launch_metrics_returns(const marlsc_episode_metrics_t& m, const float* rewards, int64_t num_envs, int W, cudaStream_t s);
int launch_metrics_fold(const marlsc_episode_metrics_t& m, const marlsc_step_io_t& io, int64_t num_envs, int W, int R, int S,
                        cudaStream_t s);

}  // namespace marlsc
