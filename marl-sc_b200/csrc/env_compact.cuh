// env_compact.cuh - the environment step of the common configurations over the compact state layout
// (MARLSC_LAYOUT_COMPACT), in env_compact.cu: K1a' places the orders and writes the pipeline block with one warp per
// (environment, warehouse) row, K1b' allocates the step's demand with one warp per environment, K1c' writes the remaining
// observation blocks and row costs with one warp per row, and K1d sums team rewards.
//
// What changed against the WIDE layout's split step (env_split.cuh) and why (ncu, profiles/r1_k1_split_65536envs.summary.txt:
// the three kernels issued 27 k warp instructions per env-step - 70 % of the row kernels' were address arithmetic of the
// per-cell ring gather - and moved 154 KB per env-step, 44 KB of it the int32 ring):
//
//   * state in the width the values need - on-hand stock and home-demand history uint16, in-transit ring uint8
//     ring[e][d][w][s] indexed by PLACEMENT time like the wide one: the orders placed at t are plane t % L. The ring was
//     first indexed by arrival time (an order placed at t with lead l in plane (t + l) % L of its warehouse row), which
//     made the arrivals and the pipeline slots of the observation plain row copies. But with a lead per cell one step's
//     orders land in every plane of a row, and single-byte stores dirty whole sectors, so K1a' wrote the row's L x S
//     bytes back to record S new ones: 10 KB per env-step at the large config. Indexed by placement time a step writes
//     one contiguous W x S plane per environment (1 KB); K1a' loads every plane of a row anyway, and finds the per-cell
//     ages of the arrivals and the pipeline slots in shared memory (multi_env.py:941-968).
//   * demand as sparse "lines" (marlsc_step_io.lines): the non-zero (order, SKU) cells, pre-sorted into 32 streams by
//     SKU % 32. Lane l walks stream l - no pass over 80 %-zero dense rows, no shuffles, 2 bytes per line instead of
//     S + 2 bytes per order.
//   * in the allocation the lane that owns SKU s owns every cell (w, s): stock [W,S] lives in shared memory, a SKU's
//     availability over the warehouses in two registers, and a trip of the allocation loop is one shipment from the
//     cheapest warehouse that has the SKU (same chains as env_alloc.cuh; demand_allocator.py:150-208).
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

// shared memory of the allocation kernel (K1b'): [region records | warp 0 | warp 1 | ...], byte offsets. The record of
// region r (compact_region_bytes each) holds everything a line of that region looks up: its perm5 chunks, its prio16 row
// and its home-table entry (uint16), so that one base address serves all three. Per warp the home-region demand plane
// [W,S] uint16 of this step (need_hist only) follows the stock [W,S] uint16, and the lost units [R] follow the shipped
// units [W,R] (they are the table's row W, lost_off bytes on). inv_row and shipq_row are the bytes of one warehouse row
// of the stock (and history) and of the shipped-unit table: the allocation loop uses them as launch constants.
__host__ __device__ constexpr int compact_region_bytes(int nch) { return nch * 64 + 20; }
struct CompactSmem {
  int t_bytes;                                  // per CTA: the region records
  int inv, hist, shipq, lostU, lostP, warp_bytes;     // per warp, from the warp's base
  int inv_row, shipq_row, lost_off;
};
__host__ __device__ inline CompactSmem compact_smem(int W, int S, int R, int nch, int pen_uniform, int need_hist) {
  CompactSmem l;
  l.t_bytes = (R * compact_region_bytes(nch) + 15) & ~15;
  int o = 0;
  l.lostP = o; o += pen_uniform ? 0 : R * 8;
  l.inv = o; o += (W * S * 2 + 15) & ~15;
  l.hist = o; o += need_hist ? (W * S * 2 + 15) & ~15 : 0;
  l.shipq = o; o += W * R * 4;
  l.lostU = o; o += R * 4;
  l.warp_bytes = (o + 15) & ~15;
  l.inv_row = S * 2;
  l.shipq_row = R * 4;
  l.lost_off = l.lostU - l.shipq;
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
