// metrics.cu - per-episode accumulators of marlsc_env_set_metrics outside the step kernels: the rewards of a COMPACT split
// step (its kernels accumulate the costs and units themselves), and the whole fold of a WIDE step's diagnostic outputs
// (reference: collect_step_info, multi_env.py:330-362, summed over an episode).
#include "env_compact.cuh"

namespace marlsc {
namespace {

constexpr unsigned FULL = 0xffffffffu;

// episode_return += rewards, one thread per (environment, warehouse)
__global__ void __launch_bounds__(256)
metrics_returns_kernel(const float* __restrict__ rewards, double* __restrict__ episode_return, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) episode_return[i] += (double)rewards[i];
}

__device__ __forceinline__ long long warp_sum(long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
  return v;
}

// One warp per environment: the float32 cost breakdown widened to float64, sum_s d_ordered and sum_{r,s} d_ship per
// warehouse, sum_{r,s} d_unfulfilled, demand as shipped + unfulfilled, and the rewards. Integer sums are exact.
__global__ void __launch_bounds__(256)
metrics_fold_kernel(const __grid_constant__ marlsc_episode_metrics_t m, const float* __restrict__ cost_breakdown,
                    const int32_t* __restrict__ ordered, const int32_t* __restrict__ ship, const int32_t* __restrict__ unfulfilled,
                    const float* __restrict__ rewards, int64_t num_envs, int W, int R, int S) {
  const int lane = threadIdx.x & 31;
  const int64_t e = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (e >= num_envs) return;
  const int RS = R * S;
  long long shipped_env = 0;
  for (int w = 0; w < W; ++w) {
    const int64_t row = e * W + w;
    long long o = 0, sh = 0;
    for (int s = lane; s < S; s += 32) o += ordered[row * S + s];
    for (int i = lane; i < RS; i += 32) sh += ship[row * RS + i];
    o = warp_sum(o);
    sh = warp_sum(sh);
    shipped_env += sh;
    if (lane == 0) {
      const float* cb = cost_breakdown + row * 4;
      m.holding_cost[row] += (double)cb[0];
      m.penalty_cost[row] += (double)cb[1];
      m.outbound_cost[row] += (double)cb[2];
      m.inbound_cost[row] += (double)cb[3];
      m.ordered_units[row] += (double)o;
      m.shipped_units[row] += (double)sh;
      m.episode_return[row] += (double)rewards[row];
    }
  }
  long long lost = 0;
  for (int i = lane; i < RS; i += 32) lost += unfulfilled[e * RS + i];
  lost = warp_sum(lost);
  if (lane == 0) {
    m.lost_units[e] += (double)lost;
    m.demand_units[e] += (double)(shipped_env + lost);
  }
}

}  // namespace

int launch_metrics_returns(const marlsc_episode_metrics_t& m, const float* rewards, int64_t num_envs, int W, cudaStream_t s) {
  const int64_t n = num_envs * W;
  metrics_returns_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(rewards, m.episode_return, n);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  MARLSC_CUDA(cudaGetLastError());
  return MARLSC_OK;
}

int launch_metrics_fold(const marlsc_episode_metrics_t& m, const marlsc_step_io_t& io, int64_t num_envs, int W, int R, int S,
                        cudaStream_t s) {
  metrics_fold_kernel<<<(unsigned)((num_envs + 7) / 8), 256, 0, s>>>(m, io.cost_breakdown, io.d_ordered, io.d_ship, io.d_unfulfilled,
                                                                     io.rewards, num_envs, W, R, S);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  MARLSC_CUDA(cudaGetLastError());
  return MARLSC_OK;
}

}  // namespace marlsc
