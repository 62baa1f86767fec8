// gae.cu - K2: reverse-time GAE(lambda) / value-target scan, and K3: per-policy advantage
// standardisation.
//
// The reference delegates both to RLlib 2.52.1 (GeneralAdvantageEstimation learner connector,
// configured at src/algorithms/ippo.py:145-160 / mappo.py:142-157 with use_gae, lambda_, gamma);
// RLlib is not vendored, so the recursion below restates its published semantics (SURVEY.md 8c):
//   target_t = r_t + gamma * ((1 - lambda) * V_{t+1} + lambda * target_{t+1}),  target_T := V_T
//   adv_t    = target_t - V_t
// with the scan restarting at episode cuts (truncation: bootstrap from the value of the final
// observation; termination: bootstrap from 0). Parity for this kernel is pinned to the NumPy
// restatement in oracle/gae_oracle.py only ("parity unpinned" at the RLlib boundary).
//
// Layout is time-major [T, N] with N = E*W columns, so a warp reads 32 consecutive columns of one
// timestep: fully coalesced, 16-17 algorithmic bytes per agent-step, HBM bound.
#include "lib_common.h"

using namespace marlsc;

namespace {

constexpr int kGaeUnroll = 4;

__global__ void __launch_bounds__(256)
gae_kernel(const float* __restrict__ rewards, const float* __restrict__ values, const uint8_t* __restrict__ cut,
           const float* __restrict__ cut_values, int T, long long N, float gamma, float lam,
           float* __restrict__ adv, float* __restrict__ targets) {
  const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  const float gl = gamma * lam, g1 = gamma * (1.0f - lam);
  float v_next = values[(long long)T * N + n];   // V(s_T)
  float tgt_next = v_next;
  int t = T - 1;
  // blocks of kGaeUnroll steps: issue all loads of the block first so they are in flight together
  for (; t >= kGaeUnroll - 1; t -= kGaeUnroll) {
    float r[kGaeUnroll], v[kGaeUnroll];
#pragma unroll
    for (int k = 0; k < kGaeUnroll; ++k) {
      r[k] = rewards[(long long)(t - k) * N + n];
      v[k] = values[(long long)(t - k) * N + n];
    }
#pragma unroll
    for (int k = 0; k < kGaeUnroll; ++k) {
      const int tt = t - k;
      if (cut && cut[tt]) {
        v_next = cut_values ? cut_values[(long long)tt * N + n] : 0.0f;
        tgt_next = v_next;
      }
      const float tgt = r[k] + (g1 * v_next + gl * tgt_next);
      targets[(long long)tt * N + n] = tgt;
      adv[(long long)tt * N + n] = tgt - v[k];
      tgt_next = tgt;
      v_next = v[k];
    }
  }
  for (; t >= 0; --t) {
    const float r = rewards[(long long)t * N + n], v = values[(long long)t * N + n];
    if (cut && cut[t]) {
      v_next = cut_values ? cut_values[(long long)t * N + n] : 0.0f;
      tgt_next = v_next;
    }
    const float tgt = r + (g1 * v_next + gl * tgt_next);
    targets[(long long)t * N + n] = tgt;
    adv[(long long)t * N + n] = tgt - v;
    tgt_next = tgt;
    v_next = v;
  }
}

// ---- standardisation: sum, sum of squares and count in double, then (x - mean) / max(1e-4, std) -----
// The three doubles are the workspace's public layout (include/marlsc_b200.h): a data-parallel caller sums them over
// its ranks between the two kernels.
struct StdWs {
  double sum, sumsq, count;
};

__global__ void __launch_bounds__(256) moments_kernel(const float* __restrict__ x, long long n, StdWs* ws) {
  double s = 0.0, q = 0.0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const double v = (double)x[i];
    s += v;
    q += v * v;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, o);
    q += __shfl_xor_sync(0xffffffffu, q, o);
  }
  __shared__ double ss[8], sq[8];
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) {
    ss[w] = s;
    sq[w] = q;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0.0, b = 0.0;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) {
      a += ss[i];
      b += sq[i];
    }
    atomicAdd(&ws->sum, a);
    atomicAdd(&ws->sumsq, b);
    if (blockIdx.x == 0) ws->count = (double)n;
  }
}

__global__ void __launch_bounds__(256) standardize_kernel(float* __restrict__ x, long long n, const StdWs* __restrict__ ws) {
  const double mean = ws->sum / ws->count;
  double var = ws->sumsq / ws->count - mean * mean;
  if (var < 0.0) var = 0.0;
  const float m = (float)mean;
  const float sd = fmaxf(1e-4f, (float)sqrt(var));
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    x[i] = (x[i] - m) / sd;
}

unsigned std_grid(long long n) {
  const long long want = (n + 255) / 256;
  return (unsigned)(want < 148 * 8 ? want : 148 * 8);
}

}  // namespace

extern "C" {

int marlsc_gae(const float* rewards, const float* values, const uint8_t* cut, const float* cut_values, int32_t T,
               int64_t N, float gamma, float lam, float* adv, float* targets, void* stream) {
  if (!rewards || !values || !adv || !targets) return set_error(MARLSC_EINVAL, "rewards, values, adv and targets must not be NULL");
  if (T < 1 || N < 1) return set_error(MARLSC_EINVAL, "T and N must be positive");
  if (cut_values && !cut) return set_error(MARLSC_EINVAL, "cut_values needs cut");
  if (!(gamma >= 0.f && gamma <= 1.f) || !(lam >= 0.f && lam <= 1.f)) return set_error(MARLSC_EINVAL, "gamma and lam must be in [0,1]");
  const int block = 256;
  const unsigned grid = (unsigned)((N + block - 1) / block);
  gae_kernel<<<grid, block, 0, static_cast<cudaStream_t>(stream)>>>(rewards, values, cut, cut_values, T, N, gamma, lam, adv, targets);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  MARLSC_CUDA(cudaGetLastError());
  return MARLSC_OK;
}

size_t marlsc_standardize_workspace_bytes(void) { return sizeof(StdWs); }

int marlsc_standardize_moments(const float* x, int64_t n, void* workspace, void* stream) {
  if (!x || !workspace) return set_error(MARLSC_EINVAL, "x and workspace must not be NULL");
  if (n < 1) return set_error(MARLSC_EINVAL, "n must be positive");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  MARLSC_CUDA(cudaMemsetAsync(workspace, 0, sizeof(StdWs), s));
  moments_kernel<<<std_grid(n), 256, 0, s>>>(x, n, static_cast<StdWs*>(workspace));
  g_launches.fetch_add(1, std::memory_order_relaxed);
  MARLSC_CUDA(cudaGetLastError());
  return MARLSC_OK;
}

int marlsc_standardize_apply(float* x, int64_t n, const void* workspace, void* stream) {
  if (!x || !workspace) return set_error(MARLSC_EINVAL, "x and workspace must not be NULL");
  if (n < 1) return set_error(MARLSC_EINVAL, "n must be positive");
  standardize_kernel<<<std_grid(n), 256, 0, static_cast<cudaStream_t>(stream)>>>(x, n, static_cast<const StdWs*>(workspace));
  g_launches.fetch_add(1, std::memory_order_relaxed);
  MARLSC_CUDA(cudaGetLastError());
  return MARLSC_OK;
}

int marlsc_standardize(float* x, int64_t n, void* workspace, void* stream) {
  const int rc = marlsc_standardize_moments(x, n, workspace, stream);
  return rc != MARLSC_OK ? rc : marlsc_standardize_apply(x, n, workspace, stream);
}

}  // extern "C"
