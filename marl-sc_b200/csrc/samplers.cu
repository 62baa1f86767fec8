// samplers.cu - K4: on-device Poisson demand sampler, K5: batched base-stock heuristic policy.
//
// K4 draws, per environment and step, what the reference's PoissonDemandSampler draws
// (src/environment/components/demand_sampler.py:105-163): per region r an order count ~ Poisson(lambda_orders[r]);
// per order a Bernoulli(probability_skus[r]) mask over SKUs and quantities max(1, Poisson(lambda_quantity[r,s])).
// Orders are emitted region-major like the reference. The random stream is Philox4x32-10 keyed by
// (seed; env, step, row, lane block), so it is reproducible and independent of the launch geometry, but it is
// NOT the reference's PCG64 stream: equality with the reference is distributional, replay/host sampling stays the
// bit-exact path. The law is the reference's at every parameter: Poisson draws invert the exact CDF (float32 search
// below rate 30, a float64 walk from the mode above) and a SKU is included with probability p to within 2^-33.
// tests/sampler_reference.py recomputes every draw from the counters; tests/test_device_samplers.py replays the
// kernels against it and checks the law against scipy.
// Output is the padded order layout marlsc_step_io accepts: env e owns rows [e*max_orders, e*max_orders + count[e]).
//
// K5 evaluates the reference's base-stock heuristic (src/experiments/run_baselines.py:133-207) for every
// environment: qty = clip(S[w,k] - on_hand - in_transit, 0, max_qty), action = 2 qty / max_qty - 1 (float32).
#include <cmath>
#include <vector>

#include "env_kernels.cuh"

namespace marlsc {

__device__ __forceinline__ void philox_round(uint32_t (&c)[4], const uint32_t (&k)[2]) {
  const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
  const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
  c[0] = hi1 ^ c[1] ^ k[0];
  c[1] = lo1;
  c[2] = hi0 ^ c[3] ^ k[1];
  c[3] = lo0;
}

__device__ __forceinline__ void philox4x32(uint32_t (&c)[4], uint64_t seed) {
  uint32_t k[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    philox_round(c, k);
    k[0] += 0x9E3779B9u;
    k[1] += 0xBB67AE85u;
  }
}

__device__ __forceinline__ float u01(uint32_t x) { return (x >> 8) * (1.0f / 16777216.0f); }   // [0,1)

constexpr float kModeRate = 30.f;   // from this rate on, Poisson inversion starts at the mode instead of at 0

// Poisson(lambda) by inversion: the smallest k with u <= P(X <= k).
// Below kModeRate: sequential search from 0 in float32. At and above: a float64 walk from the mode m = floor(lambda),
// starting from F(m) and P(m) (mode: the host's float64 values for this rate), up while u > F, down while
// u <= F - P. This stays exact where a search from 0 would need ~lambda terms and lose float32 precision on the way.
__device__ __forceinline__ int poisson_from_mode(float lambda, float u, const double* __restrict__ mode) {
  const double lam = (double)lambda, ud = (double)u;
  int k = (int)floorf(lambda);
  double F = mode[0], p = mode[1];
  if (ud > F) {
    while (ud > F) {
      ++k;
      p *= lam / (double)k;
      const double Fn = F + p;
      if (Fn == F) break;                              // the float64 sum has stopped growing (u is at most 1 - 2^-24)
      F = Fn;
    }
  } else {
    while (k > 0 && ud <= F - p) {
      F -= p;
      p *= (double)k / lam;
      --k;
    }
  }
  return k;
}

__device__ __forceinline__ int poisson_from(float lambda, float u, const double* __restrict__ mode) {
  if (lambda <= 0.f) return 0;
  if (lambda < kModeRate) {
    // float32 running sum: in the far tail the terms drop below half an ulp of F and the sum plateaus a few ulp
    // short of 1 (2-3 x 2^-24 for lambda = 1, 3, 5), below the largest uniform 1 - 2^-24 - the search then has to stop
    // where the sum stops growing instead of running on to the cap.
    float p = __expf(-lambda), F = p;
    int k = 0;
    while (u > F && k < 200) {
      ++k;
      p *= lambda / (float)k;
      const float Fn = F + p;
      if (Fn == F && (float)k > lambda) break;
      F = Fn;
    }
    return k;
  }
  return poisson_from_mode(lambda, u, mode);
}

constexpr int kCdf = 16;     // tabulated Poisson CDF entries per (region, SKU): P(X <= k), k < kCdf
struct Inclusion {           // SKU inclusion with probability p (included): t = floor(4096 p), f = round(frac(4096 p) 2^20)
  uint32_t t, f;
  float inv_f;               // float(1 / f), 0 when f == 0
};
struct DemandParams {
  const float* lam_orders;   // [R]
  const float* prob;         // [R]
  const float* lam_qty;      // [R,S], or [R] when the rate does not vary over the SKUs of a region (sku_stride 0)
  const float* cdf_qty;      // [R,S,kCdf], or [R,kCdf]: 3 KB that stay in L1 instead of 320 KB of L2 lookups
  const Inclusion* incl;     // [R]: inclusion split of prob
  const double* mode_orders; // [R,2]: F(m), P(m) at the mode of lam_orders (rates >= kModeRate only)
  const double* mode_qty;    // [R,S,2] or [R,2], like lam_qty
  int region_stride, sku_stride;   // cell (r, s) of lam_qty / cdf_qty / mode_qty is entry r * region_stride + s * sku_stride
};

// SKU inclusion with probability p from one 32-bit word w, whose low 12 bits b12 and high 20 bits b20 are uniform:
// included when b12 < t, or when b12 == t and b20 < f, with t = floor(4096 p) and f = round(frac(4096 p) * 2^20)
// (host-computed from the double p): probability p to within 2^-33. The quantity uniform is b20 / 2^20, or
// b20 * float(1 / f) for a cell included on the boundary bucket b12 == t (b20 is uniform below f there; the product
// stays below 1). When 4096 p is an integer f is 0 and this is the plain 12-bit test.
__device__ __forceinline__ bool included(uint32_t w, const Inclusion& in, float& uq) {
  const uint32_t b12 = w & 0xfffu, b20 = w >> 12;
  uq = (float)b20 * (1.0f / 1048576.0f);
  if (b12 < in.t) return true;
  if (b12 != in.t || b20 >= in.f) return false;
  uq = (float)b20 * in.inv_f;
  return true;
}

// Quantity max(1, Poisson(lambda)) by inversion: the smallest k with u <= P(X <= k), found by a four-step search of the
// tabulated CDF (same result as poisson_from's sequential search up to float rounding of the table); beyond the table
// the sequential search continues from its last entry. Rates >= kModeRate walk from the mode like poisson_from.
__device__ __forceinline__ int quantity_from(const float* __restrict__ cdf, float lambda, float u, const double* __restrict__ mode) {
  if (lambda >= kModeRate || lambda <= 0.f) return poisson_from(lambda, u, mode);
  int k = u > cdf[7] ? 8 : 0;
  k += u > cdf[k + 3] ? 4 : 0;
  k += u > cdf[k + 1] ? 2 : 0;
  k += u > cdf[k] ? 1 : 0;
  if (k == kCdf - 1 && u > cdf[kCdf - 1]) {            // tail: P(X > 15) (1e-4 at lambda 5)
    float F = cdf[kCdf - 1], p = F - cdf[kCdf - 2];
    while (u > F && k < 200) {
      ++k;
      p *= lambda / (float)k;
      const float Fn = F + p;
      if (Fn == F) break;                               // the float32 sum has stopped growing (see poisson_from)
      F = Fn;
    }
  }
  return k;
}

// test hook: the inversions K4 uses, for given (lambda, u) pairs
__global__ void poisson_inverse_kernel(const float* __restrict__ lambda, const float* __restrict__ u, long long n,
                                       const float* __restrict__ cdf, const double* __restrict__ mode, int32_t* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  out[i] = cdf ? quantity_from(cdf + i * kCdf, lambda[i], u[i], mode + 2 * i) : poisson_from(lambda[i], u[i], mode + 2 * i);
}

// one warp per environment
__global__ void __launch_bounds__(128)
sample_demand_kernel(DemandParams dp, int R, int S, long long E, uint64_t seed, long long step, int omax,
                     int32_t* __restrict__ counts, int16_t* __restrict__ region, uint8_t* __restrict__ qty,
                     int32_t* __restrict__ overflow) {
  const long long e = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (e >= E) return;
  const int lane = threadIdx.x & 31;
  int16_t* reg_e = region + e * omax;
  uint8_t* qty_e = qty + e * (long long)omax * S;
  int row = 0;                                       // rows emitted so far (warp-uniform)
  for (int r0 = 0; r0 < R; r0 += 32) {
    const int r = r0 + lane;
    int n = 0;
    if (r < R) {
      uint32_t c[4] = {(uint32_t)e, (uint32_t)(e >> 32) ^ 0x5bd1e995u, (uint32_t)step, (uint32_t)r};
      philox4x32(c, seed);
      n = poisson_from(dp.lam_orders[r], u01(c[0]), dp.mode_orders + 2 * r);
    }
    for (int l = 0; l < 32 && r0 + l < R; ++l) {      // regions in ascending order, like the reference
      const int nr = __shfl_sync(0xffffffffu, n, l);
      const int rr = r0 + l;
      const Inclusion in = dp.incl[rr];
      for (int i = 0; i < nr; ++i) {
        if (row >= omax) {                             // staging is full: drop the order and flag it
          if (lane == 0) atomicExch(overflow, 1);
          continue;
        }
        if (lane == 0) reg_e[row] = (int16_t)rr;
        for (int s0 = 0; s0 < S; s0 += 128) {          // four SKUs per lane per Philox call
          if (s0 + lane >= S) continue;
          uint32_t c[4] = {(uint32_t)e, (uint32_t)row | 0x80000000u, (uint32_t)step, (uint32_t)(s0 + lane)};
          philox4x32(c, seed);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int s = s0 + lane + 32 * j;
            if (s < S) {
              // one 32-bit word per SKU: 12 bits decide inclusion, the other 20 drive the Poisson inversion
              float uq;
              int q = 0;
              if (included(c[j], in, uq)) {
                const int cell = rr * dp.region_stride + s * dp.sku_stride;
                q = quantity_from(dp.cdf_qty + (size_t)cell * kCdf, dp.lam_qty[cell], uq, dp.mode_qty + 2 * cell);
                q = q < 1 ? 1 : (q > 255 ? 255 : q);
              }
              qty_e[(long long)row * S + s] = (uint8_t)q;
            }
          }
        }
        ++row;
      }
    }
  }
  if (lane == 0) counts[e] = row;
}

// K4 writing lines (the compact layout's demand format, include/marlsc_b200.h): the same draws as sample_demand_kernel
// (same Philox counters), but every lane appends the non-zero cells of its SKUs to its own stream instead of filling
// dense rows - the allocation kernel then walks the streams without ever scanning the 80 % zero cells. SKUs stay dealt
// round-robin (lane s % 32, slot s / 32: the lane's map word says so); ranking them by line count as the packers of
// recorded demand do would need the counts before the first entry is written, i.e. every draw twice.
__global__ void __launch_bounds__(128)
sample_demand_lines_kernel(DemandParams dp, int R, int S, long long E, uint64_t seed, long long step, int stride,
                           const int32_t* __restrict__ region_map, uint16_t* __restrict__ lines, int32_t* __restrict__ counts,
                           int32_t* __restrict__ overflow) {
  const long long e = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (e >= E) return;
  const int lane = threadIdx.x & 31;
  uint16_t* out = lines + e * (long long)stride * 32 + 2 * lane;     // entry p of this lane: out[(p >> 1) * 64 + (p & 1)]
  int row = 0, cnt = 2;                               // entries 0, 1: the lane's SKU map
  bool over = false;
  for (int r0 = 0; r0 < R; r0 += 32) {
    const int r = r0 + lane;
    int n = 0;
    if (r < R) {
      uint32_t c[4] = {(uint32_t)e, (uint32_t)(e >> 32) ^ 0x5bd1e995u, (uint32_t)step, (uint32_t)r};
      philox4x32(c, seed);
      n = poisson_from(dp.lam_orders[r], u01(c[0]), dp.mode_orders + 2 * r);
    }
    for (int l = 0; l < 32 && r0 + l < R; ++l) {      // regions in ascending order, like the reference
      const int nr = __shfl_sync(0xffffffffu, n, l);
      const int rr = r0 + l;
      const int rm = region_map ? region_map[rr] : rr;
      // The inclusion test first (included(), on the raw word), then only the cells that passed - 20 % - go through
      // the quantity inversion: a lane walks its hit bits, so a trip of the inner loop serves one hit of every lane
      // instead of one SKU slot of every lane. Orders are taken two at a time (two Philox calls in flight, hit counts
      // of a pair are better balanced over the lanes than those of one order); within a lane the first order's lines
      // still precede the second's.
      const Inclusion in = dp.incl[rr];
      const float* const cdf_r = dp.cdf_qty + (size_t)rr * dp.region_stride * kCdf;
      const float* const lam_r = dp.lam_qty + (size_t)rr * dp.region_stride;
      for (int i = 0; i < nr; i += 2) {
        const bool two = i + 1 < nr;
        uint32_t c0[4] = {(uint32_t)e, (uint32_t)row | 0x80000000u, (uint32_t)step, (uint32_t)lane};
        uint32_t c1[4] = {(uint32_t)e, (uint32_t)(row + 1) | 0x80000000u, (uint32_t)step, (uint32_t)lane};
        uint32_t hits = 0u;                           // bits 0-3: SKU slots of the first order, 4-7: of the second
        if (lane < S) {
          philox4x32(c0, seed);
          if (two) philox4x32(c1, seed);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const bool named = lane + 32 * j < S;
            float uq;
            if (named && included(c0[j], in, uq)) hits |= 1u << j;
            if (named && two && included(c1[j], in, uq)) hits |= 16u << j;
          }
        }
        while (hits) {
          const int b = __ffs((int)hits) - 1, j = b & 3;
          hits &= hits - 1u;
          const uint32_t lo = j == 0 ? c0[0] : (j == 1 ? c0[1] : (j == 2 ? c0[2] : c0[3]));
          const uint32_t hi = j == 0 ? c1[0] : (j == 1 ? c1[1] : (j == 2 ? c1[2] : c1[3]));
          const uint32_t cj = b < 4 ? lo : hi;
          const int s = lane + 32 * j;
          float uq;
          (void)included(cj, in, uq);               // the cell passed: this only recomputes its quantity uniform
          int q = quantity_from(cdf_r + (size_t)(s * dp.sku_stride) * kCdf, lam_r[s * dp.sku_stride], uq,
                                dp.mode_qty + 2 * ((size_t)rr * dp.region_stride + s * dp.sku_stride));
          q = q < 1 ? 1 : (q > 255 ? 255 : q);
          if (cnt < stride) out[(long long)(cnt >> 1) * 64 + (cnt & 1)] = (uint16_t)(q | (rm << 8) | (j << 14));
          else over = true;
          ++cnt;
        }
        row += two ? 2 : 1;
      }
    }
  }
  cnt = cnt < stride ? cnt : stride;
  const int longest = __reduce_max_sync(0xffffffffu, cnt);
  int rounds = 0;
  if (longest > 2) {                                  // an environment without demand has no rounds at all
    rounds = (longest + 1) & ~1;                      // whole round pairs
    uint32_t map = 0u;
#pragma unroll
    for (int k = 0; k < 4; ++k) map |= (uint32_t)(lane + 32 * k < S ? lane + 32 * k : 255) << (8 * k);
    out[0] = (uint16_t)(map & 0xffffu);
    out[1] = (uint16_t)(map >> 16);
    for (int c = cnt; c < rounds; ++c) out[(long long)(c >> 1) * 64 + (c & 1)] = 0;   // pad this stream to the environment's round count
  }
  if (lane == 0) counts[e] = rounds;
  if (over) atomicExch(overflow, 1);
}

// K4 for small SKU counts: one thread per environment (a warp per environment leaves 30 of 32 lanes idle at two
// SKUs). Same Philox counters and words as sample_demand_kernel, so both kernels draw identical orders.
__global__ void __launch_bounds__(128)
sample_demand_thread_kernel(DemandParams dp, int R, int S, long long E, uint64_t seed, long long step, int omax,
                            int32_t* __restrict__ counts, int16_t* __restrict__ region, uint8_t* __restrict__ qty,
                            int32_t* __restrict__ overflow) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  int16_t* reg_e = region + e * omax;
  uint8_t* qty_e = qty + e * (long long)omax * S;
  int row = 0;
  for (int r = 0; r < R; ++r) {
    uint32_t c[4] = {(uint32_t)e, (uint32_t)(e >> 32) ^ 0x5bd1e995u, (uint32_t)step, (uint32_t)r};
    philox4x32(c, seed);
    const int nr = poisson_from(dp.lam_orders[r], u01(c[0]), dp.mode_orders + 2 * r);
    const Inclusion in = dp.incl[r];
    for (int i = 0; i < nr; ++i) {
      if (row >= omax) {
        atomicExch(overflow, 1);
        continue;
      }
      reg_e[row] = (int16_t)r;
      for (int s = 0; s < S; ++s) {
        const int s0 = s & ~127, lane = s & 31, j = (s >> 5) & 3;   // the warp kernel's (block, lane, word) of SKU s
        uint32_t d[4] = {(uint32_t)e, (uint32_t)row | 0x80000000u, (uint32_t)step, (uint32_t)(s0 + lane)};
        philox4x32(d, seed);
        float uq;
        int q = 0;
        if (included(d[j], in, uq)) {
          const int cell = r * dp.region_stride + s * dp.sku_stride;
          q = quantity_from(dp.cdf_qty + (size_t)cell * kCdf, dp.lam_qty[cell], uq, dp.mode_qty + 2 * cell);
          q = q < 1 ? 1 : (q > 255 ? 255 : q);
        }
        qty_e[(long long)row * S + s] = (uint8_t)q;
      }
      ++row;
    }
  }
  counts[e] = row;
}

// K4b: actual lead times of one step, four consecutive cells per thread (one Philox call). A 32-bit word w gives
// the deviation floor(w * (2d+1) / 2^32) - d: uniform over {-d..+d} up to a bias below (2d+1) / 2^32.
__global__ void __launch_bounds__(256)
sample_lead_kernel(const int32_t* __restrict__ expected, const int32_t* __restrict__ max_dev, int S, long long WS,
                   long long n_cells, uint64_t seed, long long step, uint8_t* __restrict__ actual) {
  const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long i0 = q * 4;
  if (i0 >= n_cells) return;
  uint32_t c[4] = {(uint32_t)q, (uint32_t)(q >> 32) ^ 0x1ead71e5u, (uint32_t)step, (uint32_t)(step >> 32)};
  philox4x32(c, seed);
  uint32_t packed = 0u;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const long long i = i0 + j;
    int v = 0;
    if (i < n_cells) {
      const int cell = (int)(i % WS);
      const int d = max_dev[cell % S];
      const int dev = (int)__umulhi(c[j], (uint32_t)(2 * d + 1)) - d;
      v = expected[cell] + dev;
      v = v < 1 ? 1 : (v > 255 ? 255 : v);
    }
    packed |= (uint32_t)v << (8 * j);
  }
  if (i0 + 3 < n_cells && (reinterpret_cast<uintptr_t>(actual) & 3u) == 0) {
    reinterpret_cast<uint32_t*>(actual)[q] = packed;
  } else {
    for (int j = 0; j < 4 && i0 + j < n_cells; ++j) actual[i0 + j] = (uint8_t)(packed >> (8 * j));
  }
}

// K5: one thread per (env, warehouse, SKU) cell; IDX is 32-bit whenever the batch has fewer than 2^32 cells. The
// in-transit planes of a cell are read four at a time (independent loads in flight instead of a chain of le).
template <typename IDX>
__global__ void __launch_bounds__(256)
base_stock_policy_kernel(const __grid_constant__ DevSpec sp, const __grid_constant__ marlsc_env_state_t st,
                         const float* __restrict__ level, int level_per_env, int t, float* __restrict__ actions) {
  const IDX WS = (IDX)(sp.W * sp.S);
  const IDX idx = (IDX)blockIdx.x * (IDX)blockDim.x + (IDX)threadIdx.x;
  if (idx >= (IDX)st.num_envs * WS) return;
  const IDX e = idx / WS;
  const int i = (int)(idx - e * WS);
  const int D = sp.D;
  const int32_t* ring = static_cast<const int32_t*>(st.ring_qty) + (long long)e * (long long)WS * D + i;
  const int le = sp.lead_exp[i];
  int pending = 0;                                     // units ordered and not yet arrived before step t
  if (sp.lead_mode == MARLSC_LEAD_FIXED) {
    int row = (t - 1) % D;                             // plane of the order placed one step ago, then backwards
    const int n = le < t ? le : t;
    for (int a0 = 0; a0 < n; a0 += 4) {
      int v[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        int rr = row - k;
        rr += rr < 0 ? D : 0;
        v[k] = a0 + k < n ? ring[(long long)rr * (long long)WS] : 0;
      }
      pending += (v[0] + v[1]) + (v[2] + v[3]);
      row -= 4;
      row += row < 0 ? D : 0;
    }
  } else {
    const uint8_t* rl = st.ring_lead + (long long)e * (long long)WS * D + i;
    for (int d = 0; d < D; ++d) {
      const int tau = (t - 1) - (((t - 1 - d) % D + D) % D);
      if (tau < 0) continue;
      const int q = ring[(long long)d * (long long)WS];
      if (q > 0 && tau + (int)rl[(long long)d * (long long)WS] >= t) pending += q;
    }
  }
  const double mx = sp.action_max[i % sp.S];
  double q = (double)(level_per_env ? level[idx] : level[i]) - (double)static_cast<const int32_t*>(st.inventory)[idx] - (double)pending;
  q = q < 0.0 ? 0.0 : (q > mx ? mx : q);
  actions[idx] = (float)(2.0 * q / mx - 1.0);
}

int launch_base_stock(const DevSpec& ds, const marlsc_env_state_t& st, const float* level, int level_per_env, int t,
                      float* actions, cudaStream_t s) {
  const long long n = st.num_envs * (long long)ds.W * ds.S;
  const unsigned grid = (unsigned)((n + 255) / 256);
  if (n < (1LL << 32)) base_stock_policy_kernel<unsigned><<<grid, 256, 0, s>>>(ds, st, level, level_per_env, t, actions);
  else base_stock_policy_kernel<long long><<<grid, 256, 0, s>>>(ds, st, level, level_per_env, t, actions);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  MARLSC_CUDA(cudaGetLastError());
  return MARLSC_OK;
}

}  // namespace marlsc

using namespace marlsc;

namespace {

// F(m) and P(m) at the mode m = floor(lambda) of Poisson(lambda), in double (poisson_from_mode). The sum runs down from
// the mode until the terms stop counting, about 40 sqrt(lambda) of them; rates below kModeRate get zeros (unused).
void mode_cdf(double lam, double* out) {
  out[0] = out[1] = 0.0;
  if (!(lam >= (double)kModeRate)) return;
  const double m = std::floor(lam);
  const double pm = std::exp(-lam + m * std::log(lam) - std::lgamma(m + 1.0));
  double F = pm, p = pm;
  for (double k = m; k > 0.0; k -= 1.0) {
    p *= k / lam;
    F += p;
    if (p < F * 1e-18) break;
  }
  out[0] = F;
  out[1] = pm;
}

// the Inclusion of included() for inclusion probability p
Inclusion inclusion_split(double p) {
  const double x = p * 4096.0, t = std::floor(x);
  const double f = std::nearbyint((x - t) * 1048576.0);
  if (f >= 1048576.0) return Inclusion{(uint32_t)t + 1u, 0u, 0.f};
  return Inclusion{(uint32_t)t, (uint32_t)f, f > 0.0 ? (float)(1.0 / f) : 0.f};
}

}  // namespace

struct marlsc_demand {
  void* blob = nullptr;
  DemandParams dp{};
  int R = 0, S = 0, device = 0;
};

extern "C" {

int marlsc_demand_create(int32_t n_regions, int32_t n_skus, const double* lambda_orders, const double* probability_skus,
                         const double* lambda_quantity, int device, marlsc_demand_t** out) {
  if (!out || !lambda_orders || !probability_skus || !lambda_quantity) return set_error(MARLSC_EINVAL, "null argument");
  if (n_regions < 1 || n_skus < 1) return set_error(MARLSC_EINVAL, "n_regions and n_skus must be positive");
  // rates that do not vary over the SKUs of a region (the reference's scalar and per-region forms): one CDF row per region
  bool per_region = true;
  for (int r = 0; r < n_regions && per_region; ++r)
    for (int s = 1; s < n_skus; ++s)
      if (lambda_quantity[(size_t)r * n_skus + s] != lambda_quantity[(size_t)r * n_skus]) {
        per_region = false;
        break;
      }
  const int cols = per_region ? 1 : n_skus;
  const size_t n_cells = (size_t)n_regions * cols;
  // one upload: floats (rates, CDF tables), then the inclusion splits, then the mode CDFs in double
  const size_t n_f = (size_t)2 * n_regions + n_cells * (1 + kCdf);
  const size_t off_i = (n_f * sizeof(float) + 7) & ~(size_t)7;
  const size_t off_d = (off_i + (size_t)n_regions * sizeof(Inclusion) + 7) & ~(size_t)7;
  const size_t bytes = off_d + (size_t)2 * (n_regions + n_cells) * sizeof(double);
  std::vector<double> raw((bytes + 7) / 8);
  unsigned char* base = reinterpret_cast<unsigned char*>(raw.data());
  float* host = reinterpret_cast<float*>(base);
  Inclusion* incl = reinterpret_cast<Inclusion*>(base + off_i);
  double* mode = reinterpret_cast<double*>(base + off_d);
  for (int r = 0; r < n_regions; ++r) {
    if (!(lambda_orders[r] >= 0.0) || !(probability_skus[r] >= 0.0 && probability_skus[r] <= 1.0))
      return set_error(MARLSC_EINVAL, "lambda_orders must be >= 0 and probability_skus in [0,1]");
    host[r] = (float)lambda_orders[r];
    host[n_regions + r] = (float)probability_skus[r];
    incl[r] = inclusion_split(probability_skus[r]);
    mode_cdf((double)(float)lambda_orders[r], mode + 2 * r);
  }
  for (size_t i = 0; i < (size_t)n_regions * n_skus; ++i)
    if (!(lambda_quantity[i] >= 0.0)) return set_error(MARLSC_EINVAL, "lambda_quantity must be >= 0");
  for (size_t i = 0; i < n_cells; ++i) {
    const double lq = lambda_quantity[per_region ? i * n_skus : i];
    host[2 * n_regions + i] = (float)lq;
    // P(X <= k) for the float32 rate the kernel sees, accumulated in double
    const double lam = (double)(float)lq;
    double pk = std::exp(-lam), F = pk;
    for (int k = 0; k < kCdf; ++k) {
      if (k > 0) {
        pk *= lam / k;
        F += pk;
      }
      host[2 * n_regions + n_cells + i * kCdf + k] = (float)F;
    }
    mode_cdf(lam, mode + 2 * (n_regions + i));
  }
  marlsc_demand* d = new (std::nothrow) marlsc_demand();
  if (!d) return set_error(MARLSC_ENOMEM, "out of host memory");
  d->R = n_regions;
  d->S = n_skus;
  d->device = device;
  cudaError_t ce = cudaSetDevice(device);
  if (ce == cudaSuccess) ce = cudaMalloc(&d->blob, bytes);
  if (ce == cudaSuccess) ce = cudaMemcpy(d->blob, base, bytes, cudaMemcpyHostToDevice);
  if (ce != cudaSuccess) {
    if (d->blob) cudaFree(d->blob);
    delete d;
    return set_error(MARLSC_ECUDA, std::string("uploading demand parameters: ") + cudaGetErrorString(ce));
  }
  const float* fb = static_cast<const float*>(d->blob);
  d->dp.lam_orders = fb;
  d->dp.prob = fb + n_regions;
  d->dp.lam_qty = fb + 2 * n_regions;
  d->dp.cdf_qty = fb + 2 * n_regions + n_cells;
  d->dp.incl = reinterpret_cast<const Inclusion*>(static_cast<const unsigned char*>(d->blob) + off_i);
  d->dp.mode_orders = reinterpret_cast<const double*>(static_cast<const unsigned char*>(d->blob) + off_d);
  d->dp.mode_qty = d->dp.mode_orders + 2 * n_regions;
  d->dp.region_stride = cols;
  d->dp.sku_stride = per_region ? 0 : 1;
  *out = d;
  return MARLSC_OK;
}

void marlsc_demand_destroy(marlsc_demand_t* d) {
  if (!d) return;
  if (d->blob) cudaFree(d->blob);
  delete d;
}

int marlsc_demand_sample(marlsc_demand_t* d, int64_t num_envs, uint64_t seed, int64_t step_index, int32_t max_orders_per_env,
                         int32_t* order_counts, int16_t* order_region, uint8_t* order_qty, int32_t* overflow_flag, void* stream) {
  if (!d || !order_counts || !order_region || !order_qty || !overflow_flag) return set_error(MARLSC_EINVAL, "null argument");
  if (num_envs < 1 || max_orders_per_env < 1) return set_error(MARLSC_EINVAL, "num_envs and max_orders_per_env must be positive");
  MARLSC_CUDA(cudaSetDevice(d->device));
  if (d->S <= 16) {   // few SKUs: a thread per environment
    sample_demand_thread_kernel<<<(unsigned)((num_envs + 127) / 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(
        d->dp, d->R, d->S, num_envs, seed, step_index, max_orders_per_env, order_counts, order_region, order_qty, overflow_flag);
  } else {
    const int wpb = 4;
    const unsigned grid = (unsigned)((num_envs + wpb - 1) / wpb);
    sample_demand_kernel<<<grid, wpb * 32, 0, static_cast<cudaStream_t>(stream)>>>(
        d->dp, d->R, d->S, num_envs, seed, step_index, max_orders_per_env, order_counts, order_region, order_qty, overflow_flag);
  }
  g_launches.fetch_add(1, std::memory_order_relaxed);
  MARLSC_CUDA(cudaGetLastError());
  return MARLSC_OK;
}

int marlsc_demand_sample_lines(marlsc_demand_t* d, int64_t num_envs, uint64_t seed, int64_t step_index, int32_t line_stride,
                               const int32_t* region_map, uint16_t* lines, int32_t* line_counts, int32_t* overflow_flag,
                               void* stream) {
  if (!d || !lines || !line_counts || !overflow_flag) return set_error(MARLSC_EINVAL, "null argument");
  if (num_envs < 1 || line_stride < 2 || (line_stride & 1)) return set_error(MARLSC_EINVAL, "num_envs must be positive and line_stride positive and even");
  if (d->S > 128) return set_error(MARLSC_EUNSUPPORTED, "lines address at most 128 SKUs");
  if (!region_map && d->R > 64) return set_error(MARLSC_EUNSUPPORTED, "lines address at most 64 regions");
  MARLSC_CUDA(cudaSetDevice(d->device));
  const int wpb = 4;
  sample_demand_lines_kernel<<<(unsigned)((num_envs + wpb - 1) / wpb), wpb * 32, 0, static_cast<cudaStream_t>(stream)>>>(
      d->dp, d->R, d->S, num_envs, seed, step_index, line_stride, region_map, lines, line_counts, overflow_flag);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  MARLSC_CUDA(cudaGetLastError());
  return MARLSC_OK;
}

int marlsc_poisson_inverse(const float* lambda, const float* u, int64_t n, int32_t tabulated, int32_t* k_out, void* stream) {
  if (!lambda || !u || !k_out || n < 1) return set_error(MARLSC_EINVAL, "null argument or n < 1");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  // the tables marlsc_demand_create builds, for these rates: mode CDFs always, CDF rows when tabulated
  std::vector<float> hl((size_t)n);
  std::vector<double> hm((size_t)n * 2);
  MARLSC_CUDA(cudaMemcpyAsync(hl.data(), lambda, sizeof(float) * n, cudaMemcpyDeviceToHost, s));
  MARLSC_CUDA(cudaStreamSynchronize(s));
  for (int64_t i = 0; i < n; ++i) mode_cdf((double)hl[i], hm.data() + 2 * i);
  double* mode = nullptr;
  MARLSC_CUDA(cudaMalloc(&mode, hm.size() * sizeof(double)));
  MARLSC_CUDA(cudaMemcpyAsync(mode, hm.data(), hm.size() * sizeof(double), cudaMemcpyHostToDevice, s));
  float* cdf = nullptr;
  if (tabulated) {
    std::vector<float> hc((size_t)n * kCdf);
    for (int64_t i = 0; i < n; ++i) {
      const double lam = (double)hl[i];
      double pk = std::exp(-lam), F = pk;
      for (int k = 0; k < kCdf; ++k) {
        if (k > 0) {
          pk *= lam / k;
          F += pk;
        }
        hc[i * kCdf + k] = (float)F;
      }
    }
    MARLSC_CUDA(cudaMalloc(&cdf, hc.size() * sizeof(float)));
    MARLSC_CUDA(cudaMemcpyAsync(cdf, hc.data(), hc.size() * sizeof(float), cudaMemcpyHostToDevice, s));
  }
  poisson_inverse_kernel<<<(unsigned)((n + 127) / 128), 128, 0, s>>>(lambda, u, n, cdf, mode, k_out);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  MARLSC_CUDA(cudaGetLastError());
  MARLSC_CUDA(cudaStreamSynchronize(s));
  MARLSC_CUDA(cudaFree(mode));
  if (cdf) MARLSC_CUDA(cudaFree(cdf));
  return MARLSC_OK;
}

int marlsc_lead_sample(int64_t num_envs, int32_t n_warehouses, int32_t n_skus, const int32_t* expected_lead,
                       const int32_t* max_deviation, uint64_t seed, int64_t step_index, uint8_t* actual_lead, void* stream) {
  if (!expected_lead || !max_deviation || !actual_lead) return set_error(MARLSC_EINVAL, "null argument");
  if (num_envs < 1 || n_warehouses < 1 || n_skus < 1) return set_error(MARLSC_EINVAL, "num_envs, n_warehouses and n_skus must be positive");
  const long long WS = (long long)n_warehouses * n_skus, n = num_envs * WS;
  const unsigned grid = (unsigned)(((n + 3) / 4 + 255) / 256);
  sample_lead_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(expected_lead, max_deviation, n_skus, WS, n, seed,
                                                                          step_index, actual_lead);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  MARLSC_CUDA(cudaGetLastError());
  return MARLSC_OK;
}

}  // extern "C"
