// mlp_forward.cu - K7: forward pass of a one-hidden-layer MLP head for every agent-sample of a rollout step, fp32.
//
// What the rollout runs per env step for every agent (reference: ActorCriticRLModule._forward_actor / _forward_critic,
// src/algorithms/models/rlmodules/base.py:412-457, over an "mlp" network with one hidden layer - the IPPO configuration
// of BASELINE configs[3]: hidden_sizes [256], local observations of 14 floats, 2 action means / 1 value):
//   out = W2 act(W1 x + b1) + b2
// As two library GEMMs the hidden activations ([786,432 x 256] floats = 805 MB per network and step at 262,144 small
// environments) are written to HBM and read back, and the step of the whole rollout is bound by that traffic (1.5 of
// 1.8 ms). Here a thread owns one or two rows of x in registers and walks the hidden units: the unit's weights
// [W1[j,:], b1[j], W2[:,j]] are one shared-memory record, read as broadcast 16-byte words, the unit's activation never
// leaves the register file, and the only HBM traffic is x in and out back. Plain fp32 FFMA chains (inputs in ascending
// order per unit, units in ascending order per output), no tensor cores, no reduced precision: results agree with the
// library GEMMs to float32 rounding of a differently ordered sum (tests: rtol 1e-5).
#include <cuda_runtime.h>

#include <cstdint>
#include <string>

#include "lib_common.h"

namespace marlsc {
namespace {

// DP: input width padded to whole 16-byte words (x and W1 rows zero-padded); ROWS rows per thread (four for narrow inputs:
// a record is read once per ROWS rows); ACT 0 ReLU, 1 tanh; NO outputs.
// Shared-memory record of hidden unit j: DP floats of W1[j,:], then b1[j], W2[0,j], W2[1,j], W2[2,j] (O <= 3).
template <int DP, int ROWS, int ACT, int NO>
__global__ void __launch_bounds__(128)
mlp1_forward_kernel(const float* __restrict__ x, long long N, int D, const float* __restrict__ w1, const float* __restrict__ b1, int H,
                    const float* __restrict__ w2, const float* __restrict__ b2, int O, float* __restrict__ out) {
  extern __shared__ float4 s_rec[];
  constexpr int P = DP + 4;
  float* const s = reinterpret_cast<float*>(s_rec);
  for (int i = threadIdx.x; i < H * P; i += blockDim.x) {
    const int j = i / P, c = i - j * P;
    float v = 0.0f;
    if (c < D) v = w1[(long long)j * D + c];
    else if (c == DP) v = b1[j];
    else if (c > DP && c - DP - 1 < O) v = w2[(long long)(c - DP - 1) * H + j];
    s[i] = v;
  }
  __syncthreads();
  const float o0 = b2[0], o1 = O > 1 ? b2[1] : 0.0f, o2 = O > 2 ? b2[2] : 0.0f;
  const long long stride = (long long)gridDim.x * blockDim.x * ROWS;
  for (long long row0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * ROWS; row0 < N; row0 += stride) {
    float xr[ROWS][DP];
#pragma unroll
    for (int r = 0; r < ROWS; ++r)
#pragma unroll
      for (int d = 0; d < DP; ++d) xr[r][d] = (d < D && row0 + r < N) ? x[(row0 + r) * D + d] : 0.0f;
    float acc[ROWS][3];
#pragma unroll
    for (int r = 0; r < ROWS; ++r) {
      acc[r][0] = o0;
      acc[r][1] = o1;
      acc[r][2] = o2;
    }
#pragma unroll 2
    for (int j = 0; j < H; ++j) {
      const float4* const rec = s_rec + j * (P / 4);
      float w[DP];
#pragma unroll
      for (int q = 0; q < DP / 4; ++q) {
        const float4 t = rec[q];
        w[4 * q] = t.x;
        w[4 * q + 1] = t.y;
        w[4 * q + 2] = t.z;
        w[4 * q + 3] = t.w;
      }
      const float4 tail = rec[DP / 4];                // b1[j], W2[0..2, j]
#pragma unroll
      for (int r = 0; r < ROWS; ++r) {
        float h = tail.x;
#pragma unroll
        for (int d = 0; d < DP; ++d) h = fmaf(xr[r][d], w[d], h);
        h = ACT == 0 ? fmaxf(h, 0.0f) : tanhf(h);
        acc[r][0] = fmaf(h, tail.y, acc[r][0]);
        if (NO > 1) acc[r][1] = fmaf(h, tail.z, acc[r][1]);
        if (NO > 2) acc[r][2] = fmaf(h, tail.w, acc[r][2]);
      }
    }
#pragma unroll
    for (int r = 0; r < ROWS; ++r)
      if (row0 + r < N) {
#pragma unroll
        for (int k = 0; k < NO; ++k) out[(row0 + r) * NO + k] = acc[r][k];
      }
  }
}

template <int DP, int ROWS>
int launch_mlp1(const float* x, long long N, int D, const float* w1, const float* b1, int H, const float* w2, const float* b2, int O,
                int act, float* out, cudaStream_t s) {
  const size_t smem = (size_t)H * (DP + 4) * sizeof(float);
  int dev = 0, sms = 0, optin = 0;
  MARLSC_CUDA(cudaGetDevice(&dev));
  MARLSC_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  MARLSC_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  if ((int)smem > optin) return set_error(MARLSC_EUNSUPPORTED, "mlp1_forward: the hidden layer's weights do not fit shared memory");
  const long long want = (N + 128LL * ROWS - 1) / (128LL * ROWS);
  const unsigned grid = (unsigned)(want < (long long)sms * 8 ? (want > 0 ? want : 1) : (long long)sms * 8);
#define MARLSC_MLP1(A, K)                                                                                                  \
  {                                                                                                                        \
    if (smem > 48 * 1024)                                                                                                  \
      MARLSC_CUDA(cudaFuncSetAttribute((const void*)mlp1_forward_kernel<DP, ROWS, A, K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    mlp1_forward_kernel<DP, ROWS, A, K><<<grid, 128, smem, s>>>(x, N, D, w1, b1, H, w2, b2, O, out);                        \
  }
  if (act == 0) {
    if (O == 1) MARLSC_MLP1(0, 1) else if (O == 2) MARLSC_MLP1(0, 2) else MARLSC_MLP1(0, 3)
  } else {
    if (O == 1) MARLSC_MLP1(1, 1) else if (O == 2) MARLSC_MLP1(1, 2) else MARLSC_MLP1(1, 3)
  }
#undef MARLSC_MLP1
  g_launches.fetch_add(1, std::memory_order_relaxed);
  MARLSC_CUDA(cudaGetLastError());
  return MARLSC_OK;
}

// The same head with a wide input or output: the joint head of a centralised policy reads the global state (W x local
// width, up to 128 floats) and writes the joint action (W x S, up to 16 means). NOP: output count rounded up to 4 / 8 /
// 16 (the padding weights are zero, the padding sums are not stored). Shared-memory record of hidden unit j: DP floats
// of W1[j,:], then b1[j], then W2[0..NOP-1, j], padded to whole float4s. The record is consumed a float4 at a time, so
// only x (ROWS x DP floats) and the ROWS x NOP sums stay in registers. Units in ascending order per output as in K7;
// within a unit the inputs are summed in four interleaved partial sums.
template <int DP, int ROWS, int ACT, int NOP>
__global__ void __launch_bounds__(128)
mlp1_wide_forward_kernel(const float* __restrict__ x, long long N, int D, const float* __restrict__ w1, const float* __restrict__ b1,
                         int H, const float* __restrict__ w2, const float* __restrict__ b2, int O, float* __restrict__ out) {
  extern __shared__ float4 s_rec[];
  constexpr int P = DP + NOP + 4;
  float* const s = reinterpret_cast<float*>(s_rec);
  for (int i = threadIdx.x; i < H * P; i += blockDim.x) {
    const int j = i / P, c = i - j * P;
    float v = 0.0f;
    if (c < D) v = w1[(long long)j * D + c];
    else if (c == DP) v = b1[j];
    else if (c > DP && c - DP - 1 < O) v = w2[(long long)(c - DP - 1) * H + j];
    s[i] = v;
  }
  __syncthreads();
  float bias[NOP];
#pragma unroll
  for (int k = 0; k < NOP; ++k) bias[k] = k < O ? b2[k] : 0.0f;
  const long long stride = (long long)gridDim.x * blockDim.x * ROWS;
  for (long long row0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * ROWS; row0 < N; row0 += stride) {
    float xr[ROWS][DP];
#pragma unroll
    for (int r = 0; r < ROWS; ++r)
#pragma unroll
      for (int d = 0; d < DP; ++d) xr[r][d] = (d < D && row0 + r < N) ? x[(row0 + r) * D + d] : 0.0f;
    float acc[ROWS][NOP];
#pragma unroll
    for (int r = 0; r < ROWS; ++r)
#pragma unroll
      for (int k = 0; k < NOP; ++k) acc[r][k] = bias[k];
#pragma unroll 2
    for (int j = 0; j < H; ++j) {
      const float4* const rec = s_rec + j * (P / 4);
      const float4 t0 = rec[DP / 4];                  // b1[j], W2[0..2, j]
      // four partial sums per row (input quads q % 4): a 128-input dot product is not one 128-deep FMA chain
      float hp[ROWS][4], h[ROWS];
#pragma unroll
      for (int r = 0; r < ROWS; ++r) {
        hp[r][0] = t0.x;
        hp[r][1] = hp[r][2] = hp[r][3] = 0.0f;
      }
#pragma unroll
      for (int q = 0; q < DP / 4; ++q) {
        const float4 t = rec[q];
#pragma unroll
        for (int r = 0; r < ROWS; ++r) {
          float& a = hp[r][q & 3];
          a = fmaf(xr[r][4 * q], t.x, a);
          a = fmaf(xr[r][4 * q + 1], t.y, a);
          a = fmaf(xr[r][4 * q + 2], t.z, a);
          a = fmaf(xr[r][4 * q + 3], t.w, a);
        }
      }
#pragma unroll
      for (int r = 0; r < ROWS; ++r) {
        h[r] = (hp[r][0] + hp[r][1]) + (hp[r][2] + hp[r][3]);
        h[r] = ACT == 0 ? fmaxf(h[r], 0.0f) : tanhf(h[r]);
        acc[r][0] = fmaf(h[r], t0.y, acc[r][0]);
        acc[r][1] = fmaf(h[r], t0.z, acc[r][1]);
        acc[r][2] = fmaf(h[r], t0.w, acc[r][2]);
      }
#pragma unroll
      for (int q = 1; q < (NOP + 4) / 4; ++q) {       // W2[4q-1 .. 4q+2, j]
        const float4 t = rec[DP / 4 + q];
        const float tw[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          if (4 * q - 1 + c >= NOP) continue;
#pragma unroll
          for (int r = 0; r < ROWS; ++r) acc[r][4 * q - 1 + c] = fmaf(h[r], tw[c], acc[r][4 * q - 1 + c]);
        }
      }
    }
#pragma unroll
    for (int r = 0; r < ROWS; ++r)
      if (row0 + r < N) {
#pragma unroll
        for (int k = 0; k < NOP; ++k)
          if (k < O) out[(row0 + r) * O + k] = acc[r][k];
      }
  }
}

template <int DP, int ROWS>
int launch_mlp1_wide(const float* x, long long N, int D, const float* w1, const float* b1, int H, const float* w2, const float* b2,
                     int O, int act, float* out, cudaStream_t s) {
  const int nop = O <= 4 ? 4 : (O <= 8 ? 8 : 16);
  const size_t smem = (size_t)H * (DP + nop + 4) * sizeof(float);
  int dev = 0, sms = 0, optin = 0;
  MARLSC_CUDA(cudaGetDevice(&dev));
  MARLSC_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  MARLSC_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  if ((int)smem > optin) return set_error(MARLSC_EUNSUPPORTED, "mlp1_forward: the hidden layer's weights do not fit shared memory");
  const long long want = (N + 128LL * ROWS - 1) / (128LL * ROWS);
  const unsigned grid = (unsigned)(want < (long long)sms * 8 ? (want > 0 ? want : 1) : (long long)sms * 8);
#define MARLSC_MLP1W(A, K)                                                                                                 \
  {                                                                                                                        \
    if (smem > 48 * 1024)                                                                                                  \
      MARLSC_CUDA(cudaFuncSetAttribute((const void*)mlp1_wide_forward_kernel<DP, ROWS, A, K>,                              \
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));                           \
    mlp1_wide_forward_kernel<DP, ROWS, A, K><<<grid, 128, smem, s>>>(x, N, D, w1, b1, H, w2, b2, O, out);                  \
  }
  if (act == 0) {
    if (nop == 4) MARLSC_MLP1W(0, 4) else if (nop == 8) MARLSC_MLP1W(0, 8) else MARLSC_MLP1W(0, 16)
  } else {
    if (nop == 4) MARLSC_MLP1W(1, 4) else if (nop == 8) MARLSC_MLP1W(1, 8) else MARLSC_MLP1W(1, 16)
  }
#undef MARLSC_MLP1W
  g_launches.fetch_add(1, std::memory_order_relaxed);
  MARLSC_CUDA(cudaGetLastError());
  return MARLSC_OK;
}

// Output layer of a deeper head: out[n, :] = W h[n, :] + b with a handful of outputs (action means of a small network, the
// value). The library GEMM path treats this as a [N x H] x [H x 2] product and reads the 805 MB of hidden activations at a
// third of the HBM rate, then adds the bias in a second pass; here a warp takes a row as 16-byte words (one coalesced
// 1 KB request per 256 floats), every lane keeps NO partial dot products, five shuffle rounds finish them. With PRE the
// rows are the RAW product of the hidden layer before, whose bias and ReLU are applied on the way in: cuBLASLt runs the
// "fused" bias + ReLU epilogue of its fp32 SIMT kernels as a separate pass over the activations (0.95 ms for 805 MB, as
// long as half the GEMM), which a plain product followed by this kernel avoids.
template <int NO, bool PRE>
__global__ void __launch_bounds__(256)
linear_out_kernel(const float* __restrict__ h, long long N, int H, const float* __restrict__ pre_bias, const float* __restrict__ w,
                  const float* __restrict__ b, float* __restrict__ out) {
  extern __shared__ float4 s_w4[];                    // [NO][H / 4], then (PRE) the producing layer's bias [H / 4]
  const int H4 = H >> 2;
  for (int i = threadIdx.x; i < NO * H4; i += blockDim.x) s_w4[i] = reinterpret_cast<const float4*>(w)[i];
  if (PRE)
    for (int i = threadIdx.x; i < H4; i += blockDim.x) s_w4[NO * H4 + i] = reinterpret_cast<const float4*>(pre_bias)[i];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long row = warp; row < N; row += n_warps) {
    const float4* const hr = reinterpret_cast<const float4*>(h) + row * H4;
    float acc[NO];
#pragma unroll
    for (int k = 0; k < NO; ++k) acc[k] = 0.0f;
    for (int c = lane; c < H4; c += 32) {
      float4 v = hr[c];
      if (PRE) {                                      // h holds the raw product of the layer before: + bias, ReLU
        const float4 pb = s_w4[NO * H4 + c];
        v.x = fmaxf(v.x + pb.x, 0.0f);
        v.y = fmaxf(v.y + pb.y, 0.0f);
        v.z = fmaxf(v.z + pb.z, 0.0f);
        v.w = fmaxf(v.w + pb.w, 0.0f);
      }
#pragma unroll
      for (int k = 0; k < NO; ++k) {
        const float4 q = s_w4[k * H4 + c];
        acc[k] = fmaf(v.x, q.x, acc[k]);
        acc[k] = fmaf(v.y, q.y, acc[k]);
        acc[k] = fmaf(v.z, q.z, acc[k]);
        acc[k] = fmaf(v.w, q.w, acc[k]);
      }
    }
#pragma unroll
    for (int k = 0; k < NO; ++k)
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], o);
    if (lane == 0) {
#pragma unroll
      for (int k = 0; k < NO; ++k) out[row * NO + k] = acc[k] + b[k];
    }
  }
}

// The same output layer with 5 to 16 outputs (the joint action means of a centralised policy's deeper head). NOP: the
// output count rounded up to 8 or 16; the weight rows past O are zero in shared memory and their sums are not stored.
template <int NOP, bool PRE>
__global__ void __launch_bounds__(256)
linear_out_wide_kernel(const float* __restrict__ h, long long N, int H, const float* __restrict__ pre_bias, const float* __restrict__ w,
                       const float* __restrict__ b, int O, float* __restrict__ out) {
  extern __shared__ float4 s_w4[];                    // [NOP][H / 4], then (PRE) the producing layer's bias [H / 4]
  const int H4 = H >> 2;
  for (int i = threadIdx.x; i < NOP * H4; i += blockDim.x)
    s_w4[i] = i < O * H4 ? reinterpret_cast<const float4*>(w)[i] : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
  if (PRE)
    for (int i = threadIdx.x; i < H4; i += blockDim.x) s_w4[NOP * H4 + i] = reinterpret_cast<const float4*>(pre_bias)[i];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long row = warp; row < N; row += n_warps) {
    const float4* const hr = reinterpret_cast<const float4*>(h) + row * H4;
    float acc[NOP];
#pragma unroll
    for (int k = 0; k < NOP; ++k) acc[k] = 0.0f;
    for (int c = lane; c < H4; c += 32) {
      float4 v = hr[c];
      if (PRE) {
        const float4 pb = s_w4[NOP * H4 + c];
        v.x = fmaxf(v.x + pb.x, 0.0f);
        v.y = fmaxf(v.y + pb.y, 0.0f);
        v.z = fmaxf(v.z + pb.z, 0.0f);
        v.w = fmaxf(v.w + pb.w, 0.0f);
      }
#pragma unroll
      for (int k = 0; k < NOP; ++k) {
        const float4 q = s_w4[k * H4 + c];
        acc[k] = fmaf(v.x, q.x, acc[k]);
        acc[k] = fmaf(v.y, q.y, acc[k]);
        acc[k] = fmaf(v.z, q.z, acc[k]);
        acc[k] = fmaf(v.w, q.w, acc[k]);
      }
    }
#pragma unroll
    for (int k = 0; k < NOP; ++k)
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], o);
    if (lane == 0) {
#pragma unroll
      for (int k = 0; k < NOP; ++k)
        if (k < O) out[row * O + k] = acc[k] + b[k];
    }
  }
}

// Input layer of a deeper head: h[n, :] = act(W x[n, :] + b) for narrow inputs (14 or 56 observation floats) and up to
// 256 hidden units. The library picks unaligned small-K GEMM kernels for these shapes (0.4-0.6 ms for an 805 MB or
// 201 MB result); here a lane keeps the weight rows of its UPL hidden units in registers (unit j = lane + 32 k). A warp
// takes four or eight rows of x at a time: the rows are contiguous, so the batch is a few coalesced loads per lane, requested one
// batch ahead, parked in shared memory and read back as broadcast 16-byte words; the rows of h leave as UPL coalesced
// 128-byte stores each.

template <int UPL, int DP, int ACT>
__global__ void __launch_bounds__(256)
linear_in_kernel(const float* __restrict__ x, long long N, int D, const float* __restrict__ w, const float* __restrict__ b, int H,
                 float* __restrict__ out) {
  constexpr int kInRows = UPL <= 2 ? 8 : 4;                       // rows per batch: at least 16 independent FMA chains per lane
  __shared__ __align__(16) float s_x[8][kInRows * DP];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  float wr[UPL][DP], bias[UPL];
#pragma unroll
  for (int k = 0; k < UPL; ++k) {
    const int j = lane + 32 * k;
    bias[k] = j < H ? b[j] : 0.0f;
#pragma unroll
    for (int d = 0; d < DP; ++d) wr[k][d] = (j < H && d < D) ? w[(long long)j * D + d] : 0.0f;
  }
  float* const xs = s_x[wid];
  for (int i = lane; i < kInRows * DP; i += 32) xs[i] = 0.0f;     // the padding columns stay zero
  constexpr int kLd = (kInRows * DP + 31) / 32;                   // loads per lane and batch (D <= DP)
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
  const long long n_batches = (N + kInRows - 1) / kInRows;
  float pre[kLd];
  const auto request = [&](long long batch) {                     // the batch's kInRows x D contiguous floats
    const long long first = batch * kInRows * D, last = N * D;
#pragma unroll
    for (int q = 0; q < kLd; ++q) {
      const int i = lane + 32 * q;
      pre[q] = (i < kInRows * D && first + i < last) ? x[first + i] : 0.0f;
    }
  };
  if (warp < n_batches) request(warp);
  for (long long batch = warp; batch < n_batches; batch += n_warps) {
    __syncwarp();                                                 // the previous batch has been read out
#pragma unroll
    for (int q = 0; q < kLd; ++q) {
      const int i = lane + 32 * q;
      if (i < kInRows * D) xs[(i / D) * DP + (i % D)] = pre[q];
    }
    __syncwarp();
    if (batch + n_warps < n_batches) request(batch + n_warps);    // in flight while this batch is computed
    float h[kInRows][UPL];                                        // kInRows x UPL independent chains
#pragma unroll
    for (int r = 0; r < kInRows; ++r)
#pragma unroll
      for (int k = 0; k < UPL; ++k) h[r][k] = bias[k];
#pragma unroll
    for (int d4 = 0; d4 < DP / 4; ++d4) {
#pragma unroll
      for (int r = 0; r < kInRows; ++r) {
        const float4 v = reinterpret_cast<const float4*>(xs + r * DP)[d4];
#pragma unroll
        for (int k = 0; k < UPL; ++k) {
          h[r][k] = fmaf(v.x, wr[k][4 * d4], h[r][k]);
          h[r][k] = fmaf(v.y, wr[k][4 * d4 + 1], h[r][k]);
          h[r][k] = fmaf(v.z, wr[k][4 * d4 + 2], h[r][k]);
          h[r][k] = fmaf(v.w, wr[k][4 * d4 + 3], h[r][k]);
        }
      }
    }
#pragma unroll
    for (int r = 0; r < kInRows; ++r) {
      const long long row = batch * kInRows + r;
      if (row < N) {
        float* const o = out + row * H + lane;
#pragma unroll
        for (int k = 0; k < UPL; ++k) {
          float y = h[r][k];
          if (ACT == 0) y = fmaxf(y, 0.0f);
          if (ACT == 1) y = tanhf(y);
          if (lane + 32 * k < H) o[32 * k] = y;
        }
      }
    }
  }
}

template <int UPL, int DP>
int launch_linear_in(const float* x, long long N, int D, const float* w, const float* b, int H, int act, float* out, cudaStream_t s) {
  int dev = 0, sms = 0;
  MARLSC_CUDA(cudaGetDevice(&dev));
  MARLSC_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const long long want = (N + 7) / 8;
  const unsigned grid = (unsigned)(want < (long long)sms * 4 ? want : (long long)sms * 4);
  if (act == 0) linear_in_kernel<UPL, DP, 0><<<grid, 256, 0, s>>>(x, N, D, w, b, H, out);
  else if (act == 1) linear_in_kernel<UPL, DP, 1><<<grid, 256, 0, s>>>(x, N, D, w, b, H, out);
  else linear_in_kernel<UPL, DP, 2><<<grid, 256, 0, s>>>(x, N, D, w, b, H, out);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  MARLSC_CUDA(cudaGetLastError());
  return MARLSC_OK;
}

}  // namespace
}  // namespace marlsc

using namespace marlsc;

extern "C" int marlsc_mlp1_forward(const float* x, int64_t n_rows, int32_t in_dim, const float* w1, const float* b1, int32_t hidden,
                                   const float* w2, const float* b2, int32_t out_dim, int32_t activation, float* out, void* stream) {
  if (!x || !w1 || !b1 || !w2 || !b2 || !out) return set_error(MARLSC_EINVAL, "mlp1_forward: null pointer");
  if (n_rows < 0 || in_dim < 1 || in_dim > 128 || hidden < 1 || out_dim < 1 || out_dim > 16 || (activation != 0 && activation != 1))
    return set_error(MARLSC_EUNSUPPORTED, "mlp1_forward: in_dim <= 128, out_dim <= 16, activation 0 (ReLU) or 1 (tanh)");
  if (n_rows == 0) return MARLSC_OK;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (in_dim <= 64 && out_dim <= 3) {
    if (in_dim <= 16) return launch_mlp1<16, 4>(x, n_rows, in_dim, w1, b1, hidden, w2, b2, out_dim, activation, out, s);
    if (in_dim <= 32) return launch_mlp1<32, 2>(x, n_rows, in_dim, w1, b1, hidden, w2, b2, out_dim, activation, out, s);
    return launch_mlp1<64, 1>(x, n_rows, in_dim, w1, b1, hidden, w2, b2, out_dim, activation, out, s);
  }
  if (in_dim <= 16) return launch_mlp1_wide<16, 4>(x, n_rows, in_dim, w1, b1, hidden, w2, b2, out_dim, activation, out, s);
  if (in_dim <= 32) return launch_mlp1_wide<32, 2>(x, n_rows, in_dim, w1, b1, hidden, w2, b2, out_dim, activation, out, s);
  if (in_dim <= 64) return launch_mlp1_wide<64, 1>(x, n_rows, in_dim, w1, b1, hidden, w2, b2, out_dim, activation, out, s);
  return launch_mlp1_wide<128, 1>(x, n_rows, in_dim, w1, b1, hidden, w2, b2, out_dim, activation, out, s);
}

extern "C" int marlsc_linear_out_forward(const float* h, int64_t n_rows, int32_t in_dim, const float* pre_bias, const float* w,
                                         const float* b, int32_t out_dim, float* out, void* stream) {
  if (!h || !w || !b || !out) return set_error(MARLSC_EINVAL, "linear_out_forward: null pointer");
  if (n_rows < 0 || in_dim < 4 || (in_dim & 3) || in_dim > 2048 || out_dim < 1 || out_dim > 16 ||
      ((reinterpret_cast<uintptr_t>(h) | reinterpret_cast<uintptr_t>(w) | reinterpret_cast<uintptr_t>(pre_bias)) & 15u))
    return set_error(MARLSC_EUNSUPPORTED, "linear_out_forward: in_dim a multiple of 4 (<= 2048), out_dim <= 16, 16-byte aligned h, w, pre_bias");
  if (n_rows == 0) return MARLSC_OK;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  int dev = 0, sms = 0;
  MARLSC_CUDA(cudaGetDevice(&dev));
  MARLSC_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const long long want = (n_rows + 7) / 8;
  const unsigned grid = (unsigned)(want < (long long)sms * 8 ? want : (long long)sms * 8);
  if (out_dim > 4) {
    // up to 17 x 2048 floats: past the default 48 KB of dynamic shared memory
    const size_t smem = (size_t)((out_dim <= 8 ? 8 : 16) + (pre_bias ? 1 : 0)) * in_dim * sizeof(float);
#define MARLSC_LOUTW(K, PRE)                                                                                              \
  {                                                                                                                       \
    if (smem > 48 * 1024)                                                                                                 \
      MARLSC_CUDA(cudaFuncSetAttribute((const void*)linear_out_wide_kernel<K, PRE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    linear_out_wide_kernel<K, PRE><<<grid, 256, smem, s>>>(h, n_rows, in_dim, pre_bias, w, b, out_dim, out);              \
  }
    if (out_dim <= 8) {
      if (pre_bias) MARLSC_LOUTW(8, true) else MARLSC_LOUTW(8, false)
    } else {
      if (pre_bias) MARLSC_LOUTW(16, true) else MARLSC_LOUTW(16, false)
    }
#undef MARLSC_LOUTW
    g_launches.fetch_add(1, std::memory_order_relaxed);
    MARLSC_CUDA(cudaGetLastError());
    return MARLSC_OK;
  }
  const size_t smem = (size_t)(out_dim + (pre_bias ? 1 : 0)) * in_dim * sizeof(float);
#define MARLSC_LOUT(K)                                                                                      \
  if (pre_bias) linear_out_kernel<K, true><<<grid, 256, smem, s>>>(h, n_rows, in_dim, pre_bias, w, b, out);  \
  else linear_out_kernel<K, false><<<grid, 256, smem, s>>>(h, n_rows, in_dim, pre_bias, w, b, out);
  switch (out_dim) {
    case 1: MARLSC_LOUT(1) break;
    case 2: MARLSC_LOUT(2) break;
    case 3: MARLSC_LOUT(3) break;
    default: MARLSC_LOUT(4) break;
  }
#undef MARLSC_LOUT
  g_launches.fetch_add(1, std::memory_order_relaxed);
  MARLSC_CUDA(cudaGetLastError());
  return MARLSC_OK;
}

extern "C" int marlsc_linear_in_forward(const float* x, int64_t n_rows, int32_t in_dim, const float* w, const float* b, int32_t hidden,
                                        int32_t activation, float* out, void* stream) {
  if (!x || !w || !b || !out) return set_error(MARLSC_EINVAL, "linear_in_forward: null pointer");
  const int dp = in_dim <= 16 ? 16 : (in_dim <= 32 ? 32 : 64);
  const int upl = hidden <= 32 ? 1 : (hidden <= 64 ? 2 : (hidden <= 128 ? 4 : 8));
  if (n_rows < 0 || in_dim < 1 || in_dim > 64 || hidden < 1 || hidden > 256 || upl * dp > 128 || activation < 0 || activation > 2)
    return set_error(MARLSC_EUNSUPPORTED, "linear_in_forward: in_dim <= 64, hidden <= 256, ceil(hidden / 32) x padded in_dim <= 128");
  if (n_rows == 0) return MARLSC_OK;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
#define MARLSC_LIN(U, P) return launch_linear_in<U, P>(x, n_rows, in_dim, w, b, hidden, activation, out, s)
  if (dp == 16) {
    if (upl == 1) MARLSC_LIN(1, 16);
    if (upl == 2) MARLSC_LIN(2, 16);
    if (upl == 4) MARLSC_LIN(4, 16);
    MARLSC_LIN(8, 16);
  }
  if (dp == 32) {
    if (upl == 1) MARLSC_LIN(1, 32);
    if (upl == 2) MARLSC_LIN(2, 32);
    MARLSC_LIN(4, 32);
  }
  if (upl == 1) MARLSC_LIN(1, 64);
  MARLSC_LIN(2, 64);
#undef MARLSC_LIN
}
