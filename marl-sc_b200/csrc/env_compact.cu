// env_compact.cu - fused environment step, reset, base-stock policy and order -> line conversion over the compact
// state layout (see env_compact.cuh for the design notes).
//
// Reference semantics restated here (paths under the reference repo):
//   step order ................. src/environment/envs/multi_env.py:253-366
//   action rescale ............. multi_env.py:824-828 (direct)
//   orders / arrivals .......... multi_env.py:850-919
//   greedy allocation .......... src/environment/components/demand_allocator.py:150-208
//   home demand, rolling mean .. multi_env.py:747-793
//   lost sales ................. src/environment/components/lost_sales_handler.py:71-148 (closest, shipment)
//   cost reward ................ src/environment/components/reward_calculator.py:127-188
//   observation ................ multi_env.py:577-710, 941-968
#include "env_compact.cuh"
#include "env_split.cuh"

#ifndef MARLSC_ALLOC_CTAS
#define MARLSC_ALLOC_CTAS 4
#endif
namespace marlsc {
static inline int imin_host(int a, int b) { return a < b ? a : b; }
static inline int imax_host(int a, int b) { return a > b ? a : b; }
namespace {

constexpr unsigned FULL = 0xffffffffu;
constexpr int kSlots = kCompactMaxS / 32;   // SKU slots per lane
constexpr int kPlaneBatch = 9;              // ring planes of a row in flight per lane (times kSlots cells)

__device__ __forceinline__ uint32_t sm_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t ld_s_u8(uint32_t a) { uint32_t v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ uint32_t ld_s_u16(uint32_t a) { uint32_t v; asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ void st_s_u16(uint32_t a, uint32_t v) { asm volatile("st.shared.u16 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void red_s_add(uint32_t a, uint32_t v) { asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void red_s_add_f64(uint32_t a, double v) {   // shared-memory double add (compare-and-swap loop, like atomicAdd)
  unsigned long long old, seen;
  asm volatile("ld.shared.u64 %0, [%1];" : "=l"(old) : "r"(a) : "memory");
  do {
    seen = old;
    const unsigned long long want = (unsigned long long)__double_as_longlong(__longlong_as_double((long long)seen) + v);
    asm volatile("atom.shared.cas.b64 %0, [%1], %2, %3;" : "=l"(old) : "r"(a), "l"(seen), "l"(want) : "memory");
  } while (old != seen);
}
__device__ __forceinline__ void red_g_add(uint32_t* p, uint32_t v) { asm volatile("red.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ uint32_t ld_nc_u16(const uint16_t* p) { uint32_t v; asm volatile("ld.global.nc.u16 %0, [%1];" : "=r"(v) : "l"(p)); return v; }
__device__ __forceinline__ uint32_t ld_cg_u16(const uint16_t* p) { uint32_t v; asm volatile("ld.global.cg.u16 %0, [%1];" : "=r"(v) : "l"(p)); return v; }
__device__ __forceinline__ void prefetch_l2_bulk(const void* p, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}

__device__ __forceinline__ uint32_t ld_nc_u32(const uint32_t* p) { uint32_t v; asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(v) : "l"(p)); return v; }

// A lane's line stream (marlsc_step_io.lines): two consecutive entries per 32-bit word, words of one round pair side
// by side for the 32 lanes. The first word of a lane is its SKU map (byte k = the SKU its slot k stands for, 255 = none;
// the packers deal SKUs to lanes by line count so the 32 streams of an environment end at about the same round). Three
// words are kept requested ahead of the one being consumed. (A cp.async ring in shared memory with eight words in
// flight per lane was measured too: it removes the waits on the next word but its request / commit / wait instructions
// cost more than the waits did in this issue-bound loop: 0.73 against 0.66 ms.)
struct LineStream {
  const uint32_t* base;                               // the lane's first word; word i of the lane is base[32 i]
  uint32_t at, n;                                     // next word to request (x 32), words of the block (x 32)
  uint32_t map, cur, w1, w2, w3;
  __device__ __forceinline__ void init(const uint16_t* lines, int64_t round0, int n_rounds, int lane) {
    base = reinterpret_cast<const uint32_t*>(lines) + (round0 >> 1) * 32 + lane;
    n = (uint32_t)(n_rounds >> 1) * 32u;
    map = 0u < n ? ld_nc_u32(base) : 0xffffffffu;
    cur = 32u < n ? ld_nc_u32(base + 32) : 0u;
    w1 = 64u < n ? ld_nc_u32(base + 64) : 0u;
    w2 = 96u < n ? ld_nc_u32(base + 96) : 0u;
    w3 = 128u < n ? ld_nc_u32(base + 128) : 0u;
    at = 160u;
  }
  __device__ __forceinline__ uint32_t next() const { return cur & 0xffffu; }   // 0: the stream has ended
  __device__ __forceinline__ void pop() {
    cur >>= 16;
    if (cur == 0u) {
      cur = w1;
      w1 = w2;
      w2 = w3;
      w3 = at < n ? ld_nc_u32(base + at) : 0u;
      at += 32u;
    }
  }
};

// The SKU a lane's slot stands for (byte `slot` of its map word).
__device__ __forceinline__ uint32_t map_sku(uint32_t map, uint32_t slot) { return __byte_perm(map, 0u, 0x4440u + slot); }

// Availability masks of a lane's SKUs from the staged stock [W,S] uint16 at shared address a_inv: bit w + 16 (k & 1) of
// (k & 2 ? avhi : avlo) says warehouse w holds the SKU of slot k. Map bytes that name no SKU (255, or anything >= S in a
// malformed stream) are pointed at SKU S-1 with an empty mask: their lines, if any, count as lost and touch no memory
// outside the stock image.
__device__ __forceinline__ void owner_masks(uint32_t& map, uint32_t a_inv, int W, int S, uint32_t& avlo, uint32_t& avhi) {
  avlo = avhi = 0u;
  uint32_t fixed = 0u;
#pragma unroll
  for (int k = 0; k < kSlots; ++k) {
    uint32_t sku = (map >> (8 * k)) & 0xffu;
    const bool named = sku < (uint32_t)S;
    if (!named) sku = (uint32_t)S - 1u;
    fixed |= sku << (8 * k);
    uint32_t m = 0u;
    const uint32_t a = a_inv + 2u * sku;
    for (int w = 0; w < W; ++w) m |= (ld_s_u16(a + (uint32_t)w * 2u * (uint32_t)S) != 0u ? 1u : 0u) << w;
    if (!named) m = 0u;
    if (k & 2) avhi |= m << (16 * (k & 1)); else avlo |= m << (16 * (k & 1));
  }
  map = fixed;
}

// observation element j of a warehouse's vector (after the id prefix) with the fixed mean/std normalisation of
// multi_env.py:700-702 when enabled (reset kernel; the step kernel walks pointers instead)
__device__ __forceinline__ void put(const DevSpec& sp, bool ms, float* __restrict__ out, unsigned j, float x) {
  if (ms) x = f_mul(f_sub(x, sp.obs_mean[j]), sp.obs_std[j]);
  out[j] = x;
}

// The allocation chains of one environment (demand_allocator.py:150-208) over its line streams. A trip of the loop: if
// the lane's current line is done, take the next entry of its stream; then one shipment from the cheapest warehouse that
// holds the SKU, or the lost-sales bookkeeping when none does. Lanes only meet in the exit vote. Stock [W,S] uint16,
// shipped units [W,R] and lost units [R] live in shared memory, a lane's availability masks in two registers. The cells
// of the SKUs named by the lane's map belong to this lane alone for the duration of the chains.
template <int NCH>
__device__ __forceinline__ void allocation_chains(const DevSpec& sp, LineStream& ls, uint32_t a_perm, uint32_t a_prio, uint32_t a_home,
                                                  uint32_t a_inv, uint32_t a_shipq, uint32_t a_lostU, uint32_t a_lostP, uint32_t& avlo,
                                                  uint32_t& avhi, uint32_t* hist32) {
  const uint32_t S = sp.S, S2 = 2u * S, R4 = 4u * sp.R, map = ls.map;
  const bool pen_uniform = sp.pen_uniform != 0;
  uint32_t rem = 0u, r = 0u, sl = 0u, sku2 = 0u, cand = 0u;   // units left of the current line, its region, SKU slot, 2 x SKU, candidate bits
  while (true) {
    const uint32_t n0 = ls.next();
    if (rem == 0u && n0 != 0u) {
      ls.pop();
      rem = n0 & 0xffu;
      r = (n0 >> 8) & 0x3fu;
      sl = n0 >> 14;
      sku2 = 2u * map_sku(map, sl);
      // which warehouses hold the SKU (bit w), then the same bits in the region's priority order
      const uint32_t am = ((sl & 2u ? avhi : avlo) >> (16u * (sl & 1u))) & 0xffffu;
      const uint32_t pm = a_perm + r * (NCH * 64u);
      cand = ld_s_u16(pm + 2u * (am & 31u));
      if (NCH > 1) cand |= ld_s_u16(pm + 64u + 2u * ((am >> 5) & 31u));
      if (NCH > 2) cand |= ld_s_u16(pm + 128u + 2u * ((am >> 10) & 31u));
      if (NCH > 3) cand |= ld_s_u16(pm + 192u + 2u * ((am >> 15) & 31u));
      if (hist32) {                                   // home-region demand of this step (multi_env.py:763-768)
        const uint32_t hw = ld_s_u8(a_home + r);
        if (hw != 255u) {
          const uint32_t s = sku2 >> 1;
          if (hw != 254u) {                           // two uint16 cells share a word: add into the cell's half, nobody waits
            const uint32_t c = hw * S + s;
            red_g_add(hist32 + (c >> 1), rem << (16u * (c & 1u)));
          } else {
            uint32_t hm = sp.home_mask[r];
            while (hm) {
              const uint32_t c = (uint32_t)lowest_bit(hm) * S + s;
              hm &= hm - 1;
              red_g_add(hist32 + (c >> 1), rem << (16u * (c & 1u)));
            }
          }
        }
      }
    }
    if (rem != 0u) {
      if (cand != 0u) {                               // ship from the cheapest warehouse that has the SKU
        const uint32_t v = (uint32_t)lowest_bit(cand);
        cand &= cand - 1;
        const uint32_t w = ld_s_u8(a_prio + r * 16u + v);
        const uint32_t cell = a_inv + w * S2 + sku2;
        const uint32_t a = ld_s_u16(cell);            // the cells of a SKU belong to this lane
        const uint32_t f = rem < a ? rem : a;
        st_s_u16(cell, a - f);
        red_s_add(a_shipq + w * R4 + 4u * r, f);
        rem -= f;
        if (a == f) {                                 // emptied
          const uint32_t clr = ~(1u << (w + 16u * (sl & 1u)));
          if (sl & 2u) avhi &= clr; else avlo &= clr;
        }
      }
      if (rem != 0u && cand == 0u) {
        // no warehouse can supply the rest: lost (demand_allocator.py:205-208); units are enough when every SKU
        // carries the same penalty rate
        red_s_add(a_lostU + 4u * r, rem);
        if (!pen_uniform) red_s_add_f64(a_lostP + 8u * r, (double)rem * sp.pen_rate[sku2 >> 1]);
        rem = 0u;
      }
    }
    if (!__any_sync(FULL, (rem | ls.next()) != 0u)) break;
  }
}

// (x - mean) * (1 / std) when the kernel is instantiated with the normalisation, else x
template <bool MS>
__device__ __forceinline__ float nrm(float x, const float* __restrict__ mean, const float* __restrict__ istd, int off) {
  if (MS) return f_mul(f_sub(x, mean[off]), istd[off]);
  return x;
}

// ---------------------------------------------------------------------------------------------------------------
// K1 (compact): one warp per environment; in the allocation a lane owns the SKUs its stream's map word names. The row loops walk pointers (one add per row or
// plane, cells at constant offsets): the first version of this kernel spent 80 % of its 39 k warp instructions per
// env-step on index arithmetic.
// ---------------------------------------------------------------------------------------------------------------
// SKU slot k of a lane is valid: always below FS (= S / 32, compile time), for lanes below the remainder at FS, never above
#define VALID(k) ((k) < FS || ((k) == FS && tail))

template <int NCH, bool MS, int FS>
__global__ void __launch_bounds__(kCompactWarps * 32, 4)
env_step_compact_kernel(const __grid_constant__ DevSpec sp, const __grid_constant__ marlsc_env_state_t st,
                        const __grid_constant__ marlsc_step_io_t io, int t, int prefetch) {
  extern __shared__ __align__(16) unsigned char smem[];
  __shared__ int s_poff[kCompactMaxL];                // 32-bit word offset of pipeline slot k's plane inside a warehouse row of the ring
  const int W = sp.W, S = sp.S, R = sp.R, L = sp.L, WS = W * S;
  const CompactSmem lay = compact_smem(W, S, R, NCH, sp.pen_uniform);
  if (threadIdx.x < kCompactMaxL) s_poff[threadIdx.x] = (int)((unsigned)(t + 1 + threadIdx.x) % (unsigned)L) * (S >> 2);
  {  // per-CTA tables: availability -> priority-order permutation, priority rows, home warehouse of a region
    const int n_perm = (R * NCH * 32) >> 1, n_prio = (R * 16) >> 2, n_home = (R + 3) >> 2;
    for (int i = threadIdx.x; i < n_perm + n_prio + n_home; i += blockDim.x) {
      if (i < n_perm) reinterpret_cast<uint32_t*>(smem + lay.t_perm)[i] = reinterpret_cast<const uint32_t*>(sp.perm5)[i];
      else if (i < n_perm + n_prio) reinterpret_cast<uint32_t*>(smem + lay.t_prio)[i - n_perm] = reinterpret_cast<const uint32_t*>(sp.prio16)[i - n_perm];
      else reinterpret_cast<uint32_t*>(smem + lay.t_home)[i - n_perm - n_prio] = reinterpret_cast<const uint32_t*>(sp.home_wh)[i - n_perm - n_prio];
    }
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int64_t e = (int64_t)blockIdx.x * kCompactWarps + wid;
  if (e >= st.num_envs) return;                       // whole warps leave together; everything below is warp-local

  // this environment's lines: read first, everything the allocation loads hangs on these two values
  const int64_t round0 = io.line_counts ? e * (int64_t)io.line_stride : (int64_t)io.line_offsets[e];
  const int n_rounds = io.line_counts ? io.line_counts[e] : io.line_offsets[e + 1] - (int)round0;
  if (lane == 0 && n_rounds > 0) prefetch_l2_bulk(io.lines + round0 * 32, (uint32_t)n_rounds * 64u);   // in flight during phase 1
  // ... and this environment's state blocks on their way into L2 (one bulk prefetch each, no registers or shared
  // memory held): the row loops below then wait for L2, not DRAM
  if (prefetch) {
    if (lane == 1) prefetch_l2_bulk(static_cast<const uint8_t*>(st.ring_qty) + e * (int64_t)WS * L, (uint32_t)(WS * L));
    if (lane == 2 && !io.action_qty) prefetch_l2_bulk(io.actions + e * WS, (uint32_t)(WS * 4));
    if (lane == 3) prefetch_l2_bulk(static_cast<const uint16_t*>(st.inventory) + e * WS, (uint32_t)(WS * 2));
    if (lane == 4 && io.action_qty) prefetch_l2_bulk(io.action_qty + e * WS, (uint32_t)WS);
  }

  unsigned char* const wbase = smem + lay.t_bytes + (size_t)wid * lay.warp_bytes;
  uint16_t* const s_inv = reinterpret_cast<uint16_t*>(wbase + lay.inv);
  uint32_t* const s_shipq = reinterpret_cast<uint32_t*>(wbase + lay.shipq);
  uint32_t* const s_lostU = reinterpret_cast<uint32_t*>(wbase + lay.lostU);
  double* const s_lostP = reinterpret_cast<double*>(wbase + lay.lostP);
  const bool pen_uniform = sp.pen_uniform != 0;
  for (int i = lane; i < W * R; i += 32) s_shipq[i] = 0u;
  for (int i = lane; i < R; i += 32) {
    s_lostU[i] = 0u;
    if (!pen_uniform) s_lostP[i] = 0.0;
  }

  const bool need_hist = sp.need_hist != 0;
  const int pa = t % L;                               // plane of the orders arriving now
  const bool by_row = sp.row_rates_uniform != 0;
  const bool tail = lane < S - 32 * FS;               // this lane owns a SKU in the partly filled slot FS
  // per-lane bases (this lane's first cell); rows advance them by their strides
  uint16_t* const g_inv = pinned(static_cast<uint16_t*>(st.inventory) + e * WS + lane);
  uint8_t* const g_ring = pinned(static_cast<uint8_t*>(st.ring_qty) + e * (int64_t)WS * L + lane);
  uint16_t* const g_hist = need_hist ? pinned(static_cast<uint16_t*>(st.demand_hist) + e * (int64_t)kWindow * WS + lane) : nullptr;
  uint16_t* const hist_now = need_hist ? g_hist + (t % kWindow) * WS : nullptr;
  float* const g_obs = pinned(io.obs + e * (int64_t)W * sp.obs_dim + sp.id_off + lane);
  const float* const mean_l = MS ? sp.obs_mean + lane : nullptr;
  const float* const istd_l = MS ? sp.obs_std + lane : nullptr;
  const int obs_dim = sp.obs_dim, off_pipe = sp.off_pipe, LS = L * S;

  // ---- phase 1: per warehouse row - orders in, arrivals in (multi_env.py:287-292), pipeline block of the observation
  // (multi_env.py:941-968). In this phase lane q owns the four CONSECUTIVE SKUs 4q .. 4q+3 of a row, so a row's cells
  // and ring planes arrive as a handful of vector loads (one 32-bit load per plane: the nine planes of a row in flight
  // cost nine registers; byte loads by strided lanes cost 36 and were what kept this kernel waiting on memory).
  // Slot k of the pipeline block is plane (t + 1 + k) % L for every cell. Slots 0 .. L-2 are the planes after the
  // arrival plane, copied as they stand - four shuffles per plane turn the lane-contiguous bytes into 128-byte
  // coalesced float stores; this step only adds the order a cell places now, which lands in slot lead-1 (the byte there
  // is 0: the plane was cleared when it last arrived, and only this cell's order of exactly that lead writes it) and is
  // patched into the row right after the copy, while its sectors are still in L2 (patching a whole phase later made L2
  // re-fetch every patched sector: +37 KB of DRAM traffic per env-step). Slot L-1 is the arrival plane itself, which
  // after this step only holds the new orders of lead L.
  int rowQ = 0, rowPos = 0;                           // lane w keeps row w's ordered units / ordered cells
  double rowInb = 0.0;                                // ... or its inbound cost when the rates vary over the row
  {
    const bool mine = 4 * lane < S;                   // S % 4 == 0: a lane's four cells exist together
    const int c4 = mine ? lane : 0;
    const float4* __restrict__ act4 = io.action_qty ? nullptr : reinterpret_cast<const float4*>(io.actions + e * WS) + c4;
    const uint32_t* __restrict__ aq4 = io.action_qty ? reinterpret_cast<const uint32_t*>(io.action_qty + e * WS) + c4 : nullptr;
    const uint32_t* __restrict__ lead4 = reinterpret_cast<const uint32_t*>(sp.lead_u8) + c4;
    uint2* inv4 = reinterpret_cast<uint2*>(static_cast<uint16_t*>(st.inventory) + e * WS) + c4;
    uint32_t* row4 = reinterpret_cast<uint32_t*>(static_cast<uint8_t*>(st.ring_qty) + e * (int64_t)WS * L) + c4;
    uint2* hz4 = need_hist ? reinterpret_cast<uint2*>(hist_now - lane) + c4 : nullptr;
    float* __restrict__ out = g_obs + off_pipe;       // lane l's element of a 32-wide store group
    float* __restrict__ outc = g_obs - lane + off_pipe + 4 * c4;   // this lane's own four cells
    uint32_t a_sinv = sm_addr(s_inv) + 8u * c4;
    const int S4 = S >> 2, LS4 = LS >> 2, pa4 = pa * S4;
    int mx[4];                                        // order maxima are whole numbers <= 255 in this layout
#pragma unroll
    for (int j = 0; j < 4; ++j) mx[j] = mine ? (int)sp.action_max[4 * lane + j] : 0;
    const int sub = lane & 3, src0 = lane >> 2;       // where lane l's element of store group j lives: lane 8j + l/4, byte l%4
#pragma unroll 1
    for (int w = 0; w < W; ++w) {
      // every load of the row first: own cells, then the planes of the first batch
      float4 a4 = make_float4(0.f, 0.f, 0.f, 0.f);
      uint32_t aqw = 0u, arr4 = 0u, le4 = 0x01010101u;
      uint2 iv = make_uint2(0u, 0u);
      if (mine) {
        if (aq4) aqw = *aq4; else a4 = *act4;
        iv = *inv4;
        arr4 = row4[pa4];
        le4 = *lead4;
      }
      int q[4], le[4];
      float* dst = out;
      int moff = off_pipe;
#pragma unroll 1
      for (int k0 = 0; k0 < L; k0 += kPlaneBatch) {
        uint32_t x[kPlaneBatch];
#pragma unroll
        for (int kk = 0; kk < kPlaneBatch; ++kk) {
          const bool live = k0 + kk < L - 1;
          x[kk] = (mine && live) ? row4[s_poff[live ? k0 + kk : 0]] : 0u;
        }
        if (k0 == 0) {                                // the row's own cells: order quantity, stock, ring, history plane
          const float af[4] = {a4.x, a4.y, a4.z, a4.w};
          const uint32_t ivv[4] = {iv.x & 0xffffu, iv.x >> 16, iv.y & 0xffffu, iv.y >> 16};
          uint32_t ni[4], newarr = 0u;
          int nQ = 0, nPos = 0;
          double inb = 0.0;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            le[j] = (int)((le4 >> (8 * j)) & 0xffu);
            q[j] = 0;
            if (mine) q[j] = aq4 ? imin((int)((aqw >> (8 * j)) & 0xffu), mx[j]) : rescale_action<kCapsLean>(sp, af[j], (double)mx[j], 0, 0);
            ni[j] = ivv[j] + ((arr4 >> (8 * j)) & 0xffu);
            if (le[j] == L) newarr |= (uint32_t)q[j] << (8 * j);
            nQ += q[j];
            nPos += q[j] > 0 ? 1 : 0;
            if (!by_row && q[j] > 0) {
              const int i = w * S + 4 * lane + j;
              inb += sp.in_fixed[i] + ((double)q[j] * sp.skw[4 * lane + j]) * sp.in_var[i];
            }
          }
          if (mine) {
            asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(a_sinv), "r"(ni[0] | (ni[1] << 16)), "r"(ni[2] | (ni[3] << 16)) : "memory");
            row4[pa4] = newarr;                       // arrivals consumed, lead-L orders in
            uint8_t* rowb = reinterpret_cast<uint8_t*>(row4);
#pragma unroll
            for (int j = 0; j < 4; ++j)
              if (q[j] > 0 && le[j] < L) {
                int p2 = pa + le[j];
                p2 -= p2 >= L ? L : 0;
                rowb[p2 * S + j] = (uint8_t)q[j];
              }
            if (need_hist) *hz4 = make_uint2(0u, 0u);
          }
          if (by_row) {
            nQ = __reduce_add_sync(FULL, nQ);
            nPos = __reduce_add_sync(FULL, nPos);
            if (lane == w) {
              rowQ = nQ;
              rowPos = nPos;
            }
          } else {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) inb += __shfl_xor_sync(FULL, inb, o);
            if (lane == w) rowInb = inb;
          }
        }
#pragma unroll
        for (int kk = 0; kk < kPlaneBatch; ++kk) {
          if (k0 + kk < L) {                          // slot L-1 (x == 0): the arrival plane
#pragma unroll
            for (int j = 0; j < kSlots; ++j) {
              const uint32_t v = __shfl_sync(FULL, x[kk], 8 * j + src0);
              if (VALID(j)) dst[32 * j] = nrm<MS>((float)((v >> (8 * sub)) & 0xffu), mean_l, istd_l, moff + 32 * j);
            }
            dst += S;
            moff += S;
          }
        }
      }
      if (mine) {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (q[j] > 0) {                             // the new order's slot of the pipeline block
            const int po = (le[j] - 1) * S + j;
            outc[po] = nrm<MS>((float)q[j], mean_l - lane, istd_l - lane, off_pipe + 4 * lane + po);
          }
      }
      if (aq4) aq4 += S4; else act4 += S4;
      lead4 += S4;
      inv4 += S4;
      row4 += LS4;
      hz4 += S4;
      out += obs_dim;
      outc += obs_dim;
      a_sinv += 2u * S;
    }
  }
  __syncwarp();                                       // stock staged, history plane cleared

  // ---- phase 2: greedy allocation of this step's lines (demand_allocator.py:150-208) -----------------------------
  {
    LineStream ls;
    ls.init(io.lines, round0, n_rounds, lane);
    uint32_t avlo, avhi;
    owner_masks(ls.map, sm_addr(s_inv), W, S, avlo, avhi);
    allocation_chains<NCH>(sp, ls, sm_addr(smem + lay.t_perm), sm_addr(smem + lay.t_prio), sm_addr(smem + lay.t_home),
                           sm_addr(s_inv), sm_addr(s_shipq), sm_addr(s_lostU), sm_addr(s_lostP), avlo, avhi,
                           need_hist ? reinterpret_cast<uint32_t*>(hist_now - lane) : nullptr);
  }
  __syncwarp();

  // Outbound cost and lost-sales penalty of every warehouse (reward_calculator.py:134-142). Lanes take regions (two per
  // lane cover R <= 64). Per region the lost volume's cost is either spread over the warehouses in proportion to what
  // they shipped there (shipment handler, lost_sales_handler.py:113-148: a rate per shipped unit, one division per
  // region) or goes to the closest warehouse (closest handler, and the shipment handler's fallback when nothing was
  // shipped). Then warehouse by warehouse the lanes' partial sums meet in a shuffle reduction; lane w keeps row w's.
  double costA = 0.0;
  {
    const double pen0 = sp.pen_rate[0];
    double rate[2], lump[2];
    int close_w[2];
#pragma unroll
    for (int qq = 0; qq < 2; ++qq) {
      const int r = lane + 32 * qq;
      rate[qq] = lump[qq] = 0.0;
      close_w[qq] = -1;
      if (r < R) {
        const uint32_t lu = s_lostU[r];
        if (lu > 0u) {
          const double lpn = pen_uniform ? (double)lu * pen0 : s_lostP[r];
          uint32_t shipped_r = 0u;
          if (sp.lost_type == MARLSC_LOST_SHIPMENT)
            for (int w = 0; w < W; ++w) shipped_r += s_shipq[w * R + r];
          if (shipped_r > 0u) {
            rate[qq] = lpn / (double)shipped_r;
          } else {
            lump[qq] = lpn;
            close_w[qq] = sp.closest[r];
          }
        }
      }
    }
    for (int w = 0; w < W; ++w) {
      double c = 0.0;
#pragma unroll
      for (int qq = 0; qq < 2; ++qq) {
        const int r = lane + 32 * qq;
        if (r < R) {
          const uint32_t sq = s_shipq[w * R + r];
          if (sq > 0u) c += (double)sq * (sp.out_var[w * R + r] + rate[qq]);
          if (close_w[qq] == w) c += lump[qq];
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(FULL, c, o);
      if (lane == w) costA = c;
    }
  }

  // ---- phase 3: per warehouse row - stock out, rolling mean, the remaining observation blocks, holding cost ------
  const int hist_n = imin(t + 1, kWindow);
  double costR = 0.0;
  {
    // mean over the window = integer sum / n, rounded to float32 like NumPy's (multi_env.py:785-787): the product with
    // the double reciprocal is within 2^-52 of the quotient, far from every float32 rounding boundary of a quotient
    // of integers below 2^24 by n <= 5, so rounding it gives the correctly rounded float32 quotient
    const double rcp_n = 1.0 / (double)hist_n;
    uint32_t a_sinv = sm_addr(s_inv) + 2u * lane;
    uint16_t* inv = g_inv;
    const uint16_t* hnow = hist_now;
    const uint16_t* hold_p[kWindow - 1];
#pragma unroll
    for (int back = 1; back < kWindow; ++back) hold_p[back - 1] = need_hist ? g_hist + pmod(t - back, kWindow) * WS : nullptr;
    float* out = g_obs;
    const int off_inv = sp.off_inv, off_dh = sp.off_dh, off_rm = sp.off_rm;
    const bool inv_agg = (sp.feat & MARLSC_F_INVENTORY_AGG) != 0;
#pragma unroll 1
    for (int w = 0; w < W; ++w) {
      int vI[kSlots], vdh[kSlots], hv[kSlots][kWindow - 1];
#pragma unroll
      for (int k = 0; k < kSlots; ++k) {              // loads first
        vI[k] = VALID(k) ? (int)ld_s_u16(a_sinv + 64u * k) : 0;
        vdh[k] = VALID(k) && need_hist ? (int)ld_cg_u16(hnow + 32 * k) : 0;   // accumulated with fire-and-forget adds above
#pragma unroll
        for (int back = 1; back < kWindow; ++back)
          hv[k][back - 1] = VALID(k) && need_hist && back < hist_n ? (int)hold_p[back - 1][32 * k] : 0;
      }
      int nI = 0;
      double hold = 0.0;
#pragma unroll
      for (int k = 0; k < kSlots; ++k)
        if (VALID(k)) {
          inv[32 * k] = (uint16_t)vI[k];              // multi_env.py:307 (never negative)
          nI += vI[k];
          if (!by_row) hold += (double)vI[k] * sp.hold_rate[lane + 32 * k];
          out[off_inv + 32 * k] = nrm<MS>((float)vI[k], mean_l, istd_l, off_inv + 32 * k);
          if (off_dh >= 0) out[off_dh + 32 * k] = nrm<MS>((float)vdh[k], mean_l, istd_l, off_dh + 32 * k);
          if (off_rm >= 0) {
            const int hsum = (hv[k][0] + hv[k][1]) + (hv[k][2] + hv[k][3]) + vdh[k];
            out[off_rm + 32 * k] = nrm<MS>((float)((double)hsum * rcp_n), mean_l, istd_l, off_rm + 32 * k);
          }
        }
      nI = __reduce_add_sync(FULL, nI);
      if (lane == 0 && inv_agg) out[off_inv + S] = nrm<MS>((float)nI, mean_l, istd_l, off_inv + S);
      if (sp.id_off && lane < W) out[-sp.id_off] = lane == w ? 1.0f : 0.0f;   // obs_w[lane]: out already points at element id_off + lane
      if (by_row) {
        if (lane == w) {
          const int base = w * S;
          costR = (double)nI * sp.hold_rate[0] + ((double)rowPos * sp.in_fixed[base] + ((double)rowQ * sp.skw[0]) * sp.in_var[base]);
        }
      } else {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) hold += __shfl_xor_sync(FULL, hold, o);
        if (lane == w) costR = hold + rowInb;
      }
      a_sinv += 2u * S;
      inv += S;
      hnow += S;
#pragma unroll
      for (int back = 1; back < kWindow; ++back) hold_p[back - 1] += S;
      out += obs_dim;
    }
  }

  // ---- rewards (multi_env.py:316-327) ----------------------------------------------------------------------------
  double rew = lane < W ? -((costR + costA) * sp.scale) : 0.0;
  if (sp.scope == MARLSC_SCOPE_TEAM) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) rew += __shfl_xor_sync(FULL, rew, o);
  }
  if (lane < W) io.rewards[e * W + lane] = (float)rew;
  if (io.truncated && lane == 0) io.truncated[e] = (uint8_t)(t + 1 >= sp.episode_length);
}

// ---------------------------------------------------------------------------------------------------------------
// The same step as three row / environment kernels + the reward kernel (K1a' .. K1d). The fused kernel above keeps an
// environment's stock in shared memory from the first row to the last, which holds it to 32 warps per SM, and at that
// residency every one of its ~30 dependent memory round trips per env-step shows (ncu: 13 warps per issue slot waiting on
// the long scoreboard, 35-40 % issue utilisation, 25-30 % of DRAM bandwidth). Cut along the data dependencies, the two
// streaming parts run as short-lived warps, one per (environment, warehouse) row with every load of the row in flight at
// once, and only the allocation keeps the shared-memory scratch.
// ---------------------------------------------------------------------------------------------------------------

// K1a': one warp per (environment, warehouse) row - order quantities, arrivals, the row of the ring rewritten with the
// new orders in, history plane cleared, pipeline block of the observation row; the row's inbound cost goes to cost_rows.
// Loads: lane q reads the four consecutive cells 4q .. 4q+3 of the row and of each of its L ring planes (vector loads,
// all in flight at once). The row's L x S bytes are then laid out in shared memory in pipeline-slot order (slot k =
// plane (t + 1 + k) % L, multi_env.py:941-968; slot L-1 is the arrival plane, emptied), the new orders are dropped into
// their slots there (slot lead-1), and the image goes out twice: back to the ring as whole 32-bit words (the first
// version stored single bytes: each touched a 32-byte sector of its own, 25 L1 wavefronts per instruction), and to the
// observation as floats, lane l taking bytes l + 32 j so that every store instruction covers 128 consecutive bytes.
// POLICY: the base-stock heuristic evaluated in place of given actions (its own instantiation: the extra live values cost
// the ordinary one a resident CTA per SM)
// LT: the lead-time horizon L as a compile-time constant (1..16; the plane loops then unroll without predicates: the
// runtime-L form spent 16 instructions per plane load on them), 0 = read it from the spec.
// STATS: also add the row's inbound cost and ordered units to the episode accumulators m (marlsc_env_set_metrics; only
// instantiated with LT = 0, the other kernels ignore m).
template <bool MS, bool POLICY, int LT, bool STATS = false>
__global__ void __launch_bounds__(256)
compact_place_kernel(const __grid_constant__ DevSpec sp, const __grid_constant__ marlsc_env_state_t st,
                     const __grid_constant__ marlsc_step_io_t io, double* __restrict__ cost_rows, int t,
                     const __grid_constant__ marlsc_episode_metrics_t m) {
  extern __shared__ __align__(16) unsigned char smem[];           // [8 warps][L * S] row images
  constexpr int KMAX = LT ? LT : kCompactMaxL;
  const int W = sp.W, S = sp.S, L = LT ? LT : sp.L, WS = W * S;
  const int lane = threadIdx.x & 31;
  const unsigned row = blockIdx.x * 8u + (threadIdx.x >> 5);
  if (row >= (unsigned)st.num_envs * (unsigned)W) return;
  const unsigned eu = row / (unsigned)W;
  const int w = (int)(row - eu * (unsigned)W);
  const int64_t e = eu;
  const bool mine = 4 * lane < S;
  const int c4 = mine ? lane : 0;
  const int S4 = S >> 2, pa = t % L;
  // 32-bit word offset of pipeline slot k's plane inside the ring row: plane (t + 1 + k) % L, walked with one add per slot
  const int LS4 = L * S4;
  int po0 = (pa + 1) * S4;
  po0 = po0 == LS4 ? 0 : po0;
  const bool need_hist = sp.need_hist != 0;
  uint32_t* const row4 = reinterpret_cast<uint32_t*>(static_cast<uint8_t*>(st.ring_qty) + (e * WS + (int64_t)w * S) * L) + c4;
  // every load of the row first
  float4 a4 = make_float4(0.f, 0.f, 0.f, 0.f);
  uint32_t aqw = 0u, arr4 = 0u, le4 = 0x01010101u;
  uint2 iv = make_uint2(0u, 0u);
  uint2* const inv4 = reinterpret_cast<uint2*>(static_cast<uint16_t*>(st.inventory) + e * WS + w * S) + c4;
  uint32_t x[KMAX > 1 ? KMAX - 1 : 1];
  if (mine) {
    if (io.action_qty) aqw = reinterpret_cast<const uint32_t*>(io.action_qty + e * WS + w * S)[c4];
    else if (io.actions) a4 = reinterpret_cast<const float4*>(io.actions + e * WS + w * S)[c4];
    iv = *inv4;
    arr4 = row4[pa * S4];
    le4 = reinterpret_cast<const uint32_t*>(sp.lead_u8 + w * S)[c4];
    int po = po0;
#pragma unroll
    for (int k = 0; k < KMAX - 1; ++k)
      if (k < L - 1) {
        x[k] = row4[po];
        po += S4;
        po = po == LS4 ? 0 : po;
      }
  }
  constexpr bool policy = POLICY;                     // base-stock heuristic in place of given actions (marlsc_step_io.base_stock_level)
  float4 lv4 = make_float4(0.f, 0.f, 0.f, 0.f);
  if (policy && mine)
    lv4 = reinterpret_cast<const float4*>(io.base_stock_level + (io.base_stock_per_env ? e * WS : 0) + w * S)[c4];
  const uint32_t img = sm_addr(smem) + (threadIdx.x >> 5) * (uint32_t)(L * S);   // this warp's row image, slot-major
  if (mine) {
#pragma unroll
    for (int k = 0; k < KMAX - 1; ++k)
      if (k < L - 1) asm volatile("st.shared.u32 [%0], %1;" ::"r"(img + (uint32_t)(k * S + 4 * lane)), "r"(x[k]) : "memory");
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(img + (uint32_t)((L - 1) * S + 4 * lane)), "r"(0u) : "memory");
  }
  float af[4] = {a4.x, a4.y, a4.z, a4.w};
  const uint32_t ivv[4] = {iv.x & 0xffffu, iv.x >> 16, iv.y & 0xffffu, iv.y >> 16};
  if (policy && mine) {
    // reference make_bs_newsvendor_action_fn (run_baselines.py:188-207): order up to the level given on-hand stock and
    // everything in transit - every plane of the ring, the arrivals of this step included (the policy acts before them)
    const float lv[4] = {lv4.x, lv4.y, lv4.z, lv4.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      uint32_t pend = (arr4 >> (8 * j)) & 0xffu;
#pragma unroll
      for (int k = 0; k < KMAX - 1; ++k)
        if (k < L - 1) pend += (x[k] >> (8 * j)) & 0xffu;
      const double mxd = sp.action_max[4 * lane + j];
      double qd = (double)lv[j] - (double)ivv[j] - (double)pend;
      qd = qd < 0.0 ? 0.0 : (qd > mxd ? mxd : qd);
      af[j] = (float)(2.0 * qd / mxd - 1.0);
    }
  }
  uint32_t ni[4];
  int nQ = 0, nPos = 0;
  double inb = 0.0;
  const bool by_row = sp.row_rates_uniform != 0;
  __syncwarp();                                       // a cell's slot may lie in a word another lane has just written? no: own words only,
                                                      // but the byte stores below must follow this lane's word stores in program order
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int le = (int)((le4 >> (8 * j)) & 0xffu);
    int q = 0;
    if (mine) {
      const int mxj = (int)sp.action_max[4 * lane + j];
      q = io.action_qty ? imin((int)((aqw >> (8 * j)) & 0xffu), mxj) : rescale_action<kCapsLean>(sp, af[j], (double)mxj, 0, 0);
      if (q > 0) asm volatile("st.shared.u8 [%0], %1;" ::"r"(img + (uint32_t)((le - 1) * S + 4 * lane + j)), "r"(q) : "memory");
    }
    ni[j] = ivv[j] + ((arr4 >> (8 * j)) & 0xffu);
    nQ += q;
    nPos += q > 0 ? 1 : 0;
    if (!by_row && q > 0) {
      const int i = w * S + 4 * lane + j;
      inb += sp.in_fixed[i] + ((double)q * sp.skw[4 * lane + j]) * sp.in_var[i];
    }
  }
  if (mine) {
    *inv4 = make_uint2(ni[0] | (ni[1] << 16), ni[2] | (ni[3] << 16));
    if (need_hist)
      reinterpret_cast<uint2*>(static_cast<uint16_t*>(st.demand_hist) + e * (int64_t)kWindow * WS + (t % kWindow) * WS + w * S)[c4] = make_uint2(0u, 0u);
  }
  if (by_row) {
    nQ = __reduce_add_sync(FULL, nQ);
    nPos = __reduce_add_sync(FULL, nPos);
    if (lane == 0) cost_rows[row] = (double)nPos * sp.in_fixed[w * S] + ((double)nQ * sp.skw[0]) * sp.in_var[w * S];
  } else {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) inb += __shfl_xor_sync(FULL, inb, o);
    if (lane == 0) cost_rows[row] = inb;
  }
  if (STATS) {                                        // one warp per row: lane 0 owns the row's accumulators
    if (!by_row) nQ = __reduce_add_sync(FULL, nQ);
    if (lane == 0) {
      m.inbound_cost[row] += by_row ? (double)nPos * sp.in_fixed[w * S] + ((double)nQ * sp.skw[0]) * sp.in_var[w * S] : inb;
      m.ordered_units[row] += (double)nQ;
    }
  }
  __syncwarp();                                       // image complete
  if (mine) {                                         // the ring row, every plane as whole words
    int po = po0;
#pragma unroll
    for (int k = 0; k < KMAX; ++k)
      if (k < L) {
        uint32_t v;
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(img + (uint32_t)(k * S + 4 * lane)));
        row4[po] = v;                                 // slot L-1 is the arrival plane
        po += S4;
        po = po == LS4 ? 0 : po;
      }
  }
  // the pipeline block of the observation row
  const float* const mean_l = MS ? sp.obs_mean + sp.off_pipe + lane : nullptr;
  const float* const istd_l = MS ? sp.obs_std + sp.off_pipe + lane : nullptr;
  float* const dst = io.obs + (size_t)row * sp.obs_dim + sp.id_off + sp.off_pipe + lane;
  const uint32_t src = img + lane;
  const int n = L * S;
#pragma unroll 4
  for (int i = 0; i < n; i += 32) {                   // i + lane < n needs checking in the last trip only when n % 32 != 0
    if (i + lane < n) dst[i] = nrm<MS>((float)ld_s_u8(src + i), mean_l, istd_l, i);
  }
}

// K1b': one warp per environment - stock into shared memory, allocation chains over the environment's lines, stock back,
// outbound + lost-sales cost per warehouse to cost_alloc. A lane owns the SKUs its stream's map word names.
// STATS: also add each warehouse's outbound cost, lost-sales cost and shipped units, and the environment's lost and
// demanded units, to the episode accumulators m (marlsc_env_set_metrics; the other kernels ignore m).
template <int NCH, int FS, bool STATS = false>
__global__ void __launch_bounds__(kCompactWarps * 32, MARLSC_ALLOC_CTAS)
compact_alloc_kernel(const __grid_constant__ DevSpec sp, const __grid_constant__ marlsc_env_state_t st,
                     const __grid_constant__ marlsc_step_io_t io, const __grid_constant__ CompactSmem lay,
                     double* __restrict__ cost_alloc, int t, const __grid_constant__ marlsc_episode_metrics_t m) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int W = sp.W, S = sp.S, R = sp.R, WS = W * S;
  {
    const int n_perm = (R * NCH * 32) >> 1, n_prio = (R * 16) >> 2, n_home = (R + 3) >> 2;
    for (int i = threadIdx.x; i < n_perm + n_prio + n_home; i += blockDim.x) {
      if (i < n_perm) reinterpret_cast<uint32_t*>(smem + lay.t_perm)[i] = reinterpret_cast<const uint32_t*>(sp.perm5)[i];
      else if (i < n_perm + n_prio) reinterpret_cast<uint32_t*>(smem + lay.t_prio)[i - n_perm] = reinterpret_cast<const uint32_t*>(sp.prio16)[i - n_perm];
      else reinterpret_cast<uint32_t*>(smem + lay.t_home)[i - n_perm - n_prio] = reinterpret_cast<const uint32_t*>(sp.home_wh)[i - n_perm - n_prio];
    }
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int64_t e = (int64_t)blockIdx.x * kCompactWarps + wid;
  if (e >= st.num_envs) return;
  const bool tail = lane < S - 32 * FS;
  const int64_t round0 = io.line_counts ? e * (int64_t)io.line_stride : (int64_t)io.line_offsets[e];
  const int n_rounds = io.line_counts ? io.line_counts[e] : io.line_offsets[e + 1] - (int)round0;
  if (lane == 0 && n_rounds > 0) prefetch_l2_bulk(io.lines + round0 * 32, (uint32_t)n_rounds * 64u);   // the whole block, one request
  unsigned char* const wbase = smem + lay.t_bytes + (size_t)wid * lay.warp_bytes;
  LineStream ls;
  ls.init(io.lines, round0, n_rounds, lane);          // on their way while the stock is staged
  uint16_t* const s_inv = reinterpret_cast<uint16_t*>(wbase + lay.inv);
  uint32_t* const s_shipq = reinterpret_cast<uint32_t*>(wbase + lay.shipq);
  uint32_t* const s_lostU = reinterpret_cast<uint32_t*>(wbase + lay.lostU);
  double* const s_lostP = reinterpret_cast<double*>(wbase + lay.lostP);
  const bool pen_uniform = sp.pen_uniform != 0;
  for (int i = lane; i < W * R; i += 32) s_shipq[i] = 0u;
  for (int i = lane; i < R; i += 32) {
    s_lostU[i] = 0u;
    if (!pen_uniform) s_lostP[i] = 0.0;
  }
  // stock in: five rows in flight per lane
  uint16_t* const g_inv = pinned(static_cast<uint16_t*>(st.inventory) + e * WS + lane);
  for (int w0 = 0; w0 < W; w0 += 5) {
    uint32_t v[5][kSlots];
#pragma unroll
    for (int d = 0; d < 5; ++d)
#pragma unroll
      for (int k = 0; k < kSlots; ++k) v[d][k] = (w0 + d < W && VALID(k)) ? (uint32_t)g_inv[(w0 + d) * S + 32 * k] : 0u;
#pragma unroll
    for (int d = 0; d < 5; ++d)
#pragma unroll
      for (int k = 0; k < kSlots; ++k)
        if (w0 + d < W && VALID(k)) s_inv[(w0 + d) * S + lane + 32 * k] = (uint16_t)v[d][k];
  }
  __syncwarp();
  uint32_t avlo, avhi;                                // which warehouses hold the SKUs this lane's streams name
  owner_masks(ls.map, sm_addr(s_inv), W, S, avlo, avhi);
  const bool need_hist = sp.need_hist != 0;
  uint32_t* const hist32 = need_hist ? reinterpret_cast<uint32_t*>(static_cast<uint16_t*>(st.demand_hist) + e * (int64_t)kWindow * WS + (t % kWindow) * WS) : nullptr;
  {
    // every shared address the chains use is one of two bases plus a launch constant (the layout is a kernel parameter)
    const uint32_t a_cta = sm_addr(smem), a_warp = a_cta + (uint32_t)lay.t_bytes + (uint32_t)wid * (uint32_t)lay.warp_bytes;
    allocation_chains<NCH>(sp, ls, a_cta + (uint32_t)lay.t_perm, a_cta + (uint32_t)lay.t_prio, a_cta + (uint32_t)lay.t_home,
                           a_warp + (uint32_t)lay.inv, a_warp + (uint32_t)lay.shipq, a_warp + (uint32_t)lay.lostU,
                           a_warp + (uint32_t)lay.lostP, avlo, avhi, hist32);
  }
  __syncwarp();
  for (int w0 = 0; w0 < W; ++w0)                       // stock out (multi_env.py:307; never negative)
#pragma unroll
    for (int k = 0; k < kSlots; ++k)
      if (VALID(k)) g_inv[w0 * S + 32 * k] = s_inv[w0 * S + lane + 32 * k];
  // outbound cost and lost-sales penalty per warehouse (see the fused kernel)
  const double pen0 = sp.pen_rate[0];
  double rate[2], lump[2];
  int close_w[2];
#pragma unroll
  for (int qq = 0; qq < 2; ++qq) {
    const int r = lane + 32 * qq;
    rate[qq] = lump[qq] = 0.0;
    close_w[qq] = -1;
    if (r < R) {
      const uint32_t lu = s_lostU[r];
      if (lu > 0u) {
        const double lpn = pen_uniform ? (double)lu * pen0 : s_lostP[r];
        uint32_t shipped_r = 0u;
        if (sp.lost_type == MARLSC_LOST_SHIPMENT)
          for (int w = 0; w < W; ++w) shipped_r += s_shipq[w * R + r];
        if (shipped_r > 0u) {
          rate[qq] = lpn / (double)shipped_r;
        } else {
          lump[qq] = lpn;
          close_w[qq] = sp.closest[r];
        }
      }
    }
  }
  for (int w0 = 0; w0 < W; w0 += 4) {                  // four warehouses' table entries in flight per lane
    uint32_t sq[4][2];
    double ov[4][2];
#pragma unroll
    for (int d = 0; d < 4; ++d)
#pragma unroll
      for (int qq = 0; qq < 2; ++qq) {
        const int r = lane + 32 * qq;
        const bool ok = w0 + d < W && r < R;
        sq[d][qq] = ok ? s_shipq[(w0 + d) * R + r] : 0u;
        ov[d][qq] = ok ? sp.out_var[(w0 + d) * R + r] : 0.0;
      }
#pragma unroll
    for (int d = 0; d < 4; ++d) {
      if (w0 + d < W) {
        double c = 0.0;
        double c_out = 0.0, c_pen = 0.0;              // STATS: the two parts of c
#pragma unroll
        for (int qq = 0; qq < 2; ++qq) {
          if (sq[d][qq] > 0u) c += (double)sq[d][qq] * (ov[d][qq] + rate[qq]);
          if (close_w[qq] == w0 + d) c += lump[qq];
          if (STATS) {
            c_out += (double)sq[d][qq] * ov[d][qq];
            c_pen += (double)sq[d][qq] * rate[qq] + (close_w[qq] == w0 + d ? lump[qq] : 0.0);
          }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(FULL, c, o);
        if (lane == 0) cost_alloc[e * W + w0 + d] = c;
        if (STATS) {                                  // one warp per environment: lane 0 owns its accumulators
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) {
            c_out += __shfl_xor_sync(FULL, c_out, o);
            c_pen += __shfl_xor_sync(FULL, c_pen, o);
          }
          const uint32_t shipped = __reduce_add_sync(FULL, sq[d][0] + sq[d][1]);
          if (lane == 0) {
            const int64_t i = e * W + w0 + d;
            m.outbound_cost[i] += c_out;
            m.penalty_cost[i] += c_pen;
            m.shipped_units[i] += (double)shipped;
          }
        }
      }
    }
  }
  if (STATS) {                                        // units demanded = shipped + lost (every line is one or the other)
    uint32_t lost = 0u, shipped = 0u;
#pragma unroll
    for (int qq = 0; qq < 2; ++qq) {
      const int r = lane + 32 * qq;
      if (r < R) {
        lost += s_lostU[r];
        for (int w = 0; w < W; ++w) shipped += s_shipq[w * R + r];
      }
    }
    lost = __reduce_add_sync(FULL, lost);
    shipped = __reduce_add_sync(FULL, shipped);
    if (lane == 0) {
      m.lost_units[e] += (double)lost;
      m.demand_units[e] += (double)shipped + (double)lost;
    }
  }
}

// K1c': one warp per (environment, warehouse) row - rolling mean, the remaining observation blocks, holding cost added to
// the row's inbound cost; with agent-scope rewards also the reward itself (no K1d launch). Like K1a', lane q loads the
// four consecutive cells 4q .. 4q+3 of each plane with one vector load (six loads per lane instead of 24 two-byte ones),
// the block values go through a small shared-memory image and leave as 128-byte coalesced float stores.
#ifndef MARLSC_FEAT_CTAS
#define MARLSC_FEAT_CTAS 8
#endif
// STATS: also add the row's holding cost to the episode accumulators m (marlsc_env_set_metrics; the other kernels ignore m).
template <bool MS, bool STATS = false>
__global__ void __launch_bounds__(256, MARLSC_FEAT_CTAS)
compact_feature_kernel(const __grid_constant__ DevSpec sp, const __grid_constant__ marlsc_env_state_t st,
                       const __grid_constant__ marlsc_step_io_t io, double* __restrict__ cost_rows,
                       const double* __restrict__ cost_alloc, int t, int write_rewards,
                       const __grid_constant__ marlsc_episode_metrics_t m) {
  extern __shared__ __align__(16) unsigned char smem[];           // [8 warps][3 * S] floats: inventory | home demand | rolling mean
  const int W = sp.W, S = sp.S, WS = W * S;
  const int lane = threadIdx.x & 31;
  const unsigned row = blockIdx.x * 8u + (threadIdx.x >> 5);
  if (row >= (unsigned)st.num_envs * (unsigned)W) return;
  const unsigned eu = row / (unsigned)W;
  const int w = (int)(row - eu * (unsigned)W);
  const int64_t e = eu;
  const bool mine = 4 * lane < S;
  const int c4 = mine ? lane : 0;
  const bool need_hist = sp.need_hist != 0;
  const int hist_n = imin(t + 1, kWindow);
  const uint2* const inv4 = reinterpret_cast<const uint2*>(static_cast<const uint16_t*>(st.inventory) + e * WS + w * S) + c4;
  const uint16_t* const hist = need_hist ? static_cast<const uint16_t*>(st.demand_hist) + e * (int64_t)kWindow * WS + w * S : nullptr;
  uint2 iv = make_uint2(0u, 0u), hn = make_uint2(0u, 0u), ho[kWindow - 1];
#pragma unroll
  for (int back = 1; back < kWindow; ++back) ho[back - 1] = make_uint2(0u, 0u);
  double cost_in = 0.0, cost_al = 0.0;                // the row's cost so far: requested with everything else, used last
  if (lane == 0) {
    cost_in = cost_rows[row];
    if (write_rewards) cost_al = cost_alloc[row];
  }
  if (mine) {                                         // every load of the row first
    iv = *inv4;
    if (need_hist) {
      // this step's plane was accumulated by K1b' with red.global: read it from L2
      asm volatile("ld.global.cg.v2.u32 {%0, %1}, [%2];" : "=r"(hn.x), "=r"(hn.y) : "l"(reinterpret_cast<const uint2*>(hist + (t % kWindow) * WS) + c4));
#pragma unroll
      for (int back = 1; back < kWindow; ++back)
        if (back < hist_n) ho[back - 1] = reinterpret_cast<const uint2*>(hist + pmod(t - back, kWindow) * WS)[c4];
    }
  }
  float* const img = reinterpret_cast<float*>(smem) + (threadIdx.x >> 5) * (3 * S);
  const double rcp_n = 1.0 / (double)hist_n;          // see the fused kernel: rounds to the correctly rounded float32 quotient
  const bool by_row = sp.row_rates_uniform != 0;
  int nI = 0;
  double hold = 0.0;
  if (mine) {
    const uint32_t vI[4] = {iv.x & 0xffffu, iv.x >> 16, iv.y & 0xffffu, iv.y >> 16};
    const uint32_t vd[4] = {hn.x & 0xffffu, hn.x >> 16, hn.y & 0xffffu, hn.y >> 16};
    uint32_t hs[4] = {vd[0], vd[1], vd[2], vd[3]};
#pragma unroll
    for (int back = 1; back < kWindow; ++back) {
      hs[0] += ho[back - 1].x & 0xffffu;
      hs[1] += ho[back - 1].x >> 16;
      hs[2] += ho[back - 1].y & 0xffffu;
      hs[3] += ho[back - 1].y >> 16;
    }
    float4 fi, fd, fr;
    fi.x = (float)vI[0]; fi.y = (float)vI[1]; fi.z = (float)vI[2]; fi.w = (float)vI[3];
    fd.x = (float)vd[0]; fd.y = (float)vd[1]; fd.z = (float)vd[2]; fd.w = (float)vd[3];
    fr.x = (float)((double)hs[0] * rcp_n); fr.y = (float)((double)hs[1] * rcp_n);
    fr.z = (float)((double)hs[2] * rcp_n); fr.w = (float)((double)hs[3] * rcp_n);
    reinterpret_cast<float4*>(img)[lane] = fi;
    reinterpret_cast<float4*>(img + S)[lane] = fd;
    reinterpret_cast<float4*>(img + 2 * S)[lane] = fr;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      nI += (int)vI[j];
      if (!by_row) hold += (double)vI[j] * sp.hold_rate[4 * lane + j];
    }
  }
  nI = __reduce_add_sync(FULL, nI);
  double cost;
  if (by_row) {
    cost = (double)nI * sp.hold_rate[0];
  } else {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) hold += __shfl_xor_sync(FULL, hold, o);
    cost = hold;
  }
  float* const obs_w = io.obs + (size_t)row * sp.obs_dim;
  if (lane == 0) {
    if (STATS) m.holding_cost[row] += cost;           // one warp per row: lane 0 owns the row's accumulators
    cost += cost_in;                                  // + the inbound cost K1a' left there
    if (write_rewards) {                              // agent scope (multi_env.py:316-327): no reward kernel needed
      io.rewards[row] = (float)(-((cost + cost_al) * sp.scale));
      if (io.truncated && w == 0) io.truncated[e] = (uint8_t)(t + 1 >= sp.episode_length);
    } else {
      cost_rows[row] = cost;
    }
    if (sp.feat & MARLSC_F_INVENTORY_AGG) {
      float x = (float)nI;
      if (MS) x = f_mul(f_sub(x, sp.obs_mean[sp.off_inv + S]), sp.obs_std[sp.off_inv + S]);
      obs_w[sp.id_off + sp.off_inv + S] = x;
    }
  }
  if (sp.id_off && lane < W) obs_w[lane] = lane == w ? 1.0f : 0.0f;
  __syncwarp();                                       // image complete
  float* const out = obs_w + sp.id_off + lane;
  const int offs[3] = {sp.off_inv, sp.off_dh, sp.off_rm};
#pragma unroll
  for (int b = 0; b < 3; ++b) {
    if (offs[b] < 0) continue;
    const float* src = img + b * S + lane;
    const float* const mean_l = MS ? sp.obs_mean + offs[b] + lane : nullptr;
    const float* const istd_l = MS ? sp.obs_std + offs[b] + lane : nullptr;
#pragma unroll
    for (int k = 0; k < kSlots; ++k)                  // S <= 32 kSlots: four predicated stores, no loop scaffolding
      if (32 * k + lane < S) out[offs[b] + 32 * k] = nrm<MS>(src[32 * k], mean_l, istd_l, 32 * k);
  }
}

// K1c' with the bulk-copy engine (opt-in: MARLSC_FEATURE_BULK=1; measured slower, see below): persistent CTAs, one warp
// per warehouse row. A single thread asks the copy engine for an environment's stock block ([W,S] uint16) and its five
// history planes ([5,W,S] uint16, contiguous) - two cp.async.bulk requests (SASS UBLKCP.S.G), 12 W S bytes, completion
// counted on an mbarrier - a few environments ahead of the one the warps are reading out of shared memory; a second set
// of mbarriers hands the stages back, so no warp waits for another. The blocks are 16-byte granular when W S is a
// multiple of 8 (the launcher checks). Same arithmetic as above, bit-identical results (the parity tests run both).
// Measured at 65,536 large environments (one B200): 0.37 ms with four stages and a CTA barrier per environment,
// 0.48-0.55 ms in this form, against 0.34 ms for the register version above; the copy pipeline alone (no read-out) runs
// in 0.15 ms, the read-out without its observation stores adds 0.16 ms and the stores another 0.17 ms - the three do
// not overlap the way the 40 independent short-lived warps per SM of the register version do, so that one stays.
constexpr int kFeatStages = 5;

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_load(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes),
               "r"(bar)
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}"
               : "=r"(done)
               : "r"(bar), "r"(parity)
               : "memory");
  return done != 0u;
}

template <bool MS>
__global__ void __launch_bounds__(512)
compact_feature_bulk_kernel(const __grid_constant__ DevSpec sp, const __grid_constant__ marlsc_env_state_t st,
                            const __grid_constant__ marlsc_step_io_t io, double* __restrict__ cost_rows,
                            const double* __restrict__ cost_alloc, int t, int write_rewards) {
  extern __shared__ __align__(16) unsigned char smem[];           // kFeatStages x (stock | 5 history planes), then the mbarriers
  const int W = sp.W, S = sp.S, WS = W * S;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;         // blockDim.x = 32 W: warp w owns row w
  const bool need_hist = sp.need_hist != 0;
  const uint32_t stock_bytes = 2u * (uint32_t)WS, hist_bytes = need_hist ? (uint32_t)kWindow * stock_bytes : 0u;
  const uint32_t stage_bytes = (1u + (uint32_t)kWindow) * stock_bytes;
  const uint32_t a_smem = sm_addr(smem), a_full = a_smem + (uint32_t)kFeatStages * stage_bytes, a_empty = a_full + 8u * kFeatStages;
  if (threadIdx.x == 0) {
#pragma unroll
    for (int i = 0; i < kFeatStages; ++i) {
      mbar_init(a_full + 8u * i, 1u);
      mbar_init(a_empty + 8u * i, (uint32_t)W);       // one arrival per warp that has read the stage out
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  const int64_t n_env = st.num_envs, stride = gridDim.x;
  const uint16_t* const g_inv = static_cast<const uint16_t*>(st.inventory);
  const uint16_t* const g_hist = static_cast<const uint16_t*>(st.demand_hist);
  const auto request = [&](int64_t e, int stage) {    // thread 0: the two blocks of environment e into a stage
    const uint32_t bar = a_full + 8u * stage, dst = a_smem + (uint32_t)stage * stage_bytes;
    mbar_expect_tx(bar, stock_bytes + hist_bytes);
    bulk_load(dst, g_inv + e * WS, stock_bytes, bar);
    if (need_hist) bulk_load(dst + stock_bytes, g_hist + e * (int64_t)kWindow * WS, hist_bytes, bar);
  };
  // Trip i reads stage i % kFeatStages. Thread 0 requests trip i + kFeatStages - 2 at the start of trip i: that stage
  // was read out in trip i - 2, so the other warps had a whole trip to leave it (no warp waits for another here; the
  // warps of a CTA drift up to two environments apart).
  constexpr int kAhead = kFeatStages - 2;
  if (threadIdx.x == 0)
    for (int k = 0; k < kAhead; ++k)
      if (blockIdx.x + k * stride < n_env) request(blockIdx.x + k * stride, k);
  const int hist_n = imin(t + 1, kWindow);
  const double rcp_n = 1.0 / (double)hist_n;          // see the fused kernel: rounds to the correctly rounded float32 quotient
  const bool by_row = sp.row_rates_uniform != 0;
  const int p_now = t % kWindow;
  int it = 0;
  for (int64_t e = blockIdx.x; e < n_env; e += stride, ++it) {
    const int stage = it % kFeatStages;
    if (threadIdx.x == 0) {
      const int64_t e_next = e + (int64_t)kAhead * stride;
      if (e_next < n_env) {
        const int st_next = (it + kAhead) % kFeatStages;
        if (it >= 2) {                                // its previous tenant: trip it - 2
          const uint32_t par = (uint32_t)((it - 2) / kFeatStages) & 1u;
          while (!mbar_try_wait(a_empty + 8u * st_next, par)) {}
        }
        request(e_next, st_next);
      }
    }
    const int64_t row = e * W + w;
    double cost_in = 0.0, cost_al = 0.0;              // on their way while the stage lands
    if (lane == 0) {
      cost_in = cost_rows[row];
      if (write_rewards) cost_al = cost_alloc[row];
    }
    const uint32_t parity = (uint32_t)(it / kFeatStages) & 1u;
    while (!mbar_try_wait(a_full + 8u * stage, parity)) {}
    const uint16_t* const s_inv = reinterpret_cast<const uint16_t*>(smem + (size_t)stage * stage_bytes) + w * S;
    const uint16_t* const s_hist = s_inv + WS;        // plane p of this row: s_hist + p WS
    float* const obs_w = io.obs + (size_t)row * sp.obs_dim;
    float* const out = obs_w + sp.id_off;
    int nI = 0;
    double hold = 0.0;
    for (int i = lane; i < S; i += 32) {
      const uint32_t v = s_inv[i];
      nI += (int)v;
      if (!by_row) hold += (double)v * sp.hold_rate[i];
      if (sp.off_inv >= 0) out[sp.off_inv + i] = nrm<MS>((float)v, sp.obs_mean, sp.obs_std, sp.off_inv + i);
      if (need_hist) {
        const uint32_t d = s_hist[p_now * WS + i];
        uint32_t hs = d;
#pragma unroll
        for (int back = 1; back < kWindow; ++back)
          if (back < hist_n) hs += s_hist[pmod(t - back, kWindow) * WS + i];
        if (sp.off_dh >= 0) out[sp.off_dh + i] = nrm<MS>((float)d, sp.obs_mean, sp.obs_std, sp.off_dh + i);
        if (sp.off_rm >= 0) out[sp.off_rm + i] = nrm<MS>((float)((double)hs * rcp_n), sp.obs_mean, sp.obs_std, sp.off_rm + i);
      }
    }
    nI = __reduce_add_sync(FULL, nI);
    double cost;
    if (by_row) {
      cost = (double)nI * sp.hold_rate[0];
    } else {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) hold += __shfl_xor_sync(FULL, hold, o);
      cost = hold;
    }
    __syncwarp();
    if (lane == 0) {
      asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(a_empty + 8u * stage) : "memory");   // this warp has left the stage
      cost += cost_in;                                // + the inbound cost K1a' left there
      if (write_rewards) {                            // agent scope (multi_env.py:316-327): no reward kernel needed
        io.rewards[row] = (float)(-((cost + cost_al) * sp.scale));
        if (io.truncated && w == 0) io.truncated[e] = (uint8_t)(t + 1 >= sp.episode_length);
      } else {
        cost_rows[row] = cost;
      }
      if (sp.feat & MARLSC_F_INVENTORY_AGG) {
        float x = (float)nI;
        if (MS) x = f_mul(f_sub(x, sp.obs_mean[sp.off_inv + S]), sp.obs_std[sp.off_inv + S]);
        obs_w[sp.id_off + sp.off_inv + S] = x;
      }
    }
    if (sp.id_off && lane < W) obs_w[lane] = lane == w ? 1.0f : 0.0f;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Reset (multi_env.py:233-246): clear ring and history, load the start inventory, first observation. One thread per
// (environment, warehouse, SKU) cell; not a hot kernel.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
env_reset_compact_kernel(const __grid_constant__ DevSpec sp, const __grid_constant__ marlsc_env_state_t st,
                         const int32_t* __restrict__ init, int per_env, float* __restrict__ obs) {
  const int W = sp.W, S = sp.S, L = sp.L, WS = W * S;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= st.num_envs * (long long)WS) return;
  const long long e = idx / WS;
  const int i = (int)(idx - e * WS), w = i / S, s = i - w * S;
  const int v = init[per_env ? idx : i];
  static_cast<uint16_t*>(st.inventory)[idx] = (uint16_t)(v < 0 ? 0 : (v > 65535 ? 65535 : v));
  uint8_t* ring = static_cast<uint8_t*>(st.ring_qty) + (e * WS + (long long)w * S) * L + s;
  for (int d = 0; d < L; ++d) ring[d * S] = 0;
  if (st.demand_hist) {
    uint16_t* h = static_cast<uint16_t*>(st.demand_hist) + e * (long long)kWindow * WS + i;
    for (int b = 0; b < kWindow; ++b) h[b * WS] = 0;
  }
  const bool ms = sp.norm == MARLSC_NORM_MEANSTD;
  float* obs_w = obs + (e * W + w) * (long long)sp.obs_dim;
  float* out = obs_w + sp.id_off;
  put(sp, ms, out, (unsigned)(sp.off_inv + s), (float)v);
  for (int k = 0; k < L; ++k) put(sp, ms, out, (unsigned)(sp.off_pipe + k * S + s), 0.f);
  if (sp.off_dh >= 0) put(sp, ms, out, (unsigned)(sp.off_dh + s), 0.f);
  if (sp.off_rm >= 0) put(sp, ms, out, (unsigned)(sp.off_rm + s), 0.f);
  if (s == 0) {
    if (sp.feat & MARLSC_F_INVENTORY_AGG) {
      int tot = 0;
      for (int ss = 0; ss < S; ++ss) tot += init[(per_env ? e * WS : 0) + w * S + ss];
      put(sp, ms, out, (unsigned)(sp.off_inv + S), (float)tot);
    }
    for (int j = 0; j < sp.id_off; ++j) obs_w[j] = j == w ? 1.0f : 0.0f;
  }
}

// K5 (compact): units in transit to a cell are the sum of its ring column (every plane is an arrival still to come).
template <typename IDX>
__global__ void __launch_bounds__(256)
base_stock_compact_kernel(const __grid_constant__ DevSpec sp, const __grid_constant__ marlsc_env_state_t st,
                          const float* __restrict__ level, int level_per_env, float* __restrict__ actions) {
  const IDX WS = (IDX)(sp.W * sp.S);
  const IDX idx = (IDX)blockIdx.x * (IDX)blockDim.x + (IDX)threadIdx.x;
  if (idx >= (IDX)st.num_envs * WS) return;
  const IDX e = idx / WS;
  const int i = (int)(idx - e * WS), w = i / sp.S, s = i - w * sp.S;
  const int L = sp.L;
  const uint8_t* ring = static_cast<const uint8_t*>(st.ring_qty) + ((long long)e * (long long)WS + (long long)w * sp.S) * L + s;
  int pending = 0;
  for (int d0 = 0; d0 < L; d0 += 4) {
    int v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) v[k] = d0 + k < L ? (int)ring[(d0 + k) * sp.S] : 0;
    pending += (v[0] + v[1]) + (v[2] + v[3]);
  }
  const double mx = sp.action_max[s];
  double q = (double)(level_per_env ? level[idx] : level[i]) - (double)static_cast<const uint16_t*>(st.inventory)[idx] - (double)pending;
  q = q < 0.0 ? 0.0 : (q > mx ? mx : q);
  actions[idx] = (float)(2.0 * q / mx - 1.0);
}

// Dense order rows -> lines (padded layout): one warp per environment. Pass 1 counts the non-zero cells of every SKU;
// the SKUs are then ranked by that count (descending, ties by SKU id) and dealt to the 32 lanes in a snake (rank 0..31
// to lanes 0..31 as slot 0, ranks 32..63 to lanes 31..0 as slot 1, ...), so the streams of an environment end within a
// few entries of each other - the allocation kernel runs as long as the longest stream. Pass 2 writes the entries: a
// stream holds all lines of its slot-0 SKU, then of its slot-1 SKU, ..., each in order sequence (the chains of different
// SKUs never meet, demand_allocator.py:150-208, so only the sequence inside a SKU matters). Entry 0/1 of every lane is
// its SKU map. demand.pack_lines builds the same bytes on the host.
__global__ void __launch_bounds__(128)
lines_from_orders_kernel(const __grid_constant__ DevSpec sp, long long E, const __grid_constant__ marlsc_step_io_t io,
                         int stride, uint16_t* __restrict__ lines, int32_t* __restrict__ counts, int32_t* __restrict__ overflow) {
  __shared__ uint16_t s_cnt[4][128];     // lines of SKU s
  __shared__ uint16_t s_base[4][128];    // first entry of SKU s inside its stream
  __shared__ uint8_t s_dst[4][128];      // stream of SKU s: lane | slot << 5
  __shared__ uint8_t s_map[4][128];      // SKU of (lane, slot): index 4 lane + slot
  __shared__ uint16_t s_dcnt[4][128];    // its line count
  const int wid = threadIdx.x >> 5;
  const long long e = (long long)blockIdx.x * 4 + wid;
  if (e >= E) return;
  const int lane = threadIdx.x & 31, S = sp.S;
  const long long o_begin = io.order_counts ? e * (long long)io.order_stride : (long long)io.order_offsets[e];
  const int n_orders = io.order_counts ? io.order_counts[e] : io.order_offsets[e + 1] - (int)o_begin;
  const uint8_t* qty = static_cast<const uint8_t*>(io.order_qty) + o_begin * S + lane;
  uint16_t* const env_lines = lines + e * (long long)stride * 32;    // entry p of lane l: env_lines[(p >> 1) * 64 + 2 l + (p & 1)]
  // pass 1: lines per SKU
  int c[kSlots];
#pragma unroll
  for (int k = 0; k < kSlots; ++k) c[k] = 0;
  for (int j0 = 0; j0 < n_orders; j0 += 4) {
    uint32_t v[4][kSlots];
#pragma unroll
    for (int jj = 0; jj < 4; ++jj)
#pragma unroll
      for (int k = 0; k < kSlots; ++k) v[jj][k] = (j0 + jj < n_orders && lane + 32 * k < S) ? (uint32_t)qty[(long long)(j0 + jj) * S + 32 * k] : 0u;
#pragma unroll
    for (int jj = 0; jj < 4; ++jj)
#pragma unroll
      for (int k = 0; k < kSlots; ++k) c[k] += v[jj][k] != 0u ? 1 : 0;
  }
#pragma unroll
  for (int k = 0; k < kSlots; ++k) {
    s_cnt[wid][lane + 32 * k] = (uint16_t)c[k];
    s_map[wid][lane + 32 * k] = 255;
    s_dcnt[wid][lane + 32 * k] = 0;
  }
  __syncwarp();
  // rank -> (lane, slot)
  int rank[kSlots];
#pragma unroll
  for (int k = 0; k < kSlots; ++k) rank[k] = 0;
  for (int s2 = 0; s2 < S; ++s2) {
    const int c2 = s_cnt[wid][s2];
#pragma unroll
    for (int k = 0; k < kSlots; ++k) rank[k] += (c2 > c[k] || (c2 == c[k] && s2 < lane + 32 * k)) ? 1 : 0;
  }
#pragma unroll
  for (int k = 0; k < kSlots; ++k)
    if (lane + 32 * k < S) {
      const int row = rank[k] >> 5, col = rank[k] & 31, dl = (row & 1) ? 31 - col : col;
      s_dst[wid][lane + 32 * k] = (uint8_t)(dl | (row << 5));
      s_map[wid][4 * dl + row] = (uint8_t)(lane + 32 * k);
      s_dcnt[wid][4 * dl + row] = (uint16_t)c[k];
    }
  __syncwarp();
  uint32_t map = 0u;
  int total = 0;
#pragma unroll
  for (int k = 0; k < kSlots; ++k) {
    const uint32_t sk = s_map[wid][4 * lane + k];
    map |= sk << (8 * k);
    if (sk != 255u) s_base[wid][sk] = (uint16_t)total;
    total += s_dcnt[wid][4 * lane + k];
  }
  __syncwarp();
  // pass 2: entries
  int at[kSlots], dl[kSlots], ds[kSlots];
#pragma unroll
  for (int k = 0; k < kSlots; ++k) {
    const bool named = lane + 32 * k < S;
    at[k] = named ? 2 + (int)s_base[wid][lane + 32 * k] : 0;        // entries 0, 1 hold the map
    dl[k] = named ? s_dst[wid][lane + 32 * k] & 31 : 0;
    ds[k] = named ? s_dst[wid][lane + 32 * k] >> 5 : 0;
  }
  bool over = false;
  for (int j0 = 0; j0 < n_orders; j0 += 4) {          // four orders' cells in flight per lane
    uint32_t v[4][kSlots];
    int rg[4];
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
      const bool live = j0 + jj < n_orders;
      rg[jj] = live ? (int)io.order_region[o_begin + j0 + jj] : 0;
#pragma unroll
      for (int k = 0; k < kSlots; ++k) v[jj][k] = (live && lane + 32 * k < S) ? (uint32_t)qty[(long long)(j0 + jj) * S + 32 * k] : 0u;
    }
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
      const int r = sp.region_map ? sp.region_map[rg[jj]] : rg[jj];
#pragma unroll
      for (int k = 0; k < kSlots; ++k)
        if (v[jj][k] != 0u) {
          if (at[k] < stride) env_lines[(long long)(at[k] >> 1) * 64 + 2 * dl[k] + (at[k] & 1)] = line_entry((int)v[jj][k], r, ds[k]);
          else over = true;
          ++at[k];
        }
    }
  }
  const int longest = __reduce_max_sync(FULL, total);
  int rounds = 0;
  if (longest > 0) {                                  // an environment without demand has no rounds at all
    const int mine = imin(total + 2, stride);
    rounds = (imin(longest + 2, stride) + 1) & ~1;    // whole round pairs
    uint16_t* const out = env_lines + 2 * lane;
    out[0] = (uint16_t)(map & 0xffffu);
    out[1] = (uint16_t)(map >> 16);
    for (int p = mine; p < rounds; ++p) out[(long long)(p >> 1) * 64 + (p & 1)] = 0;     // pad this stream to the environment's round count
  }
  if (lane == 0) counts[e] = rounds;
  if (over) atomicExch(overflow, 1);
}

template <int NCH, bool MS, int FS>
int launch_step_nch(const LaunchArgs& a, const marlsc_step_io_t& io, int t, cudaStream_t s) {
  const CompactSmem lay = compact_smem(a.ds.W, a.ds.S, a.ds.R, NCH, a.ds.pen_uniform);
  const size_t smem = (size_t)lay.t_bytes + (size_t)kCompactWarps * lay.warp_bytes;
  if ((int)smem > a.max_smem_optin)
    return set_error(MARLSC_EUNSUPPORTED, "compact step: shared-memory scratch of " + std::to_string(smem) + " bytes per CTA does not fit");
  static int configured_for[kMaxDevices] = {0};       // per device: the attributes belong to the device's context
  int dev = 0;
  MARLSC_CUDA(cudaGetDevice(&dev));
  if (dev >= kMaxDevices || configured_for[dev] < (int)smem) {
    MARLSC_CUDA(cudaFuncSetAttribute((const void*)env_step_compact_kernel<NCH, MS, FS>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                     (int)cudaSharedmemCarveoutMaxShared));
    MARLSC_CUDA(cudaFuncSetAttribute((const void*)env_step_compact_kernel<NCH, MS, FS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (dev < kMaxDevices) configured_for[dev] = (int)smem;
  }
  const unsigned grid = (unsigned)((a.st.num_envs + kCompactWarps - 1) / kCompactWarps);
  // bulk L2 prefetches of an environment's state blocks need 16-byte aligned addresses and sizes
  const auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; };
  const int prefetch = a.ds.compact_prefetch && al16(a.st.ring_qty) && al16(a.st.inventory) && al16(io.actions) && al16(io.action_qty);
  env_step_compact_kernel<NCH, MS, FS><<<grid, kCompactWarps * 32, smem, s>>>(a.ds, a.st, io, t, prefetch);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  MARLSC_CUDA(cudaGetLastError());
  return MARLSC_OK;
}

template <int NCH, bool MS, int FS>
int launch_split_nch(const LaunchArgs& a, const marlsc_step_io_t& io, const SplitWork& wk, int t, cudaStream_t s) {
  const CompactSmem lay = compact_smem(a.ds.W, a.ds.S, a.ds.R, NCH, a.ds.pen_uniform);
  const size_t smem = (size_t)lay.t_bytes + (size_t)kCompactWarps * lay.warp_bytes;
  if ((int)smem > a.max_smem_optin)
    return set_error(MARLSC_EUNSUPPORTED, "compact step: shared-memory scratch of " + std::to_string(smem) + " bytes per CTA does not fit");
  static int configured_for[kMaxDevices] = {0};       // per device: the attributes belong to the device's context
  int dev = 0;
  MARLSC_CUDA(cudaGetDevice(&dev));
  if (dev >= kMaxDevices || configured_for[dev] < (int)smem) {
    MARLSC_CUDA(cudaFuncSetAttribute((const void*)compact_alloc_kernel<NCH, FS>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                     (int)cudaSharedmemCarveoutMaxShared));
    MARLSC_CUDA(cudaFuncSetAttribute((const void*)compact_alloc_kernel<NCH, FS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (dev < kMaxDevices) configured_for[dev] = (int)smem;
  }
  // episode metrics (marlsc_env_set_metrics): the STATS instantiations of K1a' (runtime lead horizon), K1b' and K1c'
  const bool stats = wk.metrics != nullptr;
  const marlsc_episode_metrics_t m = stats ? *wk.metrics : marlsc_episode_metrics_t{};
  if (stats) {
    static int stats_configured_for[kMaxDevices] = {0};
    if (dev >= kMaxDevices || stats_configured_for[dev] < (int)smem) {
      MARLSC_CUDA(cudaFuncSetAttribute((const void*)compact_alloc_kernel<NCH, FS, true>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                       (int)cudaSharedmemCarveoutMaxShared));
      MARLSC_CUDA(cudaFuncSetAttribute((const void*)compact_alloc_kernel<NCH, FS, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      if (dev < kMaxDevices) stats_configured_for[dev] = (int)smem;
    }
  }
  const int64_t rows = a.st.num_envs * a.ds.W;
  const unsigned grid_rows = (unsigned)((rows + 7) / 8);
  const unsigned grid_envs = (unsigned)((a.st.num_envs + kCompactWarps - 1) / kCompactWarps);
  if (wk.marks) MARLSC_CUDA(cudaEventRecord(wk.marks[0], s));
  {
    const bool policy = !io.actions && !io.action_qty;
    const size_t img = (size_t)8 * a.ds.L * a.ds.S;
#define MARLSC_PLACE_L(LT)                                                                                          \
  case LT:                                                                                                          \
    if (policy) compact_place_kernel<MS, true, LT><<<grid_rows, 256, img, s>>>(a.ds, a.st, io, wk.cost_rows, t, m);  \
    else compact_place_kernel<MS, false, LT><<<grid_rows, 256, img, s>>>(a.ds, a.st, io, wk.cost_rows, t, m);        \
    break;
    if (stats) {
      if (policy) compact_place_kernel<MS, true, 0, true><<<grid_rows, 256, img, s>>>(a.ds, a.st, io, wk.cost_rows, t, m);
      else compact_place_kernel<MS, false, 0, true><<<grid_rows, 256, img, s>>>(a.ds, a.st, io, wk.cost_rows, t, m);
    } else switch (a.ds.L) {
      MARLSC_PLACE_L(1) MARLSC_PLACE_L(2) MARLSC_PLACE_L(3) MARLSC_PLACE_L(4) MARLSC_PLACE_L(5) MARLSC_PLACE_L(6)
      MARLSC_PLACE_L(7) MARLSC_PLACE_L(8) MARLSC_PLACE_L(9) MARLSC_PLACE_L(10) MARLSC_PLACE_L(11) MARLSC_PLACE_L(12)
      MARLSC_PLACE_L(13) MARLSC_PLACE_L(14) MARLSC_PLACE_L(15) MARLSC_PLACE_L(16)
      default:
        if (policy) compact_place_kernel<MS, true, 0><<<grid_rows, 256, img, s>>>(a.ds, a.st, io, wk.cost_rows, t, m);
        else compact_place_kernel<MS, false, 0><<<grid_rows, 256, img, s>>>(a.ds, a.st, io, wk.cost_rows, t, m);
    }
#undef MARLSC_PLACE_L
  }
  MARLSC_CUDA(cudaGetLastError());
  if (wk.marks) MARLSC_CUDA(cudaEventRecord(wk.marks[1], s));
  if (stats) compact_alloc_kernel<NCH, FS, true><<<grid_envs, kCompactWarps * 32, smem, s>>>(a.ds, a.st, io, lay, wk.cost_alloc, t, m);
  else compact_alloc_kernel<NCH, FS><<<grid_envs, kCompactWarps * 32, smem, s>>>(a.ds, a.st, io, lay, wk.cost_alloc, t, m);
  MARLSC_CUDA(cudaGetLastError());
  if (wk.marks) MARLSC_CUDA(cudaEventRecord(wk.marks[2], s));
  const int agent_scope = a.ds.scope == MARLSC_SCOPE_AGENT;
  // bulk-copy version when an environment's blocks are 16-byte granular (W S a multiple of 8) and aligned
  const auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; };
  const size_t feat_smem = (size_t)kFeatStages * (1 + kWindow) * 2 * a.ds.W * a.ds.S + 16 * kFeatStages;
  if (!stats && a.ds.feature_bulk && al16(a.st.inventory) && al16(a.st.demand_hist) && (int)feat_smem <= a.max_smem_optin) {
    static int feat_configured[kMaxDevices] = {0};
    int sms = 0;
    MARLSC_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    if (dev >= kMaxDevices || feat_configured[dev] < (int)feat_smem) {
      MARLSC_CUDA(cudaFuncSetAttribute((const void*)compact_feature_bulk_kernel<MS>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                       (int)cudaSharedmemCarveoutMaxShared));
      MARLSC_CUDA(cudaFuncSetAttribute((const void*)compact_feature_bulk_kernel<MS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)feat_smem));
      if (dev < kMaxDevices) feat_configured[dev] = (int)feat_smem;
    }
    const int per_sm = imax_host(1, imin_host((int)(220 * 1024 / feat_smem), 2048 / (32 * a.ds.W)));
    const unsigned grid_feat = (unsigned)std::min<int64_t>(a.st.num_envs, (int64_t)sms * per_sm);
    compact_feature_bulk_kernel<MS><<<grid_feat, 32 * a.ds.W, feat_smem, s>>>(a.ds, a.st, io, wk.cost_rows, wk.cost_alloc, t, agent_scope);
  } else if (stats) {
    compact_feature_kernel<MS, true><<<grid_rows, 256, (size_t)8 * 3 * a.ds.S * sizeof(float), s>>>(a.ds, a.st, io, wk.cost_rows, wk.cost_alloc,
                                                                                                   t, agent_scope, m);
  } else {
    compact_feature_kernel<MS><<<grid_rows, 256, (size_t)8 * 3 * a.ds.S * sizeof(float), s>>>(a.ds, a.st, io, wk.cost_rows, wk.cost_alloc, t,
                                                                                             agent_scope, m);
  }
  MARLSC_CUDA(cudaGetLastError());
  if (wk.marks) MARLSC_CUDA(cudaEventRecord(wk.marks[3], s));
  if (!agent_scope) {                                 // team rewards need the sum over an environment's rows
    env_reward_kernel<<<(unsigned)((a.st.num_envs + 255) / 256), 256, 0, s>>>(a.ds, a.st.num_envs, wk.cost_alloc, wk.cost_rows,
                                                                             io.rewards, io.truncated, t);
    MARLSC_CUDA(cudaGetLastError());
  }
  if (wk.marks) MARLSC_CUDA(cudaEventRecord(wk.marks[4], s));
  g_launches.fetch_add(agent_scope ? 3 : 4, std::memory_order_relaxed);
  return MARLSC_OK;
}

template <int NCH, bool MS>
int launch_split_fs(const LaunchArgs& a, const marlsc_step_io_t& io, const SplitWork& wk, int t, cudaStream_t s) {
  switch (a.ds.S / 32) {
    case 1: return launch_split_nch<NCH, MS, 1>(a, io, wk, t, s);
    case 2: return launch_split_nch<NCH, MS, 2>(a, io, wk, t, s);
    case 3: return launch_split_nch<NCH, MS, 3>(a, io, wk, t, s);
    default: return launch_split_nch<NCH, MS, 4>(a, io, wk, t, s);
  }
}

template <int NCH, bool MS>
int launch_step_fs(const LaunchArgs& a, const marlsc_step_io_t& io, int t, cudaStream_t s) {
  switch (a.ds.S / 32) {                              // compact layouts have 32 < S <= 128
    case 1: return launch_step_nch<NCH, MS, 1>(a, io, t, s);
    case 2: return launch_step_nch<NCH, MS, 2>(a, io, t, s);
    case 3: return launch_step_nch<NCH, MS, 3>(a, io, t, s);
    default: return launch_step_nch<NCH, MS, 4>(a, io, t, s);
  }
}

}  // namespace

int launch_step_compact(const LaunchArgs& a, const marlsc_step_io_t& io, int t, cudaStream_t s) {
  const bool ms = a.ds.norm == MARLSC_NORM_MEANSTD;
  switch (a.ds.perm5_chunks) {
    case 1: return ms ? launch_step_fs<1, true>(a, io, t, s) : launch_step_fs<1, false>(a, io, t, s);
    case 2: return ms ? launch_step_fs<2, true>(a, io, t, s) : launch_step_fs<2, false>(a, io, t, s);
    case 3: return ms ? launch_step_fs<3, true>(a, io, t, s) : launch_step_fs<3, false>(a, io, t, s);
    case 4: return ms ? launch_step_fs<4, true>(a, io, t, s) : launch_step_fs<4, false>(a, io, t, s);
    default: return set_error(MARLSC_EUNSUPPORTED, "compact step needs W <= 16");
  }
}

int launch_split_compact(const LaunchArgs& a, const marlsc_step_io_t& io, const SplitWork& wk, int t, cudaStream_t s) {
  const bool ms = a.ds.norm == MARLSC_NORM_MEANSTD;
  switch (a.ds.perm5_chunks) {
    case 1: return ms ? launch_split_fs<1, true>(a, io, wk, t, s) : launch_split_fs<1, false>(a, io, wk, t, s);
    case 2: return ms ? launch_split_fs<2, true>(a, io, wk, t, s) : launch_split_fs<2, false>(a, io, wk, t, s);
    case 3: return ms ? launch_split_fs<3, true>(a, io, wk, t, s) : launch_split_fs<3, false>(a, io, wk, t, s);
    case 4: return ms ? launch_split_fs<4, true>(a, io, wk, t, s) : launch_split_fs<4, false>(a, io, wk, t, s);
    default: return set_error(MARLSC_EUNSUPPORTED, "compact step needs W <= 16");
  }
}

int launch_reset_compact(const LaunchArgs& a, const int32_t* init, int per_env, float* obs, cudaStream_t s) {
  const long long n = a.st.num_envs * (long long)a.ds.W * a.ds.S;
  env_reset_compact_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(a.ds, a.st, init, per_env, obs);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  MARLSC_CUDA(cudaGetLastError());
  return MARLSC_OK;
}

int launch_base_stock_compact(const DevSpec& ds, const marlsc_env_state_t& st, const float* level, int level_per_env, int t,
                              float* actions, cudaStream_t s) {
  (void)t;
  const long long n = st.num_envs * (long long)ds.W * ds.S;
  const unsigned grid = (unsigned)((n + 255) / 256);
  if (n < (1LL << 32)) base_stock_compact_kernel<unsigned><<<grid, 256, 0, s>>>(ds, st, level, level_per_env, actions);
  else base_stock_compact_kernel<long long><<<grid, 256, 0, s>>>(ds, st, level, level_per_env, actions);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  MARLSC_CUDA(cudaGetLastError());
  return MARLSC_OK;
}

int launch_lines_from_orders(const DevSpec& ds, int64_t num_envs, const marlsc_step_io_t& io, int32_t line_stride, uint16_t* lines,
                             int32_t* line_counts, int32_t* overflow, cudaStream_t s) {
  lines_from_orders_kernel<<<(unsigned)((num_envs + 3) / 4), 128, 0, s>>>(ds, num_envs, io, line_stride, lines, line_counts, overflow);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  MARLSC_CUDA(cudaGetLastError());
  return MARLSC_OK;
}

}  // namespace marlsc
