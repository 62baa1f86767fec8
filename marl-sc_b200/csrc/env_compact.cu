// env_compact.cu - environment step (K1a' place, K1b' allocate, K1c' features, K1d rewards), reset, base-stock policy
// and order -> line conversion over the compact state layout (see env_compact.cuh for the design notes).
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
namespace {

constexpr unsigned FULL = 0xffffffffu;
constexpr int kSlots = kCompactMaxS / 32;   // SKU slots per lane

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
__device__ __forceinline__ void prefetch_l2_bulk(const void* p, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}

__device__ __forceinline__ uint32_t ld_nc_u32(const uint32_t* p) { uint32_t v; asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(v) : "l"(p)); return v; }
__device__ __forceinline__ void ld_nc_u32_if(uint32_t& v, const uint32_t* p, bool c) {   // v = *p when c, else v stays
  asm volatile("{ .reg .pred q; setp.ne.u32 q, %2, 0; @q ld.global.nc.u32 %0, [%1]; }" : "+r"(v) : "l"(p), "r"((uint32_t)c));
}

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
  __device__ __forceinline__ void pop() {         // selects rather than a branch: nearly every trip some lane of the warp refills
    cur >>= 16;
    const bool adv = cur == 0u;
    cur = adv ? w1 : cur;
    w1 = adv ? w2 : w1;
    w2 = adv ? w3 : w2;
    w3 = adv ? 0u : w3;
    ld_nc_u32_if(w3, base + at, adv && at < n);
    at += adv ? 32u : 0u;
  }
};

// Each byte of x replaced by its top bit replicated: 0xff or 0 (prmt's sign-replicating selectors; __byte_perm
// documents only the byte-copying ones).
__device__ __forceinline__ uint32_t byte_signs(uint32_t x) { uint32_t r; asm("prmt.b32 %0, %1, 0, 0xBA98;" : "=r"(r) : "r"(x)); return r; }

// Byte `slot` of a map word.
__device__ __forceinline__ uint32_t map_sku(uint32_t map, uint32_t slot) { return __byte_perm(map, 0u, 0x4440u + slot); }

// Availability masks of a lane's SKUs from the staged stock [W,S] uint16 at shared address a_inv: bit w + 16 (k & 1) of
// (k & 2 ? avhi : avlo) says warehouse w holds the SKU of slot k. The map word is rewritten to byte k = 2 x the SKU of
// slot k (the byte offset of its cell in a stock row; S <= 128). Map bytes that name no SKU (255, or anything >= S in a
// malformed stream) are pointed at SKU S-1 with an empty mask: their lines, if any, count as lost and leave the stock
// alone (the home demand of such lines lands on SKU S-1, whose owner is another lane: the result is undefined, as for
// any stream that breaks the one-owner rule of marlsc_step_io.lines).
__device__ __forceinline__ void owner_masks(uint32_t& map, uint32_t a_inv, int W, int S, uint32_t& avlo, uint32_t& avhi) {
  avlo = avhi = 0u;
  uint32_t fixed = 0u;
#pragma unroll
  for (int k = 0; k < kSlots; ++k) {
    uint32_t sku = (map >> (8 * k)) & 0xffu;
    const bool named = sku < (uint32_t)S;
    if (!named) sku = (uint32_t)S - 1u;
    fixed |= (2u * sku) << (8 * k);
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
// of the SKUs named by the lane's map belong to this lane alone for the duration of the chains, and so do the cells
// (w, s) of this step's home-region demand plane [W,S] uint16 that follows the stock image: plain loads and stores.
// Everything a trip needs of its line is worked out once when the line is taken: the shared addresses of the SKU's
// stock cell in warehouse 0, of the region's entry in row 0 of the shipped-unit table and of the region's record
// (compact_region_bytes). From those a shipment is one multiply-add by a row stride (a launch constant) per table.
// PEN_UNIFORM: every SKU carries the same lost-sales penalty rate, so lost units are enough (else an fp64
// shared-memory add per lost line).
constexpr uint32_t kHomeNone = 0xffffu, kHomeSeveral = 0xfffeu;   // home-table entries besides a plane offset

template <int NCH, bool PEN_UNIFORM>
__device__ __forceinline__ void allocation_chains(const DevSpec& sp, const CompactSmem& lay, LineStream& ls, uint32_t a_reg0,
                                                  uint32_t a_inv, uint32_t a_shipq, uint32_t a_lostP, uint32_t& avlo,
                                                  uint32_t& avhi) {
  constexpr uint32_t kPrio = NCH * 64, kHome = NCH * 64 + 16;     // offsets inside a region record
  const uint32_t map = ls.map;
  // the current line: units left, candidate warehouses (priority order), 16 x its SKU slot (the slot's first bit in
  // avhi:avlo), stock cell in warehouse 0, shipped units of the region at warehouse 0, the region's record
  uint32_t rem = 0u, cand = 0u, sl16 = 0u, a_cell = 0u, a_sq = 0u, a_reg = 0u;
  while (true) {
    const uint32_t n0 = ls.next();
    if (rem == 0u && n0 != 0u) {
      ls.pop();
      rem = n0 & 0xffu;
      const uint32_t r = (n0 >> 8) & 0x3fu;
      sl16 = (n0 >> 10) & 0x30u;
      a_cell = a_inv + map_sku(map, n0 >> 14);
      a_sq = a_shipq + 4u * r;
      a_reg = a_reg0 + r * (uint32_t)compact_region_bytes(NCH);
      // which warehouses hold the SKU (bit w), then the same bits in the region's priority order
      const uint32_t am = ((sl16 & 32u ? avhi : avlo) >> (sl16 & 16u)) & 0xffffu;
      cand = ld_s_u16(a_reg + 2u * (am & 31u));
      if (NCH > 1) cand |= ld_s_u16(a_reg + 64u + 2u * ((am >> 5) & 31u));
      if (NCH > 2) cand |= ld_s_u16(a_reg + 128u + 2u * ((am >> 10) & 31u));
      if (NCH > 3) cand |= ld_s_u16(a_reg + 192u + 2u * ((am >> 15) & 31u));
      // home-region demand of this step (multi_env.py:763-768): the entry is the offset of the home warehouse's history
      // cell from the stock cell
      const uint32_t ho = ld_s_u16(a_reg + kHome);
      if (ho < kHomeSeveral) {
        st_s_u16(a_cell + ho, ld_s_u16(a_cell + ho) + rem);
      } else if (ho == kHomeSeveral) {
        const uint32_t h0 = (uint32_t)(lay.hist - lay.inv);
        for (uint32_t hm = sp.home_mask[r]; hm; hm &= hm - 1) {
          const uint32_t c = a_cell + h0 + (uint32_t)lowest_bit(hm) * (uint32_t)lay.inv_row;
          st_s_u16(c, ld_s_u16(c) + rem);
        }
      }
    }
    if (rem != 0u) {
      if (cand != 0u) {                               // ship from the cheapest warehouse that has the SKU
        const uint32_t v = (uint32_t)lowest_bit(cand);
        cand &= cand - 1;
        const uint32_t w = ld_s_u8(a_reg + kPrio + v);
        const uint32_t cell = a_cell + w * (uint32_t)lay.inv_row;
        const uint32_t a = ld_s_u16(cell);            // the cells of a SKU belong to this lane
        const uint32_t f = rem < a ? rem : a;
        st_s_u16(cell, a - f);
        red_s_add(a_sq + w * (uint32_t)lay.shipq_row, f);
        rem -= f;
        if (a == f) {                                 // emptied
          const uint32_t b = w + sl16;
          if (b & 32u) avhi &= ~(1u << (b & 31u)); else avlo &= ~(1u << (b & 31u));
        }
      }
      if (rem != 0u && cand == 0u) {
        // no warehouse can supply the rest: lost (demand_allocator.py:205-208)
        red_s_add(a_sq + (uint32_t)lay.lost_off, rem);
        if (!PEN_UNIFORM) red_s_add_f64(a_lostP + 2u * (a_sq - a_shipq), (double)rem * sp.pen_rate[(a_cell - a_inv) >> 1]);
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
// The step as three row / environment kernels and the reward kernel (K1a' .. K1d), cut along the data dependencies: the
// two streaming parts run as short-lived warps, one per (environment, warehouse) row with every load of the row in flight
// at once, and only the allocation keeps an environment's stock in shared memory. The same step as one fused kernel kept
// the stock there from the first row to the last, which held it to 32 warps per SM, and at that residency every one of
// its ~30 dependent memory round trips per env-step showed (ncu: 13 warps per issue slot waiting on the long scoreboard,
// 35-40 % issue utilisation, 25-30 % of DRAM bandwidth; 2.7 to 3.9 ms per step at 65,536 large environments against
// 1.73 ms split, DESIGN.md section 4).
// ---------------------------------------------------------------------------------------------------------------

// SKU slot k of a lane is valid: always below FS (= S / 32, compile time), for lanes below the remainder at FS, never above
#define VALID(k) ((k) < FS || ((k) == FS && tail))

// K1a': one warp per (environment, warehouse) row - order quantities, arrivals, the new orders into the ring, pipeline
// block of the observation row; the row's inbound cost goes to cost_rows.
// The ring is indexed by placement time (marlsc_env_state): at step t plane (t - a) % L holds the orders placed a steps
// ago, age a = 1 .. L (age L is plane t % L, the one this step overwrites). A cell with lead l receives its order of age
// l, and pipeline slot k of the observation (what arrives at t + 1 + k, multi_env.py:941-968) is its order of age
// l - 1 - k, the new one being age 0, or 0 for k >= l.
// Loads: lane q reads the four consecutive cells 4q .. 4q+3 of the row in each of the L planes (vector loads, all in
// flight at once). The (age, byte) pairs are then scattered to an image of the pipeline block in shared memory, [L][S] in
// slot order, that L scratch slots precede: age a of a cell goes to slot l - 1 - a, so the ages that are no longer in
// transit land in the scratch and slot -1 receives the arrival. Only the new orders go back to the ring - one 32-bit
// word per lane into plane t % L, a contiguous W x S block per environment - and the image goes to the observation as
// floats, lane l taking bytes l + 32 j so that every store instruction covers 128 consecutive bytes.
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
  extern __shared__ __align__(16) unsigned char smem[];           // [8 warps][2L * S]: L scratch slots, then the L pipeline slots
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
  // 32-bit word offsets inside the ring: plane p of the row is p * WS4 words from the row's word in plane 0
  const int WS4 = WS >> 2, LWS4 = L * WS4, po_new = (t % L) * WS4;
  uint32_t* const row4 = reinterpret_cast<uint32_t*>(static_cast<uint8_t*>(st.ring_qty) + e * L * WS + (int64_t)w * S) + c4;
  // every load of the row first
  float4 a4 = make_float4(0.f, 0.f, 0.f, 0.f);
  uint32_t aqw = 0u, le4 = 0x01010101u;
  uint2 iv = make_uint2(0u, 0u);
  uint2* const inv4 = reinterpret_cast<uint2*>(static_cast<uint16_t*>(st.inventory) + e * WS + w * S) + c4;
  uint32_t x[KMAX];                                   // x[a - 1]: the four cells' orders of age a
  if (mine) {
    if (io.action_qty) aqw = reinterpret_cast<const uint32_t*>(io.action_qty + e * WS + w * S)[c4];
    else if (io.actions) a4 = reinterpret_cast<const float4*>(io.actions + e * WS + w * S)[c4];
    iv = *inv4;
    le4 = reinterpret_cast<const uint32_t*>(sp.lead_u8 + w * S)[c4];
    int po = po_new;
#pragma unroll
    for (int a = 1; a <= KMAX; ++a)
      if (a <= L) {                                   // plane (t - a) % L, walked with one subtraction per age
        po = (po == 0 ? LWS4 : po) - WS4;
        x[a - 1] = row4[po];
      }
  }
  constexpr bool policy = POLICY;                     // base-stock heuristic in place of given actions (marlsc_step_io.base_stock_level)
  float4 lv4 = make_float4(0.f, 0.f, 0.f, 0.f);
  if (policy && mine)
    lv4 = reinterpret_cast<const float4*>(io.base_stock_level + (io.base_stock_per_env ? e * WS : 0) + w * S)[c4];
  const uint32_t img = sm_addr(smem) + (threadIdx.x >> 5) * (uint32_t)(2 * L * S) + (uint32_t)(L * S);   // pipeline slot 0
  const uint32_t col = img + 4u * (uint32_t)lane;     // the lane's four cells in slot 0
  uint32_t arr4 = 0u;
  if (mine) {
    // slots at or past a cell's lead hold nothing: zero the lane's word of every slot, then scatter ages 1 .. L
#pragma unroll
    for (int k = 0; k < KMAX; ++k)
      if (k < L) asm volatile("st.shared.u32 [%0], %1;" ::"r"(col + (uint32_t)(k * S)), "r"(0u) : "memory");
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int le = (int)((le4 >> (8 * j)) & 0xffu);
      uint32_t adr = col + (uint32_t)((le - 2) * S + j);                  // slot le - 1 - a of age a = 1
#pragma unroll
      for (int a = 1; a <= KMAX; ++a)
        if (a <= L) {
          asm volatile("st.shared.u8 [%0], %1;" ::"r"(adr), "r"(x[a - 1] >> (8 * j)) : "memory");
          adr -= (uint32_t)S;
        }
    }
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(arr4) : "r"(col - (uint32_t)S));   // slot -1: the arrivals (age = lead)
  }
  float af[4] = {a4.x, a4.y, a4.z, a4.w};
  const uint32_t ivv[4] = {iv.x & 0xffffu, iv.x >> 16, iv.y & 0xffffu, iv.y >> 16};
  if (policy && mine) {
    // reference make_bs_newsvendor_action_fn (run_baselines.py:188-207): order up to the level given on-hand stock and
    // everything in transit - ages 1 .. lead, the arrivals of this step included (the policy acts before them). Summed
    // from the registers, four cells at a time: byte b of (leads | 0x80 per byte) - a keeps its top bit exactly when
    // lead_b >= a (leads <= 16, no borrow crosses a byte), and the sign-replicating byte permute turns that bit into the
    // byte's mask. Bytes 0, 2 and 1, 3 add up in 16-bit halves (at most 16 x 255).
    uint32_t p02 = 0u, p13 = 0u;
#pragma unroll
    for (int a = 1; a <= KMAX; ++a)
      if (a <= L) {
        const uint32_t v = x[a - 1] & byte_signs((le4 | 0x80808080u) - 0x01010101u * (uint32_t)a);
        p02 += __byte_perm(v, 0u, 0x4240u);
        p13 += __byte_perm(v, 0u, 0x4341u);
      }
    const uint32_t pend[4] = {p02 & 0xffffu, p13 & 0xffffu, p02 >> 16, p13 >> 16};
    const float lv[4] = {lv4.x, lv4.y, lv4.z, lv4.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const double mxd = sp.action_max[4 * lane + j];
      double qd = (double)lv[j] - (double)ivv[j] - (double)pend[j];
      qd = qd < 0.0 ? 0.0 : (qd > mxd ? mxd : qd);
      af[j] = (float)(2.0 * qd / mxd - 1.0);
    }
  }
  uint32_t ni[4], qw = 0u;
  int nQ = 0, nPos = 0;
  double inb = 0.0;
  const bool by_row = sp.row_rates_uniform != 0;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int le = (int)((le4 >> (8 * j)) & 0xffu);
    int q = 0;
    if (mine) {
      const int mxj = (int)sp.action_max[4 * lane + j];
      q = io.action_qty ? imin((int)((aqw >> (8 * j)) & 0xffu), mxj) : rescale_action<kCapsLean>(sp, af[j], (double)mxj, 0, 0);
      if (q > 0) asm volatile("st.shared.u8 [%0], %1;" ::"r"(col + (uint32_t)((le - 1) * S + j)), "r"(q) : "memory");   // age 0
    }
    qw |= (uint32_t)q << (8 * j);
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
    row4[po_new] = qw;                                // every cell, 0 included: the plane held the orders of age L
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
  const bool need_hist = sp.need_hist != 0;
  {
    // region records, word by word: perm5 chunks, prio16 row, home entry = the offset of the home warehouse's history
    // cell from the stock cell of the same SKU in warehouse 0 (allocation_chains), kHomeSeveral (home_mask) or
    // kHomeNone (all kHomeNone without a history plane)
    constexpr int kWords = compact_region_bytes(NCH) / 4, kPerm = NCH * 16;
    for (int i = threadIdx.x; i < R * kWords; i += blockDim.x) {
      const int r = i / kWords, j = i - r * kWords;
      uint32_t v;
      if (j < kPerm) {
        v = reinterpret_cast<const uint32_t*>(sp.perm5)[r * kPerm + j];
      } else if (j < kPerm + 4) {
        v = reinterpret_cast<const uint32_t*>(sp.prio16)[r * 4 + j - kPerm];
      } else {
        const uint32_t hw = sp.home_wh[r];
        v = !need_hist || hw == 255u ? kHomeNone : hw == 254u ? kHomeSeveral : (uint32_t)(lay.hist - lay.inv) + hw * (uint32_t)lay.inv_row;
      }
      reinterpret_cast<uint32_t*>(smem)[i] = v;
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
  uint2* const s_hist = reinterpret_cast<uint2*>(wbase + lay.hist);   // this step's home-region demand, four cells per word pair
  if (need_hist)
    for (int i = lane; i < WS / 4; i += 32) s_hist[i] = make_uint2(0u, 0u);
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
  {
    // every shared address the chains use is one of two bases plus a launch constant (the layout is a kernel parameter)
    const uint32_t a_cta = sm_addr(smem), a_warp = a_cta + (uint32_t)lay.t_bytes + (uint32_t)wid * (uint32_t)lay.warp_bytes;
    if (pen_uniform)
      allocation_chains<NCH, true>(sp, lay, ls, a_cta, a_warp + (uint32_t)lay.inv, a_warp + (uint32_t)lay.shipq, a_warp + (uint32_t)lay.lostP,
                                   avlo, avhi);
    else
      allocation_chains<NCH, false>(sp, lay, ls, a_cta, a_warp + (uint32_t)lay.inv, a_warp + (uint32_t)lay.shipq, a_warp + (uint32_t)lay.lostP,
                                    avlo, avhi);
  }
  __syncwarp();
  for (int w0 = 0; w0 < W; ++w0)                       // stock out (multi_env.py:307; never negative)
#pragma unroll
    for (int k = 0; k < kSlots; ++k)
      if (VALID(k)) g_inv[w0 * S + 32 * k] = s_inv[w0 * S + lane + 32 * k];
  if (need_hist) {                                    // every cell of this step's history plane (K1c' reads it)
    uint2* const g_hist = reinterpret_cast<uint2*>(static_cast<uint16_t*>(st.demand_hist) + (e * kWindow + t % kWindow) * (int64_t)WS);
    for (int i = lane; i < WS / 4; i += 32) g_hist[i] = s_hist[i];
  }
  // Outbound cost and lost-sales penalty of every warehouse (reward_calculator.py:134-142). Lanes take regions (two per
  // lane cover R <= 64). Per region the lost volume's cost is either spread over the warehouses in proportion to what
  // they shipped there (shipment handler, lost_sales_handler.py:113-148: a rate per shipped unit, one division per
  // region) or goes to the closest warehouse (closest handler, and the shipment handler's fallback when nothing was
  // shipped). Then warehouse by warehouse the lanes' partial sums meet in a shuffle reduction.
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
      // this step's plane, written whole by K1b': read once, from L2
      asm volatile("ld.global.cg.v2.u32 {%0, %1}, [%2];" : "=r"(hn.x), "=r"(hn.y) : "l"(reinterpret_cast<const uint2*>(hist + (t % kWindow) * WS) + c4));
#pragma unroll
      for (int back = 1; back < kWindow; ++back)
        if (back < hist_n) ho[back - 1] = reinterpret_cast<const uint2*>(hist + pmod(t - back, kWindow) * WS)[c4];
    }
  }
  float* const img = reinterpret_cast<float*>(smem) + (threadIdx.x >> 5) * (3 * S);
  // mean over the window = integer sum / n, rounded to float32 like NumPy's (multi_env.py:785-787): the product with the
  // double reciprocal is within 2^-52 of the quotient, far from every float32 rounding boundary of a quotient of integers
  // below 2^24 by n <= 5, so rounding it gives the correctly rounded float32 quotient
  const double rcp_n = 1.0 / (double)hist_n;
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
  uint8_t* ring = static_cast<uint8_t*>(st.ring_qty) + e * L * WS + i;
  for (int d = 0; d < L; ++d) ring[(long long)d * WS] = 0;
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

// K5 (compact): units in transit to a cell are its orders of age 1 .. l (l its lead, the arrivals of step t included):
// plane (t - a) % L of the placement-indexed ring for a = 1 .. l.
template <typename IDX>
__global__ void __launch_bounds__(256)
base_stock_compact_kernel(const __grid_constant__ DevSpec sp, const __grid_constant__ marlsc_env_state_t st,
                          const float* __restrict__ level, int level_per_env, int t, float* __restrict__ actions) {
  const IDX WS = (IDX)(sp.W * sp.S);
  const IDX idx = (IDX)blockIdx.x * (IDX)blockDim.x + (IDX)threadIdx.x;
  if (idx >= (IDX)st.num_envs * WS) return;
  const IDX e = idx / WS;
  const int i = (int)(idx - e * WS), s = i % sp.S;
  const int L = sp.L, lead = sp.lead_u8[i], tl = t % L + L;            // age a <= L lives in plane (tl - a) % L
  const uint8_t* ring = static_cast<const uint8_t*>(st.ring_qty) + (long long)e * L * (long long)WS + i;
  int pending = 0;
  for (int a0 = 1; a0 <= lead; a0 += 4) {
    int v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) v[k] = a0 + k <= lead ? (int)ring[(long long)((tl - a0 - k) % L) * (long long)WS] : 0;
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
int launch_split_nch(const LaunchArgs& a, const marlsc_step_io_t& io, const SplitWork& wk, int t, cudaStream_t s) {
  const CompactSmem lay = compact_smem(a.ds.W, a.ds.S, a.ds.R, NCH, a.ds.pen_uniform, a.ds.need_hist);
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
    const size_t img = (size_t)8 * 2 * a.ds.L * a.ds.S;   // per warp: L scratch slots and the L pipeline slots
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
  if (stats) {
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

}  // namespace

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
  const long long n = st.num_envs * (long long)ds.W * ds.S;
  const unsigned grid = (unsigned)((n + 255) / 256);
  if (n < (1LL << 32)) base_stock_compact_kernel<unsigned><<<grid, 256, 0, s>>>(ds, st, level, level_per_env, t, actions);
  else base_stock_compact_kernel<long long><<<grid, 256, 0, s>>>(ds, st, level, level_per_env, t, actions);
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
