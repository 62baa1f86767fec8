// spec_build.h - host-side translation of a marlsc_env_spec_t into the kernel's DevSpec:
// validation, observation block offsets (reference: multi_env.py:444-502, 619-695), the static
// warehouse priority table of the greedy allocator (demand_allocator.py:168-173) and the per-team
// shared-memory scratch layout. Pure C++ (no CUDA) so the test-only host emulation shares it.
#pragma once
#include <algorithm>
#include <cstring>
#include <string>
#include <vector>

#include "env_core.cuh"

namespace marlsc {

struct HostTables {
  std::vector<double> action_max, out_fixed, out_var, in_fixed, in_var, hold_rate, pen_rate, skw;
  std::vector<int32_t> lead_exp, home, closest, region_map;
  std::vector<uint8_t> prio, prio_static, lead_u8;
  std::vector<uint32_t> home_mask;
  std::vector<float> obs_mean, obs_std;
  // W <= 16: warehouse-availability bits (bit w) -> the same bits in region r's priority order (bit v = the v-th
  // cheapest warehouse), four warehouse bits per lookup: [R][perm_chunks][16] (env_alloc.cuh)
  std::vector<uint16_t> prio_perm;
  // compact layout (env_compact.cu): [R][ceil(W/5)][32] availability -> priority-order bits, [R][16] priority rows,
  // [R] home warehouse of a region (255 none, 254 several)
  std::vector<uint16_t> perm5;
  std::vector<uint8_t> prio16, home_wh;
};

inline int pow2ceil(int v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}

// Lanes per environment chosen for S SKUs: one thread for tiny SKU counts, a warp slice otherwise.
inline int auto_team_size(int S) {
  if (S <= 8) return 1;
  if (S <= 16) return 4;
  if (S <= 32) return 8;
  if (S <= 64) return 16;
  return 32;
}

// SKUs per lane (power of two) for a team of G lanes.
inline int skus_per_lane(int S, int G) { return pow2ceil((S + G - 1) / G); }

// Fills ds (pointers left null) and tabs. Returns an empty string on success, else the error text.
inline std::string build_devspec(const marlsc_env_spec_t& sp, DevSpec& ds, HostTables& tb) {
  std::memset(&ds, 0, sizeof(ds));
  if (sp.abi_version != MARLSC_ABI_VERSION) return "abi_version mismatch";
  const int W = sp.n_warehouses, S = sp.n_skus, R = sp.n_regions;
  if (W < 1 || S < 1 || R < 1) return "n_warehouses, n_skus and n_regions must be positive";
  if (W > 255) return "n_warehouses > 255 is not supported";
  if (R > 32767) return "n_regions > 32767 is not supported";
  if (sp.episode_length < 1) return "episode_length must be positive";
  if (sp.max_expected_lead < 1) return "max_expected_lead must be >= 1";
  if (sp.ring_depth < sp.max_expected_lead || sp.ring_depth > 255) return "ring_depth must be in [max_expected_lead, 255]";
  if (sp.action_type < 0 || sp.action_type > 2) return "unknown action_type";
  if (sp.lead_mode < 0 || sp.lead_mode > 1) return "unknown lead_mode";
  if (sp.lost_sales_type < 0 || sp.lost_sales_type > 2) return "unknown lost_sales_type";
  if (sp.reward_scope < 0 || sp.reward_scope > 1) return "unknown reward_scope";
  if (sp.obs_norm < 0 || sp.obs_norm > 2) return "unknown obs_norm";
  if (sp.max_splits < 0) return "max_splits must be >= 0";
  if (!(sp.feature_mask & MARLSC_F_INVENTORY) || !(sp.feature_mask & MARLSC_F_PIPELINE))
    return "inventory and pipeline features must always be enabled";   // schema.py:624-630
  const uint32_t F = sp.feature_mask;
  const struct { uint32_t parent, agg; const char* name; } pairs[] = {   // schema.py:632-639
      {MARLSC_F_INVENTORY, MARLSC_F_INVENTORY_AGG, "inventory_aggregate"},
      {MARLSC_F_PIPELINE, MARLSC_F_PIPELINE_AGG, "pipeline_aggregate"},
      {MARLSC_F_DEMAND_HOME, MARLSC_F_DEMAND_HOME_AGG, "incoming_demand_home_aggregate"},
      {MARLSC_F_SHIPPED_AWAY, MARLSC_F_SHIPPED_AWAY_AGG, "units_shipped_away_aggregate"},
      {MARLSC_F_ROLLING_MEAN, MARLSC_F_ROLLING_MEAN_AGG, "rolling_demand_mean_aggregate"},
      {MARLSC_F_FORECAST, MARLSC_F_FORECAST_AGG, "demand_forecast_aggregate"}};
  for (const auto& pr : pairs)
    if ((F & pr.agg) && !(F & pr.parent)) return std::string(pr.name) + " needs its parent feature";
  if (!sp.action_max || !sp.out_fixed || !sp.out_var || !sp.in_fixed || !sp.in_var || !sp.hold_rate ||
      !sp.pen_rate || !sp.sku_weights || !sp.expected_lead || !sp.home_region || !sp.closest_wh)
    return "a required table pointer is NULL";
  if (sp.lost_sales_type == MARLSC_LOST_COST && !(sp.lost_alpha > 0.0)) return "lost_alpha must be > 0";
  const int Rraw = sp.region_map ? sp.n_regions_raw : R;
  if (Rraw < 1 || Rraw > 32767) return "n_regions_raw out of range";

  tb.action_max.assign(sp.action_max, sp.action_max + S);
  tb.out_fixed.assign(sp.out_fixed, sp.out_fixed + W * R);
  tb.out_var.assign(sp.out_var, sp.out_var + W * R);
  tb.in_fixed.assign(sp.in_fixed, sp.in_fixed + W * S);
  tb.in_var.assign(sp.in_var, sp.in_var + W * S);
  tb.hold_rate.assign(sp.hold_rate, sp.hold_rate + S);
  tb.pen_rate.assign(sp.pen_rate, sp.pen_rate + S);
  tb.skw.assign(sp.sku_weights, sp.sku_weights + S);
  tb.lead_exp.assign(sp.expected_lead, sp.expected_lead + W * S);
  tb.home.assign(sp.home_region, sp.home_region + W);
  tb.closest.assign(sp.closest_wh, sp.closest_wh + R);
  tb.region_map.clear();
  if (sp.region_map) tb.region_map.assign(sp.region_map, sp.region_map + Rraw);
  int lmax = 0;
  for (int v : tb.lead_exp) {
    if (v < 1) return "expected lead times must be >= 1";
    lmax = std::max(lmax, v);
  }
  if (lmax != sp.max_expected_lead) return "max_expected_lead does not match expected_lead";
  for (int v : tb.home) if (v < 0 || v >= R) return "home_region out of range";
  for (int v : tb.closest) if (v < 0 || v >= W) return "closest_wh out of range";
  for (int v : tb.region_map) if (v < 0 || v >= R) return "region_map entry out of range";

  // static priority: when the fixed cost column is constant the order never depends on the weight
  const int Wp = (W + 3) & ~3;                                   // priority rows are padded to whole 32-bit words
  tb.prio.assign((size_t)R * Wp, 0);
  tb.prio_static.assign(R, 0);
  for (int r = 0; r < R; ++r) {
    bool constant = true;
    for (int w = 1; w < W; ++w) constant = constant && tb.out_fixed[w * R + r] == tb.out_fixed[r];
    tb.prio_static[r] = constant ? 1 : 0;
    std::vector<int> idx(W);
    for (int w = 0; w < W; ++w) idx[w] = w;
    std::stable_sort(idx.begin(), idx.end(), [&](int a, int b) { return tb.out_var[a * R + r] < tb.out_var[b * R + r]; });
    for (int w = 0; w < W; ++w) tb.prio[(size_t)r * Wp + w] = (uint8_t)idx[w];
  }
  tb.prio_perm.clear();
  ds.perm_chunks = 0;
  if (W <= 16) {
    const int nc = (W + 3) / 4;
    ds.perm_chunks = nc;
    tb.prio_perm.assign((size_t)R * nc * 16, 0);
    for (int r = 0; r < R; ++r)
      for (int v = 0; v < W; ++v) {
        const int w = tb.prio[(size_t)r * Wp + v];
        for (int m = 0; m < 16; ++m)
          if ((m >> (w % 4)) & 1) tb.prio_perm[((size_t)r * nc + w / 4) * 16 + m] |= (uint16_t)(1u << v);
      }
  }
  tb.perm5.clear();
  tb.prio16.clear();
  ds.perm5_chunks = 0;
  if (W <= 16) {
    const int nc = (W + 4) / 5;
    ds.perm5_chunks = nc;
    tb.perm5.assign((size_t)R * nc * 32, 0);
    tb.prio16.assign((size_t)R * 16, 0);
    for (int r = 0; r < R; ++r)
      for (int v = 0; v < W; ++v) {
        const int w = tb.prio[(size_t)r * Wp + v];
        tb.prio16[(size_t)r * 16 + v] = (uint8_t)w;
        for (int m = 0; m < 32; ++m)
          if ((m >> (w % 5)) & 1) tb.perm5[((size_t)r * nc + w / 5) * 32 + m] |= (uint16_t)(1u << v);
      }
  }
  tb.home_wh.assign(R, 255);
  for (int w = 0; w < W; ++w) {
    uint8_t& h = tb.home_wh[tb.home[w]];
    h = h == 255 ? (uint8_t)w : (uint8_t)254;
  }
  ds.pen_uniform = 1;
  for (int s = 1; s < S; ++s) ds.pen_uniform = ds.pen_uniform && tb.pen_rate[s] == tb.pen_rate[0];
  // holding and inbound rates that do not vary over the SKUs of a warehouse row: K1c sums integers per row
  ds.row_rates_uniform = 1;
  for (int s = 1; s < S; ++s) ds.row_rates_uniform = ds.row_rates_uniform && tb.hold_rate[s] == tb.hold_rate[0] && tb.skw[s] == tb.skw[0];
  for (int w = 0; w < W; ++w)
    for (int s = 1; s < S; ++s)
      ds.row_rates_uniform = ds.row_rates_uniform && tb.in_fixed[w * S + s] == tb.in_fixed[w * S] && tb.in_var[w * S + s] == tb.in_var[w * S];

  tb.home_mask.clear();
  if (W <= 32) {
    tb.home_mask.assign(R, 0u);
    for (int w = 0; w < W; ++w) tb.home_mask[tb.home[w]] |= (1u << w);
  }
  tb.lead_u8.resize((size_t)W * S);
  for (int i = 0; i < W * S; ++i) {
    if (tb.lead_exp[i] > 255) return "expected lead times above 255 are not supported";
    tb.lead_u8[i] = (uint8_t)tb.lead_exp[i];
  }
  bool unit = true;
  for (double v : tb.skw) unit = unit && (v == 1.0);

  ds.W = W; ds.S = S; ds.R = R; ds.Rraw = Rraw;
  ds.unit_weights = unit ? 1 : 0;
  ds.L = sp.max_expected_lead; ds.D = sp.ring_depth; ds.episode_length = sp.episode_length;
  ds.action_type = sp.action_type; ds.lead_mode = sp.lead_mode; ds.lost_type = sp.lost_sales_type;
  ds.scope = sp.reward_scope; ds.max_splits = sp.max_splits; ds.norm = sp.obs_norm;
  ds.id_off = sp.include_warehouse_id ? W : 0;
  ds.feat = F; ds.scale = sp.scale_factor; ds.alpha = sp.lost_alpha > 0.0 ? sp.lost_alpha : 1.0;
  ds.need_ship = (F & (MARLSC_F_SHIPPED_HOME | MARLSC_F_SHIPPED_AWAY | MARLSC_F_STOCKOUT)) ? 1 : 0;
  ds.need_hist = ((F & (MARLSC_F_ROLLING_MEAN | MARLSC_F_DAYS_OF_SUPPLY | MARLSC_F_DEMAND_VARIABILITY |
                        MARLSC_F_DEMAND_HISTORY)) || sp.action_type != MARLSC_ACTION_DIRECT) ? 1 : 0;
  ds.need_fcst = (F & (MARLSC_F_FORECAST | MARLSC_F_NET_INV_POSITION)) ? 1 : 0;
  const bool need_dh = ds.need_hist || (F & (MARLSC_F_DEMAND_HOME | MARLSC_F_STOCKOUT));
  ds.dh_mode = ds.need_hist ? 1 : (need_dh ? 2 : 0);
  ds.has_fixed = 0;
  for (double v : tb.out_fixed) if (v != 0.0) ds.has_fixed = 1;

  // observation layout, block order of multi_env.py:619-695
  int o = 0;
  auto block = [&](bool on, int n, bool agg) { int at = -1; if (on) { at = o; o += n + (agg ? 1 : 0); } return at; };
  ds.off_inv = block(true, S, F & MARLSC_F_INVENTORY_AGG);
  ds.off_pipe = block(true, ds.L * S, F & MARLSC_F_PIPELINE_AGG);
  ds.off_dh = block(F & MARLSC_F_DEMAND_HOME, S, F & MARLSC_F_DEMAND_HOME_AGG);
  ds.off_sh = block(F & MARLSC_F_SHIPPED_HOME, S, false);
  ds.off_sa = block(F & MARLSC_F_SHIPPED_AWAY, S, F & MARLSC_F_SHIPPED_AWAY_AGG);
  ds.off_so = block(F & MARLSC_F_STOCKOUT, S, false);
  ds.off_rm = block(F & MARLSC_F_ROLLING_MEAN, S, F & MARLSC_F_ROLLING_MEAN_AGG);
  ds.off_fc = block(F & MARLSC_F_FORECAST, S, F & MARLSC_F_FORECAST_AGG);
  ds.off_dos = block(F & MARLSC_F_DAYS_OF_SUPPLY, S, false);
  ds.off_nip = block(F & MARLSC_F_NET_INV_POSITION, S, false);
  ds.off_dv = block(F & MARLSC_F_DEMAND_VARIABILITY, S, false);
  ds.off_hist = block(F & MARLSC_F_DEMAND_HISTORY, kWindow * S, false);
  const int dim_noid = o;
  ds.obs_dim = o + ds.id_off;
  tb.obs_mean.clear();
  tb.obs_std.clear();
  if (sp.obs_norm == MARLSC_NORM_MEANSTD) {
    if (!sp.obs_mean || !sp.obs_std) return "obs_norm MEANSTD needs obs_mean and obs_std";
    tb.obs_mean.assign(sp.obs_mean, sp.obs_mean + dim_noid);
    tb.obs_std.assign(sp.obs_std, sp.obs_std + dim_noid);
    for (float& v : tb.obs_std) v = 1.0f / v;                  // kernels multiply by the reciprocal
  }

  // per-CTA lookup tables staged in shared memory (byte offsets, 16-byte aligned blocks)
  {
    int o = 0;
    auto blk = [&](int bytes) { const int at = o; o = (o + bytes + 15) & ~15; return at; };
    ds.t_skw = blk(S * 8);
    ds.t_pen = blk(S * 8);
    ds.t_hold = blk(S * 8);
    ds.t_prio = blk(R * ((W + 3) & ~3));
    ds.t_pstat = blk(R);
    ds.t_hmask = blk(W <= 32 ? R * 4 : 0);
    ds.t_lead = blk(W * S);
    ds.t_bytes = o;
  }
  // per-team scratch
  ds.och = S <= 16 ? 16 : std::max(8, std::min(64, (1280 / S) & ~1));
  int d = 0;
  ds.d_lostW = d; d += R;
  ds.d_lostP = d; d += R;
  ds.d_ctot = d; d += W;
  ds.d_shipw = d; if (!unit) d += W * R;
  ds.d_words = d | 1;
  int w = 0;
  const int WS = W * S;
  ds.w_inv = w; w += WS;
  ds.w_dh = w; if (ds.dh_mode == 2) w += WS;
  ds.w_sh = w; if (ds.need_ship) w += WS;
  ds.w_st = w; if (ds.need_ship) w += WS;
  ds.w_shipq = w; w += W * R;
  ds.w_cnt = w; if (ds.has_fixed) w += W * R;
  ds.w_lostN = w; w += R;
  ds.w_prio = w; w += (W + 3) / 4;
  ds.w_sreg = w; w += (ds.och + 1) / 2;
  ds.w_sqty = w; w += (ds.och * S + 8 + 3) / 4;
  ds.w_words = w | 1;
  return std::string();
}

inline void bind_tables(DevSpec& ds, const double* action_max, const double* out_fixed, const double* out_var,
                        const double* in_fixed, const double* in_var, const double* hold_rate,
                        const double* pen_rate, const double* skw, const int32_t* lead_exp, const int32_t* home,
                        const int32_t* closest, const int32_t* region_map, const uint8_t* prio,
                        const uint8_t* prio_static, const uint32_t* home_mask, const uint8_t* lead_u8,
                        const float* obs_mean, const float* obs_std) {
  ds.action_max = action_max; ds.out_fixed = out_fixed; ds.out_var = out_var; ds.in_fixed = in_fixed;
  ds.in_var = in_var; ds.hold_rate = hold_rate; ds.pen_rate = pen_rate; ds.skw = skw; ds.lead_exp = lead_exp;
  ds.home = home; ds.closest = closest; ds.region_map = region_map; ds.prio = prio; ds.prio_static = prio_static; ds.home_mask = home_mask; ds.lead_u8 = lead_u8;
  ds.obs_mean = obs_mean; ds.obs_std = obs_std;
}

}  // namespace marlsc
