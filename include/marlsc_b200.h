/*
 * marlsc_b200.h - C ABI of the B200-native batched inventory-environment hot path.
 *
 * The reference (Jakoebly/marl-sc) is pure Python and has no FFI of its own; its boundary for this
 * path is three Python contracts (SURVEY.md section 8b). Every entry point below names the
 * reference interface it replaces (paths relative to the reference repo root). Plain pointers and
 * sizes only - no torch types. All device pointers must belong to the device the handle was created
 * on. Every call is asynchronous on the given stream unless stated otherwise; the caller owns all
 * buffers. Return value: 0 on success, a negative MARLSC_E* code otherwise (text via
 * marlsc_last_error()). The Python host layer turns these into ValueError / RuntimeError to match
 * the reference's exception conventions.
 *
 * There is no CPU fallback anywhere behind this header.
 */
#ifndef MARLSC_B200_H
#define MARLSC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MARLSC_ABI_VERSION 2

enum {
  MARLSC_OK = 0,
  MARLSC_EINVAL = -1,   /* bad argument / shape (reference raises ValueError) */
  MARLSC_ECUDA = -2,    /* CUDA runtime error */
  MARLSC_ENOMEM = -3,
  MARLSC_EUNSUPPORTED = -4
};

/* action space (reference: src/environment/envs/multi_env.py:824-846) */
enum { MARLSC_ACTION_DIRECT = 0, MARLSC_ACTION_DEMAND_CENTERED = 1, MARLSC_ACTION_BASE_STOCK = 2 };
/* lead-time sampler (reference: src/environment/components/lead_time_sampler.py:97-108,169-197) */
enum { MARLSC_LEAD_FIXED = 0, MARLSC_LEAD_STOCHASTIC = 1 };
/* lost-sales handler (reference: src/environment/components/lost_sales_handler.py:71,113,172) */
enum { MARLSC_LOST_CLOSEST = 0, MARLSC_LOST_SHIPMENT = 1, MARLSC_LOST_COST = 2 };
/* reward scope (reference: src/environment/components/reward_calculator.py:186-188) */
enum { MARLSC_SCOPE_AGENT = 0, MARLSC_SCOPE_TEAM = 1 };
/* observation normalisation done inside the env (reference: multi_env.py:591,607-610,700-702) */
enum { MARLSC_NORM_OFF = 0, MARLSC_NORM_RATIO = 1, MARLSC_NORM_MEANSTD = 2 };

/* feature toggles, same names as the reference FeatureConfig (src/config/schema.py:598-617);
 * block order in the observation follows multi_env.py:619-695 */
enum {
  MARLSC_F_INVENTORY = 1u << 0,
  MARLSC_F_INVENTORY_AGG = 1u << 1,
  MARLSC_F_PIPELINE = 1u << 2,
  MARLSC_F_PIPELINE_AGG = 1u << 3,
  MARLSC_F_DEMAND_HOME = 1u << 4,
  MARLSC_F_DEMAND_HOME_AGG = 1u << 5,
  MARLSC_F_SHIPPED_HOME = 1u << 6,
  MARLSC_F_SHIPPED_AWAY = 1u << 7,
  MARLSC_F_SHIPPED_AWAY_AGG = 1u << 8,
  MARLSC_F_STOCKOUT = 1u << 9,
  MARLSC_F_ROLLING_MEAN = 1u << 10,
  MARLSC_F_ROLLING_MEAN_AGG = 1u << 11,
  MARLSC_F_FORECAST = 1u << 12,
  MARLSC_F_FORECAST_AGG = 1u << 13,
  MARLSC_F_DAYS_OF_SUPPLY = 1u << 14,
  MARLSC_F_NET_INV_POSITION = 1u << 15,
  MARLSC_F_DEMAND_VARIABILITY = 1u << 16,
  MARLSC_F_DEMAND_HISTORY = 1u << 17
};

#define MARLSC_ROLLING_WINDOW 5 /* multi_env.py:147 */

/*
 * Static description of one environment family. Replaces the reference's EnvironmentContext
 * (src/environment/context.py:30-65) plus the constructor state of the five registry components
 * (src/environment/registry.py:300-308) and of InventoryEnvironment (multi_env.py:58-190).
 * All table pointers are HOST pointers; marlsc_env_create copies them to the device.
 */
typedef struct marlsc_env_spec {
  int32_t abi_version;          /* MARLSC_ABI_VERSION */
  int32_t n_warehouses;         /* W (= agents) */
  int32_t n_skus;               /* S */
  int32_t n_regions;            /* R, regions the cost tables are defined on */
  int32_t n_regions_raw;        /* length of region_map (== R when region_map is NULL) */
  int32_t episode_length;
  int32_t max_expected_lead;    /* L = max(expected_lead) (lead_time_sampler.py:128-131) */
  int32_t ring_depth;           /* D > max actual lead time; in-transit ring depth */
  int32_t action_type;          /* MARLSC_ACTION_* */
  int32_t lead_mode;            /* MARLSC_LEAD_* */
  int32_t lost_sales_type;      /* MARLSC_LOST_* */
  int32_t reward_scope;         /* MARLSC_SCOPE_* */
  int32_t max_splits;           /* demand_allocator.py:113-116 ("default" resolved to W-1) */
  int32_t obs_norm;             /* MARLSC_NORM_* */
  int32_t include_warehouse_id; /* one-hot id prepended (multi_env.py:705-708) */
  uint32_t feature_mask;        /* MARLSC_F_* */
  double scale_factor;          /* reward_calculator.py:179-180 */
  double lost_alpha;            /* softmax temperature of the "cost" handler */
  const double* action_max;     /* [S] max_order_quantities | max_quantity_adjustment | max_stock_level */
  const double* out_fixed;      /* [W,R] */
  const double* out_var;        /* [W,R] */
  const double* in_fixed;       /* [W,S] */
  const double* in_var;         /* [W,S] */
  const double* hold_rate;      /* [S] per-unit holding rate (list value, or scalar * sku weight) */
  const double* pen_rate;       /* [S] per-unit penalty rate (same rule) */
  const double* sku_weights;    /* [S] */
  const int32_t* expected_lead; /* [W,S] */
  const int32_t* home_region;   /* [W] argmin_r distances[w,r] (multi_env.py:144) */
  const int32_t* closest_wh;    /* [R] argmin_w distances[w,r] (lost_sales_handler.py:36) */
  const int32_t* region_map;    /* [n_regions_raw] raw -> included region (preprocessor.py:382-441) or NULL */
  const float* obs_mean;        /* [obs_dim without id] or NULL (multi_env.py:700-702) */
  const float* obs_std;         /* idem */
} marlsc_env_spec_t;

typedef struct marlsc_env marlsc_env_t; /* opaque handle */

/*
 * State layouts. WIDE is the general one (every configuration). COMPACT stores the same state in the width the
 * values need; it exists for the common configurations
 * (marlsc_env_layout() tells which one a handle uses; marlsc_env_set_layout() can force WIDE before the first reset):
 * fixed lead times, direct action space with order maxima <= 255, unit SKU weights, no outbound fixed costs, static
 * warehouse priority, non-binding split limit, inventory / pipeline / home-demand / rolling-mean feature blocks,
 * normalisation off or fixed mean-std, 32 < S <= 128 (a multiple of 4), W <= 16, R <= 64, L <= 16. The caller guarantees
 * on-hand stock stays below 65536 (initial stock + episode_length * max order quantity bounds it).
 */
enum { MARLSC_LAYOUT_WIDE = 0, MARLSC_LAYOUT_COMPACT = 1 };

/*
 * Struct-of-arrays state of E environments, all DEVICE pointers owned by the caller
 * (reference state: multi_env.py:175-186). Layout is env-major so one environment's slice of
 * every array is contiguous.
 *                 WIDE                                              COMPACT
 *   inventory    int32 [E,W,S]                                      uint16 [E,W,S]
 *   ring_qty     int32 [E,D,W,S], order placed at step tau lives    uint8 [E,L,W,S], order placed at step tau lives in
 *                in plane tau % D (D = ring_depth)                  plane tau % L (L = max_expected_lead); every cell's
 *                                                                   quantity, 0 included, is written each step
 *   ring_lead    uint8 [E,D,W,S] actual lead of that order;         unused (NULL)
 *                NULL when lead_mode is FIXED
 *   demand_hist  int32 [E,5,W,S] home-region demand of the last     uint16 [E,5,W,S]
 *                5 steps, plane t % 5; may be NULL when
 *                marlsc_env_needs_history() == 0
 *   forecast     float [E,W,S] EMA demand forecast; may be NULL     unused (NULL)
 *                when marlsc_env_needs_forecast() == 0
 */
typedef struct marlsc_env_state {
  int64_t num_envs;
  void* inventory;
  void* ring_qty;
  uint8_t* ring_lead;
  void* demand_hist;
  float* forecast;
  int32_t layout;        /* MARLSC_LAYOUT_*: must equal marlsc_env_layout() of the handle the state is used with */
} marlsc_env_state_t;

/*
 * Inputs and outputs of one step. Demand is a CSR list of orders per environment in the order the
 * reference sampler emits them (demand_sampler.py:128-163): order j of env e is row
 * order_offsets[e] + j; an all-zero row is a legal no-op order.
 */
typedef struct marlsc_step_io {
  const float* actions;          /* [E,W,S] in [-1,1] (multi_env.py:253) */
  const int32_t* order_offsets;  /* [E+1] */
  const int16_t* order_region;   /* [n_orders] raw region ids */
  const void* order_qty;         /* [n_orders,S] uint8 or uint16, see order_qty_bytes. The kernel stages rows as
                                    aligned 32-bit words: the allocation must extend at least 4 bytes past the last row */
  int32_t order_qty_bytes;       /* 1 or 2 */
  const uint8_t* actual_lead;    /* [E,W,S] this step's sampled lead times (stochastic) or NULL */
  float* rewards;                /* [E,W] */
  float* obs;                    /* [E,W,obs_dim] local observations == centralised-critic state */
  uint8_t* truncated;            /* [E] or NULL (multi_env.py:327) */
  /* optional diagnostics (reference: collect_step_info, multi_env.py:330-362); NULL to skip.
   * The d_* accumulators must be zeroed by the caller before the step. */
  float* cost_breakdown;         /* [E,W,4] holding, penalty, outbound, inbound (unscaled) */
  int32_t* d_ordered;            /* [E,W,S] */
  int32_t* d_ship;               /* [E,W,R,S] units shipped per warehouse-region-SKU */
  int32_t* d_ship_count;         /* [E,W,R] */
  int32_t* d_unfulfilled;        /* [E,R,S] */
  int32_t* d_lost_orders;        /* [E,R] */
  float* d_lost_sales;           /* [E,W,S] needs d_unfulfilled */
  /* padded order layout (what marlsc_demand_sample writes): when order_counts != NULL, env e owns rows
   * [e*order_stride, e*order_stride + order_counts[e]) of order_region / order_qty and order_offsets is ignored */
  const int32_t* order_counts;   /* [E] or NULL */
  int32_t order_stride;
  /* Sparse demand ("lines"), the native input of the COMPACT layout: the non-zero (order, SKU) cells of the step's orders
   * (region ids already mapped through region_map), regrouped into 32 streams per environment. A stream carries the cells
   * of up to four SKUs - "slots" 0..3 - and each SKU belongs to exactly one (stream, slot). Entries 0 and 1 of a stream are
   * its SKU map: four bytes, byte k = the SKU slot k stands for, 255 = none. The other entries are lines:
   * quantity (1..255) | region << 8 | slot << 14; 0 = padding. The lines of one SKU must appear in the order the reference
   * allocator meets them (order index ascending, demand_allocator.py:150-208); how different SKUs of a stream interleave
   * is free (their allocations never meet). The packers rank an environment's SKUs by line count and deal them to the
   * streams in a snake so that the 32 streams end within a few entries of each other: the allocation kernel runs as long
   * as the longest stream, and the block is as many rounds long. A "round" is one entry of each of the 32 streams
   * (64 bytes); rounds come in pairs: entries 2i and 2i+1 of stream l are the low and high half of 32-bit word l of pair
   * i, i.e. entry p of stream l is uint16 lines[(r0 + (p & ~1)) * 32 + 2 l + (p & 1)] for an environment whose rounds
   * start at r0. An environment owns the (even number of) rounds [line_offsets[e], line_offsets[e+1]) - or, in the
   * padded layout (line_counts != NULL, line_stride even), rounds [e*line_stride, e*line_stride + line_counts[e]); an
   * environment without demand owns no rounds (no map either). Streams shorter than the environment's round count are
   * padded with 0 at their end. When lines != NULL the order_* fields are ignored; a COMPACT handle given dense orders
   * converts them with marlsc_lines_from_orders into a library-owned buffer first. WIDE handles take dense orders only.
   * Build lines on the host with marlsc_b200.demand.pack_lines, on the device with marlsc_lines_from_orders (both
   * balanced, byte-identical) or marlsc_demand_sample_lines (SKU s on stream s % 32, slot s / 32). */
  const uint16_t* lines;         /* [n_rounds, 32] or NULL */
  const int32_t* line_offsets;   /* [E+1] */
  const int32_t* line_counts;    /* [E] or NULL */
  int32_t line_stride;
  /* Integer order quantities instead of float actions (direct action space, COMPACT layout): uint8 [E,W,S], the quantity
   * itself (clipped to the SKU's maximum), a quarter of the bytes of `actions` for callers that decide in units. */
  const uint8_t* action_qty;     /* [E,W,S] or NULL; replaces actions when set */
  /* Base-stock heuristic evaluated inside the step (COMPACT layout, split step): when actions and action_qty are both
   * NULL and base_stock_level is set, every cell's action is what marlsc_policy_base_stock would have produced from the
   * state before this step - 2 clip(level - on_hand - in_transit, 0, max_qty) / max_qty - 1 in float32 - and is rescaled
   * like any other action. Saves the policy launch and two passes over the action tensor. */
  const float* base_stock_level; /* device float32 [W,S], or [E,W,S] when base_stock_per_env != 0; or NULL */
  int32_t base_stock_per_env;
} marlsc_step_io_t;

/* ---- lifecycle ------------------------------------------------------------------------------ */

/* Replaces InventoryEnvironment.__init__ + create_environment_context + get_* registry calls
 * (multi_env.py:58-190, context.py:143-209, registry.py:26-289). Synchronous. */
int marlsc_env_create(const marlsc_env_spec_t* spec, int device, marlsc_env_t** out);
void marlsc_env_destroy(marlsc_env_t* env);

/* Width of one warehouse's observation (multi_env.py:444-502). */
int32_t marlsc_env_obs_dim(const marlsc_env_t* env);
int32_t marlsc_env_needs_history(const marlsc_env_t* env);
int32_t marlsc_env_needs_forecast(const marlsc_env_t* env);
/* Threads cooperating on one environment (1..64, power of two; 64 = two warps, lean launches only, generic
 * launches then use 32). 0 restores the automatic choice. */
int marlsc_env_set_team_size(marlsc_env_t* env, int32_t threads_per_env);
int32_t marlsc_env_team_size(const marlsc_env_t* env);
/* The library holds a lean and a generic instantiation of the step kernel and picks the lean one when
 * the configuration allows it; on != 0 forces the generic one (used by the parity tests). */
int marlsc_env_set_generic(marlsc_env_t* env, int32_t on);
/* WIDE only. Lean launches of teams of 8+ lanes run the step as four kernels (place / allocate / features /
 * rewards, see csrc/env_split.cuh); on != 0 keeps them in the single fused kernel (used for comparisons and by the
 * tests). A COMPACT handle has one step: there on != 0 returns MARLSC_EUNSUPPORTED (force MARLSC_LAYOUT_WIDE first)
 * and on == 0 is accepted. */
int marlsc_env_set_fused(marlsc_env_t* env, int32_t on);
/* State layout of this handle (MARLSC_LAYOUT_*): COMPACT when the configuration qualifies, else WIDE. */
int32_t marlsc_env_layout(const marlsc_env_t* env);
/* Force a layout before the state is allocated / first reset: MARLSC_LAYOUT_WIDE is always possible (needed for the
 * diagnostic outputs, explicit team sizes and the generic / fused test switches, which are WIDE only);
 * MARLSC_LAYOUT_COMPACT fails with MARLSC_EUNSUPPORTED when the configuration does not qualify. */
int marlsc_env_set_layout(marlsc_env_t* env, int32_t layout);
/* Rounds per environment of the library-owned line buffer a COMPACT handle converts dense orders into (default 128;
 * a stream that needs more sets an overflow flag that fails the NEXT call on the handle). */
int marlsc_env_set_line_stride(marlsc_env_t* env, int32_t rounds);
/* Measurement aid: with on != 0 every marlsc_env_step records CUDA events on its stream around each kernel it
 * launches. marlsc_env_last_timing waits for the last timed step and writes the per-launch durations in
 * milliseconds (split step: place, allocate, features, rewards; WIDE fused step: one entry); returns how many, or a
 * negative error code. A COMPACT step is timed when it is given lines (marlsc_step_io.lines), not with dense orders. */
int marlsc_env_set_timing(marlsc_env_t* env, int32_t on);
int marlsc_env_last_timing(marlsc_env_t* env, float* ms, int32_t capacity);

/* ---- the hot path --------------------------------------------------------------------------- */

/* Replaces InventoryEnvironment.reset (multi_env.py:192-251): state cleared, inventory set from
 * init_inventory (device int32, [E,W,S], or [W,S] broadcast when per_env == 0), first observation
 * written to obs [E,W,obs_dim]. */
int marlsc_env_reset(marlsc_env_t* env, const marlsc_env_state_t* state, const int32_t* init_inventory,
                     int32_t per_env, float* obs, void* stream);

/* Replaces InventoryEnvironment.step (multi_env.py:253-366) for all E environments at timestep t
 * (the pre-increment timestep of the reference; all environments share it, multi_env.py:325-327). */
int marlsc_env_step(marlsc_env_t* env, const marlsc_env_state_t* state, const marlsc_step_io_t* io,
                    int32_t t, void* stream);

/* Same step driven from HOST buffers (the reference-facing call: numpy in, numpy out): copies
 * actions / demand / lead times host->device into caller-provided device staging, steps, and copies
 * rewards (and obs when obs_host != NULL) back. host pointers should be pinned. Returns after the
 * device->host copies are complete. */
typedef struct marlsc_host_step {
  const float* actions;          /* host [E,W,S] */
  const int32_t* order_offsets;  /* host [E+1] */
  const int16_t* order_region;   /* host [n_orders] */
  const void* order_qty;         /* host [n_orders,S] */
  int64_t n_orders;
  const uint8_t* actual_lead;    /* host [E,W,S] or NULL */
  float* rewards;                /* host [E,W] */
  float* obs;                    /* host [E,W,obs_dim] or NULL */
  /* COMPACT layout: sparse demand lines instead of dense orders, integer quantities instead of float actions
   * (see marlsc_step_io); the staging sets then need lines / line_offsets / action_qty device buffers */
  const uint16_t* lines;         /* host [n_rounds,32] or NULL */
  const int32_t* line_offsets;   /* host [E+1] */
  int64_t n_rounds;
  const uint8_t* action_qty;     /* host [E,W,S] or NULL */
} marlsc_host_step_t;
int marlsc_env_step_host(marlsc_env_t* env, const marlsc_env_state_t* state, const marlsc_step_io_t* dev_staging,
                         const marlsc_host_step_t* host, int32_t t, void* stream);

/* A rollout segment of n_steps consecutive timesteps t0 .. t0+n_steps-1 driven from HOST buffers, with
 * the host->device copies of step i+1 overlapped with the kernel of step i (two device staging sets, an
 * internal copy stream). host[i] describes step i (pinned memory strongly recommended); staging[0..1] are
 * two device staging sets like the one marlsc_env_step_host takes, except that rewards / obs of step i
 * are written to rewards_dev + i*E*W (time-major rollout buffer) and obs_dev[i & 1]; rewards are copied
 * back to host[i].rewards. Returns after everything is on the host. Replaces n_steps calls of
 * InventoryEnvironment.step (multi_env.py:253-366) made from host-side actions and demand. */
int marlsc_env_rollout_host(marlsc_env_t* env, const marlsc_env_state_t* state, const marlsc_step_io_t staging[2],
                            const marlsc_host_step_t* host, int32_t n_steps, int32_t t0, float* rewards_dev,
                            void* stream);

/* ---- per-episode metrics ---------------------------------------------------------------------------- */

/* What an inventory study reports about an episode (reference: collect_step_info, multi_env.py:330-362, summed over the
 * steps by the reference's baseline runs and seed evaluations): float64 DEVICE accumulators owned by the caller, summed
 * over the steps since the last marlsc_env_reset. Costs are unscaled, with the definitions of marlsc_step_io.cost_breakdown.
 * Per environment, demand_units == sum_w shipped_units + lost_units exactly; with agent-scope rewards
 * episode_return ~= -scale_factor * (holding + penalty + outbound + inbound) row by row. */
typedef struct marlsc_episode_metrics {
  double* holding_cost;    /* [E,W] */
  double* penalty_cost;    /* [E,W] lost-sales cost as the configured handler attributes it */
  double* outbound_cost;   /* [E,W] */
  double* inbound_cost;    /* [E,W] */
  double* ordered_units;   /* [E,W] units placed (after rescale / clipping) */
  double* shipped_units;   /* [E,W] units shipped from the warehouse to any region */
  double* episode_return;  /* [E,W] sum of the float32 rewards the steps wrote */
  double* demand_units;    /* [E]   units demanded (after the region map) */
  double* lost_units;      /* [E]   units not fulfilled */
} marlsc_episode_metrics_t;

/* Register accumulators with the handle (it keeps a copy of the pointers; every one is required, else MARLSC_EINVAL),
 * or m == NULL to stop accumulating. While set, marlsc_env_reset zeroes them on its stream (cudaMemsetAsync) and every
 * step the handle runs (marlsc_env_step, marlsc_env_step_host, marlsc_env_rollout_host) adds to them, for the
 * num_envs of the state it is given. Observations, rewards and state are the same as without metrics.
 *   COMPACT: the step's kernels accumulate as they go, plus one small launch that adds the rewards.
 *   WIDE:    the step's diagnostic outputs are folded into the accumulators by one extra launch, so marlsc_step_io must
 *            carry cost_breakdown, d_ordered, d_ship and d_unfulfilled (else MARLSC_EINVAL); that selects the generic
 *            step kernel. d_ship and d_unfulfilled accumulate, so the caller zeroes them before every step, which
 *            marlsc_env_rollout_host cannot do: it returns MARLSC_EUNSUPPORTED on a WIDE handle with metrics. */
int marlsc_env_set_metrics(marlsc_env_t* env, const marlsc_episode_metrics_t* m);

/* ---- on-device samplers and heuristic policies (SURVEY.md section 8f) -------------------------------- */

/* Device Poisson demand sampler: same distribution as the reference's PoissonDemandSampler
 * (src/environment/components/demand_sampler.py:105-163; parameters broadcast to [R], [R], [R,S]), Philox
 * counter-based stream keyed by (seed, env, step) - reproducible, but not the reference's PCG64 stream. */
typedef struct marlsc_demand marlsc_demand_t;
int marlsc_demand_create(int32_t n_regions, int32_t n_skus, const double* lambda_orders, const double* probability_skus,
                         const double* lambda_quantity, int device, marlsc_demand_t** out);
void marlsc_demand_destroy(marlsc_demand_t* d);
/* Draw one step of orders for num_envs environments into the padded layout: order_counts [E],
 * order_region [E*max_orders_per_env], order_qty uint8 [E*max_orders_per_env, S]. Orders beyond
 * max_orders_per_env are dropped and *overflow_flag (device int32, caller-zeroed) is set to 1. */
int marlsc_demand_sample(marlsc_demand_t* d, int64_t num_envs, uint64_t seed, int64_t step_index, int32_t max_orders_per_env,
                         int32_t* order_counts, int16_t* order_region, uint8_t* order_qty, int32_t* overflow_flag, void* stream);

/* The same draw written as lines (padded layout): lines [E*line_stride, 32], line_counts [E]; region ids are mapped
 * through region_map (device int32 [n_regions], or NULL). Identical orders to marlsc_demand_sample for the same
 * (seed, step). A stream longer than line_stride is cut and *overflow_flag set. S <= 128, n_regions (mapped) <= 64. */
int marlsc_demand_sample_lines(marlsc_demand_t* d, int64_t num_envs, uint64_t seed, int64_t step_index, int32_t line_stride,
                               const int32_t* region_map, uint16_t* lines, int32_t* line_counts, int32_t* overflow_flag,
                               void* stream);

/* Dense orders (CSR or padded, as in marlsc_step_io) -> lines in the padded layout for a COMPACT handle: lines
 * [E*line_stride, 32], line_counts [E] (device). Applies the handle's region_map. overflow_flag (device int32,
 * caller-zeroed) is set when a stream needs more than line_stride rounds (the surplus is dropped). */
int marlsc_lines_from_orders(marlsc_env_t* env, int64_t num_envs, const marlsc_step_io_t* orders, int32_t line_stride,
                             uint16_t* lines, int32_t* line_counts, int32_t* overflow_flag, void* stream);

/* Test hook: the Poisson inversion K4 uses, evaluated for n given (lambda, u) pairs (device float32 arrays):
 * k_out[i] = the order count drawn from uniform u[i] at rate lambda[i] (tabulated == 0), or the quantity drawn through
 * the tabulated-CDF search the per-SKU quantities use (tabulated != 0). Rates >= 30 take the float64 walk from the
 * mode in both cases. Synchronises the stream. */
int marlsc_poisson_inverse(const float* lambda, const float* u, int64_t n, int32_t tabulated, int32_t* k_out, void* stream);

/* Device lead-time sampler: the distribution of the reference's StochasticLeadTimeSampler.sample
 * (src/environment/components/lead_time_sampler.py:169-197): actual = max(1, expected[w,s] + U{-d[s]..+d[s]}),
 * independently per environment, warehouse, SKU and step (the reference also draws every step). expected_lead
 * int32 [W,S] and max_deviation int32 [S] are DEVICE pointers; actual_lead uint8 [E,W,S] is what
 * marlsc_step_io.actual_lead takes. Philox stream keyed by (seed, cell, step); not the reference's PCG64 stream. */
int marlsc_lead_sample(int64_t num_envs, int32_t n_warehouses, int32_t n_skus, const int32_t* expected_lead,
                       const int32_t* max_deviation, uint64_t seed, int64_t step_index, uint8_t* actual_lead, void* stream);

/* Batched base-stock heuristic (reference: make_bs_newsvendor_action_fn, src/experiments/run_baselines.py:133-207):
 * actions[e,w,s] = 2*clip(level[w,s] - on_hand - in_transit, 0, max_qty[s])/max_qty[s] - 1 evaluated before step t.
 * level: device float32 [W,S]; actions: device float32 [E,W,S]. Direct action space only. */
int marlsc_policy_base_stock(marlsc_env_t* env, const marlsc_env_state_t* state, const float* level, int32_t t,
                             float* actions, void* stream);
/* The same with one level per environment, level [E,W,S] (the rolling-mean "BS-Adaptive" heuristic,
 * src/experiments/run_baselines.py:209-293, derives its levels from each environment's own demand history). */
int marlsc_policy_base_stock_per_env(marlsc_env_t* env, const marlsc_env_state_t* state, const float* level, int32_t t,
                                     float* actions, void* stream);

/* Reverse-time GAE(lambda) / value-target scan over a rollout segment, one column per
 * (environment, agent). Replaces RLlib's GeneralAdvantageEstimation connector that the reference
 * configures through use_gae / lambda_ / gamma (src/algorithms/ippo.py:145-160, mappo.py:142-157).
 *   rewards [T,N], values [T+1,N] (values[T] = bootstrap V(s_T)), N = E*W columns
 *   cut [T] host-side flags: cut[t] != 0 means an episode ended (truncation) after step t; the scan
 *   restarts there and bootstraps from cut_values[t,:] (V of the final observation), or from 0 when
 *   cut_values is NULL (termination semantics).
 *   adv, targets [T,N] out. */
int marlsc_gae(const float* rewards, const float* values, const uint8_t* cut, const float* cut_values,
               int32_t T, int64_t N, float gamma, float lam, float* adv, float* targets, void* stream);

/* Per-policy advantage standardisation (x - mean) / max(1e-4, std) in place over n values
 * (RLlib learner connector). workspace: device, >= marlsc_standardize_workspace_bytes(). */
size_t marlsc_standardize_workspace_bytes(void);
int marlsc_standardize(float* x, int64_t n, void* workspace, void* stream);

/* K7 - forward pass of a one-hidden-layer MLP head over every agent-sample of a rollout step (reference:
 * ActorCriticRLModule._forward_actor / _forward_critic over an "mlp" network with one hidden layer,
 * src/algorithms/models/rlmodules/base.py:412-457; IPPO model sizes config_files/algorithms/ippo.yaml):
 *   out[n, :] = W2 act(W1 x[n, :] + b1) + b2,   activation 0 = ReLU, 1 = tanh, float32 throughout.
 * x [n_rows, in_dim], w1 [hidden, in_dim], b1 [hidden], w2 [out_dim, hidden], b2 [out_dim] (torch.nn.Linear layouts),
 * out [n_rows, out_dim], all on the device, contiguous. in_dim <= 128, out_dim <= 16 (action means of a 2-3 SKU network or
 * the value; the joint head of a centralised (CPPO) policy: W x local width inputs, W x S outputs); anything else:
 * MARLSC_EUNSUPPORTED, use the library GEMMs. The hidden activations stay in registers. in_dim <= 64 with out_dim <= 3 runs
 * the narrow kernel; wider heads a second form whose shared memory holds hidden x (in_dim padded to 16 / 32 / 64 / 128 +
 * out_dim padded to 4 / 8 / 16 + 4) floats, MARLSC_EUNSUPPORTED past the device's per-block limit. */
int marlsc_mlp1_forward(const float* x, int64_t n_rows, int32_t in_dim, const float* w1, const float* b1, int32_t hidden,
                        const float* w2, const float* b2, int32_t out_dim, int32_t activation, float* out, void* stream);

/* K7a - input layer of a deeper MLP head during rollouts: out[n, :] = act(W x[n, :] + b), activation 0 ReLU, 1 tanh,
 * 2 none (the first nn.Linear of the reference's "mlp" networks, rlmodules/base.py:412-457). x [n_rows, in_dim],
 * w [hidden, in_dim], b [hidden], out [n_rows, hidden], float32, device, contiguous; in_dim <= 64, hidden <= 256 and
 * ceil(hidden / 32) x (in_dim padded to 16 / 32 / 64) <= 128, else MARLSC_EUNSUPPORTED. */
int marlsc_linear_in_forward(const float* x, int64_t n_rows, int32_t in_dim, const float* w, const float* b, int32_t hidden,
                             int32_t activation, float* out, void* stream);

/* K7b - output layer of a deeper MLP head during rollouts: out[n, :] = W a[n, :] + b for out_dim <= 16 (the last
 * nn.Linear of the reference's "mlp" networks, rlmodules/base.py:412-457, e.g. MAPPO's actor [14, 256, 256, 2] and
 * critic [56, 64, 64, 1], config_files/algorithms/mappo.yaml:43-55), where a = h, or - with pre_bias != NULL -
 * a = relu(h + pre_bias): h is then the RAW product of the hidden layer before, whose bias [in_dim] and ReLU are applied
 * on the way in (saves the separate epilogue pass the library GEMM runs over the activations). h [n_rows, in_dim]
 * (in_dim a multiple of 4, <= 2048), w [out_dim, in_dim], b [out_dim], out [n_rows, out_dim], float32, device,
 * contiguous, h / w / pre_bias 16-byte aligned. One pass over h at the HBM rate. out_dim 5 to 16 (the joint action means
 * of a centralised policy's deeper head) runs a second form that pads the outputs to 8 or 16; anything past 16 outputs is
 * MARLSC_EUNSUPPORTED. */
int marlsc_linear_out_forward(const float* h, int64_t n_rows, int32_t in_dim, const float* pre_bias, const float* w, const float* b,
                              int32_t out_dim, float* out, void* stream);

/* K6 - PPO objective of one minibatch, forward and backward (RLlib PPOTorchLearner as the reference configures it,
 * src/algorithms/ippo.py:145-160; hysteretic_beta < 0 disables the weighting of learners/hysteretic_learner.py:39-42):
 *   L_p = -mean_p(min(ratio adv, clip(ratio, 1-c, 1+c) adv)) + vf_loss_coeff mean_p(min((value - target)^2, vf_clip_param))
 *         + kl_coeff mean_p(KL(old || new))                 (use_kl_loss, ippo.py:146; skipped when mean_old is NULL)
 * with ratio = exp(logp(actions | mean, max(log_std_p, logstd_floor)) - logp_old) of a diagonal Gaussian, summed over the
 * n_policies policies: 1 with parameter sharing (ippo.py:106-110), else one per warehouse (ippo.py:111-115) with sample i
 * belonging to policy i % n_policies, each policy averaging over its own samples. All arrays on the device: mean, actions,
 * mean_old, grad_mean [n_samples, action_dim]; logp_old, adv, value, targets, grad_value [n_samples]; log_std,
 * log_std_old (already floored) [n_policies, action_dim]. Writes dL/dmean and dL/dvalue; sums (float64
 * [n_policies, 3 + action_dim], zeroed by the call) receives per policy the sum of the surrogate, of the clipped value
 * loss, of the KL term, and dL/dlog_std. The entropy bonus only depends on log_std and is left to the caller. */
int marlsc_ppo_loss(const float* mean, const float* actions, const float* log_std, int32_t n_policies, float logstd_floor,
                    const float* logp_old, const float* adv, const float* value, const float* targets, const float* mean_old,
                    const float* log_std_old, float kl_coeff, int64_t n_samples, int32_t action_dim, float clip_param,
                    float vf_clip_param, float vf_loss_coeff, float hysteretic_beta, float* grad_mean, float* grad_value,
                    double* sums, void* stream);

/* ---- misc ----------------------------------------------------------------------------------- */
const char* marlsc_last_error(void);
int32_t marlsc_abi_version(void);
/* number of kernels this library has launched since load (bench.py reports it as gpu_launches) */
int64_t marlsc_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* MARLSC_B200_H */
