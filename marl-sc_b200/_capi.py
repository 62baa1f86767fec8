"""ctypes binding of the C ABI declared in include/marlsc_b200.h.

The shared library is the product: if it is missing this module raises instead of falling back to
anything on the CPU.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmarlsc_b200.so")
ABI_VERSION = 2
LAYOUT_WIDE, LAYOUT_COMPACT = 0, 1

# enums (include/marlsc_b200.h)
ACTION = {"direct": 0, "demand_centered": 1, "base_stock": 2}
NORM = {"off": 0, "meanstd": 0, "ratio": 1, "meanstd_custom": 2, "meanstd_grouped": 2}
FEATURE_BITS = {
    "inventory": 1 << 0, "inventory_aggregate": 1 << 1, "pipeline": 1 << 2, "pipeline_aggregate": 1 << 3,
    "incoming_demand_home": 1 << 4, "incoming_demand_home_aggregate": 1 << 5, "units_shipped_home": 1 << 6,
    "units_shipped_away": 1 << 7, "units_shipped_away_aggregate": 1 << 8, "stockout": 1 << 9,
    "rolling_demand_mean": 1 << 10, "rolling_demand_mean_aggregate": 1 << 11, "demand_forecast": 1 << 12,
    "demand_forecast_aggregate": 1 << 13, "days_of_supply": 1 << 14, "net_inventory_position": 1 << 15,
    "demand_variability": 1 << 16, "demand_history": 1 << 17,
}

_pd = C.POINTER(C.c_double)
_pi = C.POINTER(C.c_int32)
_pf = C.POINTER(C.c_float)


class EnvSpecC(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("n_warehouses", C.c_int32), ("n_skus", C.c_int32), ("n_regions", C.c_int32),
        ("n_regions_raw", C.c_int32), ("episode_length", C.c_int32), ("max_expected_lead", C.c_int32),
        ("ring_depth", C.c_int32), ("action_type", C.c_int32), ("lead_mode", C.c_int32),
        ("lost_sales_type", C.c_int32), ("reward_scope", C.c_int32), ("max_splits", C.c_int32),
        ("obs_norm", C.c_int32), ("include_warehouse_id", C.c_int32), ("feature_mask", C.c_uint32),
        ("scale_factor", C.c_double), ("lost_alpha", C.c_double),
        ("action_max", _pd), ("out_fixed", _pd), ("out_var", _pd), ("in_fixed", _pd), ("in_var", _pd),
        ("hold_rate", _pd), ("pen_rate", _pd), ("sku_weights", _pd),
        ("expected_lead", _pi), ("home_region", _pi), ("closest_wh", _pi), ("region_map", _pi),
        ("obs_mean", _pf), ("obs_std", _pf),
    ]


class EnvStateC(C.Structure):
    _fields_ = [("num_envs", C.c_int64), ("inventory", C.c_void_p), ("ring_qty", C.c_void_p),
                ("ring_lead", C.c_void_p), ("demand_hist", C.c_void_p), ("forecast", C.c_void_p), ("layout", C.c_int32)]


class StepIOC(C.Structure):
    _fields_ = [("actions", C.c_void_p), ("order_offsets", C.c_void_p), ("order_region", C.c_void_p),
                ("order_qty", C.c_void_p), ("order_qty_bytes", C.c_int32), ("actual_lead", C.c_void_p),
                ("rewards", C.c_void_p), ("obs", C.c_void_p), ("truncated", C.c_void_p),
                ("cost_breakdown", C.c_void_p), ("d_ordered", C.c_void_p), ("d_ship", C.c_void_p),
                ("d_ship_count", C.c_void_p), ("d_unfulfilled", C.c_void_p), ("d_lost_orders", C.c_void_p),
                ("d_lost_sales", C.c_void_p), ("order_counts", C.c_void_p), ("order_stride", C.c_int32),
                ("lines", C.c_void_p), ("line_offsets", C.c_void_p), ("line_counts", C.c_void_p), ("line_stride", C.c_int32),
                ("action_qty", C.c_void_p), ("base_stock_level", C.c_void_p), ("base_stock_per_env", C.c_int32)]


class HostStepC(C.Structure):
    _fields_ = [("actions", C.c_void_p), ("order_offsets", C.c_void_p), ("order_region", C.c_void_p),
                ("order_qty", C.c_void_p), ("n_orders", C.c_int64), ("actual_lead", C.c_void_p),
                ("rewards", C.c_void_p), ("obs", C.c_void_p), ("lines", C.c_void_p), ("line_offsets", C.c_void_p),
                ("n_rounds", C.c_int64), ("action_qty", C.c_void_p)]


class EpisodeMetricsC(C.Structure):
    """marlsc_episode_metrics: float64 device accumulators, [E,W] except demand_units / lost_units [E]."""
    _fields_ = [("holding_cost", C.c_void_p), ("penalty_cost", C.c_void_p), ("outbound_cost", C.c_void_p),
                ("inbound_cost", C.c_void_p), ("ordered_units", C.c_void_p), ("shipped_units", C.c_void_p),
                ("episode_return", C.c_void_p), ("demand_units", C.c_void_p), ("lost_units", C.c_void_p)]


class MarlscError(RuntimeError):
    pass


_lib: Optional[C.CDLL] = None


def lib() -> C.CDLL:
    """Load libmarlsc_b200.so (built by ``__graft_entry__.build()``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: the CUDA library is the only implementation of this path (no CPU "
            "fallback). Build it with `python -c 'import __graft_entry__ as g; g.build()'` from the repo root.")
    import torch  # noqa: F401  (loads the CUDA runtime the library links against)
    L = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    L.marlsc_env_create.argtypes = [C.POINTER(EnvSpecC), C.c_int, C.POINTER(vp)]
    L.marlsc_env_create.restype = C.c_int
    L.marlsc_env_destroy.argtypes = [vp]
    L.marlsc_env_destroy.restype = None
    for fn in ("marlsc_env_obs_dim", "marlsc_env_needs_history", "marlsc_env_needs_forecast", "marlsc_env_team_size"):
        getattr(L, fn).argtypes = [vp]
        getattr(L, fn).restype = i32
    L.marlsc_env_layout.argtypes = [vp]
    L.marlsc_env_layout.restype = i32
    L.marlsc_env_set_layout.argtypes = [vp, i32]
    L.marlsc_env_set_layout.restype = C.c_int
    L.marlsc_env_set_line_stride.argtypes = [vp, i32]
    L.marlsc_env_set_line_stride.restype = C.c_int
    L.marlsc_lines_from_orders.argtypes = [vp, i64, C.POINTER(StepIOC), i32, vp, vp, vp, vp]
    L.marlsc_lines_from_orders.restype = C.c_int
    L.marlsc_demand_sample_lines.argtypes = [vp, i64, C.c_uint64, i64, i32, vp, vp, vp, vp, vp]
    L.marlsc_demand_sample_lines.restype = C.c_int
    L.marlsc_env_set_team_size.argtypes = [vp, i32]
    L.marlsc_env_set_team_size.restype = C.c_int
    L.marlsc_env_set_generic.argtypes = [vp, i32]
    L.marlsc_env_set_generic.restype = C.c_int
    L.marlsc_env_set_fused.argtypes = [vp, i32]
    L.marlsc_env_set_fused.restype = C.c_int
    L.marlsc_env_set_metrics.argtypes = [vp, C.POINTER(EpisodeMetricsC)]
    L.marlsc_env_set_metrics.restype = C.c_int
    L.marlsc_env_set_timing.argtypes = [vp, i32]
    L.marlsc_env_set_timing.restype = C.c_int
    L.marlsc_env_last_timing.argtypes = [vp, C.POINTER(C.c_float), i32]
    L.marlsc_env_last_timing.restype = C.c_int
    L.marlsc_env_reset.argtypes = [vp, C.POINTER(EnvStateC), vp, i32, vp, vp]
    L.marlsc_env_reset.restype = C.c_int
    L.marlsc_env_step.argtypes = [vp, C.POINTER(EnvStateC), C.POINTER(StepIOC), i32, vp]
    L.marlsc_env_step.restype = C.c_int
    L.marlsc_env_step_host.argtypes = [vp, C.POINTER(EnvStateC), C.POINTER(StepIOC), C.POINTER(HostStepC), i32, vp]
    L.marlsc_env_step_host.restype = C.c_int
    L.marlsc_env_rollout_host.argtypes = [vp, C.POINTER(EnvStateC), C.POINTER(StepIOC), C.POINTER(HostStepC), i32, i32, vp, vp]
    L.marlsc_env_rollout_host.restype = C.c_int
    L.marlsc_demand_create.argtypes = [i32, i32, _pd, _pd, _pd, C.c_int, C.POINTER(vp)]
    L.marlsc_demand_create.restype = C.c_int
    L.marlsc_demand_destroy.argtypes = [vp]
    L.marlsc_demand_destroy.restype = None
    L.marlsc_demand_sample.argtypes = [vp, i64, C.c_uint64, i64, i32, vp, vp, vp, vp, vp]
    L.marlsc_demand_sample.restype = C.c_int
    L.marlsc_poisson_inverse.argtypes = [vp, vp, i64, i32, vp, vp]
    L.marlsc_poisson_inverse.restype = C.c_int
    L.marlsc_lead_sample.argtypes = [i64, i32, i32, vp, vp, C.c_uint64, i64, vp, vp]
    L.marlsc_lead_sample.restype = C.c_int
    L.marlsc_policy_base_stock.argtypes = [vp, C.POINTER(EnvStateC), vp, i32, vp, vp]
    L.marlsc_policy_base_stock.restype = C.c_int
    L.marlsc_policy_base_stock_per_env.argtypes = [vp, C.POINTER(EnvStateC), vp, i32, vp, vp]
    L.marlsc_policy_base_stock_per_env.restype = C.c_int
    L.marlsc_gae.argtypes = [vp, vp, vp, vp, i32, i64, C.c_float, C.c_float, vp, vp, vp]
    L.marlsc_gae.restype = C.c_int
    L.marlsc_mlp1_forward.argtypes = [vp, i64, i32, vp, vp, i32, vp, vp, i32, i32, vp, vp]
    L.marlsc_mlp1_forward.restype = C.c_int
    L.marlsc_linear_out_forward.argtypes = [vp, i64, i32, vp, vp, vp, i32, vp, vp]
    L.marlsc_linear_out_forward.restype = C.c_int
    L.marlsc_linear_in_forward.argtypes = [vp, i64, i32, vp, vp, i32, i32, vp, vp]
    L.marlsc_linear_in_forward.restype = C.c_int
    L.marlsc_ppo_loss.argtypes = [vp, vp, vp, i32, C.c_float, vp, vp, vp, vp, vp, vp, C.c_float, i64, i32, C.c_float, C.c_float,
                                  C.c_float, C.c_float, vp, vp, vp, vp]
    L.marlsc_ppo_loss.restype = C.c_int
    L.marlsc_standardize_workspace_bytes.argtypes = []
    L.marlsc_standardize_workspace_bytes.restype = C.c_size_t
    L.marlsc_standardize.argtypes = [vp, i64, vp, vp]
    L.marlsc_standardize.restype = C.c_int
    L.marlsc_standardize_moments.argtypes = [vp, i64, vp, vp]
    L.marlsc_standardize_moments.restype = C.c_int
    L.marlsc_standardize_apply.argtypes = [vp, i64, vp, vp]
    L.marlsc_standardize_apply.restype = C.c_int
    L.marlsc_last_error.argtypes = []
    L.marlsc_last_error.restype = C.c_char_p
    L.marlsc_abi_version.argtypes = []
    L.marlsc_abi_version.restype = i32
    L.marlsc_launch_count.argtypes = []
    L.marlsc_launch_count.restype = i64
    if L.marlsc_abi_version() != ABI_VERSION:
        raise ImportError(f"{LIB_PATH} has ABI {L.marlsc_abi_version()}, expected {ABI_VERSION}; rebuild it")
    _lib = L
    return L


def check(rc: int) -> None:
    """0 -> ok; MARLSC_EINVAL -> ValueError (the reference raises ValueError for bad input); else RuntimeError."""
    if rc == 0:
        return
    msg = (lib().marlsc_last_error() or b"").decode("utf-8", "replace")
    if rc == -1:
        raise ValueError(msg)
    raise MarlscError(f"marlsc error {rc}: {msg}")
