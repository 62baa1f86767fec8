"""Reference harness (TEST INFRASTRUCTURE ONLY - never imported by the product path).

Drives the *unmodified* reference environment from a checkout of Jakoebly/marl-sc named by the
``MARLSC_REFERENCE_ROOT`` environment variable (or its copy under ``oracle/_ref``) so that golden
trajectories can be generated. What it recorded is committed under ``tests/golden/`` by
``tests/golden/make_golden.py`` and checked without it. Two tests compare with the live reference
(its YAML files, its SeedManager): they run when MARLSC_REFERENCE_ROOT is set, fail when it names no
checkout, and skip when it is unset. ``bench.py`` times the reference through it when it is present.

What is exercised (reference file:line):
  * ``InventoryEnvironment.reset/step``            src/environment/envs/multi_env.py:192-366
  * component registry                             src/environment/registry.py:26-308
  * ``load_environment_config``                    src/config/loader.py:117
  * ``SeedManager.derive_env_seed``                src/utils/seed_manager.py:166-186

Recipe (SURVEY.md appendix B): a shim directory provides ``gymnasium.spaces.Box`` and
``pettingzoo.ParallelEnv`` (no arithmetic in either); demand / lead-time draws are recorded from
the reference's own samplers so they can be replayed into the CUDA path and the oracle.

The allocator's ``np.argsort`` tie-break is SIMD-dispatch dependent for >= 4 warehouses, so the
process that imports numpy for golden generation must have ``NPY_DISABLE_CPU_FEATURES`` set
(``STABLE_SORT_ENV`` below); ``make_golden.py`` re-execs itself with it.
"""
from __future__ import annotations

import copy
import os
import sys
from typing import Any, Dict, List, Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
_SHIM = os.path.join(_HERE, "ref_shim")


def _find_root() -> str:
    """The reference tree: MARLSC_REFERENCE_ROOT, else oracle/_ref - the unmodified copy of the env path that
    oracle/make_ref.py makes so that the reference itself can be timed where no checkout is at hand (git-ignored)."""
    env_root, ref_copy = os.environ.get("MARLSC_REFERENCE_ROOT"), os.path.join(_HERE, "_ref")
    for c in (env_root, ref_copy):
        if c and os.path.isdir(os.path.join(c, "src", "environment")):
            return c
    return env_root or ref_copy


REF_ROOT = _find_root()

STABLE_SORT_ENV = {
    "NPY_DISABLE_CPU_FEATURES": "AVX512F AVX512CD AVX512_SKX AVX512_CLX AVX512_CNL AVX512_ICL AVX512_SPR AVX2 FMA3"
}


def available() -> bool:
    return os.path.isdir(os.path.join(REF_ROOT, "src", "environment"))


def activate() -> None:
    """Put the shim and the reference on sys.path (idempotent)."""
    if not available():
        raise RuntimeError(f"reference tree not found at {REF_ROOT}")
    for p in (REF_ROOT, _SHIM):
        if p not in sys.path:
            sys.path.insert(0, p)


class _Chdir:
    def __init__(self, path):
        self.path = path

    def __enter__(self):
        self.prev = os.getcwd()
        os.chdir(self.path)

    def __exit__(self, *a):
        os.chdir(self.prev)


def load_env_config(yaml_rel_path: str):
    """Validated reference ``EnvironmentConfig`` from a YAML shipped with the reference."""
    activate()
    from src.config.loader import load_environment_config

    with _Chdir(REF_ROOT):  # feature_config_path inside the YAML is relative to the repo root
        return load_environment_config(yaml_rel_path)


def env_config_from_dict(env_dict: Dict[str, Any], allow_region_mismatch: bool = False):
    """Reference ``EnvironmentConfig`` from a plain dict in the reference's YAML layout.

    With ``allow_region_mismatch`` the top-level validator that rejects ``n_regions != n_warehouses``
    (src/config/schema.py:670-675) is bypassed by validating the sub-models and using
    ``model_construct`` (SURVEY.md appendix B); ``max_splits: default`` is resolved by hand because
    the post-validator (schema.py:840-848) is skipped too.
    """
    activate()
    from pydantic import TypeAdapter
    from src.config import schema as S

    d = copy.deepcopy(env_dict)
    d.pop("feature_config_path", None)
    if not allow_region_mismatch:
        return TypeAdapter(S.EnvironmentConfig).validate_python(d)
    parts = dict(
        n_warehouses=d["n_warehouses"], n_skus=d["n_skus"], n_regions=d["n_regions"],
        episode_length=d["episode_length"], max_wh_capacities=d["max_wh_capacities"],
        action_space=TypeAdapter(S.ActionSpaceConfig).validate_python(d["action_space"]),
        initial_inventory=TypeAdapter(S.InitialInventoryConfig).validate_python(d["initial_inventory"]),
        cost_structure=TypeAdapter(S.CostStructureConfig).validate_python(d["cost_structure"]),
        components=TypeAdapter(S.ComponentsConfig).validate_python(d["components"]),
        data_source=TypeAdapter(S.DataSourceConfig).validate_python(d["data_source"]),
        features=TypeAdapter(S.FeatureConfig).validate_python(d.get("features", {})),
    )
    cfg = S.EnvironmentConfig.model_construct(**parts)
    alloc = cfg.components.demand_allocator
    if alloc.params.get("max_splits") == "default":
        alloc.params["max_splits"] = cfg.n_warehouses - 1
    return cfg


def make_env(cfg, seed: Optional[int], env_meta: Optional[Dict[str, Any]] = None):
    activate()
    from src.environment.envs.multi_env import InventoryEnvironment

    return InventoryEnvironment(cfg, seed=seed, env_meta=env_meta)


def attach_empirical_sampler(env, frame, data_mode: str = "train"):
    """Give a reference env the reference's own EmpiricalDemandSampler over ``frame`` (columns timestep, region_id,
    order_id, sku_id, quantity): the raw CSVs its preprocessing needs are not shipped, everything after the frame is."""
    activate()
    from src.data.preprocessor import PreprocessedData
    from src.environment.components.demand_sampler import EmpiricalDemandSampler

    ctx = env.context if hasattr(env, "context") else None
    if ctx is None:
        from src.environment.context import create_environment_context
        ctx = create_environment_context(env.env_config)
    ctx.preprocessed_data = PreprocessedData(demand_data=frame, val_demand_data=None)
    ctx.data_mode = data_mode
    ctx.episode_length = env.env_config.episode_length
    env.demand_sampler = EmpiricalDemandSampler(ctx, None)
    return env.demand_sampler


def reference_map_excluded_regions(order_region_ids, warehouse_to_region_df, selected_region_ids):
    """The reference's DataProcessor.map_excluded_regions (src/data/preprocessor.py:382-441) without its CSV-loading
    constructor."""
    activate()
    from src.data.preprocessor import DataProcessor

    proc = object.__new__(DataProcessor)
    proc.warehouse_to_region_df = warehouse_to_region_df
    proc.selected_region_ids = selected_region_ids
    return proc.map_excluded_regions(order_region_ids)


def derive_env_seed(base: int, worker: int, idx: int) -> int:
    activate()
    from src.utils.seed_manager import SeedManager

    return SeedManager.derive_env_seed(base, worker, idx)


class DemandRecorder:
    """Wraps ``env.demand_sampler.sample`` and keeps every order it emitted."""

    def __init__(self, env):
        self.steps: List[List[tuple]] = []
        self._inner = env.demand_sampler.sample
        env.demand_sampler.sample = self._sample  # instance attribute shadows the method

    def _sample(self, timestep):
        orders = self._inner(timestep)
        self.steps.append([(int(o.region_id), o.sku_demands.copy()) for o in orders])
        return orders


class LeadTimeRecorder:
    def __init__(self, env):
        self.steps: List[Any] = []
        self._inner = env.lead_time_sampler.sample
        env.lead_time_sampler.sample = self._sample

    def _sample(self):
        lt = self._inner()
        self.steps.append(lt.copy())
        return lt


class ReplayDemand:
    """Stand-in for ``env.demand_sampler`` that replays recorded orders.

    Not a ``StochasticComponent`` so ``reset()`` leaves it alone (multi_env.py:543-546).
    """

    def __init__(self, steps):
        activate()
        from src.environment.components.demand_sampler import Order

        self._Order = Order
        self.steps = steps

    def sample(self, timestep):
        return [self._Order(region_id=r, sku_demands=q.copy()) for r, q in self.steps[timestep]]


def base_stock_policy(env, level):
    """The reference's base-stock heuristic (src/experiments/run_baselines.py:188-207) for given levels [W,S]:
    order up to the level, clipped to the order maximum, as a float32 action."""
    import numpy as np

    maxq = np.asarray(env.env_config.action_space.params.max_order_quantities, dtype=np.float64)
    qty = np.clip(level - env.inventory - env._compute_pending_matrix(), 0.0, maxq)
    return (2.0 * qty / maxq - 1.0).astype(np.float32)


def run_episode(env, actions, reset: bool = True, policy=None) -> Dict[str, Any]:
    """Step the reference env through ``actions[T, W, S]`` (float32 in [-1, 1]) and dump everything.
    With ``policy`` (env -> float32 [W,S]) the actions are computed from the env's state step by step and written
    into ``actions``.

    Returns per-step stacks of the quantities listed in SURVEY.md section 8c ("parity classes").
    """
    import numpy as np

    W, S = env.n_warehouses, env.n_skus
    T = actions.shape[0]
    env.collect_step_info = True
    out: Dict[str, list] = {k: [] for k in (
        "inventory", "pending", "ordered", "fulfilled", "unfulfilled", "ship_counts", "ship_qty",
        "ship_by_sku", "lost_orders", "lost_sales", "cost_hold", "cost_pen", "cost_out", "cost_in",
        "rewards", "obs_local", "trunc")}
    if reset:
        obs, _ = env.reset()
    else:
        obs = env._get_observations()
    D = env._compute_local_obs_dim()
    res: Dict[str, Any] = {
        "init_inventory": env.inventory.copy(),
        "obs0_local": np.stack([np.asarray(obs[a][:D], dtype=np.float64) for a in env.agents]),
    }
    for t in range(T):
        if policy is not None:
            actions[t] = policy(env)
        act = {a: actions[t, i].astype(np.float32) for i, a in enumerate(env.agents)}
        obs, rew, term, trunc, infos = env.step(act)
        info = infos[env.agents[0]]
        out["inventory"].append(env.inventory.copy())
        out["pending"].append(env._compute_pending_matrix().astype(np.float64))
        out["ordered"].append(info["order_quantities"])
        out["fulfilled"].append(info["fulfilled_per_warehouse"])
        out["unfulfilled"].append(info["unfulfilled_demands"])
        out["ship_counts"].append(info["shipment_counts"])
        out["ship_qty"].append(info["shipment_quantities"])
        out["ship_by_sku"].append(info["shipment_quantities_by_sku"])
        out["lost_orders"].append(info["lost_order_counts"])
        out["lost_sales"].append(info["lost_sales"])
        out["cost_hold"].append(info["holding_cost"])
        out["cost_pen"].append(info["penalty_cost"])
        out["cost_out"].append(info["outbound_shipment_cost"])
        out["cost_in"].append(info["inbound_shipment_cost"])
        out["rewards"].append(np.array([rew[a] for a in env.agents], dtype=np.float64))
        out["obs_local"].append(np.stack([np.asarray(obs[a][:D], dtype=np.float64) for a in env.agents]))
        # every agent's observation must be [local_i | local_0 .. local_{W-1}] (multi_env.py:567-573)
        glob = np.concatenate([np.asarray(obs[a][:D]) for a in env.agents])
        for a in env.agents:
            assert np.array_equal(np.asarray(obs[a][D:]), glob)
        out["trunc"].append(bool(trunc[env.agents[0]]))
        assert not any(term.values())
    for k, v in out.items():
        res[k] = np.stack([np.asarray(x) for x in v])
    return res
