"""Generate tests/golden/*.npz from the UNMODIFIED reference env (needs a checkout of Jakoebly/marl-sc).

    MARLSC_REFERENCE_ROOT=<marl-sc checkout> python tests/golden/make_golden.py [scenario ...]

For every scenario in scenarios.py this steps ``n_envs`` reference ``InventoryEnvironment`` instances
(src/environment/envs/multi_env.py of the checkout) seeded ``derive_env_seed(base_seed, 0, i)``
(src/utils/seed_manager.py:166-186) with pre-sampled float32 actions, records the demand orders and
lead times its own samplers drew, and stores inputs + every per-step output (SURVEY.md section 8c
parity classes). The committed vectors are what pins ``oracle/inventory_oracle.py`` and, through it,
the CUDA path; no test needs the checkout itself.

numpy's argsort tie-break is SIMD-dispatch dependent, so the script re-execs itself with
NPY_DISABLE_CPU_FEATURES set (see oracle/ref_harness.py).
"""
from __future__ import annotations

import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

from oracle import ref_harness as H  # noqa: E402

if os.environ.get("NPY_DISABLE_CPU_FEATURES") != H.STABLE_SORT_ENV["NPY_DISABLE_CPU_FEATURES"]:
    os.execvpe(sys.executable, [sys.executable] + sys.argv, {**os.environ, **H.STABLE_SORT_ENV})

import numpy as np  # noqa: E402

import scenarios as SC  # noqa: E402

GRID = np.array([-1.0, 1.0, 0.0, 0.5, -0.5, 0.25, -0.25, 0.3, 0.75, -0.75, 0.125, 0.9], dtype=np.float32)


def make_actions(seed, shape):
    rng = np.random.default_rng(seed)
    a = rng.uniform(-1, 1, shape).astype(np.float32)
    pick = rng.random(shape) < 0.15            # exact grid points exercise round-half-even and the clip
    a[pick] = GRID[rng.integers(0, len(GRID), size=int(pick.sum()))]
    return a


def check_small_default_matches_yaml():
    ref = H.load_env_config("config_files/environments/env_symmetric_3WH2SKU.yaml")
    mine = H.env_config_from_dict(SC.small_default())
    assert ref.model_dump() == mine.model_dump(), "small_default() drifted from the reference YAML"


def generate(name: str) -> str:
    sc = SC.scenario(name)
    env_dict = sc["env"]
    ref_dict = env_dict
    emp = None
    if sc.get("empirical"):
        # the reference env is built with a placeholder sampler and then given the reference's own EmpiricalDemandSampler
        # over a synthetic frame whose region ids went through the reference's map_excluded_regions
        import copy
        ref_dict = copy.deepcopy(env_dict)
        ref_dict["components"]["demand_sampler"] = dict(type="poisson", params=dict(lambda_orders=1.0, probability_skus=0.1, lambda_quantity=1.0))
        raw, wtr, all_ids, selected = SC.empirical_frame(n_included=env_dict["n_regions"], n_skus=env_dict["n_skus"])
        mapped = H.reference_map_excluded_regions(raw["region_raw"], wtr, selected)
        sel_index = {rid: i for i, rid in enumerate(selected)}
        frame = raw.assign(region_id=mapped.map(sel_index).astype(int))[["timestep", "region_id", "order_id", "sku_id", "quantity"]]
        frame = frame.sort_values(["timestep", "region_id", "order_id", "sku_id"]).reset_index(drop=True)   # preprocessor.py:694
        raw_index = {rid: i for i, rid in enumerate(all_ids)}
        emp = dict(frame=frame, raw=raw, wtr=wtr, all_ids=all_ids, selected=selected,
                   region_map=np.asarray([sel_index[H.reference_map_excluded_regions(
                       raw["region_raw"].iloc[:0].reindex([0]).fillna(rid), wtr, selected).iloc[0]] for rid in all_ids], dtype=np.int32),
                   raw_region_index=raw["region_raw"].map(raw_index).to_numpy(dtype=np.int16))
    cfg = H.env_config_from_dict(ref_dict, allow_region_mismatch=sc["allow_region_mismatch"])
    N, T = sc["n_envs"], sc["steps"]
    W, S, R = env_dict["n_warehouses"], env_dict["n_skus"], env_dict["n_regions"]
    actions = make_actions(sc["action_seed"], (N, T, W, S))
    policy = None
    if sc.get("policy") == "base_stock":
        # levels as the benchmark's: L E[D] + z sqrt(L E[D]) with E[D] of the regions a warehouse serves first
        p = env_dict["components"]["demand_sampler"]["params"]
        lam_o, prob, lam_q = np.asarray(p["lambda_orders"], float), np.asarray(p["probability_skus"], float), np.asarray(p["lambda_quantity"], float)
        out_var = np.asarray(env_dict["cost_structure"]["shipment_cost"]["outbound_variable"], float)
        first = np.argsort(out_var, axis=0, kind="stable")[0]
        ed = np.zeros((W, S))
        for r in range(R):
            ed[first[r]] += lam_o[r] * prob[r] * lam_q[r]
        lead = np.asarray(env_dict["components"]["lead_time_sampler"]["params"]["expected_lead_times"], float)
        level = lead * ed + 2.0 * np.sqrt(lead * ed)
        policy = lambda env: H.base_stock_policy(env, level)   # noqa: E731
    stochastic = env_dict["components"]["lead_time_sampler"]["type"] == "stochastic"

    probe = H.make_env(cfg, seed=0, env_meta=dict(include_warehouse_id=False))
    stats = SC.obs_stats_for(sc, probe._compute_local_obs_dim())
    meta = dict(obs_normalization=sc["obs_normalization"], obs_stats=stats,
                include_warehouse_id=sc["include_warehouse_id"])

    keys = None
    stacks = {}
    ptr, regions, qtys, leads, seeds = [0], [], [], [], []
    for i in range(N):
        seed = H.derive_env_seed(sc["base_seed"], 0, i)
        seeds.append(seed)
        env = H.make_env(cfg, seed=seed, env_meta=meta)
        if emp is not None:
            H.attach_empirical_sampler(env, emp["frame"])
        dem = H.DemandRecorder(env)
        ltr = H.LeadTimeRecorder(env)
        res = H.run_episode(env, actions[i], policy=policy)
        if emp is not None:
            starts = stacks.setdefault("window_start", [])
            starts.append(np.asarray(env.demand_sampler.available_timesteps.index(env.demand_sampler._start_timestep)))
        assert len(dem.steps) == T and len(ltr.steps) == T
        for step in dem.steps:
            for r, q in step:
                regions.append(r)
                qtys.append(q)
            ptr.append(len(regions))
        leads.append(np.stack(ltr.steps))
        keys = keys or [k for k in res.keys() if not (sc.get("lite") and k in ("ship_by_sku", "fulfilled", "ship_qty"))]
        for k in keys:
            stacks.setdefault(k, []).append(res[k])

    out = {k: np.stack(v) for k, v in stacks.items()}
    int_keys = ("init_inventory", "inventory", "pending", "ordered", "fulfilled", "unfulfilled",
                "ship_counts", "ship_qty", "ship_by_sku", "lost_orders")
    for k in int_keys:
        if k not in out:
            continue
        assert np.array_equal(out[k], np.round(out[k])), k
        out[k] = out[k].astype(np.int32)
    if sc.get("lite"):
        # float32 is what the reference emits (multi_env.py:569). Most entries are small whole numbers: stored as int16
        # plus the (index, value) list of the others, which compresses five times better than the float array
        obs = out.pop("obs_local").astype(np.float32)
        out["obs0_local"] = out["obs0_local"].astype(np.float32)
        whole = (obs == np.round(obs)) & (np.abs(obs) < 32000)
        out["obs_shape"] = np.asarray(obs.shape, dtype=np.int64)
        out["obs_whole"] = np.where(whole, obs, 0).astype(np.int16)
        out["obs_frac_idx"] = np.flatnonzero(~whole).astype(np.int64)
        out["obs_frac_val"] = obs.reshape(-1)[~whole.reshape(-1)]
    if env_dict["components"]["lost_sales_handler"]["type"] == "closest":
        assert np.array_equal(out["lost_sales"], np.round(out["lost_sales"]))
    qty_arr = np.asarray(qtys, dtype=np.float64).reshape(-1, S)
    assert np.array_equal(qty_arr, np.round(qty_arr)) and qty_arr.max(initial=0) < 32767
    payload = dict(
        env_json=np.array(json.dumps(env_dict)),
        meta_json=np.array(json.dumps(dict(
            obs_normalization=sc["obs_normalization"], include_warehouse_id=sc["include_warehouse_id"],
            allow_region_mismatch=sc["allow_region_mismatch"], base_seed=sc["base_seed"],
            n_envs=N, steps=T, stochastic_lead=stochastic, lite=bool(sc.get("lite")), policy=sc.get("policy"),
            empirical=bool(sc.get("empirical")),
            numpy=np.__version__, reference="Jakoebly/marl-sc"))),
        env_seeds=np.asarray(seeds, dtype=np.int64),
        actions=actions,
        order_ptr=np.asarray(ptr, dtype=np.int64),          # CSR over (env, step): row = i*T + t
        order_region=np.asarray(regions, dtype=np.int16),
        order_qty=qty_arr.astype(np.int16),
        lead_times=np.stack(leads).astype(np.int8),          # [N, T, W, S] actual lead times drawn
        **out)
    if stats is not None:
        payload["obs_mean"], payload["obs_std"] = stats
    if emp is not None:
        # the RAW frame (region ids as indices into all_region_ids), the cost table the mapping rule reads, and what the
        # reference's map_excluded_regions made of every raw region
        raw = emp["raw"]
        order_ids, order_codes = np.unique(raw["order_id"].to_numpy(dtype=str), return_inverse=True)
        payload.update(
            frame_timestep=raw["timestep"].to_numpy(dtype=np.int32), frame_region_raw=emp["raw_region_index"],
            frame_order=order_codes.astype(np.int32), frame_sku=raw["sku_id"].to_numpy(dtype=np.int16),
            frame_qty=raw["quantity"].to_numpy(dtype=np.float32),
            all_region_ids=np.array(emp["all_ids"]), selected_region_ids=np.array(emp["selected"]),
            wtr_source=emp["wtr"]["sourcenodeid"].to_numpy(dtype=str), wtr_dest=emp["wtr"]["destinationregionid"].to_numpy(dtype=str),
            wtr_cost=emp["wtr"]["fixed_costs"].to_numpy(dtype=np.float64), region_map=emp["region_map"])
    path = os.path.join(HERE, f"{name}.npz")
    np.savez_compressed(path, **payload)
    print(f"{name}: {N} envs x {T} steps, {len(regions)} orders, {os.path.getsize(path) / 1024:.0f} KiB")
    return path


if __name__ == "__main__":
    check_small_default_matches_yaml()
    for nm in (sys.argv[1:] or list(SC.SCENARIOS)):
        generate(nm)
