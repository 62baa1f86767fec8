"""CPU tests of the host-side boundary: YAML/config schema, component registry, seed derivation,
order packing, spec building, policy modules and the C ABI's exported symbols."""
import ctypes
import os
import pathlib
import re

import numpy as np
import pytest
import torch
import yaml

import marlsc_b200  # noqa: F401
from golden.scenarios import allfeat_ratio_stochastic, large_network, small_default
from marlsc_b200 import registry
from marlsc_b200.config import (ConfigFileError, ConfigValidationError, algorithm_config_from_dict,
                                environment_config_from_dict, load_algorithm_config, load_environment_config)
from marlsc_b200.demand import pack_orders
from marlsc_b200.seeds import ENVIRONMENT_SEEDS, SeedManager
from marlsc_b200.spec import build_env_spec, local_obs_dim
from oracle import ref_harness

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = ref_harness.REF_ROOT           # a checkout of the reference project (MARLSC_REFERENCE_ROOT), or its copy in oracle/_ref
# the live comparisons run when a checkout is named (and fail if it is not one); without one they skip
REF_GIVEN = bool(os.environ.get("MARLSC_REFERENCE_ROOT"))
NO_REF = "compares with a checkout of the reference project: set MARLSC_REFERENCE_ROOT"

IPPO = dict(algorithm=dict(
    name="ippo",
    shared=dict(num_iterations=300, checkpoint_freq=100, batch_size=8000, num_epochs=20, num_minibatches=10,
                learning_rate=5e-4, num_env_runners=2, num_envs_per_env_runner=10),
    algorithm_specific=dict(use_gae=True, lam=0.95, gamma=0.99, clip_param=0.1, vf_clip_param=800.0, logstd_init=-1.15,
                            logstd_floor=-3.5, obs_normalization="meanstd_custom", parameter_sharing=True,
                            networks=dict(shared_layers=None, use_mu_sigma_head=False,
                                          actor=dict(type="mlp", config=dict(hidden_sizes=[256], activation="relu")),
                                          critic=dict(type="mlp", config=dict(hidden_sizes=[256], activation="relu"))))))


# ------------------------------------------------------------------ config
def test_env_yaml_roundtrip(tmp_path):
    feats = tmp_path / "features.yaml"
    env = small_default()
    feats.write_text(yaml.safe_dump(dict(features=env.pop("features"))))
    env["feature_config_path"] = str(feats)
    path = tmp_path / "env.yaml"
    path.write_text(yaml.safe_dump(dict(environment=env)))
    cfg = load_environment_config(str(path))
    assert (cfg.n_warehouses, cfg.n_skus, cfg.n_regions) == (3, 2, 3)
    assert cfg.components.demand_allocator.params["max_splits"] == 2          # "default" -> W-1
    assert cfg.features.rolling_demand_mean and not cfg.features.stockout


@pytest.mark.skipif(not REF_GIVEN, reason=NO_REF)
def test_reference_yaml_files_load_unmodified():
    import glob
    cwd = os.getcwd()
    os.chdir(REF)
    try:
        envs = glob.glob("config_files/environments/*.yaml")
        assert envs, f"no config_files/environments/*.yaml under {REF}"
        for f in envs:
            cfg = load_environment_config(f)
            assert cfg.n_regions == cfg.n_warehouses
        for f in ("ippo", "mappo", "ippo_test", "mappo_test", "cppo"):
            algo = load_algorithm_config(f"config_files/algorithms/{f}.yaml")
            assert 0.9 <= algo.algorithm_specific.gamma <= 1.0 and algo.shared.batch_size > 0
    finally:
        os.chdir(cwd)


def test_legacy_max_order_quantities_migration():
    env = small_default()
    env.pop("action_space")
    env["max_order_quantities"] = 40
    cfg = environment_config_from_dict(env)
    assert cfg.action_space.type == "direct" and cfg.action_space.params.max_order_quantities == [40, 40]


def test_validation_rules():
    env = small_default()
    env["n_regions"] = 5
    with pytest.raises(ConfigValidationError, match="must equal n_warehouses"):
        environment_config_from_dict(env)
    env = small_default()
    env["features"]["pipeline"] = False
    with pytest.raises(ConfigValidationError, match="pipeline must always be enabled"):
        environment_config_from_dict(env)
    env = small_default()
    env["features"]["pipeline_aggregate"] = True
    env["features"]["incoming_demand_home_aggregate"] = True
    with pytest.raises(ConfigValidationError, match="cannot be enabled"):
        environment_config_from_dict(env)
    env = small_default()
    env["components"]["demand_allocator"]["params"]["max_splits"] = 3
    with pytest.raises(ConfigValidationError, match="max_splits must be <"):
        environment_config_from_dict(env)
    env = small_default()
    env["components"]["lost_sales_handler"]["type"] = "nearest"
    with pytest.raises(ConfigValidationError):
        environment_config_from_dict(env)
    with pytest.raises(ConfigFileError):
        load_environment_config("/nonexistent/env.yaml")
    big = large_network()
    big["allow_region_mismatch"] = True
    assert environment_config_from_dict(big).n_regions == 50


def test_algorithm_config():
    algo = algorithm_config_from_dict(IPPO)
    assert algo.name == "ippo" and algo.algorithm_specific.lam == 0.95
    assert algo.algorithm_specific.critic_obs_type == "local"
    bad = algorithm_config_from_dict
    d = {"algorithm": {**IPPO["algorithm"], "name": "mappo"}}
    assert bad(d).algorithm_specific.critic_obs_type == "global"
    d = {"algorithm": {**IPPO["algorithm"], "shared": {**IPPO["algorithm"]["shared"], "num_minibatches": 7}}}
    with pytest.raises(ConfigValidationError, match="divisible"):
        bad(d)


# ------------------------------------------------------------------ registry / components
def test_registry_names_and_errors():
    assert set(registry.DEMAND_SAMPLER_REGISTRY) >= {"poisson", "empirical"}
    assert set(registry.DEMAND_ALLOCATOR_REGISTRY) == {"greedy"}
    assert set(registry.LEAD_TIME_SAMPLER_REGISTRY) == {"fixed", "stochastic"}
    assert set(registry.LOST_SALES_HANDLER_REGISTRY) == {"closest", "shipment", "cost"}
    assert set(registry.REWARD_CALCULATOR_REGISTRY) == {"cost"}
    cfg = environment_config_from_dict(small_default())
    alloc = registry.get_demand_allocator(cfg)
    assert alloc.max_splits == 2
    lt = registry.get_lead_time_sampler(cfg)
    assert lt.get_max_expected() == 3 and np.array_equal(lt.sample(), lt.get_expected())
    cfg.components.reward_calculator.__dict__["type"] = "profit"
    with pytest.raises(ValueError, match=r"Unknown reward calculator: profit\. Available: \['cost'\]"):
        registry.get_reward_calculator(cfg)


def test_custom_component_registration():
    from marlsc_b200.components import ShipmentLostSalesHandler

    class Mine(ShipmentLostSalesHandler):
        pass
    registry.register_lost_sales_handler("mine", Mine)
    try:
        cfg = environment_config_from_dict(small_default())
        cfg.components.lost_sales_handler.__dict__["type"] = "mine"
        assert isinstance(registry.get_lost_sales_handler(cfg), Mine)
    finally:
        registry.LOST_SALES_HANDLER_REGISTRY.pop("mine")


@pytest.mark.skipif(not (REF_GIVEN or ref_harness.available()), reason=NO_REF)
def test_seed_manager_matches_reference():
    from oracle import ref_harness as H
    H.activate()
    from src.utils.seed_manager import SeedManager as RefSM
    a, b = SeedManager(123, ENVIRONMENT_SEEDS), RefSM(123, ENVIRONMENT_SEEDS)
    for _ in range(3):
        a.advance_episode()
        b.advance_episode()
        for name in ENVIRONMENT_SEEDS:
            assert a.get_seed_int(name) == b.get_seed_int(name)
            assert a.get_rng(name).integers(0, 1 << 30) == b.get_rng(name).integers(0, 1 << 30)
    assert SeedManager.derive_env_seed(7, 1, 5) == RefSM.derive_env_seed(7, 1, 5)
    assert a.spawn_child_seeds("inventory", 4) == b.spawn_child_seeds("inventory", 4)


def test_seed_manager_matches_recorded_reference_streams():
    """What the reference's SeedManager gave, as recorded in every golden file: the per-environment seeds
    derive_env_seed(base_seed, 0, i), and the first episode's "inventory" stream (uniform initial stock) and
    "lead_time_sampler" stream (stochastic lead times, sampled through our registry component)."""
    from golden_io import NAMES, Golden
    streams = 0
    for name in NAMES + ["empirical_regionmap"]:
        g = Golden(name)
        seeds = [SeedManager.derive_env_seed(g.meta["base_seed"], 0, i) for i in range(g.N)]
        assert seeds == g["env_seeds"].tolist(), name
        ic = g.env["initial_inventory"]
        cfg = environment_config_from_dict(g.env) if g.meta["stochastic_lead"] else None
        for i, seed in enumerate(seeds):
            sm = SeedManager(seed, ENVIRONMENT_SEEDS)
            sm.advance_episode()                              # what the first reset() does (multi_env.py:218-231)
            if ic["type"] == "uniform":
                drawn = sm.get_rng("inventory").integers(ic["params"]["min"], ic["params"]["max"] + 1, size=(g.W, g.S))
                assert np.array_equal(drawn, g["init_inventory"][i]), (name, i)
                streams += 1
            if cfg is not None:
                lt = registry.get_lead_time_sampler(cfg)
                lt.reset(sm.get_rng("lead_time_sampler"))
                for t in range(g.T):
                    assert np.array_equal(lt.sample(), g["lead_times"][i, t]), (name, i, t)
                streams += 1
    assert streams == 24                                      # 8 initial stocks, 16 lead-time trajectories


def test_seed_manager_basics():
    sm = SeedManager(None, ENVIRONMENT_SEEDS)
    assert sm.get_seed_int("inventory") is None
    with pytest.raises(ValueError, match="not in registry"):
        SeedManager(1, ENVIRONMENT_SEEDS).get_rng("train")
    s1, s2 = SeedManager(5, ENVIRONMENT_SEEDS), SeedManager(5, ENVIRONMENT_SEEDS)
    assert s1.get_rng("demand_sampler").random() == s2.get_rng("demand_sampler").random()


def test_poisson_sampler_stream_is_golden():
    """Seeded like the reference env, the host sampler must emit the orders recorded from the reference."""
    from golden_io import Golden
    g = Golden("small_default")
    cfg = environment_config_from_dict(g.env)
    for i in (0, 5):
        sm = SeedManager(int(g["env_seeds"][i]), ENVIRONMENT_SEEDS)
        sm.advance_episode()
        smp = registry.get_demand_sampler(cfg)
        smp.reset(sm.get_rng("demand_sampler"))
        for t in range(5):
            got = smp.sample(t)
            exp = g.orders(i, t)
            assert len(got) == len(exp)
            for o, (r, q) in zip(got, exp):
                assert o.region_id == r and np.array_equal(o.sku_demands, q)


# ------------------------------------------------------------------ packing / spec
def test_pack_orders():
    b = pack_orders([[(1, [0, 3]), (2, [7, 0])], [], [(0, [1, 1])]], 2)
    assert b.offsets.tolist() == [0, 2, 2, 3] and b.region.tolist() == [1, 2, 0]
    assert b.qty.dtype == np.uint8 and b.qty[:3].tolist() == [[0, 3], [7, 0], [1, 1]]
    assert (b.qty.size * b.qty.itemsize) % 16 == 0
    assert pack_orders([[(0, [300, 1])]], 2).qty.dtype == np.uint16
    with pytest.raises(ValueError):
        pack_orders([[(0, [-1, 1])]], 2)
    empty = pack_orders([[], []], 4)
    assert empty.n_orders == 0 and empty.qty.nbytes >= 16


def test_spec_tables():
    cfg = environment_config_from_dict(allfeat_ratio_stochastic())
    sp = build_env_spec(cfg, "ratio", None, True)
    s = sp.scalars
    assert s["lead_mode"] == 1 and s["ring_depth"] == 4 + 2 and s["max_expected_lead"] == 4
    assert s["action_type"] == 1 and s["lost_sales_type"] == 0 and s["reward_scope"] == 1 and s["max_splits"] == 1
    assert sp.tables["home_region"].tolist() == [0, 1, 2]
    assert np.allclose(sp.tables["pen_rate"], 4.0 * np.array([0.5, 1.0, 2.0, 1.5, 0.25]))   # scalar * sku weight
    assert np.allclose(sp.tables["hold_rate"], [0.5, 1.0, 0.25, 2.0, 1.5])                    # list: as is
    assert local_obs_dim(cfg.features, 5, 4, 3, True) == 3 + 5 + 1 + 20 + 1 + 6 + 5 + 6 + 5 + 6 + 6 + 5 + 5 + 5 + 25
    with pytest.raises(ValueError, match="obs_stats must have shape"):
        build_env_spec(cfg, "meanstd_custom", (np.zeros(3), np.ones(3)), False)
    with pytest.raises(ValueError, match="Unknown obs_normalization"):
        build_env_spec(cfg, "zscore")


# ------------------------------------------------------------------ C ABI
def test_library_exports_every_declared_symbol():
    from marlsc_b200 import _capi
    header = open(os.path.join(ROOT, "include", "marlsc_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(marlsc_[a-z_0-9]+)\s*\(", header)))
    assert "marlsc_env_step" in declared and "marlsc_gae" in declared and len(declared) >= 14
    lib = ctypes.CDLL(_capi.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/marlsc_b200.h but not exported"
    assert _capi.lib().marlsc_abi_version() == _capi.ABI_VERSION


def test_no_cpu_fallback():
    from marlsc_b200.envs import BatchedInventoryEnv
    from marlsc_b200.rollout import compute_gae
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError, match="no CPU implementation"):
        BatchedInventoryEnv(environment_config_from_dict(small_default()), 4)
    with pytest.raises(RuntimeError, match="no CPU implementation"):
        compute_gae(torch.zeros(3, 4), torch.zeros(4, 4), 0.99, 0.95)


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "marl-sc_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in text and "from oracle" not in text and "tests/emu" not in text.replace("tests/emu/emu.cpp", "")


# ------------------------------------------------------------------ policy modules
def test_actor_critic_shapes_and_split_critic():
    from marlsc_b200.rollout import ActorCritic
    algo = algorithm_config_from_dict({"algorithm": {**IPPO["algorithm"], "name": "mappo"}})
    pol = ActorCritic.from_algorithm_config(algo, local_obs_dim=14, n_warehouses=3, action_dim=2)
    obs = torch.randn(7, 3, 14)
    act, logp, val = pol.act(obs)
    assert act.shape == (7, 3, 2) and logp.shape == (7, 3) and val.shape == (7, 3)
    assert float(act.abs().max()) <= 1.0
    full = torch.cat([obs, obs.reshape(7, 1, 42).expand(7, 3, 42)], dim=2)        # reference layout
    assert torch.allclose(pol.value(obs), pol.critic(full).squeeze(-1), atol=1e-5)
    assert torch.allclose(pol.std(), torch.full((2,), float(np.exp(-1.15))), atol=1e-6)
    pol.log_std.data.fill_(-10.0)
    assert torch.allclose(pol.std(), torch.full((2,), float(np.exp(-3.5))), atol=1e-7)   # floor


def test_shard_envs():
    from marlsc_b200.rollout import shard_envs
    parts = [shard_envs(10, r, 4) for r in range(4)]
    assert [len(p) for p in parts] == [3, 3, 2, 2]
    assert sorted(i for p in parts for i in p) == list(range(10))


def test_independent_policies_equal_separate_modules():
    """parameter_sharing=False (reference ippo.py:111-115): the stacked-weight module must equal W separate MLPs with
    the same weights, the loss must be the sum of the per-policy mean losses, and grad_clip must act per policy."""
    from marlsc_b200.rollout import ActorCritic, PPOLearner, mlp
    torch.manual_seed(1)
    W, D, S, B = 3, 7, 2, 41
    pol = ActorCritic(D, W, S, actor_hidden=(8,), critic_hidden=(8,), critic_obs_type="global", parameter_sharing=False,
                      logstd_floor=-3.0)
    assert pol.n_policies == W and pol.log_std.shape == (W, S)
    obs = torch.randn(B, W, D)
    mean = pol.action_mean(obs)
    val = pol.value(obs)
    full = torch.cat([obs, obs.reshape(B, 1, W * D).expand(B, W, W * D)], dim=2)
    for w in range(W):
        a = mlp(D, (8,), S)
        a[0].weight.data, a[0].bias.data = pol.actor[0].weight.data[w].t(), pol.actor[0].bias.data[w, 0]
        a[2].weight.data, a[2].bias.data = pol.actor[2].weight.data[w].t(), pol.actor[2].bias.data[w, 0]
        assert torch.allclose(a(obs[:, w]), mean[:, w], atol=1e-5)
        c = mlp(D * (1 + W), (8,), 1)
        c[0].weight.data, c[0].bias.data = pol.critic[0].weight.data[w].t(), pol.critic[0].bias.data[w, 0]
        c[2].weight.data, c[2].bias.data = pol.critic[2].weight.data[w].t(), pol.critic[2].bias.data[w, 0]
        assert torch.allclose(c(full[:, w]).squeeze(-1), val[:, w], atol=1e-5)
    learner = PPOLearner(pol, fused_loss=False, grad_clip=0.05, use_kl_loss=True)
    with torch.no_grad():
        actions = mean + 0.5 * torch.randn_like(mean)
        logp_old = pol.log_prob(mean, actions) + 0.2 * torch.randn(B, W)
        mean_old = mean + 0.1 * torch.randn_like(mean)
        ls_old = pol.clamped_log_std() - 0.1
    adv, tgt = torch.randn(B, W), torch.randn(B, W)
    out = learner.loss(obs, actions, logp_old, adv, tgt, mean_old, ls_old)
    # per-policy pieces by hand
    ratio = (pol.log_prob(mean, actions) - logp_old).exp()
    surr = torch.minimum(ratio * adv, ratio.clamp(0.8, 1.2) * adv)
    assert torch.allclose(out["policy"], -sum(surr[:, w].mean() for w in range(W)), atol=1e-6)
    learner.buckets.zero()
    out["total"].backward()
    learner._clip()
    for w in range(W):                                  # every policy's own gradient norm is clipped to 0.05
        sq = sum(float(p.grad[w].pow(2).sum()) for p in learner.params)
        assert sq ** 0.5 <= 0.05 * (1 + 1e-4)


def test_learner_update_loop_and_kl_adaptation():
    """num_epochs x num_minibatches with a fresh on-device permutation per epoch (reference ippo.py:149-152) on a
    synthetic rollout; at the behaviour parameters the first minibatch has ratio 1 and KL 0."""
    from marlsc_b200.rollout import ActorCritic, PPOLearner
    from marlsc_b200.rollout.collector import Rollout
    torch.manual_seed(2)
    T, E, W, D, S = 6, 10, 3, 5, 2
    pol = ActorCritic(D, W, S, actor_hidden=(8,), critic_hidden=(8,))
    obs = torch.randn(T + 1, E, W, D)
    with torch.no_grad():
        act, raw, logp, val, mean = pol.act(obs[:T], return_raw=True)
    assert float((raw - act).abs().max()) > 0          # some samples were clipped; the batch keeps the raw ones
    ro = Rollout(obs, raw, logp, torch.randn(T, E, W), torch.randn(T + 1, E, W), torch.randn(T, E, W), torch.randn(T, E, W),
                 torch.zeros(T, dtype=torch.uint8), mean, pol.clamped_log_std().detach().reshape(1, S).clone())
    learner = PPOLearner(pol, lr=1e-3, fused_loss=False, use_kl_loss=True, num_epochs=3, num_minibatches=4, seed=1)
    first = learner.loss(obs[:T].reshape(T * E, W, D), raw.reshape(T * E, W, S), logp.reshape(T * E, W),
                         ro.advantages.reshape(T * E, W), ro.targets.reshape(T * E, W), mean.reshape(T * E, W, S), ro.log_std_old)
    assert abs(float(first["kl"])) < 1e-6
    assert torch.allclose(first["policy"], -ro.advantages.mean(), atol=1e-5)     # ratio == 1 everywhere
    before = [p.detach().clone() for p in pol.parameters()]
    stats = learner.update(ro)
    assert stats["minibatches"] == 12 and np.isfinite(stats["total"])
    assert any(not torch.equal(a, b.detach()) for a, b in zip(before, pol.parameters()))
    assert stats["kl_coeff"] in (0.1, 0.2, 0.30000000000000004)


def test_running_meanstd_filter_and_column_standardisation():
    from marlsc_b200.rollout import MeanStdFilter, standardize_columns_
    torch.manual_seed(0)
    flt = MeanStdFilter(4, "cpu")
    chunks = [torch.randn(5, 3, 4) * 3 + 7 for _ in range(6)]
    for c in chunks:
        flt(c.clone())
    allx = torch.cat(chunks).reshape(-1, 4).double()
    assert torch.allclose(flt.mean, allx.mean(0), atol=1e-9)
    assert torch.allclose(torch.sqrt(flt.m2 / (flt.count - 1)), allx.std(0), atol=1e-9)
    x = torch.randn(7, 5, 3) * torch.tensor([1.0, 5.0, 0.0]) + torch.tensor([0.0, 2.0, 1.0])
    standardize_columns_(x, 3)
    assert torch.allclose(x.reshape(-1, 3).mean(0), torch.zeros(3), atol=1e-5)
    assert torch.allclose(x.reshape(-1, 3).std(0, unbiased=False)[:2], torch.ones(2), atol=1e-4)


# ------------------------------------------------------------------ empirical demand + excluded-region mapping (A7, A12)
def _empirical_golden():
    import pandas as pd
    z = np.load(os.path.join(ROOT, "tests", "golden", "empirical_regionmap.npz"))
    wtr = pd.DataFrame(dict(sourcenodeid=z["wtr_source"], destinationregionid=z["wtr_dest"], fixed_costs=z["wtr_cost"]))
    raw = pd.DataFrame(dict(timestep=z["frame_timestep"], region_id=z["frame_region_raw"].astype(int), order_id=z["frame_order"],
                            sku_id=z["frame_sku"].astype(int), quantity=z["frame_qty"].astype(float)))
    return z, wtr, raw


def test_region_map_builder_matches_reference_mapping():
    """build_region_map against what the reference's DataProcessor.map_excluded_regions (preprocessor.py:382-441) made of
    every raw region of the golden frame - shared-warehouse argmin of the mean fixed cost, both fallbacks included."""
    from marlsc_b200.data import build_region_map, map_excluded_regions
    import pandas as pd
    z, wtr, _ = _empirical_golden()
    all_ids, selected = list(z["all_region_ids"]), list(z["selected_region_ids"])
    rmap = build_region_map(all_ids, wtr, selected)
    assert np.array_equal(rmap, z["region_map"])
    assert all(rmap[all_ids.index(s)] == i for i, s in enumerate(selected))          # included regions map to themselves
    assert len(set(rmap)) > 3 and rmap.count(0) > 2                                  # the rule spreads them; fallbacks hit region 0
    ser = pd.Series(all_ids)
    mapped = map_excluded_regions(ser, wtr, selected)
    assert [selected.index(x) for x in mapped] == rmap


def test_empirical_sampler_replays_reference_orders():
    """pack_demand_frame + EmpiricalDemandSampler over the RAW golden frame with the region map applied must emit, for
    the reference's seeds, exactly the orders the reference's EmpiricalDemandSampler emitted (window start from the
    same rng.integers draw, (region_id, order_id) grouping order, duplicate SKU rows summed, SKU ids >= n_skus dropped)."""
    from golden_io import Golden
    from marlsc_b200.components import EmpiricalDemandSampler
    from marlsc_b200.context import create_environment_context
    from marlsc_b200.data import PreprocessedData, pack_demand_frame
    from marlsc_b200.seeds import ENVIRONMENT_SEEDS, SeedManager
    z, wtr, raw = _empirical_golden()
    g = Golden("empirical_regionmap")
    rmap = z["region_map"]
    mapped = raw.assign(region_id=rmap[raw["region_id"].to_numpy()])                 # what the reference's preprocessing stores
    frame = pack_demand_frame(mapped, g.S)
    assert frame.n_timesteps == 40 and frame.order_qty.dtype == np.uint8
    with pytest.raises(Exception, match="requires data_source.type='real_world'"):   # the reference's rule, unless lifted
        environment_config_from_dict(dict(g.env, allow_region_mismatch=True))
    cfg = environment_config_from_dict(dict(g.env, allow_region_mismatch=True, allow_empirical_frame=True))
    ctx = create_environment_context(cfg, preprocessed_data=PreprocessedData(mapped))
    for i in range(g.N):
        sm = SeedManager(root_seed=int(z["env_seeds"][i]), seed_registry=ENVIRONMENT_SEEDS)
        sm.advance_episode()
        smp = EmpiricalDemandSampler(ctx, cfg.components.demand_sampler)
        smp.reset(sm.get_rng("demand_sampler"))
        assert smp.start_index() == int(z["window_start"][i])
        for t in range(g.T):
            mine = smp.sample(t)
            ref = g.orders(i, t)
            assert len(mine) == len(ref)
            for o, (r, q) in zip(mine, ref):
                assert o.region_id == r and np.array_equal(o.sku_demands, q)
    # too short a frame fails like the reference
    with pytest.raises(ValueError, match="episode_length"):
        EmpiricalDemandSampler(create_environment_context(cfg, preprocessed_data=PreprocessedData(mapped[mapped["timestep"] < 10])),
                               cfg.components.demand_sampler)
    with pytest.raises(ValueError, match="requires preprocessed_data"):
        EmpiricalDemandSampler(create_environment_context(cfg), cfg.components.demand_sampler)


# ------------------------------------------------------------------ boundary hygiene
def test_ctypes_structs_match_the_header_layout(tmp_path):
    """sizeof / offsetof of every struct of include/marlsc_b200.h as the C compiler lays them out against the ctypes
    mirrors in _capi.py (a binding that is a field short reads garbage; INTEGRATION.md's stub is generated from these)."""
    import subprocess
    from marlsc_b200 import _capi
    structs = {"marlsc_env_spec_t": _capi.EnvSpecC, "marlsc_env_state_t": _capi.EnvStateC, "marlsc_step_io_t": _capi.StepIOC,
               "marlsc_host_step_t": _capi.HostStepC}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "marlsc_b200.h"', 'int main(void) {']
    for cname, cls in structs.items():
        lines.append(f'  printf("{cname} %zu\\n", sizeof({cname}));')
        for fname, _ in cls._fields_:
            lines.append(f'  printf("{cname}.{fname} %zu\\n", offsetof({cname}, {fname}));')
    lines += ['  return 0;', '}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    got = dict(l.split() for l in subprocess.check_output([str(exe)], text=True).splitlines())
    for cname, cls in structs.items():
        assert int(got[cname]) == ctypes.sizeof(cls), cname
        for fname, _ in cls._fields_:
            assert int(got[f"{cname}.{fname}"]) == getattr(cls, fname).offset, f"{cname}.{fname}"
    # and the header has no field the mirrors lack
    hdr = open(os.path.join(ROOT, "include", "marlsc_b200.h")).read()
    for cname, cls in structs.items():
        body = re.search(r"typedef struct \w+ \{([^}]*)\} " + cname + ";", hdr).group(1)
        body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
        names = re.findall(r"(\w+)\s*;", body)
        assert names == [f for f, _ in cls._fields_], cname


def test_registry_rejects_classes_without_spec_fields_and_meanstd_warns():
    class HostOnlyAllocator:                     # the reference's kind of component: arithmetic in Python
        def allocate(self, orders, inventories):
            return None
    with pytest.raises(TypeError, match="spec_fields"):
        registry.register_demand_allocator("host_only", HostOnlyAllocator)
    assert "host_only" not in registry.DEMAND_ALLOCATOR_REGISTRY
    from marlsc_b200.spec import build_env_spec
    cfg = environment_config_from_dict(small_default())
    with pytest.warns(UserWarning, match="running filter"):
        spec = build_env_spec(cfg, obs_normalization="meanstd")
    assert spec.scalars["obs_norm"] == 0


def test_integration_md_stub_structs_match_the_binding():
    """The reference-side ctypes stub printed in INTEGRATION.md must lay its structs out exactly like the binding the
    tests use (round 1's stub was two fields short of marlsc_step_io_t)."""
    from marlsc_b200 import _capi
    md = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    block = md[md.index("# src/environment/envs/_b200.py"):]
    block = block[:block.index("def make_env")]
    block = "\n".join(l for l in block.splitlines() if not l.startswith("lib = "))
    ns = {}
    exec(block, ns)
    for mine, theirs in ((ns["Spec"], _capi.EnvSpecC), (ns["State"], _capi.EnvStateC), (ns["StepIO"], _capi.StepIOC)):
        assert [f for f, _ in mine._fields_] == [f for f, _ in theirs._fields_]
        assert ctypes.sizeof(mine) == ctypes.sizeof(theirs)
        for f, _ in mine._fields_:
            assert getattr(mine, f).offset == getattr(theirs, f).offset, f
    assert "abi_version=2" in md and _capi.ABI_VERSION == 2


def test_pack_lines_roundtrip_and_balance():
    """Sparse demand lines (include/marlsc_b200.h, marlsc_step_io.lines): every (order, SKU) cell appears once, the lines
    of a SKU keep the order sequence the reference allocator meets them in (demand_allocator.py:150-208), every SKU has
    one (stream, slot), and the balanced dealing shortens an environment's block."""
    from marlsc_b200.demand import pack_lines, pack_orders, unpack_lines
    rng = np.random.default_rng(3)
    S, E = 100, 9
    per_env = []
    for e in range(E):
        n = 0 if e == 4 else int(rng.integers(1, 70))
        orders = sorted(((int(rng.integers(0, 50)), ((rng.random(S) < 0.2) * rng.integers(1, 9, S)).astype(np.int64)) for _ in range(n)),
                        key=lambda x: x[0])
        per_env.append(orders)
    batch = pack_orders(per_env, S)
    region_map = [(r * 7) % 50 for r in range(50)]
    rounds = {}
    for balance in (True, False):
        lb = pack_lines(batch, region_map=region_map, balance=balance)
        rounds[balance] = np.diff(lb.offsets)
        assert np.all(rounds[balance] % 2 == 0) and lb.lines.shape[1] == 32 and lb.lines.dtype == np.uint16
        total = 0
        for e in range(E):
            exp = {}
            for r, q in per_env[e]:
                for sku in np.nonzero(q)[0]:
                    exp.setdefault(int(sku), []).append((region_map[r], int(q[sku])))
            assert unpack_lines(lb, e) == exp, (e, balance)
            total += sum(len(v) for v in exp.values())
            r0, r1 = lb.offsets[e], lb.offsets[e + 1]
            if r1 > r0:                                   # SKU maps: every SKU named exactly once
                hdr = lb.lines[r0:r0 + 2].reshape(1, 32, 2)[0]       # entries 0, 1 of every lane
                ids = np.concatenate([hdr[:, 0] & 0xff, hdr[:, 0] >> 8, hdr[:, 1] & 0xff, hdr[:, 1] >> 8])
                assert sorted(ids[ids != 255].tolist()) == list(range(S))
        assert lb.n_lines == total
        assert rounds[balance][4] == 0                    # an environment without demand owns no rounds
    assert rounds[True].sum() < rounds[False].sum()
    longest = [max(sum(len(v) for k, v in unpack_lines(pack_lines(batch, balance=False), e).items() if k % 32 == l) for l in range(32)) for e in range(E)]
    assert np.array_equal(rounds[False], np.where(np.array(longest) > 0, (np.array(longest) + 3) & ~1, 0))


def test_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (no GPU needed): one JSON line with the reference arm's keys - the same metric / unit /
    config as the GPU arm, `impl`, a `cpu_baseline` describing this run and an `e2e` object with zero copy bytes. Runs the
    reference's own env modules when oracle/_ref is populated (build() does that when MARLSC_REFERENCE_ROOT names a marl-sc
    checkout), else the oracle port."""
    import json
    import subprocess
    import sys
    root = pathlib.Path(__file__).resolve().parents[1]
    out = subprocess.run([sys.executable, str(root / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=str(root))
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "agent_steps_per_sec_env_step_plus_gae"
    assert line["unit"] == "agent-steps/s" and line["higher_is_better"] is True and line["value"] > 0
    assert line["steps"] == 1 and line["warmup"] == 1 and line["n_gpus"] == 1
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    assert line["e2e"] == dict(value=line["value"], unit=line["unit"], h2d_bytes_per_step=0, d2h_bytes_per_step=0)
    assert "BASELINE configs[2]" in line["config"]["workload"]


def test_bench_dump_outputs_writes_a_fixed_environment_sample(tmp_path, monkeypatch):
    """`bench.py --dump-outputs`: under the byte cap every array keeps the same seeded sample of environments (float32,
    float64 kept), a second run writes identical files, and a batch that fits is written whole."""
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 20)
    E, W, D, T = 4096, 3, 40, 20
    obs, rew = torch.randn(E, W, D), torch.randn(T, E, W, dtype=torch.float64)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), dict(observations=(obs, 0), rewards=(rew, 1)), E)
    o, r = np.load(tmp_path / "a" / "observations.npy"), np.load(tmp_path / "a" / "rewards.npy")
    k = o.shape[0]
    assert 0 < k < E and r.shape == (T, k, W) and o.dtype == np.float32 and r.dtype == np.float64
    assert o.nbytes + r.nbytes <= bench.DUMP_BYTES
    idx = np.flatnonzero(np.isin(obs[:, 0, 0].numpy(), o[:, 0, 0]))                # the sampled environments
    assert len(idx) == k and np.array_equal(o, obs[idx].numpy()) and np.array_equal(r, rew[:, idx].numpy())
    for name in ("observations", "rewards"):
        assert np.array_equal(np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy"))
    bench.dump_outputs(str(tmp_path / "whole"), dict(rewards=(rew[:, :64], 1)), 64)
    assert np.array_equal(np.load(tmp_path / "whole" / "rewards.npy"), rew[:, :64].numpy())
    monkeypatch.setattr(bench, "DUMP_BYTES", 100)                # one environment's observations alone are 480 bytes
    with pytest.raises(ValueError, match="exceed"):
        bench.dump_outputs(str(tmp_path / "none"), dict(observations=(obs, 0)), E)


def test_line_streams_carry_the_allocation_the_oracle_computes():
    """The contract of the sparse demand format (include/marlsc_b200.h): with the lean capability set the greedy allocation
    of one SKU never looks at another SKU, so walking every SKU's lines - in stream sequence, down the region's warehouse
    priority list - gives the stock the sequential allocator of the reference ends with (demand_allocator.py:150-208,
    as restated in the oracle). Checked on the CPU from `pack_lines` output alone, balanced and round-robin dealing."""
    from marlsc_b200.demand import pack_lines, pack_orders, unpack_lines
    from oracle.inventory_oracle import OracleEnv
    from parity_common import _lean_env_dict
    rng = np.random.default_rng(21)
    W, S, R = 6, 40, 9
    env_dict = _lean_env_dict(rng, W, S, R, "shipment", True, 3)
    out_var = np.asarray(env_dict["cost_structure"]["shipment_cost"]["outbound_variable"])       # [W, R]
    E = 5
    per_env = []
    for e in range(E):
        orders = [(int(rng.integers(0, R)), np.where(rng.random(S) < 0.4, rng.integers(1, 9, S), 0).astype(float))
                  for _ in range(int(rng.integers(0, 25)))]
        per_env.append(orders)
    batch = pack_orders(per_env, S)
    for balance in (True, False):
        lines = pack_lines(batch, balance=balance)
        for e in range(E):
            o = OracleEnv(env_dict)
            o.reset(np.full((W, S), 5))
            want = o.step(np.full((W, S), -1.0, dtype=np.float32), per_env[e])        # action -1: nothing is ordered
            stock = np.full((W, S), 5, dtype=np.int64)                                 # leads >= 1: nothing arrives at t = 0
            for sku, seq in unpack_lines(lines, e).items():
                for region, qty in seq:
                    for w in np.argsort(out_var[:, region], kind="stable"):            # cheapest warehouse first
                        take = min(qty, stock[w, sku])
                        stock[w, sku] -= take
                        qty -= take
                        if qty == 0:
                            break
            assert np.array_equal(stock, want["inventory"]), (e, balance)
