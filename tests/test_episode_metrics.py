"""-m gpu: per-episode metrics (marlsc_env_set_metrics, BatchedInventoryEnv(episode_metrics=True), rollout.evaluate) against
the oracle, the golden trajectories, the other state layout and the step without metrics."""
import ctypes as C

import numpy as np
import pytest
import torch

from golden_io import NAMES, Golden
from parity_common import _lean_env_dict, spec_for, step_orders

pytestmark = pytest.mark.gpu

UNITS = ("ordered_units", "shipped_units", "demand_units", "lost_units")
COSTS = ("holding_cost", "penalty_cost", "outbound_cost", "inbound_cost")


def _metrics(env):
    return {k: v.cpu().numpy() for k, v in env.episode_metrics().items()}


@pytest.mark.parametrize("W,S,R,lost,pen_uniform,max_orders,lead_hi,variant", [
    (7, 68, 9, "closest", False, 9, 3, "float"),             # per-SKU penalties, three SKUs on some lanes (ragged)
    (10, 100, 50, "shipment", True, 30, 6, "qty"),           # uint8 order quantities
    (10, 100, 50, "shipment", False, 30, 6, "policy"),       # base-stock heuristic evaluated inside the step
    (6, 64, 12, "shipment", True, 20, 4, "team"),            # team-scope rewards (the reward kernel K1d)
    (10, 100, 50, "closest", True, 30, 6, "region_map"),     # 50 raw regions mapped onto 10
])
def test_compact_metrics_vs_oracle(W, S, R, lost, pen_uniform, max_orders, lead_hi, variant):
    """Two episodes with a reset between them, scarce stock (lines split and lost), empty environments and a batch that
    does not fill the last CTA: unit metrics equal the oracle's per-step sums exactly, costs to 1e-9, the return to the
    sum of the float32 rewards, and the second episode starts from zero."""
    from marlsc_b200.config import environment_config_from_dict
    from marlsc_b200.demand import pack_orders
    from marlsc_b200.envs import BatchedInventoryEnv
    from oracle.inventory_oracle import OracleEnv
    rng = np.random.default_rng(W * 100 + S + len(variant))
    R_cost = 10 if variant == "region_map" else R
    env_dict = _lean_env_dict(rng, W, S, R_cost, lost, pen_uniform, lead_hi, scope="team" if variant == "team" else "agent")
    cfg = environment_config_from_dict(dict(env_dict, allow_region_mismatch=True))
    region_map = [int(x) for x in rng.integers(0, R_cost, R)] if variant == "region_map" else None
    E = 11
    env = BatchedInventoryEnv(cfg, E, device="cuda:0", host_samplers=False, region_map=region_map, layout="compact",
                              episode_metrics=True)
    assert env.layout == "compact"
    oracles = [OracleEnv(env_dict) for _ in range(E)]
    maxq = np.asarray(env_dict["action_space"]["params"]["max_order_quantities"])
    level = torch.from_numpy(rng.uniform(0, 40, (E, W, S)).astype(np.float32)).cuda()
    lost_any = False
    for episode in range(2):
        env.reset()
        for o in oracles:
            o.reset(np.full((W, S), 6))
        exp = {k: np.zeros((E, W)) for k in ("ordered_units", "shipped_units") + COSTS}
        exp.update(demand_units=np.zeros(E), lost_units=np.zeros(E))
        ret = np.zeros((E, W))
        done = False
        t = 0
        while not done:
            per_env = []
            for i in range(E):
                if i == 1 or (i == 3 and t % 2):
                    per_env.append([])
                    continue
                orders = []
                for _ in range(int(rng.integers(max_orders // 2, max_orders + 1))):
                    q = np.where(rng.random(S) < 0.3, rng.integers(1, 12, S), 0)
                    if rng.random() < 0.1:
                        q[:] = 0
                    orders.append((int(rng.integers(0, R)), q.astype(float)))
                per_env.append(orders)
            batch = pack_orders(per_env, S)
            if variant == "qty":
                qa = rng.integers(0, 40, (E, W, S)).astype(np.uint8)
                act = (2.0 * np.minimum(qa, maxq) / maxq - 1.0).astype(np.float32)
                _, rew, done = env.step(torch.from_numpy(qa).cuda(), orders=batch)
            elif variant == "policy":
                act = env.base_stock_actions(level).cpu().numpy()       # the policy kernel, from the same state
                _, rew, done = env.step(None, orders=batch, base_stock_level=level)
            else:
                act = rng.uniform(-1, 1, (E, W, S)).astype(np.float32)
                _, rew, done = env.step(torch.from_numpy(act).cuda(), orders=batch)
            ret += rew.double().cpu().numpy()
            for i, o in enumerate(oracles):
                mapped = [(region_map[rg], q) for rg, q in per_env[i]] if region_map else per_env[i]
                out = o.step(act[i], mapped)
                exp["ordered_units"][i] += out["ordered"].sum(1)
                exp["shipped_units"][i] += out["ship_qty"].sum(1)
                exp["lost_units"][i] += out["unfulfilled"].sum()
                exp["demand_units"][i] += sum(q.sum() for _, q in per_env[i])
                for k, ok in zip(COSTS, ("cost_hold", "cost_pen", "cost_out", "cost_in")):
                    exp[k][i] += out[ok]
                lost_any = lost_any or out["lost_orders"].sum() > 0
            t += 1
        got = _metrics(env)
        for k in UNITS:
            assert np.array_equal(got[k], exp[k]), (episode, k)
        for k in COSTS:
            np.testing.assert_allclose(got[k], exp[k], rtol=1e-9, atol=1e-9, err_msg=f"episode {episode} {k}")
        np.testing.assert_allclose(got["episode_return"], ret, rtol=1e-6)
        assert np.array_equal(got["demand_units"], got["shipped_units"].sum(1) + got["lost_units"])
        if variant != "team":
            np.testing.assert_allclose(got["episode_return"], -0.1 * got["total_cost"], rtol=1e-6)
    assert lost_any, "workload was meant to lose sales"
    env.close()


def _golden_layouts(g):
    from marlsc_b200.envs import BatchedInventoryEnv
    cfg, _ = spec_for(g)
    env = BatchedInventoryEnv(cfg, 1, device="cuda:0", host_samplers=False)
    auto = env.layout
    env.close()
    return [None, "wide"] if auto == "compact" else [None]


@pytest.mark.parametrize("name", NAMES)
def test_metrics_match_golden_sums(name):
    """Every layout a golden scenario runs on (automatic choice, and WIDE): the metrics equal the per-step sums of what
    the reference recorded."""
    from marlsc_b200.envs import BatchedInventoryEnv
    g = Golden(name)
    cfg, _ = spec_for(g)
    meta = dict(obs_normalization=g.meta["obs_normalization"], obs_stats=g.obs_stats, include_warehouse_id=g.meta["include_warehouse_id"])
    ptr = g["order_ptr"]
    demand = np.array([g["order_qty"][ptr[i * g.T]:ptr[i * g.T + g.T]].astype(np.float64).sum() for i in range(g.N)])
    for layout in _golden_layouts(g):
        env = BatchedInventoryEnv(cfg, g.N, device="cuda:0", env_meta=meta, host_samplers=False, layout=layout, episode_metrics=True)
        env.reset(init_inventory=torch.from_numpy(g["init_inventory"]))
        ret = np.zeros((g.N, g.W))
        for t in range(g.T):
            lead = g["lead_times"][:, t].astype(np.uint8) if g.meta["stochastic_lead"] else None
            _, rew, _ = env.step(torch.from_numpy(g["actions"][:, t]).to("cuda:0"), orders=step_orders(g, t), actual_lead=lead)
            ret += rew.double().cpu().numpy()
        got = _metrics(env)
        what = f"{name} ({env.layout})"
        for k, gk in zip(COSTS, ("cost_hold", "cost_pen", "cost_out", "cost_in")):
            np.testing.assert_allclose(got[k], g[gk].sum(1), rtol=1e-5, atol=1e-5, err_msg=f"{what} {k}")
        assert np.array_equal(got["ordered_units"], g["ordered"].astype(np.float64).sum((1, 3))), what
        assert np.array_equal(got["lost_units"], g["unfulfilled"].astype(np.float64).sum((1, 2, 3))), what
        assert np.array_equal(got["demand_units"], demand), what
        if "ship_qty" in g.z:
            assert np.array_equal(got["shipped_units"], g["ship_qty"].astype(np.float64).sum((1, 3))), what
        else:                                                # "lite" files carry no shipment cube
            assert np.array_equal(got["shipped_units"].sum(1), demand - got["lost_units"]), what
        np.testing.assert_allclose(got["episode_return"], ret, rtol=1e-6, err_msg=what)
        env.close()


def _large_cfg(episode_length=20):
    from golden.scenarios import large_network
    from marlsc_b200.config import environment_config_from_dict
    d = large_network()
    d["episode_length"] = episode_length
    return environment_config_from_dict(dict(d, allow_region_mismatch=True))


@pytest.mark.parametrize("policy", ["random", "base_stock"])
def test_compact_metrics_equal_wide_metrics(policy):
    """The large shape, same device-drawn demand and the same actions on both layouts: units exact, costs to 1e-6 (WIDE
    folds its float32 per-step cost breakdown)."""
    from marlsc_b200.envs import BatchedInventoryEnv
    from marlsc_b200.rollout import base_stock_levels
    cfg, E = _large_cfg(), 1000
    a = BatchedInventoryEnv(cfg, E, device="cuda:0", host_samplers=False, device_demand=True, demand_seed=3, episode_metrics=True)
    b = BatchedInventoryEnv(cfg, E, device="cuda:0", host_samplers=False, device_demand=True, demand_seed=3, episode_metrics=True,
                            layout="wide")
    assert a.layout == "compact" and b.layout == "wide"
    a.reset()
    b.reset()
    level = torch.from_numpy(base_stock_levels(a, 2.0).astype(np.float32)).cuda()
    gen = torch.Generator(device="cuda:0").manual_seed(4)
    done = False
    while not done:
        if policy == "random":
            act = torch.rand((E, 10, 100), device="cuda:0", generator=gen) * 2 - 1
            a.step(act)
        else:
            act = b.base_stock_actions(level)
            a.step(None, base_stock_level=level)
        _, _, done = b.step(act)
    ga, gb = _metrics(a), _metrics(b)
    for k in UNITS:
        assert np.array_equal(ga[k], gb[k]), k
    for k in COSTS + ("episode_return",):
        np.testing.assert_allclose(ga[k], gb[k], rtol=1e-6, atol=1e-6, err_msg=k)
    assert ga["demand_units"].sum() > 0
    if policy == "base_stock":                               # random actions overstock; the z = 2 levels run short
        assert ga["lost_units"].sum() > 0
    a.close()
    b.close()


def test_metrics_do_not_perturb_the_step():
    """Metrics on against metrics off, the split step and then the in-step base-stock policy: observations, rewards,
    truncation and state bit-identical every step. Then the same episode through marlsc_env_rollout_host
    (HostRollout.run_lines) and through step() accumulates the same metrics."""
    from marlsc_b200.demand import pack_lines, pack_orders
    from marlsc_b200.envs import BatchedInventoryEnv, HostRollout
    cfg, E = _large_cfg(16), 333
    a = BatchedInventoryEnv(cfg, E, device="cuda:0", host_samplers=False, device_demand=True, demand_seed=9, seed=1)
    b = BatchedInventoryEnv(cfg, E, device="cuda:0", host_samplers=False, device_demand=True, demand_seed=9, seed=1, episode_metrics=True)
    assert a.layout == b.layout == "compact"
    assert torch.equal(a.reset(), b.reset())
    gen = torch.Generator(device="cuda:0").manual_seed(2)
    level = torch.rand((E, 10, 100), device="cuda:0", generator=gen) * 30
    for t in range(16):
        if t < 8:
            act = torch.rand((E, 10, 100), device="cuda:0", generator=gen) * 2 - 1
            oa, ra, da = a.step(act)
            ob, rb, db = b.step(act)
        else:
            oa, ra, da = a.step(None, base_stock_level=level)
            ob, rb, db = b.step(None, base_stock_level=level)
        assert torch.equal(oa, ob) and torch.equal(ra, rb) and da == db, t
        assert torch.equal(a.truncated, b.truncated) and torch.equal(a.inventory, b.inventory), t
        assert torch.equal(a.ring_qty, b.ring_qty) and torch.equal(a.demand_hist, b.demand_hist), t
    a.close()
    b.close()

    # host rollout against step(): uint8 quantities and host-packed lines
    rng = np.random.default_rng(5)
    E, T = 37, 16
    c = BatchedInventoryEnv(cfg, E, device="cuda:0", host_samplers=False, episode_metrics=True, seed=2)
    d = BatchedInventoryEnv(cfg, E, device="cuda:0", host_samplers=False, episode_metrics=True, seed=2)
    W, S, R = 10, 100, c.n_regions
    batches = []
    for t in range(T):
        per_env = [[(int(rng.integers(0, R)), np.where(rng.random(S) < 0.3, rng.integers(1, 12, S), 0).astype(float))
                    for _ in range(int(rng.integers(0, 40)))] for _ in range(E)]
        batches.append(pack_lines(pack_orders(per_env, S), c.spec.tables["region_map"]))
    qty = [torch.from_numpy(rng.integers(0, 30, (E, W, S)).astype(np.uint8)) for _ in range(T)]
    c.reset()
    d.reset()
    hr = HostRollout(c, max_rounds_per_step=max(max(lb.n_rounds for lb in batches), 1))
    rew_host = torch.empty((T, E, W)).pin_memory()
    rew_dev = torch.empty((T, E, W), device="cuda:0")
    hr.run_lines([q.pin_memory() for q in qty], [torch.from_numpy(lb.offsets).pin_memory() for lb in batches],
                 [torch.from_numpy(lb.lines.view(np.int16)).pin_memory() for lb in batches], [lb.n_rounds for lb in batches],
                 rew_host, rew_dev)
    for t in range(T):
        d.step(qty[t].cuda(), orders=batches[t])
    mc, md = _metrics(c), _metrics(d)
    for k in mc:
        assert np.array_equal(mc[k], md[k]), k
    assert mc["demand_units"].sum() > 0
    c.close()
    d.close()


def test_evaluate_base_stock_known_answer_and_actor_critic():
    """evaluate() of the base-stock policy (z = 2) on BASELINE config #1, seeded like the dict adapter, reproduces the
    reference's first three episode returns; evaluate() of an ActorCritic equals a hand-written deterministic loop."""
    from golden.scenarios import small_default
    from marlsc_b200.config import environment_config_from_dict
    from marlsc_b200.envs import BatchedInventoryEnv
    from marlsc_b200.rollout import ActorCritic, base_stock_levels, evaluate
    cfg = environment_config_from_dict(small_default())
    env = BatchedInventoryEnv(cfg, 1, device="cuda:0", env_seeds=[123], env_meta={"data_mode": "train"}, episode_metrics=True)
    res = evaluate(env, base_stock_levels(env, 2.0), 3)
    np.testing.assert_allclose(res["episode_return"].sum(-1)[:, 0].cpu().numpy(), [-158.8005, -165.7435, -170.5540], atol=2e-3)
    assert res["fill_rate"].shape == (3, 1) and 0.0 < float(res["fill_rate"].min()) <= 1.0
    s = res.summary()
    assert s["episode_return"]["mean"] == pytest.approx(float(res["episode_return"].sum(-1).mean()))
    env.close()

    E = 64
    torch.manual_seed(0)
    a = BatchedInventoryEnv(cfg, E, device="cuda:0", host_samplers=False, device_demand=True, demand_seed=4, seed=8, episode_metrics=True)
    b = BatchedInventoryEnv(cfg, E, device="cuda:0", host_samplers=False, device_demand=True, demand_seed=4, seed=8)
    ac = ActorCritic(a.obs_dim, a.n_warehouses, a.n_skus, actor_hidden=(32,), logstd_init=0.5).cuda()
    res = evaluate(a, ac, 2)
    for ep in range(2):
        obs, done, total = b.reset(), False, torch.zeros((E, 3), dtype=torch.float64, device="cuda:0")
        while not done:
            with torch.no_grad():
                act = ac.action_mean(obs).clamp(-1.0, 1.0)
            obs, rew, done = b.step(act.contiguous())
            total += rew.double()
        assert torch.equal(res["episode_return"][ep], total), ep
    a.close()
    b.close()


def test_metrics_refuse_unsupported_combinations():
    """The compact fused kernel does not accumulate metrics (either order of the two switches), and a WIDE step with
    metrics needs the diagnostic outputs."""
    from marlsc_b200 import _capi
    from marlsc_b200.demand import pack_orders
    from marlsc_b200.envs import BatchedInventoryEnv
    cfg = _large_cfg()
    with pytest.raises(ValueError, match="fused"):
        BatchedInventoryEnv(cfg, 8, device="cuda:0", host_samplers=False, layout="compact", fused_kernel=True, episode_metrics=True)
    L = _capi.lib()
    env = BatchedInventoryEnv(cfg, 8, device="cuda:0", host_samplers=False, layout="compact", fused_kernel=True)
    bufs = [torch.zeros(80, dtype=torch.float64, device="cuda:0") for _ in range(9)]
    m = _capi.EpisodeMetricsC(*[t.data_ptr() for t in bufs])
    assert L.marlsc_env_set_metrics(env._h, C.byref(m)) == -4           # MARLSC_EUNSUPPORTED
    env.close()
    env = BatchedInventoryEnv(cfg, 8, device="cuda:0", host_samplers=False, episode_metrics=True)
    assert L.marlsc_env_set_fused(env._h, 1) == -4
    partial = _capi.EpisodeMetricsC(*[t.data_ptr() for t in bufs[:8]])
    assert L.marlsc_env_set_metrics(env._h, C.byref(partial)) == -1     # MARLSC_EINVAL: a pointer is missing
    env.close()
    env = BatchedInventoryEnv(cfg, 8, device="cuda:0", host_samplers=False, layout="wide")    # no diagnostic buffers
    _capi.check(L.marlsc_env_set_metrics(env._h, C.byref(m)))
    env.reset()
    with pytest.raises(ValueError, match="d_ordered"):
        env.step(torch.zeros((8, 10, 100), device="cuda:0"), orders=pack_orders([[] for _ in range(8)], 100))
    env.close()
