"""-m gpu: the CUDA library (through its C ABI via marlsc_b200) against the reference's golden
trajectories and the oracle. Integer quantities bit-exact; costs / rewards / observations / GAE to
rtol 1e-5 (BASELINE.json north_star)."""
import numpy as np
import pytest
import torch

from golden_io import NAMES, Golden
from parity_common import _lean_env_dict  # noqa: F401  (shared with the CPU tests)
from parity_common import compare_step, spec_for, step_orders

pytestmark = pytest.mark.gpu


def _run(g, team_size=0, region_map=None, region_shift=None, steps=None, diagnostics=True, generic=False, fused=False, layout=None):
    from marlsc_b200.envs import BatchedInventoryEnv
    cfg, _ = spec_for(g)
    meta = dict(obs_normalization=g.meta["obs_normalization"], obs_stats=g.obs_stats,
                include_warehouse_id=g.meta["include_warehouse_id"])
    env = BatchedInventoryEnv(cfg, g.N, device="cuda:0", env_meta=meta, host_samplers=False, diagnostics=diagnostics,
                              team_size=team_size, region_map=region_map, generic_kernel=generic, fused_kernel=fused, layout=layout)
    # poison the state so reset has to clear it
    env.ring_qty.fill_(5)
    env.inventory.fill_(123)
    obs0 = env.reset(init_inventory=torch.from_numpy(g["init_inventory"]))
    np.testing.assert_allclose(obs0.cpu().numpy(), g["obs0_local"], rtol=1e-5, atol=1e-6)
    stochastic = g.meta["stochastic_lead"]
    for t in range(steps or g.T):
        act = torch.from_numpy(g["actions"][:, t]).to("cuda:0")
        lead = g["lead_times"][:, t].astype(np.uint8) if stochastic else None
        obs, rew, trunc = env.step(act, orders=step_orders(g, t, region_shift), actual_lead=lead)
        out = {k: v.cpu().numpy() for k, v in env.diag.items()}
        out.update(inventory=env.inventory.cpu().numpy(), rewards=rew.cpu().numpy(), obs=obs.cpu().numpy(),
                   trunc=env.truncated.cpu().numpy())
        assert bool(trunc) == bool(g["trunc"][0, t])
        compare_step(g, t, out, what=f"cuda team={env.team_size} layout={env.layout} ")
    layout_used = env.layout
    env.close()
    return layout_used


@pytest.mark.parametrize("name", NAMES)
def test_cuda_matches_reference_auto_team(name):
    _run(Golden(name))


@pytest.mark.parametrize("mode", ["auto", "split", "fused", "generic"])
@pytest.mark.parametrize("name", NAMES)
def test_cuda_without_diagnostics(name, mode):
    """No diagnostic outputs. ``auto``: the compact layout and its step where the configuration qualifies (the large
    networks), else the wide lean path; ``split``: the wide layout's lean path - the four-kernel split step for teams of
    8+ lanes, else the lean fused kernel; ``fused`` keeps lean launches in the wide fused kernel; ``generic`` forces the
    generic instantiation."""
    used = _run(Golden(name), diagnostics=False, generic=mode == "generic", fused=mode == "fused",
                layout="wide" if mode == "split" else None)
    if name.startswith("large_network"):
        assert used == ("compact" if mode == "auto" else "wide")


@pytest.mark.parametrize("team", [1, 2, 4, 8, 16, 32])
@pytest.mark.parametrize("name", ["allfeat_ratio_stochastic", "basestock_cost_meanstd"])
def test_cuda_team_sizes_small(name, team):
    _run(Golden(name), team_size=team)


@pytest.mark.parametrize("team", [16, 32])
def test_cuda_team_sizes_large(team):
    _run(Golden("large_network"), team_size=team, steps=6)


@pytest.mark.parametrize("mode", ["split", "fused", "diagnostics"])
def test_cuda_two_warp_team_large(mode):
    """64 lanes per environment (two warps): the lean paths without diagnostics, the 32-lane generic fallback
    with them."""
    _run(Golden("large_network"), team_size=64, steps=8, diagnostics=mode == "diagnostics", fused=mode == "fused")


@pytest.mark.parametrize("team", [8, 16, 32])
@pytest.mark.parametrize("name", ["small_default", "regions_ne_warehouses"])
def test_cuda_split_step_small_shapes(name, team):
    """The split step on the small networks (teams wider than the automatic choice, one SKU per lane)."""
    _run(Golden(name), team_size=team, diagnostics=False)


def test_tiny_network_takes_the_split_step_automatically():
    """A network with a handful of SKUs (BASELINE configs[1]: 3 warehouses x 2 SKUs) runs the split step with 8-lane teams
    by default (up to 4,096 environments; larger batches keep the thread-per-environment kernel); launches the split step does not cover
    (here: the fused-kernel switch) fall back to a thread per environment. Both paths against the golden trajectory, and
    against each other on a ragged batch."""
    from golden.scenarios import small_default
    from marlsc_b200.config import environment_config_from_dict
    from marlsc_b200.envs import BatchedInventoryEnv
    g = Golden("small_default")
    _run(g, diagnostics=False)                       # automatic choice
    _run(g, diagnostics=False, fused=True)           # thread per environment
    cfg = environment_config_from_dict(small_default())
    E = 301
    a = BatchedInventoryEnv(cfg, E, device="cuda:0", host_samplers=False, device_demand=True, demand_seed=3)
    b = BatchedInventoryEnv(cfg, E, device="cuda:0", host_samplers=False, device_demand=True, demand_seed=3, team_size=1)
    assert a.team_size == 8 and b.team_size == 1 and a.layout == b.layout == "wide"
    assert torch.equal(a.reset(), b.reset())
    gen = torch.Generator(device="cuda:0").manual_seed(0)
    for t in range(40):
        act = torch.rand((E, a.n_warehouses, a.n_skus), device="cuda:0", generator=gen) * 2 - 1
        oa, ra, _ = a.step(act)
        ob, rb, _ = b.step(act)
        assert torch.equal(a.inventory, b.inventory) and torch.equal(a.ring_qty, b.ring_qty), t
        np.testing.assert_allclose(ra.cpu().numpy(), rb.cpu().numpy(), rtol=1e-6, atol=1e-6)
        np.testing.assert_allclose(oa.cpu().numpy(), ob.cpu().numpy(), rtol=1e-6, atol=1e-6)


@pytest.mark.parametrize("fused", [False, True])
@pytest.mark.parametrize("team", [0, 64])
@pytest.mark.parametrize("fixed_cost", [0.0, 2.0])
def test_lean_equals_generic_under_stockouts(fixed_cost, team, fused):
    """The lean instantiation allocates through independent per-lane SKU chains (one or two warps per
    environment); the generic one walks every order warehouse by warehouse (and is itself pinned to the golden
    trajectories). On a scarce-inventory large network (constant splitting, lost sales) both must agree exactly."""
    from golden.scenarios import large_network
    from marlsc_b200.config import environment_config_from_dict
    from marlsc_b200.context import create_environment_context
    from marlsc_b200.demand import pack_orders
    from marlsc_b200.envs import BatchedInventoryEnv
    from marlsc_b200.registry import get_demand_sampler
    d = large_network()
    d["allow_region_mismatch"] = True
    d["initial_inventory"] = dict(type="custom", params=dict(values=4))
    if fixed_cost:
        d["cost_structure"]["shipment_cost"]["outbound_fixed"] = [[fixed_cost] * 50] * 10
    cfg = environment_config_from_dict(d)
    E, T = 48, 16
    rng = np.random.default_rng(5)
    samplers = []
    for i in range(E):
        smp = get_demand_sampler(cfg, context=create_environment_context(cfg))
        smp.reset(np.random.default_rng(100 + i))
        samplers.append(smp)
    lean = BatchedInventoryEnv(cfg, E, device="cuda:0", host_samplers=False, team_size=team, fused_kernel=fused)
    gen = BatchedInventoryEnv(cfg, E, device="cuda:0", host_samplers=False, generic_kernel=True)
    o1, o2 = lean.reset().clone(), gen.reset().clone()
    assert torch.equal(o1, o2)
    lost_any = False
    for t in range(T):
        act = torch.from_numpy(rng.uniform(-1, -0.6, (E, 10, 100)).astype(np.float32)).cuda()
        orders = pack_orders([smp.sample(t) for smp in samplers], 100)
        ob1, r1, _ = lean.step(act, orders=orders)
        ob2, r2, _ = gen.step(act, orders=orders)
        assert torch.equal(lean.inventory.to(torch.int32), gen.inventory), f"inventory differs at step {t}"
        if lean.layout == gen.layout:
            assert torch.equal(lean.ring_qty, gen.ring_qty)
        else:                                           # compact ring is indexed by arrival time: compare what is in transit
            assert torch.equal(lean.pending_matrix(), gen.pending_matrix())
        np.testing.assert_allclose(r1.cpu().numpy(), r2.cpu().numpy(), rtol=1e-6, atol=1e-6)
        np.testing.assert_allclose(ob1.cpu().numpy(), ob2.cpu().numpy(), rtol=1e-6, atol=1e-6)
        lost_any = lost_any or bool((lean.inventory == 0).any())
    assert lost_any, "workload was meant to run out of stock"
    assert lean.layout == ("compact" if (fixed_cost == 0.0 and team == 0 and not fused) else "wide")


def test_cuda_region_map():
    g = Golden("small_default")
    R = g.R
    _run(g, region_map=list(range(R)) * 2, region_shift=lambda i, t, j: R * ((i + t + j) % 2), steps=20)


def test_host_samplers_replay_reference_streams():
    """Seeded like the reference (derive_env_seed), the host-side samplers draw the same initial
    inventory, orders and lead times, so no demand has to be fed in to land on the golden trajectory."""
    from marlsc_b200.envs import BatchedInventoryEnv
    for name in ("small_default", "allfeat_ratio_stochastic"):
        g = Golden(name)
        cfg, _ = spec_for(g)
        meta = dict(obs_normalization=g.meta["obs_normalization"], obs_stats=g.obs_stats,
                    include_warehouse_id=g.meta["include_warehouse_id"])
        env = BatchedInventoryEnv(cfg, g.N, device="cuda:0", env_meta=meta, seed=g.meta["base_seed"], diagnostics=True)
        env.reset()
        assert np.array_equal(env.inventory.cpu().numpy(), g["init_inventory"])
        for t in range(min(g.T, 25)):
            obs, rew, _ = env.step(torch.from_numpy(g["actions"][:, t]).to("cuda:0"))
            assert np.array_equal(env.inventory.cpu().numpy(), g["inventory"][:, t])
            np.testing.assert_allclose(rew.cpu().numpy(), g["rewards"][:, t], rtol=1e-5, atol=1e-6)
        env.close()


def test_dict_adapter_matches_reference():
    from marlsc_b200.envs import InventoryEnvironment
    g = Golden("small_default")
    cfg, _ = spec_for(g)
    env = InventoryEnvironment(cfg, seed=int(g["env_seeds"][3]))
    obs, infos = env.reset()
    D = env._compute_local_obs_dim()
    assert set(obs) == {"warehouse_0", "warehouse_1", "warehouse_2"} and obs["warehouse_0"].shape == ((1 + g.W) * D,)
    env.collect_step_info = True
    for t in range(10):
        act = {a: g["actions"][3, t, i] for i, a in enumerate(env.agents)}
        obs, rew, term, trunc, infos = env.step(act)
        np.testing.assert_allclose([rew[a] for a in env.agents], g["rewards"][3, t], rtol=1e-5, atol=1e-6)
        assert np.array_equal(env.inventory, g["inventory"][3, t])
        assert np.array_equal(env._compute_pending_matrix(), g["pending"][3, t])
        info = infos["warehouse_0"]
        assert np.array_equal(info["shipment_quantities_by_sku"], g["ship_by_sku"][3, t])
        np.testing.assert_allclose(info["lost_sales"], g["lost_sales"][3, t], rtol=1e-5, atol=1e-6)
        loc = np.stack([obs[a][:D] for a in env.agents])
        np.testing.assert_allclose(loc, g["obs_local"][3, t], rtol=1e-5, atol=1e-6)
        assert np.array_equal(obs["warehouse_1"][D:], loc.reshape(-1))
        assert not any(term.values()) and not any(trunc.values())


def test_centralized_wrapper_matches_reference_trajectory():
    """CentralizedEnvWrapper (reference: src/environment/envs/single_env.py): global observation, flat joint action,
    summed reward - against the same golden trajectory as the dict adapter."""
    from marlsc_b200.envs import CentralizedEnvWrapper
    g = Golden("small_default")
    cfg, _ = spec_for(g)
    env = CentralizedEnvWrapper(cfg, seed=int(g["env_seeds"][5]))
    obs, info = env.reset()
    assert obs.shape == env.observation_space.shape == (g.W * env._local_obs_dim,)
    assert env.action_space.shape == (g.W * g.S,)
    np.testing.assert_allclose(obs, g["obs0_local"][5].reshape(-1), rtol=1e-5, atol=1e-6)
    for t in range(12):
        obs, rew, term, trunc, info = env.step(g["actions"][5, t].reshape(-1))
        np.testing.assert_allclose(obs, g["obs_local"][5, t].reshape(-1), rtol=1e-5, atol=1e-6)
        np.testing.assert_allclose(rew, g["rewards"][5, t].sum(), rtol=1e-5, atol=1e-6)
        assert not term and not trunc
    assert env.agents == ["warehouse_0", "warehouse_1", "warehouse_2"] and env.episode_length == cfg.episode_length


def test_errors_are_loud():
    from marlsc_b200.envs import BatchedInventoryEnv
    g = Golden("small_default")
    cfg, _ = spec_for(g)
    env = BatchedInventoryEnv(cfg, 4, device="cuda:0", host_samplers=False)
    env.reset()
    with pytest.raises(ValueError):
        env.step(torch.zeros((4, 3, 3), device="cuda:0"))
    with pytest.raises(ValueError):
        env.step(torch.zeros((4, 3, 2), dtype=torch.float64, device="cuda:0"))
    with pytest.raises(RuntimeError):
        env.step(torch.zeros((4, 3, 2), device="cuda:0"))      # no demand source configured
    env.close()


@pytest.mark.parametrize("T,N,cuts", [(1, 5, False), (7, 1, False), (37, 1000, True), (100, 12288, True), (33, 333, True)])
def test_gae_matches_oracle(T, N, cuts):
    from marlsc_b200.rollout import compute_gae
    from oracle.gae_oracle import gae_targets
    rng = np.random.default_rng(T * 7 + N)
    r = rng.normal(-1.5, 1.0, (T, N)).astype(np.float32)
    v = rng.normal(-30, 5.0, (T + 1, N)).astype(np.float32)
    cut = np.zeros(T, np.uint8)
    cv = rng.normal(-30, 5.0, (T, N)).astype(np.float32)
    if cuts:
        cut[rng.integers(0, T, size=3)] = 1
    for gamma, lam, use_cv in ((0.99, 0.95, True), (0.95, 0.9, False), (1.0, 1.0, True)):
        a_ref, t_ref = gae_targets(r, v, gamma, lam, cut.astype(bool) if cuts else None, cv if (cuts and use_cv) else None)
        a, tg = compute_gae(torch.from_numpy(r).cuda(), torch.from_numpy(v).cuda(), gamma, lam,
                            torch.from_numpy(cut).cuda() if cuts else None,
                            torch.from_numpy(cv).cuda() if (cuts and use_cv) else None)
        np.testing.assert_allclose(tg.cpu().numpy(), t_ref, rtol=1e-5, atol=1e-5)
        np.testing.assert_allclose(a.cpu().numpy(), a_ref, rtol=1e-5, atol=1e-4)


def test_gae_shapes_env_agent():
    from marlsc_b200.rollout import compute_gae
    r = torch.randn(8, 16, 3, device="cuda")
    v = torch.randn(9, 16, 3, device="cuda")
    a, tg = compute_gae(r, v, 0.99, 0.95)
    assert a.shape == r.shape and tg.shape == r.shape
    a2, _ = compute_gae(r.reshape(8, 48), v.reshape(9, 48), 0.99, 0.95)
    assert torch.equal(a.reshape(8, 48), a2)


def test_standardize_matches_oracle():
    from marlsc_b200.rollout import standardize_
    from oracle.gae_oracle import standardize
    for n in (1, 31, 4097, 1 << 20):
        x = np.random.default_rng(n).normal(2.0, 3.0, n).astype(np.float32)
        y = standardize_(torch.from_numpy(x).cuda()).cpu().numpy()
        np.testing.assert_allclose(y, standardize(x), rtol=1e-4, atol=2e-5)


def test_rollout_collector_matches_manual_loop():
    """Collector = policy forward -> fused step -> buffer -> GAE; its buffers must equal a hand-rolled
    loop over the same env seeds, and its GAE the oracle's."""
    from golden.scenarios import small_default
    from marlsc_b200.config import environment_config_from_dict
    from marlsc_b200.envs import BatchedInventoryEnv
    from marlsc_b200.rollout import ActorCritic, PPOLearner, RolloutCollector
    from oracle.gae_oracle import gae_targets
    d = small_default()
    d["episode_length"] = 12
    cfg = environment_config_from_dict(d)
    torch.manual_seed(0)
    E, T = 32, 30                                   # crosses two episode boundaries
    env = BatchedInventoryEnv(cfg, E, device="cuda:0", seed=11, env_meta=dict(include_warehouse_id=True))
    pol = ActorCritic(env.obs_dim, 3, 2, actor_hidden=(32,), critic_hidden=(32,), critic_obs_type="global").cuda()
    col = RolloutCollector(env, pol, T, gamma=0.97, lam=0.9, standardize_advantages=False, seed=5)
    ro = col.collect()
    assert ro.cut.cpu().tolist() == [1 if (t + 1) % 12 == 0 else 0 for t in range(T)]
    # same thing by hand on a second env with the same seeds
    env2 = BatchedInventoryEnv(cfg, E, device="cuda:0", seed=11, env_meta=dict(include_warehouse_id=True))
    gen = torch.Generator(device="cuda:0")
    gen.manual_seed(5)
    obs = env2.reset().clone()
    rewards, values, cut_vals = [], [], {}
    with torch.no_grad():
        for t in range(T):
            act, logp, val = pol.act(obs, generator=gen)
            assert torch.equal(obs, ro.obs[t]) and torch.allclose(logp, ro.logp[t])
            o, r, trunc = env2.step(act.contiguous())
            rewards.append(r.clone())
            values.append(val)
            obs = o.clone()
            if trunc:
                cut_vals[t] = pol.value(obs)
                obs = env2.reset().clone()
        values.append(pol.value(obs))
    r = torch.stack(rewards).reshape(T, -1).cpu().numpy()
    v = torch.stack(values).reshape(T + 1, -1).cpu().numpy()
    assert np.array_equal(r, ro.rewards.reshape(T, -1).cpu().numpy())
    cv = np.zeros_like(r)
    for t, x in cut_vals.items():
        cv[t] = x.reshape(-1).cpu().numpy()
    a_ref, t_ref = gae_targets(r, v, 0.97, 0.9, ro.cut.cpu().numpy().astype(bool), cv)
    np.testing.assert_allclose(ro.targets.reshape(T, -1).cpu().numpy(), t_ref, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(ro.advantages.reshape(T, -1).cpu().numpy(), a_ref, rtol=1e-5, atol=1e-4)
    # one learner step runs and changes the weights
    learner = PPOLearner(pol, lr=1e-3, grad_clip=5.0)
    before = pol.log_std.detach().clone()
    stats = learner.minibatch_step(ro, slice(0, 10), slice(0, 16))
    assert np.isfinite(stats["total"]) and not torch.equal(before, pol.log_std.detach())


def test_pipelined_host_rollout_equals_stepwise():
    """marlsc_env_rollout_host (double-buffered host->device copies overlapping the step kernels) must
    give exactly what step-by-step calls give."""
    from marlsc_b200.envs import BatchedInventoryEnv, HostRollout
    g = Golden("small_default")
    cfg, _ = spec_for(g)
    T = 24
    env = BatchedInventoryEnv(cfg, g.N, device="cuda:0", host_samplers=False)
    env.reset(init_inventory=torch.from_numpy(g["init_inventory"]))
    batches = [step_orders(g, t) for t in range(T)]
    hr = HostRollout(env, max(b.n_orders for b in batches))
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()   # noqa: E731
    acts = [pin(g["actions"][:, t]) for t in range(T)]
    offs = [pin(b.offsets) for b in batches]
    regs = [pin(b.region) for b in batches]
    qtys = [pin(b.qty) for b in batches]
    r_host = torch.empty((T, g.N, g.W)).pin_memory()
    r_dev = torch.empty((T, g.N, g.W), device="cuda:0")
    obs = hr.run(acts, offs, regs, qtys, [b.n_orders for b in batches], r_host, r_dev)
    np.testing.assert_allclose(r_host.numpy(), np.moveaxis(g["rewards"][:, :T], 0, 1), rtol=1e-5, atol=1e-6)
    assert torch.equal(r_host, r_dev.cpu())
    assert np.array_equal(env.inventory.cpu().numpy(), g["inventory"][:, T - 1])
    np.testing.assert_allclose(obs.cpu().numpy(), g["obs_local"][:, T - 1], rtol=1e-5, atol=1e-6)
    assert env.timestep == T


# ---------------------------------------------------------------------------- K4 / K5 (SURVEY.md section 8f)
def _small_env(E, **kw):
    from golden.scenarios import small_default
    from marlsc_b200.config import environment_config_from_dict
    from marlsc_b200.envs import BatchedInventoryEnv
    cfg = environment_config_from_dict(small_default())
    return cfg, BatchedInventoryEnv(cfg, E, device="cuda:0", **kw)


def test_device_demand_matches_reference_distribution():
    """Philox stream != PCG64 stream, so the device sampler is checked distributionally against the reference
    sampler's law: order counts ~ Poisson(lambda_orders), SKU inclusion ~ Bernoulli(p), quantities ~
    max(1, Poisson(lambda_quantity)); 5-sigma bands on the moments and a chi-square on the quantity histogram."""
    from scipy import stats
    E = 8192
    cfg, env = _small_env(E, host_samplers=False, device_demand=True, demand_seed=7)
    env.sample_device_demand()
    d = env._dd
    counts = d["counts"].cpu().numpy()
    omax, S, R = d["omax"], 2, 3
    region = d["region"].cpu().numpy().reshape(E, omax)
    qty = d["qty"].cpu().numpy()[:E * omax * S].reshape(E, omax, S)
    assert not env.demand_overflowed()
    valid = np.arange(omax)[None, :] < counts[:, None]
    lam_o, p, lam_q = 4.0, 0.667, 5.0
    n = E * R
    per_region = np.stack([((region == r) & valid).sum(1) for r in range(R)], 1)
    assert abs(per_region.mean() - lam_o) < 5 * np.sqrt(lam_o / n)
    assert abs(per_region.var() - lam_o) < 0.15                                     # Poisson: variance = mean
    assert all((np.diff(region[e][:counts[e]]) >= 0).all() for e in range(0, E, 97))   # region-major like the reference
    q = qty[valid]                                                                   # [n_orders, S]
    inc = (q > 0).mean()
    assert abs(inc - p) < 5 * np.sqrt(p * (1 - p) / q.size)
    nz = q[q > 0].astype(int)
    ks = np.arange(1, 16)
    pmf = stats.poisson.pmf(ks, lam_q)
    pmf[0] += stats.poisson.pmf(0, lam_q)                                            # max(1, .)
    pmf = np.append(pmf, 1 - pmf.sum())                                              # tail bucket >= 16
    obs = np.array([(nz == k).sum() for k in ks] + [(nz >= 16).sum()])
    chi2 = ((obs - nz.size * pmf) ** 2 / (nz.size * pmf)).sum()
    assert chi2 < stats.chi2.ppf(1 - 1e-6, len(pmf) - 1), chi2
    # reproducible: same seed and step index -> same draw; next step differs
    a = d["qty"].clone()
    env._demand_step = 0
    env.sample_device_demand()
    assert torch.equal(a, d["qty"])
    env.sample_device_demand()
    assert not torch.equal(a, d["qty"])
    env.close()


def test_device_lead_times_match_reference_distribution():
    """K4b against the law of the reference's StochasticLeadTimeSampler (lead_time_sampler.py:169-197):
    actual = max(1, expected + U{-d[s]..+d[s]}), independent per environment / cell / step; then a stepped
    environment that draws its own lead times equals one fed the same draws explicitly."""
    from scipy import stats
    from marlsc_b200.envs import BatchedInventoryEnv
    g = Golden("allfeat_ratio_stochastic")
    cfg, _ = spec_for(g)
    meta = dict(obs_normalization=g.meta["obs_normalization"], obs_stats=g.obs_stats,
                include_warehouse_id=g.meta["include_warehouse_id"])
    E = 6000
    env = BatchedInventoryEnv(cfg, E, device="cuda:0", env_meta=meta, host_samplers=False)
    env.enable_device_leads(seed=3)
    a = env.sample_device_leads().cpu().numpy().astype(int)
    exp = np.asarray(env.expected_lead_times, dtype=int)
    md = np.array([0, 1, 2, 1, 0])
    assert a.min() >= 1
    for w in range(3):
        for s in range(5):
            d, x = md[s], a[:, w, s]
            support = np.arange(exp[w, s] - d, exp[w, s] + d + 1)
            pmf = np.full(len(support), 1.0 / len(support))
            clipped = np.maximum(1, support)                     # deviations below 1 pile up on 1
            vals = np.unique(clipped)
            p = np.array([pmf[clipped == v].sum() for v in vals])
            assert set(np.unique(x)) <= set(vals), (w, s)
            if len(vals) > 1:
                obs = np.array([(x == v).sum() for v in vals])
                chi2 = ((obs - E * p) ** 2 / (E * p)).sum()
                assert chi2 < stats.chi2.ppf(1 - 1e-6, len(vals) - 1), (w, s, chi2)
    # cells are independent: neighbouring SKUs of the same warehouse are uncorrelated
    c = np.corrcoef(a[:, 0, 1], a[:, 0, 2])[0, 1]
    assert abs(c) < 5 / np.sqrt(E)
    env._dl["step"] = 0
    b = env.sample_device_leads().clone()
    assert np.array_equal(b.cpu().numpy(), a)                    # same seed and step -> same draw
    assert not torch.equal(env.sample_device_leads(), b)         # the next step differs
    # stepping: own draws vs the same draws fed explicitly
    fed = BatchedInventoryEnv(cfg, E, device="cuda:0", env_meta=meta, host_samplers=False)
    init = torch.randint(0, 30, (E, 3, 5), dtype=torch.int32, device="cuda:0")
    env.reset(init_inventory=init)
    fed.reset(init_inventory=init)
    env._dl["step"] = 10
    from marlsc_b200.demand import pack_orders
    rng = np.random.default_rng(2)
    for t in range(6):
        big = pack_orders([g.orders(i % g.N, t) for i in range(E)], 5)
        act = torch.from_numpy(rng.uniform(-1, 1, (E, 3, 5)).astype(np.float32)).cuda()
        ob1, r1, _ = env.step(act, orders=big)
        ob2, r2, _ = fed.step(act, orders=big, actual_lead=env._dl["actual"])
        assert torch.equal(env.inventory, fed.inventory) and torch.equal(env.ring_qty, fed.ring_qty)
        assert torch.equal(env.ring_lead, fed.ring_lead) and torch.equal(ob1, ob2) and torch.equal(r1, r2)
    assert int(env.ring_lead.max()) > 1
    env.close()
    fed.close()


def test_step_with_device_demand_equals_same_orders_fed_as_csr():
    """The padded order layout the sampler writes and the CSR layout must drive K1 to the same result."""
    from marlsc_b200.demand import OrderBatch
    E = 64
    cfg, a = _small_env(E, host_samplers=False, device_demand=True, demand_seed=3)
    _, b = _small_env(E, host_samplers=False)
    a.reset()
    b.reset()
    g = torch.Generator(device="cuda:0").manual_seed(0)
    for t in range(15):
        act = torch.rand((E, 3, 2), device="cuda:0", generator=g) * 2 - 1
        oa, ra, _ = a.step(act)
        d = a._dd
        counts = d["counts"].cpu().numpy()
        omax = d["omax"]
        region = d["region"].cpu().numpy().reshape(E, omax)
        qty = d["qty"].cpu().numpy()[:E * omax * 2].reshape(E, omax, 2)
        per_env = [[(int(region[e, j]), qty[e, j]) for j in range(counts[e])] for e in range(E)]
        from marlsc_b200.demand import pack_orders
        ob, rb, _ = b.step(act, orders=pack_orders(per_env, 2))
        assert torch.equal(a.inventory, b.inventory) and torch.equal(ra, rb) and torch.equal(oa, ob)
    a.close()
    b.close()


def test_base_stock_policy_kernel_matches_reference_formula():
    from marlsc_b200.rollout import base_stock_levels
    E = 32
    cfg, env = _small_env(E, seed=5)
    level = base_stock_levels(env, 2.0)
    # reference: S = L*E[D] + z*sqrt(L*E[D]), E[D] = 4 * 0.667 * 5 for every (w,k), L = 3
    ed = 4 * 0.667 * 5
    assert np.allclose(level, 3 * ed + 2.0 * np.sqrt(3 * ed))
    env.reset()
    lvl = torch.from_numpy(level).float()
    rng = np.random.default_rng(0)
    for t in range(12):
        act = env.base_stock_actions(lvl)
        inv = env.inventory.cpu().numpy().astype(np.float64)
        pend = env.pending_matrix().cpu().numpy().astype(np.float64)
        qty = np.clip(level[None] - inv - pend, 0.0, 40.0)                       # run_baselines.py:196-203
        exp = (2.0 * qty / 40.0 - 1.0).astype(np.float32)
        np.testing.assert_allclose(act.cpu().numpy(), exp, rtol=1e-6, atol=1e-6)
        env.step(act)
    env.close()


def test_config1_base_stock_returns_match_reference_numbers():
    """BASELINE config #1: default small env, single env, heuristic base-stock policy z=2, eval seed 123.
    The reference's first three episode returns (BASELINE.md, measured from the reference itself) are
    -158.8005, -165.7435, -170.5540; the drop-in adapter seeded the same way must reproduce them."""
    from golden.scenarios import small_default
    from marlsc_b200.config import environment_config_from_dict
    from marlsc_b200.envs import InventoryEnvironment
    from marlsc_b200.rollout import base_stock_levels
    cfg = environment_config_from_dict(small_default())
    env = InventoryEnvironment(cfg, seed=123, env_meta={"data_mode": "train"})
    level = base_stock_levels(env._batch, 2.0)
    got = []
    for ep in range(3):
        obs, _ = env.reset()
        total, done = 0.0, False
        while not done:
            inv, pipe = env.inventory, env._compute_pending_matrix().astype(float)
            actions = {}
            for w, agent in enumerate(env.agents):
                qty = np.clip(level[w] - inv[w] - pipe[w], 0.0, 40.0)
                actions[agent] = (2.0 * qty / 40.0 - 1.0).astype(np.float32)
            obs, rew, term, trunc, _ = env.step(actions)
            total += sum(rew.values())
            done = all(trunc.values())
        got.append(total)
    np.testing.assert_allclose(got, [-158.8005, -165.7435, -170.5540], atol=2e-3)


def test_device_baseline_rollout_statistics():
    """Whole base-stock episodes on the device (K5 -> K4 -> K1 per step, no host round trip): the mean
    episode return over many envs must sit where the reference's 20-episode estimate does (-165.40 +- 10.89)."""
    from marlsc_b200.rollout import base_stock_levels, baseline_rollout
    cfg, env = _small_env(2048, host_samplers=False, device_demand=True, demand_seed=11)
    ret = baseline_rollout(env, base_stock_levels(env, 2.0), num_episodes=1)      # [1, E, W]
    per_env = ret.sum(-1).reshape(-1).cpu().numpy()
    assert abs(per_env.mean() - (-165.4)) < 3.0, per_env.mean()
    assert 5.0 < per_env.std() < 20.0
    env.close()


@pytest.mark.parametrize("team", [0, 2, 8])
def test_cuda_edge_cases_vs_oracle(team):
    """Odd shapes (W4 S7 R6), weight-dependent priority, softmax lost-sales handler, stochastic leads, base-stock
    actions, environments with no orders, all-zero orders, quantities that need 16 bits, an env count that does
    not fill the last CTA, more steps than the ring is deep, and a reset in the middle - CUDA vs the oracle."""
    from marlsc_b200.config import environment_config_from_dict
    from marlsc_b200.demand import pack_orders
    from marlsc_b200.envs import BatchedInventoryEnv
    from oracle.inventory_oracle import OracleEnv
    W, S, R = 4, 7, 6
    rng = np.random.default_rng(42)
    env_dict = dict(
        action_space=dict(type="base_stock", params=dict(max_stock_level=[int(x) for x in rng.integers(200, 900, S)])),
        n_warehouses=W, n_skus=S, n_regions=R, episode_length=14, max_wh_capacities=[1e7] * W,
        initial_inventory=dict(type="custom", params=dict(values=150)),
        cost_structure=dict(
            holding_cost=0.5, penalty_cost=[float(x) for x in rng.integers(1, 9, S)],
            shipment_cost=dict(
                outbound_fixed=(rng.integers(0, 8, (W, R)) * 0.5).tolist(), outbound_variable=(rng.integers(1, 16, (W, R)) / 16).tolist(),
                inbound_fixed=(rng.integers(0, 3, (W, S)) * 1.0).tolist(), inbound_variable=(rng.integers(1, 5, (W, S)) * 0.25).tolist()),
            sku_weights=[0.5, 1.0, 2.0, 0.25, 1.5, 1.0, 4.0], distances=(rng.integers(10, 500, (W, R)) * 1.0).tolist()),
        components=dict(
            demand_sampler=dict(type="poisson", params=dict(lambda_orders=1.0, probability_skus=0.5, lambda_quantity=5.0)),
            demand_allocator=dict(type="greedy", params=dict(max_splits=2)),
            lead_time_sampler=dict(type="stochastic", params=dict(
                expected_lead_times=rng.integers(1, 5, (W, S)).tolist(), deviation=dict(type="uniform", max_deviation=2))),
            lost_sales_handler=dict(type="cost", params=dict(alpha=3.0)),
            reward_calculator=dict(type="cost", params=dict(scope="team", scale_factor=0.1, cost_weights=[0.25] * 4))),
        data_source=dict(type="custom"),
        features=dict(inventory=True, pipeline=True, incoming_demand_home=True, units_shipped_home=True, units_shipped_away=True,
                      stockout=True, rolling_demand_mean=True, demand_forecast=True, days_of_supply=True,
                      net_inventory_position=True, demand_variability=True, demand_history=True, inventory_aggregate=False,
                      pipeline_aggregate=True, incoming_demand_home_aggregate=False, units_shipped_away_aggregate=True,
                      rolling_demand_mean_aggregate=True, demand_forecast_aggregate=False))
    cfg = environment_config_from_dict(dict(env_dict, allow_region_mismatch=True))
    E, T = 5, 26
    env = BatchedInventoryEnv(cfg, E, device="cuda:0", host_samplers=False, diagnostics=True, team_size=team,
                              env_meta=dict(include_warehouse_id=True))
    oracles = [OracleEnv(env_dict, include_warehouse_id=True) for _ in range(E)]
    lead_exp = np.asarray(env_dict["components"]["lead_time_sampler"]["params"]["expected_lead_times"])

    def reset_all():
        obs = env.reset().cpu().numpy()
        for i, o in enumerate(oracles):
            np.testing.assert_allclose(obs[i], o.reset(np.full((W, S), 150)), rtol=1e-5, atol=1e-6)
    reset_all()
    for t in range(T):
        if t == 14:                                   # episode over (truncated at t = 13): start the next one
            reset_all()
        per_env = []
        for i in range(E):
            if i == 1 or (i == 3 and t % 2):          # envs without any order this step
                per_env.append([])
                continue
            orders = []
            for _ in range(int(rng.integers(1, 9))):
                q = np.where(rng.random(S) < 0.5, rng.integers(1, 700 if i == 4 else 40, S), 0)
                if rng.random() < 0.15:
                    q[:] = 0                          # all-zero order: legal no-op
                orders.append((int(rng.integers(0, R)), q.astype(float)))
            per_env.append(orders)
        batch = pack_orders(per_env, S)
        assert batch.qty_bytes == 2
        act = rng.uniform(-1, 1, (E, W, S)).astype(np.float32)
        leads = np.maximum(1, lead_exp[None] + rng.integers(-2, 3, (E, W, S))).astype(np.uint8)
        obs, rew, trunc = env.step(torch.from_numpy(act).cuda(), orders=batch, actual_lead=leads)
        d = {k: v.cpu().numpy() for k, v in env.diag.items()}
        inv, r, ob = env.inventory.cpu().numpy(), rew.cpu().numpy(), obs.cpu().numpy()
        for i, o in enumerate(oracles):
            out = o.step(act[i], per_env[i], leads[i])
            assert np.array_equal(inv[i], out["inventory"]), (t, i)
            assert np.array_equal(d["ordered"][i], out["ordered"])
            assert np.array_equal(d["ship_by_sku"][i], out["ship_by_sku"])
            assert np.array_equal(d["ship_counts"][i], out["ship_counts"])
            assert np.array_equal(d["unfulfilled"][i], out["unfulfilled"])
            assert np.array_equal(d["lost_orders"][i], out["lost_orders"])
            np.testing.assert_allclose(d["lost_sales"][i], out["lost_sales"], rtol=1e-5, atol=1e-5)
            np.testing.assert_allclose(r[i], out["rewards"], rtol=1e-5, atol=1e-5)
            np.testing.assert_allclose(ob[i], out["obs_local"], rtol=1e-5, atol=2e-5, err_msg=f"obs t={t} env={i}")
            assert bool(trunc) == bool(out["trunc"])
    env.close()


@pytest.mark.parametrize("W,S,R,lost,pen_uniform,max_orders", [
    (3, 20, 5, "shipment", True, 9),       # one SKU per lane, one permutation chunk
    (7, 70, 9, "closest", False, 9),       # four SKUs per lane (ragged: S % 32 != 0), per-SKU penalties -> fp64 lost sums
    (10, 100, 50, "shipment", False, 80),  # the large shape; more than 64 orders in a step -> two mask passes
    (16, 200, 70, "shipment", True, 40),   # eight SKUs per lane, four permutation chunks, R > 64 -> generic cost epilogue
])
def test_one_warp_split_step_vs_oracle(W, S, R, lost, pen_uniform, max_orders):
    """The split step with one-warp teams (K1a / env_alloc_warp_kernel / K1c) against the oracle on shapes that reach every
    instantiation of the allocation kernel, with scarce stock (most lines are split or lost), environments without
    orders, all-zero orders, a batch that does not fill the last CTA and a mid-run reset."""
    from marlsc_b200.config import environment_config_from_dict
    from marlsc_b200.demand import pack_orders
    from marlsc_b200.envs import BatchedInventoryEnv
    from oracle.inventory_oracle import OracleEnv
    rng = np.random.default_rng(W * 1000 + S)
    out_var = np.stack([rng.permutation(W) for _ in range(R)], 1) * 0.05 + 0.05          # tie-free -> static priority
    pen = 4.0 if pen_uniform else [float(x) for x in rng.integers(1, 9, S)]
    env_dict = dict(
        action_space=dict(type="direct", params=dict(max_order_quantities=[int(x) for x in rng.integers(5, 30, S)])),
        n_warehouses=W, n_skus=S, n_regions=R, episode_length=9, max_wh_capacities=[1e7] * W,
        initial_inventory=dict(type="custom", params=dict(values=6)),
        cost_structure=dict(
            holding_cost=0.5, penalty_cost=pen,
            shipment_cost=dict(outbound_fixed=np.zeros((W, R)).tolist(), outbound_variable=out_var.tolist(),
                               inbound_fixed=np.full((W, S), 0.5).tolist(), inbound_variable=np.full((W, S), 0.25).tolist()),
            sku_weights=[1.0] * S, distances=(rng.integers(10, 500, (W, R)) * 1.0).tolist()),
        components=dict(
            demand_sampler=dict(type="poisson", params=dict(lambda_orders=1.0, probability_skus=0.3, lambda_quantity=5.0)),
            demand_allocator=dict(type="greedy", params=dict(max_splits=W - 1)),
            lead_time_sampler=dict(type="fixed", params=dict(expected_lead_times=rng.integers(1, 4, (W, S)).tolist())),
            lost_sales_handler=dict(type=lost, params=None),
            reward_calculator=dict(type="cost", params=dict(scope="agent", scale_factor=0.1, cost_weights=[0.25] * 4))),
        data_source=dict(type="custom"),
        features=dict(inventory=True, pipeline=True, incoming_demand_home=False, units_shipped_home=False, units_shipped_away=False,
                      stockout=False, rolling_demand_mean=True, demand_forecast=False, days_of_supply=False,
                      net_inventory_position=False, demand_variability=False, demand_history=False, inventory_aggregate=True,
                      pipeline_aggregate=False, incoming_demand_home_aggregate=False, units_shipped_away_aggregate=False,
                      rolling_demand_mean_aggregate=False, demand_forecast_aggregate=False))
    cfg = environment_config_from_dict(dict(env_dict, allow_region_mismatch=True))
    E, T = 6, 13
    env = BatchedInventoryEnv(cfg, E, device="cuda:0", host_samplers=False, team_size=32)
    assert env.team_size == 32
    oracles = [OracleEnv(env_dict) for _ in range(E)]

    def reset_all():
        obs = env.reset().cpu().numpy()
        for i, o in enumerate(oracles):
            np.testing.assert_allclose(obs[i], o.reset(np.full((W, S), 6)), rtol=1e-5, atol=1e-6)
    reset_all()
    lost_any = False
    for t in range(T):
        if t == 9:
            reset_all()
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
        assert batch.qty_bytes == 1
        act = rng.uniform(-1, 1, (E, W, S)).astype(np.float32)
        obs, rew, trunc = env.step(torch.from_numpy(act).cuda(), orders=batch)
        inv, r, ob = env.inventory.cpu().numpy(), rew.cpu().numpy(), obs.cpu().numpy()
        for i, o in enumerate(oracles):
            out = o.step(act[i], per_env[i])
            assert np.array_equal(inv[i], out["inventory"]), (t, i)
            np.testing.assert_allclose(r[i], out["rewards"], rtol=1e-5, atol=1e-5, err_msg=f"rewards t={t} env={i}")
            np.testing.assert_allclose(ob[i], out["obs_local"], rtol=1e-5, atol=2e-5, err_msg=f"obs t={t} env={i}")
            assert bool(trunc) == bool(out["trunc"])
            lost_any = lost_any or out["lost_orders"].sum() > 0
    assert lost_any, "workload was meant to lose sales"
    env.close()


def test_device_obs_statistics_match_the_reference_estimator():
    """compute_obs_statistics (reference: src/utils/obs_stats.py:11-168) on the device: its float64 column sums must
    reproduce np.mean / np.std (the reference's estimator) of the very observations the same seeds produce, both per
    column and grouped, and an environment normalised with them must come out standardised."""
    from golden.scenarios import small_default
    from marlsc_b200.config import environment_config_from_dict
    from marlsc_b200.envs import BatchedInventoryEnv
    from marlsc_b200.rollout import compute_obs_statistics
    from marlsc_b200.seeds import EXPERIMENT_SEEDS, SeedManager
    cfg = environment_config_from_dict(small_default())
    n_ep = 64
    mean, std = compute_obs_statistics(cfg, SeedManager(root_seed=11, seed_registry=EXPERIMENT_SEEDS), n_episodes=n_ep)
    gmean, gstd = compute_obs_statistics(cfg, SeedManager(root_seed=11, seed_registry=EXPERIMENT_SEEDS), mode="meanstd_grouped",
                                         n_episodes=n_ep)
    # the same loop by hand, observations kept
    env_seed, action_seed = SeedManager(root_seed=11, seed_registry=EXPERIMENT_SEEDS).spawn_child_seeds("obs_stats", 2)
    env = BatchedInventoryEnv(cfg, n_ep, device="cuda:0", host_samplers=False)
    env.enable_device_demand(seed=int(env_seed))
    gen = torch.Generator(device="cuda:0")
    gen.manual_seed(int(action_seed))
    rows = [env.reset().reshape(-1, env.obs_dim).cpu().numpy().copy()]
    for _ in range(env.episode_length):
        act = torch.rand((n_ep, 3, 2), device="cuda:0", generator=gen) * 2.0 - 1.0
        rows.append(env.step(act)[0].reshape(-1, env.obs_dim).cpu().numpy().copy())
    allobs = np.concatenate(rows).astype(np.float32)
    assert allobs.shape[0] == n_ep * (cfg.episode_length + 1) * 3
    np.testing.assert_allclose(mean, allobs.astype(np.float64).mean(0), rtol=1e-5, atol=1e-6)
    ref_std = allobs.astype(np.float64).std(0)
    np.testing.assert_allclose(std, np.where(ref_std < 1e-8, 1.0, ref_std), rtol=1e-4, atol=1e-6)
    # grouped: inventory (2 SKU columns + aggregate), pipeline (3 x 2), rolling mean (2) for the default features
    S, L = 2, env.max_expected_lead_time
    assert gmean[0] == gmean[1] and gstd[0] == gstd[1]
    np.testing.assert_allclose(gmean[0], allobs[:, :S].astype(np.float64).mean(), rtol=1e-5)
    np.testing.assert_allclose(gstd[0], allobs[:, :S].astype(np.float64).std(), rtol=1e-4)
    np.testing.assert_allclose(gmean[S], allobs[:, S].astype(np.float64).mean(), rtol=1e-5)          # the aggregate column
    pipe = allobs[:, S + 1:S + 1 + L * S].astype(np.float64)
    np.testing.assert_allclose(gmean[S + 1:S + 1 + L * S], pipe.mean(), rtol=1e-5)
    np.testing.assert_allclose(gstd[S + 1:S + 1 + L * S], pipe.std(), rtol=1e-4)
    env.close()
    # an environment normalised with the statistics comes out standardised on the same trajectory
    norm = BatchedInventoryEnv(cfg, n_ep, device="cuda:0", host_samplers=False,
                               env_meta=dict(obs_normalization="meanstd_custom", obs_stats=(mean, std)))
    norm.enable_device_demand(seed=int(env_seed))
    gen.manual_seed(int(action_seed))
    rows = [norm.reset().reshape(-1, norm.obs_dim).cpu().numpy().copy()]
    for _ in range(norm.episode_length):
        act = torch.rand((n_ep, 3, 2), device="cuda:0", generator=gen) * 2.0 - 1.0
        rows.append(norm.step(act)[0].reshape(-1, norm.obs_dim).cpu().numpy().copy())
    z = np.concatenate(rows).astype(np.float64)
    live = ref_std >= 1e-8
    assert np.abs(z.mean(0)[live]).max() < 1e-3 and np.abs(z.std(0)[live] - 1).max() < 1e-3
    norm.close()


@pytest.mark.parametrize("S,beta", [(2, None), (2, 0.4), (37, None)])
def test_fused_ppo_loss_matches_pytorch(S, beta):
    """K6 (marlsc_ppo_loss) against the same objective in plain PyTorch fp32 with autograd: loss terms and the
    gradients of every parameter, with ratios on both sides of the clip range, advantages of both signs, value errors
    beyond vf_clip and a log_std entry below its floor. rtol 1e-4 (fp32 sums in a different order)."""
    from marlsc_b200.rollout import ActorCritic, PPOLearner
    torch.manual_seed(3)
    W, D, B = 3, 11, 700
    pol = ActorCritic(D, W, S, actor_hidden=(32,), critic_hidden=(32,), logstd_floor=-1.0).cuda()
    with torch.no_grad():
        pol.log_std.copy_(torch.linspace(-1.5, 0.5, S))            # the first entries sit below the floor
    obs = torch.randn(B, W, D, device="cuda")
    with torch.no_grad():
        mean = pol.action_mean(obs)
        actions = mean + torch.randn_like(mean) * 0.8
        logp_old = pol.log_prob(mean, actions) + torch.randn(B, W, device="cuda") * 0.3     # ratios well outside [0.8, 1.2] too
        adv = torch.randn(B, W, device="cuda")
        targets = pol.value(obs) + torch.randn(B, W, device="cuda") * 4.0                    # squared errors beyond vf_clip = 10
    fused = PPOLearner(pol, hysteretic_beta=beta, fused_loss=True)
    ref = PPOLearner(pol, hysteretic_beta=beta, fused_loss=False)
    out_f = fused.loss(obs, actions, logp_old, adv, targets)
    pol.zero_grad()
    out_f["total"].backward()
    g_f = [p.grad.clone() for p in pol.parameters()]
    out_r = ref.loss(obs, actions, logp_old, adv, targets)
    pol.zero_grad()
    out_r["total"].backward()
    g_r = [p.grad.clone() for p in pol.parameters()]
    for k in ("total", "policy", "vf", "entropy"):
        np.testing.assert_allclose(float(out_f[k].detach()), float(out_r[k].detach()), rtol=1e-4, atol=1e-6, err_msg=k)
    assert float((pol.log_std.grad != 0).sum()) > 0
    for (name, _), a, b in zip(pol.named_parameters(), g_f, g_r):
        np.testing.assert_allclose(a.cpu().numpy(), b.cpu().numpy(), rtol=1e-4, atol=1e-6, err_msg=name)


def test_adaptive_constant_and_random_baselines_match_reference_formulas():
    """BS-Adaptive / constant / random baselines (reference: src/experiments/run_baselines.py:73-293) for a batch of
    environments against the reference formulas evaluated in NumPy on the same states."""
    from golden.scenarios import small_default
    from marlsc_b200.config import environment_config_from_dict
    from marlsc_b200.envs import BatchedInventoryEnv
    from marlsc_b200.rollout import AdaptiveBaseStock, constant_actions, random_actions
    cfg = environment_config_from_dict(small_default())
    E, z, H = 37, 1.5, 4
    env = BatchedInventoryEnv(cfg, E, device="cuda:0", host_samplers=False)
    env.enable_device_demand(seed=9)
    env.reset()
    pol = AdaptiveBaseStock(env, z, H)
    lead = np.asarray(env.expected_lead_times, dtype=float)
    mx = np.asarray(cfg.action_space.params.max_order_quantities, dtype=float)
    hist = []
    for t in range(12):
        a = pol.actions().cpu().numpy()
        if t > 0:
            hist.append(env.demand_hist[:, (t - 1) % 5].cpu().numpy().astype(float))
        if not hist:
            assert np.all(a == -1.0)
        else:
            win = np.array(hist[-H:])
            mean = win.mean(0)
            var = win.var(0) if len(win) > 1 else mean.copy()
            level = lead * mean + z * np.sqrt(lead * var)
            ring = env.ring_qty.cpu().numpy()
            pend = np.zeros_like(mean)
            for k in range(1, int(lead.max()) + 1):          # orders placed at t - k still in transit when lead > k - 1 ... >= k
                if t - k >= 0:
                    pend += ring[:, (t - k) % env.ring_depth] * (lead >= k)[None]
            qty = np.clip(level - env.inventory.cpu().numpy() - pend, 0.0, mx)
            np.testing.assert_allclose(a, (2.0 * qty / mx - 1.0).astype(np.float32), rtol=1e-5, atol=2e-6, err_msg=f"t={t}")
        env.step(torch.from_numpy(a).cuda())
    c = constant_actions(env, np.array([[3.0, 500.0], [0.0, 7.0], [-2.0, 1.0]]))
    exp = (2.0 * np.clip(np.array([[3.0, 500.0], [0.0, 7.0], [-2.0, 1.0]]), 0.0, mx) / mx - 1.0).astype(np.float32)
    assert c.shape == (E, 3, 2) and np.array_equal(c[5].cpu().numpy(), exp)
    g = torch.Generator(device="cuda:0")
    g.manual_seed(1)
    r = random_actions(env, g)
    assert r.shape == (E, 3, 2) and float(r.min()) >= -1.0 and float(r.max()) < 1.0 and abs(float(r.mean())) < 0.2
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("D,H,O,act,N", [(14, 256, 2, "relu", 70001), (14, 256, 1, "relu", 257), (3, 17, 3, "tanh", 1000),
                                         (32, 64, 1, "relu", 4099), (56, 64, 1, "tanh", 513), (64, 300, 3, "relu", 130)])
def test_fused_mlp_forward_matches_pytorch(D, H, O, act, N):
    """K7 (marlsc_mlp1_forward: one-hidden-layer head, hidden activations in registers; reference network: mlp of
    rlmodules/base.py:412-457) against the same nn.Sequential evaluated by PyTorch in float32 (cuBLAS TF32 off) - rows that
    do not fill the last thread pair / CTA, every input-width instantiation, both activations."""
    from marlsc_b200.rollout.policy import forward_mlp, mlp
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.manual_seed(D * 1000 + H)
    net = mlp(D, (H,), O, act).cuda()
    x = torch.randn((N // 3 + 1, 3, D), device="cuda:0")[: N // 3 + 1]
    with torch.no_grad():
        got = forward_mlp(net, x)
        want = net(x)
    assert got.shape == want.shape
    torch.testing.assert_close(got, want, rtol=1e-5, atol=2e-6)
    # with autograd on, the PyTorch modules run (the learner's path)
    y = forward_mlp(net, x[:4])
    assert y.requires_grad


@pytest.mark.parametrize("D,hidden,O,N", [(14, (256, 256), 2, 50001), (56, (64, 64), 1, 4097), (10, (32, 20, 8), 4, 333),
                                          (30, (100, 64), 3, 1000), (64, (48, 16), 1, 77), (3, (250, 4), 2, 999)])
def test_deeper_mlp_rollout_forward_matches_pytorch(D, hidden, O, N):
    """Heads with more than one hidden layer (MAPPO's actor and critic, mappo.yaml:43-55): hidden layers through the library
    GEMM with bias + ReLU in its epilogue, the input layer through K7a (marlsc_linear_in_forward, every register
    tiling it instantiates) and the output layer through K7b (marlsc_linear_out_forward) - against the same nn.Sequential
    in PyTorch float32."""
    from marlsc_b200.rollout.policy import forward_mlp, mlp
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.manual_seed(D + N)
    net = mlp(D, hidden, O, "relu").cuda()
    x = torch.randn((N, D), device="cuda:0")
    with torch.no_grad():
        got, want = forward_mlp(net, x), net(x)
    torch.testing.assert_close(got, want, rtol=1e-5, atol=2e-6)


def test_global_critic_rollout_path_matches_autograd_path():
    """MAPPO's centralised critic (critic_obs_type 'global', mappo.py:142-157): without autograd the value runs through the
    library's layer kernels over [local | global] rows, with autograd through PyTorch's split first layer - same numbers."""
    from marlsc_b200.rollout import ActorCritic
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.manual_seed(5)
    pol = ActorCritic(14, 3, 2, actor_hidden=(256, 256), critic_hidden=(64, 64), critic_obs_type="global", parameter_sharing=True).cuda()
    obs = torch.randn((1001, 3, 14), device="cuda:0")
    with torch.no_grad():
        fast = pol.value(obs)
        mean_fast = pol.action_mean(obs)
    slow, mean_slow = pol.value(obs), pol.action_mean(obs)
    assert slow.requires_grad and not fast.requires_grad
    torch.testing.assert_close(fast, slow.detach(), rtol=1e-5, atol=2e-6)
    torch.testing.assert_close(mean_fast, mean_slow.detach(), rtol=1e-5, atol=2e-6)


def test_fresh_rollout_has_ratio_one_and_zero_kl():
    """The collector stores the RAW Gaussian sample the log-prob refers to and sends only its clipped copy to the env
    (RLlib clip_actions=True, reference ippo.py:183-188): on the first minibatch of a fresh rollout the probability
    ratio is exactly 1, so the surrogate equals -mean(advantages) and the KL term vanishes."""
    from golden.scenarios import small_default
    from marlsc_b200.config import environment_config_from_dict
    from marlsc_b200.envs import BatchedInventoryEnv
    from marlsc_b200.rollout import ActorCritic, PPOLearner, RolloutCollector
    cfg = environment_config_from_dict(small_default())
    torch.manual_seed(0)
    E, T = 64, 20
    env = BatchedInventoryEnv(cfg, E, device="cuda:0", seed=3, env_meta=dict(include_warehouse_id=True))
    pol = ActorCritic(env.obs_dim, 3, 2, actor_hidden=(32,), critic_hidden=(32,), logstd_init=0.0).cuda()   # std 1: ~32 % clipped
    col = RolloutCollector(env, pol, T, seed=1, keep_dist_inputs=True)
    ro = col.collect()
    assert float((ro.actions.abs() > 1).float().mean()) > 0.1          # raw samples are kept
    learner = PPOLearner(pol, use_kl_loss=True, fused_loss=True)
    sl = (slice(0, 10), slice(0, 32))
    out = learner.loss(ro.obs[sl].flatten(0, 1), ro.actions[sl].flatten(0, 1), ro.logp[sl].flatten(0, 1),
                       ro.advantages[sl].flatten(0, 1), ro.targets[sl].flatten(0, 1), ro.mean_old[sl].flatten(0, 1), ro.log_std_old)
    np.testing.assert_allclose(float(out["policy"]), -float(ro.advantages[sl].mean()), rtol=1e-4, atol=1e-5)
    assert abs(float(out["kl"])) < 1e-5
    stats = learner.update(ro, num_epochs=2, num_minibatches=4)
    assert stats["minibatches"] == 8 and np.isfinite(stats["total"])
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("sharing", [True, False])
def test_fused_ppo_loss_with_kl_and_independent_policies(sharing):
    """K6 with the KL penalty (use_kl_loss, reference mappo.yaml:21) and with one policy per warehouse
    (parameter_sharing=False, ippo.py:111-115) against the same objective in plain PyTorch with autograd."""
    from marlsc_b200.rollout import ActorCritic, PPOLearner
    torch.manual_seed(5)
    W, D, S, B = 3, 9, 4, 500
    pol = ActorCritic(D, W, S, actor_hidden=(16,), critic_hidden=(16,), critic_obs_type="global", logstd_floor=-1.0,
                      parameter_sharing=sharing).cuda()
    with torch.no_grad():
        pol.log_std.copy_(torch.linspace(-1.5, 0.5, pol.log_std.numel()).reshape(pol.log_std.shape))
    obs = torch.randn(B, W, D, device="cuda")
    with torch.no_grad():
        mean = pol.action_mean(obs)
        actions = mean + torch.randn_like(mean) * 0.8
        logp_old = pol.log_prob(mean, actions) + torch.randn(B, W, device="cuda") * 0.3
        adv = torch.randn(B, W, device="cuda")
        targets = pol.value(obs) + torch.randn(B, W, device="cuda") * 4.0
        mean_old = mean + 0.2 * torch.randn_like(mean)
        ls_old = (pol.clamped_log_std() + 0.1 * torch.randn_like(pol.log_std)).reshape(pol.n_policies, S)
    fused = PPOLearner(pol, fused_loss=True, use_kl_loss=True, kl_coeff=0.3)
    ref = PPOLearner(pol, fused_loss=False, use_kl_loss=True, kl_coeff=0.3)
    grads = []
    outs = []
    for lr_ in (fused, ref):
        out = lr_.loss(obs, actions, logp_old, adv, targets, mean_old, ls_old)
        pol.zero_grad()
        out["total"].backward()
        grads.append([p.grad.clone() for p in pol.parameters()])
        outs.append(out)
    for k in ("total", "policy", "vf", "entropy", "kl"):
        np.testing.assert_allclose(float(outs[0][k].detach()), float(outs[1][k].detach()), rtol=1e-4, atol=1e-6, err_msg=k)
    for (name, _), a, b in zip(pol.named_parameters(), grads[0], grads[1]):
        np.testing.assert_allclose(a.cpu().numpy(), b.cpu().numpy(), rtol=2e-4, atol=2e-6, err_msg=name)


@pytest.mark.gpu
def test_poisson_inversion_survives_the_largest_uniform():
    """The float32 CDF sum of the device Poisson inversion plateaus a few ulp below 1; with the largest 24-bit uniform
    (1 - 2^-24) the search must stop where the sum stops growing, not run to its 200 cap (which used to hand a region
    200 orders about once per 10^7 draws)."""
    from marlsc_b200 import _capi
    lam = torch.tensor([0.25, 1.0, 3.0, 5.0, 12.0, 29.0], device="cuda")
    u = torch.full_like(lam, 1.0 - 2.0 ** -24)
    for tab in (0, 1):
        out = torch.zeros(lam.numel(), dtype=torch.int32, device="cuda")
        _capi.check(_capi.lib().marlsc_poisson_inverse(lam.data_ptr(), u.data_ptr(), lam.numel(), tab, out.data_ptr(),
                                                       torch.cuda.current_stream().cuda_stream))
        k = out.cpu().numpy()
        # far in the tail, but nowhere near the cap: P(X >= k) at these k is ~1e-7
        bound = np.array([8, 12, 20, 25, 40, 70])
        assert (k <= bound).all() and (k >= np.array([3, 6, 10, 14, 25, 50])).all(), (tab, k)
    # and ordinary uniforms still invert exactly like the float64 CDF
    from scipy.stats import poisson
    g = torch.Generator(device="cuda").manual_seed(1)
    lam2 = torch.tensor([1.0, 3.0, 5.0], device="cuda").repeat_interleave(4000)
    u2 = torch.rand(lam2.numel(), device="cuda", generator=g) * 0.999
    out = torch.zeros(lam2.numel(), dtype=torch.int32, device="cuda")
    _capi.check(_capi.lib().marlsc_poisson_inverse(lam2.data_ptr(), u2.data_ptr(), lam2.numel(), 0, out.data_ptr(),
                                                   torch.cuda.current_stream().cuda_stream))
    ref = poisson.ppf(u2.cpu().numpy().astype(np.float64), lam2.cpu().numpy().astype(np.float64))
    assert (out.cpu().numpy() != ref).mean() < 2e-3        # only draws within float32 rounding of a CDF step differ


@pytest.mark.parametrize("W,S,R,lost,pen_uniform,max_orders,lead_hi,variant", [
    (7, 68, 9, "closest", False, 9, 3, "lines"),            # ragged last slot, per-SKU penalties (float64 lost sums), W in two chunks
    (10, 100, 50, "shipment", False, 80, 10, "lines"),      # the large shape, leads up to 10 (ring wraps), > 64 orders per step
    (16, 128, 64, "shipment", True, 40, 16, "lines"),       # every limit of the layout at once: W 16, S 128, R 64, L 16
    (5, 36, 3, "shipment", True, 12, 1, "lines"),           # a single ring plane (L = 1), one warehouse chunk
    (10, 100, 50, "shipment", True, 30, 6, "dense"),        # dense order rows converted on the device (marlsc_lines_from_orders)
    (10, 100, 50, "closest", True, 30, 6, "qty_actions"),   # integer order quantities instead of float actions
    (6, 64, 12, "shipment", True, 20, 4, "norm_id_team"),   # fixed mean/std normalisation, one-hot id, team reward, home-demand block
    (10, 100, 50, "shipment", True, 30, 6, "region_map"),   # 50 raw regions mapped onto 10 included ones (preprocessor.py:382-441)
])
def test_compact_step_vs_oracle(W, S, R, lost, pen_uniform, max_orders, lead_hi, variant):
    """The compact layout's kernels (csrc/env_compact.cu: the step K1a'-K1d) against the oracle: scarce stock (most lines
    are split or lost), environments without orders, all-zero orders, a batch that does not fill the last CTA, a mid-run
    reset, ring wrap-around, and every way of feeding it (lines packed on the host, dense rows converted on the device,
    integer quantity actions, a region map)."""
    from marlsc_b200.config import environment_config_from_dict
    from marlsc_b200.demand import pack_orders
    from marlsc_b200.envs import BatchedInventoryEnv, DeviceOrders
    from oracle.inventory_oracle import OracleEnv
    rng = np.random.default_rng(W * 1000 + S + len(variant))
    norm = variant == "norm_id_team"
    R_cost = 10 if variant == "region_map" else R                 # regions the cost tables are defined on
    env_dict = _lean_env_dict(rng, W, S, R_cost, lost, pen_uniform, lead_hi, scope="team" if norm else "agent", demand_home=norm)
    env_dict["episode_length"] = 2 * lead_hi + 5
    cfg = environment_config_from_dict(dict(env_dict, allow_region_mismatch=True))
    region_map = [int(x) for x in rng.integers(0, R_cost, R)] if variant == "region_map" else None
    meta, okw = {}, {}
    if norm:
        dim = S + 1 + lead_hi * S + S + S
        stats = (rng.uniform(0, 5, dim).astype(np.float32), rng.uniform(0.5, 3, dim).astype(np.float32))
        meta = dict(obs_normalization="meanstd_custom", obs_stats=stats, include_warehouse_id=True)
        okw = dict(obs_normalization="meanstd_custom", obs_stats=stats, include_warehouse_id=True)
    E, T = 11, 2 * lead_hi + 7
    env = BatchedInventoryEnv(cfg, E, device="cuda:0", host_samplers=False, env_meta=meta, region_map=region_map,
                              layout="compact")
    assert env.layout == "compact"
    oracles = [OracleEnv(env_dict, **okw) for _ in range(E)]
    maxq = np.asarray(env_dict["action_space"]["params"]["max_order_quantities"])

    def reset_all():
        obs = env.reset().cpu().numpy()
        for i, o in enumerate(oracles):
            np.testing.assert_allclose(obs[i], o.reset(np.full((W, S), 6)), rtol=1e-5, atol=1e-6)
    env.ring_qty.fill_(7)                                          # reset has to clear the state
    env.inventory.fill_(99)
    reset_all()
    lost_any = False
    for t in range(T):
        if env.timestep >= env.episode_length or t == lead_hi + 3:
            reset_all()
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
        if variant == "qty_actions":
            qa = rng.integers(0, 40, (E, W, S)).astype(np.uint8)                   # some above the SKU's maximum: clipped
            act_dev = torch.from_numpy(qa).cuda()
            act = (2.0 * np.minimum(qa, maxq) / maxq - 1.0).astype(np.float32)      # the float action with the same quantity
        else:
            act = rng.uniform(-1, 1, (E, W, S)).astype(np.float32)
            act_dev = torch.from_numpy(act).cuda()
        feed = DeviceOrders.from_host(batch, "cuda:0") if variant == "dense" else batch
        obs, rew, trunc = env.step(act_dev, orders=feed)
        inv, r, ob = env.inventory.cpu().numpy(), rew.cpu().numpy(), obs.cpu().numpy()
        pend = env.pending_matrix().cpu().numpy()
        for i, o in enumerate(oracles):
            mapped = [(region_map[rg], q) for rg, q in per_env[i]] if region_map else per_env[i]
            out = o.step(act[i], mapped)
            assert np.array_equal(inv[i], out["inventory"]), (t, i)
            assert np.array_equal(pend[i], out["pending"]), (t, i)
            np.testing.assert_allclose(r[i], out["rewards"], rtol=1e-5, atol=1e-5, err_msg=f"rewards t={t} env={i}")
            np.testing.assert_allclose(ob[i], out["obs_local"], rtol=1e-5, atol=2e-5, err_msg=f"obs t={t} env={i}")
            assert bool(trunc) == bool(out["trunc"])
            lost_any = lost_any or out["lost_orders"].sum() > 0
    assert lost_any, "workload was meant to lose sales"
    env.close()


def test_lines_from_orders_matches_host_packer():
    """marlsc_lines_from_orders (device) and demand.pack_lines (host) build byte-identical blocks: same ranking of SKUs by
    line count, same snake dealing, same sequence inside a stream - for ragged SKU counts, an empty environment and
    with a region map."""
    from marlsc_b200.config import environment_config_from_dict
    from marlsc_b200.demand import pack_lines, pack_orders
    from marlsc_b200.envs import BatchedInventoryEnv, DeviceOrders
    for S, R, W in ((100, 50, 10), (68, 9, 7), (128, 64, 16)):
        E = 13
        rng = np.random.default_rng(S)
        cfg = environment_config_from_dict(dict(_lean_env_dict(rng, W, S, R, "shipment", True, 6), allow_region_mismatch=True))
        env = BatchedInventoryEnv(cfg, E, device="cuda:0", host_samplers=False, layout="compact")
        per_env = []
        for e in range(E):
            n = 0 if e == 5 else int(rng.integers(1, 90))
            per_env.append(sorted(((int(rng.integers(0, R)), np.where(rng.random(S) < 0.25, rng.integers(1, 200, S), 0).astype(float))
                                   for _ in range(n)), key=lambda x: x[0]))
        batch = pack_orders(per_env, S)
        host = pack_lines(batch)
        dev = env.lines_from_orders(DeviceOrders.from_host(batch, "cuda:0"))
        assert np.array_equal(dev.offsets.cpu().numpy(), host.offsets)
        n = host.n_rounds
        assert np.array_equal(dev.lines.cpu().numpy().view(np.uint16)[:n], host.lines[:n])
        assert dev.n_lines == host.n_lines
        env.close()


def test_compact_device_demand_lines_and_in_step_base_stock():
    """All-device pipeline on the compact layout: (i) the sampler writing lines (marlsc_demand_sample_lines) draws the
    orders the dense sampler draws for the same (seed, step) - an environment fed the dense rows ends in the same state;
    (ii) the base-stock heuristic evaluated inside the step (marlsc_step_io.base_stock_level) equals the policy kernel
    (marlsc_policy_base_stock) followed by a step with its actions."""
    from golden.scenarios import large_network
    from marlsc_b200 import _capi
    from marlsc_b200.config import environment_config_from_dict
    from marlsc_b200.envs import BatchedInventoryEnv, DeviceOrders
    d = large_network()
    d["episode_length"] = 30
    cfg = environment_config_from_dict(dict(d, allow_region_mismatch=True))
    E = 37
    a = BatchedInventoryEnv(cfg, E, device="cuda:0", host_samplers=False, device_demand=True, demand_seed=5)     # lines, in-step policy
    b = BatchedInventoryEnv(cfg, E, device="cuda:0", host_samplers=False)                                        # dense rows, policy kernel
    assert a.layout == b.layout == "compact" and "lines" in a._dd
    smp = a.spec.components["demand_sampler"]
    lam_o, prob, lam_q = smp.dense_params()
    omax = 128
    L = _capi.lib()
    h = __import__("ctypes").c_void_p()
    import ctypes as C
    dbl = lambda x: np.ascontiguousarray(x, dtype=np.float64).ctypes.data_as(C.POINTER(C.c_double))   # noqa: E731
    keep = [np.ascontiguousarray(v, np.float64) for v in (lam_o, prob, lam_q)]
    _capi.check(L.marlsc_demand_create(50, 100, dbl(keep[0]), dbl(keep[1]), dbl(keep[2]), 0, C.byref(h)))
    counts = torch.zeros(E, dtype=torch.int32, device="cuda")
    region = torch.zeros(E * omax, dtype=torch.int16, device="cuda")
    qty = torch.zeros(E * omax * 100 + 16, dtype=torch.uint8, device="cuda")
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")
    rng = np.random.default_rng(0)
    level = torch.from_numpy(rng.uniform(5, 60, (10, 100)).astype(np.float32)).cuda()
    a.reset()
    b.reset()
    for t in range(24):
        _capi.check(L.marlsc_demand_sample(h, E, 5, t, omax, counts.data_ptr(), region.data_ptr(), qty.data_ptr(), flag.data_ptr(),
                                           torch.cuda.current_stream().cuda_stream))
        cnt = counts.cpu().numpy()
        offs = np.zeros(E + 1, np.int32)
        offs[1:] = np.cumsum(cnt)
        rows = np.concatenate([np.arange(e * omax, e * omax + cnt[e]) for e in range(E)])
        reg = region.cpu().numpy()[rows]
        q = qty.cpu().numpy()[:E * omax * 100].reshape(E * omax, 100)[rows]
        pad = np.zeros((-(q.size)) % 16 + 16, np.uint8)
        dense = DeviceOrders(torch.from_numpy(offs).cuda(), torch.from_numpy(reg).cuda(),
                             torch.from_numpy(np.concatenate([q.reshape(-1), pad])).cuda(), int(offs[-1]))
        oa, ra, _ = a.step(None, base_stock_level=level)                              # K4 lines + policy inside K1a'
        ob, rb, _ = b.step(b.base_stock_actions(level), orders=dense)                 # K5, then K1 on the dense rows
        assert torch.equal(a.inventory, b.inventory), t
        assert torch.equal(a.ring_qty, b.ring_qty), t
        assert torch.equal(oa, ob) and torch.equal(ra, rb), t
    assert not a.demand_overflowed() and int(flag.item()) == 0
    L.marlsc_demand_destroy(h)
    a.close()
    b.close()


def test_empirical_demand_with_region_map_matches_reference():
    """Golden scenario of SURVEY 8a rows A7 + A12: the reference env with its own EmpiricalDemandSampler over a demand
    frame whose 50 raw regions went through the reference's map_excluded_regions. Here: the RAW frame packed by
    pack_demand_frame, the region map from build_region_map, environments seeded like the reference's (window starts
    from the same NumPy stream), orders sliced from the frame on the device - trajectories must match bit-exactly."""
    import pandas as pd
    from marlsc_b200.config import environment_config_from_dict
    from marlsc_b200.data import PreprocessedData, build_region_map
    from marlsc_b200.envs import BatchedInventoryEnv
    g = Golden("empirical_regionmap")
    z = g.z
    wtr = pd.DataFrame(dict(sourcenodeid=z["wtr_source"], destinationregionid=z["wtr_dest"], fixed_costs=z["wtr_cost"]))
    raw = pd.DataFrame(dict(timestep=z["frame_timestep"], region_id=z["frame_region_raw"].astype(int), order_id=z["frame_order"],
                            sku_id=z["frame_sku"].astype(int), quantity=z["frame_qty"].astype(float)))
    rmap = build_region_map(list(z["all_region_ids"]), wtr, list(z["selected_region_ids"]))
    cfg = environment_config_from_dict(dict(g.env, allow_region_mismatch=True, allow_empirical_frame=True))
    for layout in ("compact", "wide"):
        env = BatchedInventoryEnv(cfg, g.N, device="cuda:0", env_seeds=[int(s) for s in z["env_seeds"]], region_map=rmap,
                                  env_meta=dict(preprocessed_data=PreprocessedData(raw)), layout=layout)
        assert env.layout == layout
        obs0 = env.reset()
        np.testing.assert_allclose(obs0.cpu().numpy(), g["obs0_local"], rtol=1e-5, atol=1e-6)
        assert env._frame_start is None
        for t in range(g.T):
            obs, rew, trunc = env.step(torch.from_numpy(g["actions"][:, t]).cuda())
            if t == 0:
                assert env._frame_start.cpu().tolist() == [int(x) for x in z["window_start"]]
            out = dict(inventory=env.inventory.cpu().numpy(), rewards=rew.cpu().numpy(), obs=obs.cpu().numpy(),
                       trunc=env.truncated.cpu().numpy())
            compare_step(g, t, out, what=f"empirical {layout} ")
            assert np.array_equal(env.pending_matrix().cpu().numpy(), g["pending"][:, t])
        env.close()


def test_config2_4096_envs_100_steps_strided_oracle_check():
    """BASELINE configs[1]: the default small env batched to 4,096 instances, T = 100, uniform float32 actions, demand from
    the device sampler; 64 strided environments - the first and the last of the batch (last CTA) among them - are
    replayed through the oracle with the orders the sampler drew for them: inventory exact, rewards / observations 1e-5."""
    from golden.scenarios import small_default
    from marlsc_b200.config import environment_config_from_dict
    from marlsc_b200.envs import BatchedInventoryEnv
    from oracle.inventory_oracle import OracleEnv
    env_dict = small_default()
    cfg = environment_config_from_dict(env_dict)
    E, T = 4096, 100
    env = BatchedInventoryEnv(cfg, E, device="cuda:0", host_samplers=False, device_demand=True, demand_seed=2)
    picks = np.unique(np.concatenate([np.arange(0, E, 65), [E - 1, E - 2, E - 127, E - 128, E - 129]]))
    assert len(picks) >= 64
    obs = env.reset()
    init = env.inventory.cpu().numpy()
    oracles = {}
    for i in picks:
        o = OracleEnv(env_dict)
        np.testing.assert_allclose(obs[i].cpu().numpy(), o.reset(init[i]), rtol=1e-5, atol=1e-6)
        oracles[int(i)] = o
    gen = torch.Generator(device="cuda:0").manual_seed(0)
    d = env._dd
    omax = d["omax"]
    for t in range(T):
        act = torch.rand((E, 3, 2), device="cuda:0", generator=gen) * 2 - 1
        obs, rew, trunc = env.step(act)
        counts = d["counts"].cpu().numpy()
        region = d["region"].cpu().numpy().reshape(E, omax)
        qty = d["qty"].cpu().numpy()[:E * omax * 2].reshape(E, omax, 2)
        a_h, inv, r, ob = act.cpu().numpy(), env.inventory.cpu().numpy(), rew.cpu().numpy(), obs.cpu().numpy()
        for i, o in oracles.items():
            out = o.step(a_h[i], [(int(region[i, j]), qty[i, j].astype(float)) for j in range(counts[i])])
            assert np.array_equal(inv[i], out["inventory"]), (t, i)
            np.testing.assert_allclose(r[i], out["rewards"], rtol=1e-5, atol=1e-6, err_msg=f"t={t} env={i}")
            np.testing.assert_allclose(ob[i], out["obs_local"], rtol=1e-5, atol=1e-6, err_msg=f"t={t} env={i}")
            assert bool(trunc) == bool(out["trunc"])
    assert bool(trunc) and not env.demand_overflowed()
    env.close()


def test_graphed_episode_equals_eager_steps():
    """reset + T steps captured in one CUDA graph (rollout/graph.py) must reproduce the eager step-by-step results, and a
    replay after the actions were overwritten in place must follow the new actions."""
    from golden.scenarios import small_default
    from marlsc_b200.config import environment_config_from_dict
    from marlsc_b200.envs import BatchedInventoryEnv, DeviceOrders
    from marlsc_b200.rollout import GraphedEpisode
    g = Golden("small_default")
    cfg = environment_config_from_dict(small_default())
    E, T = g.N, 30
    orders = [DeviceOrders.from_host(step_orders(g, t), "cuda:0") for t in range(T)]
    act = torch.from_numpy(np.ascontiguousarray(g["actions"][:, :T].transpose(1, 0, 2, 3))).cuda()
    init = torch.from_numpy(g["init_inventory"])
    env = BatchedInventoryEnv(cfg, E, device="cuda:0", host_samplers=False)
    ep = GraphedEpisode(env, act, orders, init_inventory=init)
    rew = ep.replay().clone()
    torch.cuda.synchronize()
    for t in range(T):
        np.testing.assert_allclose(rew[t].cpu().numpy(), g["rewards"][:, t], rtol=1e-5, atol=1e-6)
        np.testing.assert_allclose(ep.obs[t + 1].cpu().numpy(), g["obs_local"][:, t], rtol=1e-5, atol=1e-6)
    assert np.array_equal(env.inventory.cpu().numpy(), g["inventory"][:, T - 1])
    act.mul_(0.5)                                     # new actions in the same buffer: the replay must pick them up
    rew2 = ep.replay().clone()
    ref = BatchedInventoryEnv(cfg, E, device="cuda:0", host_samplers=False)
    ref.reset(init_inventory=init)
    for t in range(T):
        _, r, _ = ref.step(act[t], orders=orders[t])
        assert torch.equal(r, rew2[t])
    assert not torch.equal(rew, rew2)
