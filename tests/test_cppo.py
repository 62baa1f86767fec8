"""-m gpu: CPPO on the device. The widened K7 / K7b against PyTorch float32, the collector with a CentralizedActorCritic
against a hand-written loop and against CentralizedEnvWrapper, K6 against loss_reference on the joint action,
evaluate() of a centralised policy, and a short learning run."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _small_cfg(**over):
    from golden.scenarios import small_default
    from marlsc_b200.config import environment_config_from_dict
    d = small_default()
    d.update(over)
    return environment_config_from_dict(d)


@pytest.mark.parametrize("act", ["relu", "tanh"])
@pytest.mark.parametrize("O", [1, 6, 15, 16])
@pytest.mark.parametrize("D", [12, 22, 33, 78, 128])
def test_wide_k7_matches_pytorch(D, O, act):
    """marlsc_mlp1_forward past the narrow envelope (the joint heads of a centralised policy: in <= 128, out <= 16) against
    the same nn.Sequential in PyTorch float32 (TF32 off), with a row count that does not fill the last CTA - every input
    padding of the wide form, including the ones with four (12 inputs) and two (22) rows per thread."""
    from marlsc_b200.rollout.policy import _fused_mlp1, mlp
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.manual_seed(D * 100 + O)
    net = mlp(D, (256,), O, act).cuda()
    x = torch.randn((3000 + D, D), device="cuda:0")
    with torch.no_grad():
        got = _fused_mlp1(list(net), x, max_in=128, max_out=16)
        want = net(x)
    assert got is not None and got.shape == want.shape
    torch.testing.assert_close(got, want, rtol=1e-5, atol=2e-6)


@pytest.mark.parametrize("pre", [False, True])
@pytest.mark.parametrize("H", [256, 2048])
@pytest.mark.parametrize("O", [5, 8, 15, 16])
def test_wide_k7b_matches_pytorch(O, H, pre):
    """marlsc_linear_out_forward with 5-16 outputs, with and without the producing layer's bias + ReLU applied on the way in
    (2048 inputs: the weights need more than the default 48 KB of shared memory)."""
    from marlsc_b200.rollout.policy import _linear_out, _linear_out_ok
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.manual_seed(O * 7 + H)
    m = torch.nn.Linear(H, O).cuda()
    h = torch.randn((1001, H), device="cuda:0")
    pb = torch.randn(H, device="cuda:0") if pre else None
    with torch.no_grad():
        assert _linear_out_ok(m, h, max_out=16)
        got = _linear_out(h, m, pre_bias=pb)
        want = m(torch.relu(h + pb) if pre else h)
    torch.testing.assert_close(got, want, rtol=1e-5, atol=2e-5 if H == 2048 else 2e-6)


@pytest.mark.parametrize("D,H,O", [(78, 512, 15), (78, 512, 1), (33, 1024, 6)])
def test_head_too_wide_for_shared_memory_takes_the_library_path(D, H, O):
    """A one-hidden-layer head whose weights do not fit K7's shared memory runs through the library GEMM + K7b in the
    rollout forward, with the same numbers as the nn.Sequential; K7 itself refuses the head."""
    from marlsc_b200 import _capi
    from marlsc_b200.rollout.policy import _central_forward, _fused_mlp1, _mlp1_smem_bytes, mlp
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.manual_seed(H + O)
    assert _mlp1_smem_bytes(D, H, O) > torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    net = mlp(D, (H,), O).cuda()
    x = torch.randn((2049, D), device="cuda:0")
    with torch.no_grad():
        got, want = _central_forward(net, x), net(x)
        with pytest.raises(_capi.MarlscError):
            _fused_mlp1(list(net), x, max_in=128, max_out=16)
    torch.testing.assert_close(got, want, rtol=1e-5, atol=2e-6)


@pytest.mark.parametrize("hidden", [(256,), (64, 64)])
def test_centralized_rollout_forward_matches_autograd_path(hidden):
    """The rollout forward (K7 for one hidden layer; library GEMMs + K7b for two) against the PyTorch modules."""
    from marlsc_b200.rollout import CentralizedActorCritic
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.manual_seed(3)
    pol = CentralizedActorCritic(11, 3, 2, actor_hidden=hidden, critic_hidden=hidden).cuda()
    obs = torch.randn((4097, 3, 11), device="cuda:0")
    with torch.no_grad():
        fast_m, fast_v = pol.action_mean(obs), pol.value(obs)
    slow_m, slow_v = pol.action_mean(obs), pol.value(obs)
    assert slow_m.requires_grad and not fast_m.requires_grad
    torch.testing.assert_close(fast_m, slow_m.detach(), rtol=1e-5, atol=2e-6)
    torch.testing.assert_close(fast_v, slow_v.detach(), rtol=1e-5, atol=2e-6)


def test_centralized_collector_matches_manual_loop():
    """Collector with a CentralizedActorCritic = policy forward on the global state -> step -> reward summed over the
    warehouses -> GAE over the environments; its buffers equal a hand-written loop over the same env seeds, and its GAE the
    oracle's on the summed rewards. The horizon crosses two episode boundaries."""
    from marlsc_b200.envs import BatchedInventoryEnv
    from marlsc_b200.rollout import CentralizedActorCritic, PPOLearner, RolloutCollector
    from oracle.gae_oracle import gae_targets
    cfg = _small_cfg(episode_length=12)
    torch.manual_seed(0)
    E, T, W, S = 32, 30, 3, 2
    env = BatchedInventoryEnv(cfg, E, device="cuda:0", seed=11)
    pol = CentralizedActorCritic(env.obs_dim, W, S, actor_hidden=(32,), critic_hidden=(32,)).cuda()
    col = RolloutCollector(env, pol, T, gamma=0.97, lam=0.9, standardize_advantages=False, seed=5, keep_dist_inputs=True)
    ro = col.collect()
    assert ro.cut.cpu().tolist() == [1 if (t + 1) % 12 == 0 else 0 for t in range(T)]
    assert ro.actions.shape == (T, E, W * S) and ro.mean_old.shape == (T, E, W * S) and ro.log_std_old.shape == (1, W * S)
    assert ro.logp.shape == ro.rewards.shape == ro.advantages.shape == ro.targets.shape == (T, E)
    assert ro.values.shape == (T + 1, E)
    env2 = BatchedInventoryEnv(cfg, E, device="cuda:0", seed=11)
    gen = torch.Generator(device="cuda:0")
    gen.manual_seed(5)
    obs = env2.reset().clone()
    rewards, values, cut_vals = [], [], {}
    with torch.no_grad():
        for t in range(T):
            act, raw, logp, val, mean = pol.act(obs, generator=gen, return_raw=True)
            assert torch.equal(obs, ro.obs[t]) and torch.equal(raw, ro.actions[t]) and torch.equal(logp, ro.logp[t])
            assert torch.equal(mean, ro.mean_old[t]) and torch.equal(val, ro.values[t])
            assert act.shape == (E, W, S) and torch.equal(act.reshape(E, W * S), raw.clamp(-1, 1))
            o, r, trunc = env2.step(act.contiguous())
            rewards.append(r.sum(1))
            values.append(val)
            obs = o.clone()
            if trunc:
                cut_vals[t] = pol.value(obs)
                obs = env2.reset().clone()
        values.append(pol.value(obs))
    r = torch.stack(rewards).cpu().numpy()
    v = torch.stack(values).cpu().numpy()
    assert np.array_equal(r, ro.rewards.cpu().numpy())
    assert np.array_equal(v, ro.values.cpu().numpy())
    cv = np.zeros_like(r)
    for t, x in cut_vals.items():
        cv[t] = x.cpu().numpy()
    assert np.array_equal(cv, col.cut_values.cpu().numpy())
    a_ref, t_ref = gae_targets(r, v, 0.97, 0.9, ro.cut.cpu().numpy().astype(bool), cv)
    np.testing.assert_allclose(ro.targets.cpu().numpy(), t_ref, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(ro.advantages.cpu().numpy(), a_ref, rtol=1e-5, atol=1e-4)
    # a learner step over a minibatch of the rollout runs (K6 with one policy and W*S actions) and moves the weights
    learner = PPOLearner(pol, lr=1e-3, grad_clip=5.0, use_kl_loss=True)
    before = pol.log_std.detach().clone()
    stats = learner.minibatch_step(ro, slice(0, 10), slice(0, 16))
    assert np.isfinite(stats["total"]) and not torch.equal(before, pol.log_std.detach())


def test_centralized_collector_matches_the_wrapper():
    """Per environment, the collector's global observations and summed rewards equal CentralizedEnvWrapper (the reference's
    single-agent view) driven with the same seed and the same joint actions."""
    from marlsc_b200.envs import BatchedInventoryEnv, CentralizedEnvWrapper
    from marlsc_b200.rollout import CentralizedActorCritic, RolloutCollector
    from marlsc_b200.seeds import SeedManager
    cfg = _small_cfg(episode_length=12)
    torch.manual_seed(1)
    E, T, W = 4, 11, 3
    env = BatchedInventoryEnv(cfg, E, device="cuda:0", seed=11)
    pol = CentralizedActorCritic(env.obs_dim, W, 2, actor_hidden=(32,), critic_hidden=(32,), logstd_init=-0.5).cuda()
    ro = RolloutCollector(env, pol, T, seed=2).collect()
    obs = ro.obs.cpu().numpy().reshape(T + 1, E, -1)
    joint = ro.actions.clamp(-1, 1).cpu().numpy()
    rew = ro.rewards.cpu().numpy()
    for e in range(E):
        w = CentralizedEnvWrapper(cfg, seed=SeedManager.derive_env_seed(11, 0, e))
        o, _ = w.reset()
        np.testing.assert_allclose(o, obs[0, e], rtol=1e-5, atol=1e-6)
        for t in range(T):
            o, r, term, trunc, _ = w.step(joint[t, e])
            np.testing.assert_allclose(o, obs[t + 1, e], rtol=1e-5, atol=1e-6)
            np.testing.assert_allclose(r, rew[t, e], rtol=1e-5, atol=1e-5)
            assert not term and not trunc


@pytest.mark.parametrize("W,S,D", [(3, 2, 11), (3, 5, 26)])
def test_k6_matches_loss_reference_on_the_joint_action(W, S, D):
    """K6 with one policy over W*S actions against the PyTorch objective: loss terms and every parameter gradient."""
    from marlsc_b200.rollout import CentralizedActorCritic, PPOLearner
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.manual_seed(W * S)
    pol = CentralizedActorCritic(D, W, S, actor_hidden=(64,), critic_hidden=(64,), logstd_init=-0.3).cuda()
    B = 3001
    obs = torch.randn((B, W, D), device="cuda:0")
    with torch.no_grad():
        mean = pol.action_mean(obs)
        actions = mean + 0.6 * torch.randn_like(mean)
        logp_old = pol.log_prob(mean, actions) + 0.3 * torch.randn(B, device="cuda:0")
        mean_old = mean + 0.1 * torch.randn_like(mean)
        ls_old = (pol.clamped_log_std() - 0.1).reshape(1, W * S)
    adv, tgt = torch.randn(B, device="cuda:0"), torch.randn(B, device="cuda:0") + pol.value(obs).detach()
    out, grads = {}, {}
    for fused in (True, False):
        learner = PPOLearner(pol, fused_loss=fused, use_kl_loss=True, hysteretic_beta=0.5, vf_clip_param=1.0)
        for p in pol.parameters():
            p.grad = None
        res = learner.loss(obs, actions, logp_old, adv, tgt, mean_old, ls_old)
        res["total"].backward()
        out[fused] = {k: float(v) for k, v in res.items()}
        grads[fused] = [p.grad.detach().clone() for p in pol.parameters()]
    for k in ("total", "policy", "vf", "kl", "entropy"):
        assert out[True][k] == pytest.approx(out[False][k], rel=1e-4, abs=1e-6), k
    for a, b in zip(grads[True], grads[False]):
        torch.testing.assert_close(a, b, rtol=1e-4, atol=1e-6)


def test_evaluate_centralized_policy_matches_manual_loop():
    from marlsc_b200.envs import BatchedInventoryEnv
    from marlsc_b200.rollout import CentralizedActorCritic, MeanStdFilter, evaluate
    cfg = _small_cfg()
    E = 64
    torch.manual_seed(0)
    a = BatchedInventoryEnv(cfg, E, device="cuda:0", host_samplers=False, device_demand=True, demand_seed=4, seed=8, episode_metrics=True)
    b = BatchedInventoryEnv(cfg, E, device="cuda:0", host_samplers=False, device_demand=True, demand_seed=4, seed=8)
    pol = CentralizedActorCritic(a.obs_dim, 3, 2, actor_hidden=(32,), logstd_init=0.5).cuda()
    res = evaluate(a, pol, 2)
    for ep in range(2):
        obs, done, total = b.reset(), False, torch.zeros((E, 3), dtype=torch.float64, device="cuda:0")
        while not done:
            with torch.no_grad():
                act = pol.actor(obs.reshape(E, -1)).clamp(-1.0, 1.0).reshape(E, 3, 2)
            obs, rew, done = b.step(act.contiguous())
            total += rew.double()
        torch.testing.assert_close(res["episode_return"][ep], total, rtol=1e-6, atol=1e-4)
    # with a frozen global-state filter the policy sees the normalised [E, W*D] state; the env's buffer stays raw
    flt = MeanStdFilter(3 * a.obs_dim, "cuda:0", update=False)
    flt.count.fill_(10.0)
    flt.mean.uniform_(0, 5)
    flt.m2.uniform_(9, 90)
    res = evaluate(a, pol, 1, obs_filter=flt)
    obs, done, total = b.reset(), False, torch.zeros((E, 3), dtype=torch.float64, device="cuda:0")
    while not done:
        with torch.no_grad():
            x = flt(obs.clone().reshape(E, -1))
            act = pol.actor(x).clamp(-1.0, 1.0).reshape(E, 3, 2)
        obs, rew, done = b.step(act.contiguous())
        total += rew.double()
    torch.testing.assert_close(res["episode_return"][0], total, rtol=1e-6, atol=1e-4)
    a.close()
    b.close()


def test_cppo_learns_on_the_small_config():
    """3 x 2 config, 4,096 environments, device demand: 20 PPO updates of a CentralizedActorCritic lower the mean total cost
    of the deterministic policy."""
    from marlsc_b200.envs import BatchedInventoryEnv
    from marlsc_b200.rollout import CentralizedActorCritic, MeanStdFilter, PPOLearner, RolloutCollector, evaluate
    cfg = _small_cfg()
    E = 4096
    torch.manual_seed(0)
    env = BatchedInventoryEnv(cfg, E, device="cuda:0", host_samplers=False, device_demand=True, demand_seed=1, seed=1)
    ev = BatchedInventoryEnv(cfg, 1024, device="cuda:0", host_samplers=False, device_demand=True, demand_seed=9, seed=9,
                             episode_metrics=True)
    W, D = env.n_warehouses, env.obs_dim
    pol = CentralizedActorCritic(D, W, env.n_skus, actor_hidden=(64,), critic_hidden=(64,), logstd_init=-0.5).cuda()
    flt = MeanStdFilter(W * D, "cuda:0")
    col = RolloutCollector(env, pol, 25, gamma=0.99, lam=0.95, seed=3, obs_filter=flt)
    learner = PPOLearner(pol, lr=1e-3, num_epochs=4, num_minibatches=4, grad_clip=1.0, vf_clip_param=1e4, vf_loss_coeff=0.01)
    frozen = MeanStdFilter(W * D, "cuda:0", update=False)

    def cost():
        frozen.load_state_dict(flt.state_dict())
        return evaluate(ev, pol, 1, obs_filter=frozen).summary()["total_cost"]["mean"]

    col.collect()                                   # the filter's statistics come from the first rollout
    before = cost()
    for _ in range(20):
        stats = learner.update(col.collect())
        assert np.isfinite(stats["total"])
    after = cost()
    assert after < before, (before, after)
    env.close()
    ev.close()
