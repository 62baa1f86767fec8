"""CPPO without a device: CentralizedActorCritic built from a CPPO config, its action layout against
CentralizedEnvWrapper's, its log-prob, the learner on a synthetic CPPO rollout, and the C limits of the widened K7 / K7b."""
import ctypes
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import marlsc_b200  # noqa: F401
from marlsc_b200 import _capi
from marlsc_b200.config import algorithm_config_from_dict
from marlsc_b200.envs import CentralizedEnvWrapper
from marlsc_b200.rollout import ActorCritic, CentralizedActorCritic, PPOLearner, env_meta_from_algorithm_config
from marlsc_b200.rollout.collector import Rollout

EUNSUPPORTED = -4                      # MARLSC_EUNSUPPORTED (include/marlsc_b200.h)

# shaped like the reference's config_files/algorithms/cppo.yaml
CPPO = dict(algorithm=dict(
    name="cppo",
    shared=dict(num_iterations=300, checkpoint_freq=100, batch_size=8000, num_epochs=20, num_minibatches=10,
                learning_rate=5e-4, num_env_runners=2, num_envs_per_env_runner=10),
    algorithm_specific=dict(use_gae=True, lam=0.95, gamma=0.99, clip_param=0.1, vf_clip_param=800.0, logstd_init=-1.15,
                            logstd_floor=-3.5, obs_normalization="meanstd",
                            networks=dict(shared_layers=None, use_mu_sigma_head=False,
                                          actor=dict(type="mlp", config=dict(hidden_sizes=[64], activation="relu")),
                                          critic=dict(type="mlp", config=dict(hidden_sizes=[48], activation="relu"))))))


def test_from_algorithm_config_builds_the_joint_heads():
    algo = algorithm_config_from_dict(CPPO)
    W, D, S = 3, 11, 2
    pol = CentralizedActorCritic.from_algorithm_config(algo, local_obs_dim=D, n_warehouses=W, action_dim=S)
    lin = [m for m in pol.actor if isinstance(m, torch.nn.Linear)]
    assert [(m.in_features, m.out_features) for m in lin] == [(W * D, 64), (64, W * S)]
    lin = [m for m in pol.critic if isinstance(m, torch.nn.Linear)]
    assert [(m.in_features, m.out_features) for m in lin] == [(W * D, 48), (48, 1)]
    assert pol.log_std.shape == (W * S,) and pol.n_policies == 1
    assert torch.allclose(pol.std(), torch.full((W * S,), float(np.exp(-1.15))), atol=1e-6)
    pol.log_std.data.fill_(-10.0)
    assert torch.allclose(pol.std(), torch.full((W * S,), float(np.exp(-3.5))), atol=1e-7)      # floor
    # the env of a CPPO run carries no warehouse id
    assert "include_warehouse_id" not in env_meta_from_algorithm_config(algo)
    assert env_meta_from_algorithm_config(algo)["obs_normalization"] == "meanstd"


def test_actor_critic_rejects_a_cppo_config():
    algo = algorithm_config_from_dict(CPPO)
    with pytest.raises(ValueError, match="CentralizedActorCritic"):
        ActorCritic.from_algorithm_config(algo, local_obs_dim=11, n_warehouses=3, action_dim=2)
    ippo = algorithm_config_from_dict({"algorithm": {**CPPO["algorithm"], "name": "ippo"}})
    with pytest.raises(ValueError, match="ActorCritic"):
        CentralizedActorCritic.from_algorithm_config(ippo, local_obs_dim=11, n_warehouses=3, action_dim=2)


def test_act_shapes_and_joint_action_layout():
    torch.manual_seed(0)
    E, W, D, S = 7, 3, 5, 4
    pol = CentralizedActorCritic(D, W, S, actor_hidden=(16,), critic_hidden=(16,))
    obs = torch.randn(E, W, D)
    act, raw, logp, val, mean = pol.act(obs, return_raw=True)
    assert act.shape == (E, W, S) and raw.shape == (E, W * S) and mean.shape == (E, W * S)
    assert logp.shape == (E,) and val.shape == (E,)
    assert torch.equal(mean, pol.actor(obs.reshape(E, W * D)))
    assert torch.equal(val, pol.critic(obs.reshape(E, W * D)).squeeze(-1))
    a2, lp2, v2 = pol.act(obs)
    assert a2.shape == (E, W, S) and lp2.shape == (E,) and v2.shape == (E,)
    # entry w*S + s of the joint vector is (warehouse w, SKU s): what the wrapper hands each agent
    wrapper = SimpleNamespace(n_warehouses=W, n_skus=S, env=SimpleNamespace(agents=[f"warehouse_{w}" for w in range(W)]))
    for e in range(E):
        split = CentralizedEnvWrapper._split_action(wrapper, raw[e].detach().clamp(-1, 1).numpy())
        for w in range(W):
            assert np.array_equal(split[f"warehouse_{w}"], act[e, w].detach().numpy())
    with pytest.raises(ValueError, match="obs must be"):
        pol.action_mean(torch.randn(E, W * D))


def test_log_prob_is_the_diagonal_gaussian():
    torch.manual_seed(1)
    W, D, S = 3, 6, 5
    pol = CentralizedActorCritic(D, W, S, actor_hidden=(8,), critic_hidden=(8,), logstd_init=-0.7, logstd_floor=-1.0)
    pol.log_std.data[:4] = -3.0                                          # below the floor: clamped
    obs = torch.randn(11, W, D)
    with torch.no_grad():
        mean = pol.action_mean(obs)
        raw = mean + torch.randn_like(mean)
        want = torch.distributions.Normal(mean, pol.clamped_log_std().exp()).log_prob(raw).sum(-1)
        assert torch.allclose(pol.log_prob(mean, raw), want, atol=1e-5)
        assert torch.allclose(pol.entropy(), torch.distributions.Normal(mean[0], pol.std()).entropy().sum(), atol=1e-5)


def test_learner_update_on_a_cppo_rollout():
    """The same loop as for the multi-agent policies, one sample per environment: at the behaviour parameters the first
    minibatch has ratio 1 and KL 0."""
    torch.manual_seed(2)
    T, E, W, D, S = 6, 10, 3, 5, 2
    pol = CentralizedActorCritic(D, W, S, actor_hidden=(8,), critic_hidden=(8,))
    obs = torch.randn(T + 1, E, W, D)
    with torch.no_grad():
        act, raw, logp, val, mean = pol.act(obs[:T], return_raw=True)
    assert raw.shape == (T, E, W * S) and logp.shape == (T, E)
    ro = Rollout(obs, raw, logp, torch.randn(T, E), torch.randn(T + 1, E), torch.randn(T, E), torch.randn(T, E),
                 torch.zeros(T, dtype=torch.uint8), mean, pol.clamped_log_std().detach().reshape(1, W * S).clone())
    learner = PPOLearner(pol, lr=1e-3, fused_loss=False, use_kl_loss=True, num_epochs=3, num_minibatches=4, seed=1)
    first = learner.loss(obs[:T].reshape(T * E, W, D), raw.reshape(T * E, W * S), logp.reshape(T * E),
                         ro.advantages.reshape(T * E), ro.targets.reshape(T * E), mean.reshape(T * E, W * S), ro.log_std_old)
    assert abs(float(first["kl"])) < 1e-6
    assert torch.allclose(first["policy"], -ro.advantages.mean(), atol=1e-5)     # ratio == 1 everywhere
    before = [p.detach().clone() for p in pol.parameters()]
    stats = learner.update(ro)
    assert stats["minibatches"] == 12 and np.isfinite(stats["total"])
    assert all(not torch.equal(a, b.detach()) for a, b in zip(before, pol.parameters()))


def test_fused_learner_rejects_joint_actions_past_k6():
    pol = CentralizedActorCritic(4, 9, 57, actor_hidden=(8,), critic_hidden=(8,))         # 513 joint actions
    with pytest.raises(ValueError, match="512"):
        PPOLearner(pol, fused_loss=True)
    PPOLearner(pol, fused_loss=False)
    PPOLearner(CentralizedActorCritic(4, 8, 64, actor_hidden=(8,), critic_hidden=(8,)), fused_loss=True)   # 512


def test_widened_head_kernels_reject_past_their_limits_without_a_device():
    L = _capi.lib()
    buf = (ctypes.c_float * 64)()
    p = ctypes.addressof(buf) + (-ctypes.addressof(buf)) % 16        # 16-byte aligned, never dereferenced
    # K7: 129 inputs or 17 outputs
    assert L.marlsc_mlp1_forward(p, 10, 129, p, p, 8, p, p, 4, 0, p, None) == EUNSUPPORTED
    assert L.marlsc_mlp1_forward(p, 10, 33, p, p, 8, p, p, 17, 0, p, None) == EUNSUPPORTED
    assert L.marlsc_mlp1_forward(p, 10, 33, p, p, 8, p, p, 6, 2, p, None) == EUNSUPPORTED    # no such activation
    # K7b: 17 outputs, with and without pre_bias
    assert L.marlsc_linear_out_forward(p, 10, 64, None, p, p, 17, p, None) == EUNSUPPORTED
    assert L.marlsc_linear_out_forward(p, 10, 64, p, p, p, 17, p, None) == EUNSUPPORTED
    # the new limits themselves pass the argument checks; no rows means no device work
    assert L.marlsc_mlp1_forward(p, 0, 128, p, p, 8, p, p, 16, 1, p, None) == 0
    assert L.marlsc_linear_out_forward(p, 0, 64, p, p, p, 16, p, None) == 0
