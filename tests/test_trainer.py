"""-m gpu: the environment snapshot (bit-for-bit continuation after a restore, refusal of a different environment), the
trainer's learning-rate schedule, learning, files, checkpoints and resume, and tools/train.py."""
import copy
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import yaml

from golden.scenarios import allfeat_ratio_stochastic, basestock_cost_meanstd, large_network, small_default

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _cfg(d):
    from marlsc_b200.config import environment_config_from_dict
    return environment_config_from_dict(d)


# ------------------------------------------------------------------ environment snapshot
def _compact():
    from marlsc_b200.envs import BatchedInventoryEnv
    cfg = _cfg(dict(large_network(episode_length=12), allow_region_mismatch=True))
    env = BatchedInventoryEnv(cfg, 8, device="cuda:0", seed=3, host_samplers=False, device_demand=True, demand_seed=5,
                              episode_metrics=True)
    assert env.layout == "compact"
    return env


def _wide_device_leads():
    from marlsc_b200.envs import BatchedInventoryEnv
    d = allfeat_ratio_stochastic()
    d["episode_length"] = 12
    env = BatchedInventoryEnv(_cfg(d), 16, device="cuda:0", seed=4, host_samplers=False, device_demand=True, demand_seed=6,
                              layout="wide", episode_metrics=True)
    env.enable_device_leads(seed=8)
    assert env.layout == "wide" and env.ring_lead is not None and env.forecast is not None and env.demand_hist is not None
    return env


def _wide_host_samplers():
    from marlsc_b200.envs import BatchedInventoryEnv
    d = basestock_cost_meanstd()
    d["episode_length"] = 12
    d["initial_inventory"] = dict(type="uniform", params=dict(min=5, max=40))
    env = BatchedInventoryEnv(_cfg(d), 16, device="cuda:0", seed=9, layout="wide", episode_metrics=True)
    assert env.layout == "wide" and env.stochastic_lead
    return env


def _record(env, actions):
    """Step with the given actions (resetting at the end of an episode); every step's observations, rewards, state
    tensors and metric accumulators."""
    from marlsc_b200.envs.batched_env import _SNAPSHOT_TENSORS
    out = []
    for a in actions:
        obs, rew, done = env.step(a)
        rec = dict(obs=obs.clone(), rew=rew.clone(), timestep=env.timestep)
        rec.update({k: getattr(env, k).clone() for k in _SNAPSHOT_TENSORS if getattr(env, k) is not None})
        rec.update({"m_" + k: v.clone() for k, v in env.episode_metrics().items()})
        if done:
            rec["reset_obs"] = env.reset().clone()
            rec["reset_inventory"] = env.inventory.clone()
        out.append(rec)
    return out


@pytest.mark.parametrize("make", [_compact, _wide_device_leads, _wide_host_samplers],
                         ids=["compact_device_demand", "wide_device_leads", "wide_host_samplers"])
def test_snapshot_continues_bit_for_bit(make):
    env = make()
    E, W, S = env.num_envs, env.n_warehouses, env.n_skus
    g = torch.Generator(device="cuda:0")
    g.manual_seed(1)
    acts = [torch.rand((E, W, S), device="cuda:0", generator=g) * 2 - 1 for _ in range(12 + 4)]
    env.reset()
    for a in acts[:5]:                                  # mid-episode
        env.step(a)
    sd = env.state_dict()
    want = _record(env, acts[5:])                       # past the end of the episode, through a reset and 4 more steps
    assert any("reset_obs" in r for r in want) and want[-1]["timestep"] == 4
    fresh = make()
    fresh.load_state_dict(sd)
    got = _record(fresh, acts[5:])
    for t, (a, b) in enumerate(zip(want, got)):
        assert a.keys() == b.keys()
        for k in a:
            if isinstance(a[k], torch.Tensor):
                assert torch.equal(a[k], b[k]), (t, k)
            else:
                assert a[k] == b[k], (t, k)
    env.close()
    fresh.close()


def test_snapshot_refuses_a_different_environment():
    from marlsc_b200.envs import BatchedInventoryEnv

    def big(episode_length=12):
        return _cfg(dict(large_network(episode_length=episode_length), allow_region_mismatch=True))
    cfg = big()
    a = BatchedInventoryEnv(cfg, 4, device="cuda:0", seed=1)
    assert a.layout == "compact"
    a.reset()
    sd = a.state_dict()
    with pytest.raises(ValueError, match="layout"):
        BatchedInventoryEnv(cfg, 4, device="cuda:0", seed=1, layout="wide").load_state_dict(sd)
    with pytest.raises(ValueError, match="num_envs"):
        BatchedInventoryEnv(cfg, 8, device="cuda:0", seed=1).load_state_dict(sd)
    with pytest.raises(ValueError, match="spec"):
        BatchedInventoryEnv(big(13), 4, device="cuda:0", seed=1).load_state_dict(sd)
    with pytest.raises(ValueError, match="episode_metrics"):
        BatchedInventoryEnv(cfg, 4, device="cuda:0", seed=1, episode_metrics=True).load_state_dict(sd)
    with pytest.raises(ValueError, match="device_demand"):
        BatchedInventoryEnv(cfg, 4, device="cuda:0", seed=1, device_demand=True).load_state_dict(sd)
    with pytest.raises(ValueError, match="host_samplers"):
        BatchedInventoryEnv(cfg, 4, device="cuda:0", seed=1, host_samplers=False).load_state_dict(sd)
    BatchedInventoryEnv(cfg, 4, device="cuda:0", seed=1).load_state_dict(sd)


# ------------------------------------------------------------------ trainer
def _algo(name="ippo", lr=1e-3, iters=4, ckpt=2, batch=None, epochs=2, minibatches=2, norm="meanstd", hidden=32,
          sharing=True, **specific):
    from marlsc_b200.config import algorithm_config_from_dict
    net = dict(shared_layers=None, use_mu_sigma_head=False,
               actor=dict(type="mlp", config=dict(hidden_sizes=[hidden], activation="relu")),
               critic=dict(type="mlp", config=dict(hidden_sizes=[hidden], activation="relu")))
    sp = dict(use_gae=True, lam=0.95, gamma=0.99, clip_param=0.2, vf_clip_param=1e4, vf_loss_coeff=0.01, grad_clip=1.0,
              logstd_init=-0.5, logstd_floor=-3.5, obs_normalization=norm, networks=net)
    if name != "cppo":
        sp["parameter_sharing"] = sharing
    sp.update(specific)
    return algorithm_config_from_dict(dict(algorithm=dict(
        name=name, shared=dict(num_iterations=iters, checkpoint_freq=ckpt, batch_size=batch or 1024, num_epochs=epochs,
                               num_minibatches=minibatches, learning_rate=lr, eval_interval=1, num_eval_episodes=1),
        algorithm_specific=sp)))


def _lines(path):
    with open(os.path.join(path, "training_metrics.jsonl")) as f:
        return [json.loads(ln) for ln in f]


def test_learning_rate_follows_the_schedule(tmp_path):
    from marlsc_b200.rollout import Trainer, lr_schedule
    sched = [[0, 1e-3], [2048, 5e-4], [4096, 1e-4]]
    tr = Trainer(_cfg(small_default()), _algo(lr=sched, iters=6, ckpt=6), 256, str(tmp_path), horizon=4, num_eval_envs=64)
    assert tr.steps_per_iteration == 1024
    f, seen = lr_schedule(sched), []
    tr.run(log=lambda line: seen.append((line["iteration"], line["lr"], tr.learner.opt.param_groups[0]["lr"])))
    assert [s[0] for s in seen] == list(range(1, 7))
    for it, logged, opt_lr in seen:
        assert logged == opt_lr == f((it - 1) * 1024)
    assert [s[1] for s in seen][:4] == pytest.approx([1e-3, 7.5e-4, 5e-4, 3e-4])
    assert seen[-1][1] == pytest.approx(1e-4)


def test_ippo_learns_and_writes_its_files(tmp_path):
    """IPPO on the 3 x 2 config, parameter sharing, meanstd_custom, 4,096 environments, 20 iterations: the evaluated total
    cost falls; one metrics line per iteration, the periodic / best / final checkpoints, best = highest logged return."""
    from marlsc_b200.rollout import Trainer, evaluate
    out = tmp_path / "ippo"
    algo = _algo(iters=20, ckpt=5, batch=4096 * 25, epochs=4, minibatches=4, norm="meanstd_custom", hidden=64)
    tr = Trainer(_cfg(small_default()), algo, 4096, str(out))
    assert tr.horizon == 25 and tr.eval_env.num_envs == 1024 and tr.obs_stats is not None
    before = evaluate(tr.eval_env, tr.policy, 1).summary()["total_cost"]["mean"]
    tr.run()
    lines = _lines(out)
    assert [ln["iteration"] for ln in lines] == list(range(1, 21))
    assert [ln["env_steps"] for ln in lines] == [i * 4096 * 25 for i in range(1, 21)]
    assert all(np.isfinite(ln["learner"]["total"]) and ln["collect_s"] > 0 and ln["update_s"] > 0 for ln in lines)
    after = np.mean([ln["eval"]["total_cost"]["mean"] for ln in lines[-3:]])
    assert after < before, (before, after)
    for name in ("checkpoint_5.pt", "checkpoint_10.pt", "checkpoint_15.pt", "checkpoint_20.pt", "checkpoint_final.pt",
                 "checkpoint_best.pt"):
        assert (out / name).exists(), name
    rets = [ln["eval"]["episode_return"]["mean"] for ln in lines]
    best = torch.load(out / "checkpoint_best.pt", map_location="cpu", weights_only=False)
    assert best["iteration"] == int(np.argmax(rets)) + 1 and best["best_return"] == max(rets)
    assert torch.load(out / "checkpoint_final.pt", map_location="cpu", weights_only=False)["iteration"] == 20


@pytest.mark.parametrize("name,norm", [("mappo", "meanstd_grouped"), ("cppo", "meanstd")])
def test_mappo_and_cppo_run(name, norm, tmp_path):
    from marlsc_b200.rollout import CentralizedActorCritic, Trainer
    tr = Trainer(_cfg(small_default()), _algo(name, iters=2, ckpt=1, norm=norm, use_kl_loss=True), 256, str(tmp_path),
                 horizon=4, num_eval_envs=32)
    assert isinstance(tr.policy, CentralizedActorCritic) == (name == "cppo")
    tr.run()
    lines = _lines(tmp_path)
    assert len(lines) == 2 and all("eval" in ln and np.isfinite(ln["learner"]["total"]) for ln in lines)
    for f in ("checkpoint_1.pt", "checkpoint_2.pt", "checkpoint_final.pt", "checkpoint_best.pt"):
        assert (tmp_path / f).exists(), f


def test_resume_continues_the_run(tmp_path):
    """k + 1 = 3 iterations with a checkpoint at k = 2, against a resume from that checkpoint running iteration 3: the same
    rollout bit for bit, parameters after the update to rtol 1e-5 (K6 and the advantage standardisation sum with atomics),
    and the same iteration, env steps and learning rate in the metrics line."""
    from marlsc_b200.rollout import Trainer
    keys = ("obs", "actions", "logp", "rewards", "values")

    def record(tr, store):
        orig = tr.collector.collect

        def collect():
            ro = orig()
            store.append({k: getattr(ro, k).clone() for k in keys})
            return ro
        tr.collector.collect = collect

    algo = _algo(lr=[[0, 1e-3], [4096, 1e-4]], iters=3, ckpt=2, sharing=False, use_kl_loss=True)
    a = Trainer(_cfg(small_default()), algo, 256, str(tmp_path / "a"), horizon=6, num_eval_envs=64, seed=3)
    ra, rb = [], []
    record(a, ra)
    a.run()
    b = Trainer.resume(str(tmp_path / "a" / "checkpoint_2.pt"), out_dir=str(tmp_path / "b"))
    assert b.iteration == 2 and b.horizon == 6 and b.num_envs == 256
    record(b, rb)
    b.run()
    assert len(ra) == 3 and len(rb) == 1
    for k in keys:
        assert torch.equal(ra[2][k], rb[0][k]), k
    for (n, p), q in zip(a.policy.named_parameters(), b.policy.parameters()):
        torch.testing.assert_close(p, q, rtol=1e-5, atol=1e-6, msg=n)
    la, lb = _lines(tmp_path / "a"), _lines(tmp_path / "b")
    assert len(lb) == 1
    for k in ("iteration", "env_steps", "lr"):
        assert la[2][k] == lb[0][k], k
    # resuming into the run's own directory keeps its metrics up to the checkpoint
    c = Trainer.resume(str(tmp_path / "a" / "checkpoint_2.pt"))
    assert [ln["iteration"] for ln in _lines(tmp_path / "a")] == [1, 2] and c.iteration == 2


def test_train_cli_runs_two_iterations(tmp_path):
    env_yaml, algo_yaml = tmp_path / "env.yaml", tmp_path / "algo.yaml"
    env_yaml.write_text(yaml.safe_dump(dict(environment=small_default())))
    from test_host_logic import IPPO
    d = copy.deepcopy(IPPO)
    d["algorithm"]["shared"].update(num_iterations=2, checkpoint_freq=1, batch_size=256 * 4, num_epochs=2, num_minibatches=2)
    algo_yaml.write_text(yaml.safe_dump(d))
    out = tmp_path / "run"
    res = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "train.py"), "--env-config", str(env_yaml),
                          "--algo-config", str(algo_yaml), "--num-envs", "256", "--out", str(out), "--eval-envs", "32"],
                         capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout + res.stderr
    assert "power limit" in res.stdout and "iter     2" in res.stdout
    assert len(_lines(out)) == 2 and (out / "checkpoint_final.pt").exists()
