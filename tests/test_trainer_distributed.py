"""-m gpu: data-parallel training on two ranks - NCCL on cuda:0 / cuda:1 when two GPUs are visible, gloo with both ranks on
cuda:0 otherwise. The K3 split and the advantage standardisation over both ranks, the learner's averaged update and statistics,
the merged observation filter, the trainer (identical parameters, one metrics file, sharded checkpoints, resume) and
tools/train.py under torch.distributed.run. Every rank is a child process joined with a timeout and terminated if it is still
alive, so no process outlives its test."""
import copy
import json
import os
import signal
import socket
import subprocess
import sys
import traceback

import pytest
import torch
import yaml

from golden.scenarios import small_default

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORLD = 2


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _entry(name, rank, port, out, args):
    import torch.distributed as dist
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        two = torch.cuda.device_count() >= WORLD
        dev = torch.device("cuda", rank if two else 0)
        torch.cuda.set_device(dev)
        if two:
            dist.init_process_group("nccl", rank=rank, world_size=WORLD, device_id=dev)
        else:
            dist.init_process_group("gloo", rank=rank, world_size=WORLD)
        import marlsc_b200  # noqa: F401
        globals()[name](rank, dev, out, *args)
        dist.destroy_process_group()
    except BaseException:
        traceback.print_exc()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(1)


def _spawn(name, out, *args, timeout=600):
    """Run ``name(rank, device, out, *args)`` on two ranks; fail unless both exit 0 within ``timeout`` seconds."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    port = _free_port()
    procs = [ctx.Process(target=_entry, args=(name, r, port, str(out), args)) for r in range(WORLD)]
    try:
        for p in procs:
            p.start()
        for p in procs:
            p.join(timeout)
        assert [p.exitcode for p in procs] == [0] * WORLD, [p.exitcode for p in procs]
    finally:
        for p in procs:
            if p.is_alive():
                p.terminate()
                p.join(10)
            if p.is_alive():
                p.kill()
                p.join(10)


def _load(out, rank):
    return torch.load(os.path.join(str(out), f"rank{rank}.pt"), map_location="cpu", weights_only=False)


# ------------------------------------------------------------------ 1. K3 split and the standardisation over the ranks
def _exact_values(n, seed, dev):
    """Multiples of 1/64 below 16 in magnitude: every partial sum of x and x^2 is exact in float64, so K3's sums do not depend
    on the order its atomics land in, and two runs can be compared bit for bit."""
    g = torch.Generator(device=dev).manual_seed(seed)
    return (torch.randint(-1024, 1024, (n,), device=dev, generator=g) / 64.0).float()


def _standardize_worker(rank, dev, out):
    import torch.distributed as dist
    from marlsc_b200 import _capi
    from marlsc_b200.rollout import standardize_, standardize_columns_
    L = _capi.lib()
    ws = torch.zeros(int(L.marlsc_standardize_workspace_bytes()), dtype=torch.uint8, device=dev)
    assert ws.numel() >= 24
    stream = torch.cuda.current_stream(dev).cuda_stream
    for n in (1, 300, 1 << 20):
        x = _exact_values(n, 7 + n, dev)
        a, b = x.clone(), x.clone()
        _capi.check(L.marlsc_standardize(a.data_ptr(), n, ws.data_ptr(), stream))
        _capi.check(L.marlsc_standardize_moments(b.data_ptr(), n, ws.data_ptr(), stream))
        torch.cuda.synchronize(dev)
        m = ws[:24].view(torch.float64).cpu()
        assert m[2].item() == n and m[0].item() == float(x.double().sum()) and m[1].item() == float((x.double() ** 2).sum())
        _capi.check(L.marlsc_standardize_apply(b.data_ptr(), n, ws.data_ptr(), stream))
        assert torch.equal(a, b), n
    # over the group: each rank's values standardised as its slice of both ranks' values together
    sizes = (5000, 5000)
    xs = [torch.randn(s, generator=torch.Generator().manual_seed(50 + r)).to(dev) * (r + 1) + r for r, s in enumerate(sizes)]
    mine = standardize_(xs[rank].clone(), dist.group.WORLD)
    whole = standardize_(torch.cat(xs))
    torch.testing.assert_close(mine, whole[rank * sizes[0]:(rank + 1) * sizes[0]], rtol=1e-6, atol=1e-6)
    # per column (independent policies): [T, E, W], the ranks' environments side by side
    cols = [torch.randn(6, 40, 3, generator=torch.Generator().manual_seed(70 + r)).to(dev) * torch.tensor([1.0, 5.0, 0.2]).to(dev) + r
            for r in range(WORLD)]
    mine = standardize_columns_(cols[rank].clone(), 3, dist.group.WORLD)
    whole = standardize_columns_(torch.cat(cols, dim=1), 3)
    torch.testing.assert_close(mine, whole[:, rank * 40:(rank + 1) * 40], rtol=1e-6, atol=1e-6)


def test_standardize_split_and_across_ranks(tmp_path):
    _spawn("_standardize_worker", tmp_path)


# ------------------------------------------------------------------ 2. learner
W, S, D, T, E = 3, 2, 9, 4, 16


def _policy(dev):
    from marlsc_b200.rollout import ActorCritic
    torch.manual_seed(0)
    return ActorCritic(D, W, S, actor_hidden=(32,), critic_hidden=(32,), logstd_init=-0.5).to(dev)


def _rollout(pol, seed, dev):
    """A synthetic rollout of T steps x E environments (behaviour = the initial policy)."""
    from marlsc_b200.rollout import Rollout
    g = torch.Generator().manual_seed(seed)
    obs = torch.randn(T + 1, E, W, D, generator=g).to(dev)
    with torch.no_grad():
        mean = pol.action_mean(obs[:T])
        act = mean + 0.4 * torch.randn(mean.shape, generator=g).to(dev)
        logp = pol.log_prob(mean, act)
    adv, tgt = torch.randn(T, E, W, generator=g).to(dev), torch.randn(T, E, W, generator=g).to(dev)
    return Rollout(obs, act, logp, torch.zeros(T, E, W, device=dev), torch.zeros(T + 1, E, W, device=dev), adv, tgt,
                   torch.zeros(T, dtype=torch.uint8, device=dev), mean.clone(), pol.clamped_log_std().detach().reshape(1, S).clone())


def _learner(pol):
    from marlsc_b200.rollout import PPOLearner
    # a small kl_target so that the coefficient moves: the adapted value must agree across the ranks
    return PPOLearner(pol, lr=1e-2, grad_clip=1.0, use_kl_loss=True, kl_target=1e-4, num_epochs=1, num_minibatches=2)


def _learner_worker(rank, dev, out):
    pol = _policy(dev)
    learner = _learner(pol)
    ro = _rollout(pol, 100 + rank, dev)
    stats = learner.update(ro, shuffle=False)
    torch.save(dict(rollout={k: getattr(ro, k).cpu() for k in ("obs", "actions", "logp", "advantages", "targets", "mean_old",
                                                               "log_std_old")},
                    stats=stats, kl_coeff=learner.kl_coeff, params=[p.detach().cpu() for p in pol.parameters()]),
               os.path.join(out, f"rank{rank}.pt"))


def test_learner_update_on_two_ranks_equals_one_process_on_the_joined_minibatches(tmp_path):
    _spawn("_learner_worker", tmp_path)
    r = [_load(tmp_path, k) for k in range(WORLD)]
    assert r[0]["stats"] == r[1]["stats"] and r[0]["kl_coeff"] == r[1]["kl_coeff"]
    for a, b in zip(r[0]["params"], r[1]["params"]):
        assert torch.equal(a, b)
    # one process: step_on over the concatenation of the ranks' k-th minibatches (shuffle=False: contiguous rows)
    dev = torch.device("cuda", 0)
    pol = _policy(dev)
    learner = _learner(pol)
    n, mb = T * E, T * E // 2
    flat = lambda x: x[:T].reshape(n, *x.shape[2:])                            # noqa: E731
    sums = {}
    for k in range(2):
        part = {name: torch.cat([flat(q["rollout"][name])[k * mb:(k + 1) * mb] for q in r]).to(dev)
                for name in ("obs", "actions", "logp", "advantages", "targets", "mean_old")}
        o = learner.step_on(part["obs"], part["actions"], part["logp"], part["advantages"], part["targets"], part["mean_old"],
                            r[0]["rollout"]["log_std_old"].to(dev))
        for name, v in o.items():
            sums[name] = sums.get(name, 0.0) + float(v.detach()) / 2
    kl_coeff = 0.2 * (1.5 if sums["kl"] > 2e-4 else 0.5 if sums["kl"] < 0.5e-4 else 1.0)
    assert r[0]["kl_coeff"] == kl_coeff
    for name, v in sums.items():
        assert r[0]["stats"][name] == pytest.approx(v, rel=1e-5, abs=1e-6), name
    for a, b in zip(r[0]["params"], pol.parameters()):
        torch.testing.assert_close(a, b.detach().cpu(), rtol=1e-5, atol=1e-6)


# ------------------------------------------------------------------ 3. observation filter
def _filter_worker(rank, dev, out):
    import torch.distributed as dist
    from marlsc_b200.config import environment_config_from_dict
    from marlsc_b200.envs import BatchedInventoryEnv
    from marlsc_b200.rollout import ActorCritic, MeanStdFilter, RolloutCollector
    env = BatchedInventoryEnv(environment_config_from_dict(small_default()), 16 + 8 * rank, device=dev, seed=rank,
                              host_samplers=False, device_demand=True, demand_seed=1 + rank)
    torch.manual_seed(0)
    pol = ActorCritic(env.obs_dim, env.n_warehouses, env.n_skus, actor_hidden=(16,), critic_hidden=(16,)).to(dev)
    flt = MeanStdFilter(env.obs_dim, dev)
    flt(torch.randn(50, env.obs_dim, generator=torch.Generator().manual_seed(3)).to(dev) * 4 + 2)   # the same prior on both
    col = RolloutCollector(env, pol, 5, seed=rank, obs_filter=flt, process_group=dist.group.WORLD)
    seen = []
    orig = flt.sync

    def sync(group=None):
        seen.append(dict(synced=[t.clone() for t in flt.synced], buffer=[t.clone() for t in flt.buffer]))
        orig(group)
    flt.sync = sync
    for _ in range(2):                       # the second collection starts from the first one's merge
        col.collect()
        seen[-1]["after"] = [t.clone() for t in (flt.count, flt.mean, flt.m2)]
    torch.save(seen, os.path.join(out, f"rank{rank}.pt"))


def test_filters_are_merged_after_each_collection(tmp_path):
    from marlsc_b200.rollout.obs_filter import merge_buffers
    _spawn("_filter_worker", tmp_path)
    r = [_load(tmp_path, k) for k in range(WORLD)]
    dev = torch.device("cuda", 0)
    assert len(r[0]) == len(r[1]) == 2
    for it in range(2):
        a, b = r[0][it], r[1][it]
        for x, y in zip(a["after"], b["after"]):
            assert torch.equal(x, y)                                  # bit-identical on every rank
        for x, y in zip(a["synced"], b["synced"]):
            assert torch.equal(x, y)
        assert a["buffer"][0] != b["buffer"][0]                       # 16 and 24 environments: different buffers
        want = merge_buffers(tuple(t.to(dev) for t in a["synced"]), [tuple(t.to(dev) for t in q[it]["buffer"]) for q in r])
        for x, y in zip(a["after"], want):
            assert torch.equal(x, y.cpu())
        if it == 1:
            for x, y in zip(a["synced"], r[0][0]["after"]):
                assert torch.equal(x, y)


# ------------------------------------------------------------------ 4. trainer
def _algo(name, iters, ckpt, norm="meanstd", **specific):
    from marlsc_b200.config import algorithm_config_from_dict
    net = dict(shared_layers=None, use_mu_sigma_head=False,
               actor=dict(type="mlp", config=dict(hidden_sizes=[32], activation="relu")),
               critic=dict(type="mlp", config=dict(hidden_sizes=[32], activation="relu")))
    sp = dict(use_gae=True, lam=0.95, gamma=0.99, clip_param=0.2, vf_clip_param=1e4, vf_loss_coeff=0.01, grad_clip=1.0,
              logstd_init=-0.5, logstd_floor=-3.5, obs_normalization=norm, networks=net, **specific)
    if name != "cppo":
        sp["parameter_sharing"] = False
    return algorithm_config_from_dict(dict(algorithm=dict(
        name=name, shared=dict(num_iterations=iters, checkpoint_freq=ckpt, batch_size=1024, num_epochs=2, num_minibatches=2,
                               learning_rate=[[0, 1e-3], [2048, 1e-4]], eval_interval=1, num_eval_episodes=1),
        algorithm_specific=sp)))


def _trainer_worker(rank, dev, out):
    from marlsc_b200.config import environment_config_from_dict
    from marlsc_b200.rollout import Trainer
    keys = ("obs", "actions", "logp", "rewards", "values")
    cfg = environment_config_from_dict(small_default())
    res = {}

    def record(tr, store):
        orig = tr.collector.collect

        def collect():
            ro = orig()
            store.append({k: getattr(ro, k).clone() for k in keys})
            return ro
        tr.collector.collect = collect

    def flat(tr):
        return torch.cat([p.detach().reshape(-1) for p in tr.policy.parameters()]).cpu()

    for name, iters, ckpt in (("ippo", 3, 2), ("cppo", 2, 1)):
        run = os.path.join(out, name)
        a = Trainer(cfg, _algo(name, iters, ckpt, use_kl_loss=True), 256, run, horizon=4, num_eval_envs=33, seed=3)
        assert a.env.num_envs == 128 and a.eval_env.num_envs == (17, 16)[rank] and a.steps_per_iteration == 1024
        params, ra = [], []
        record(a, ra)
        a.run(log=lambda line: params.append(flat(a)))
        res[name] = dict(params=params)
        if name == "ippo":
            b = Trainer.resume(os.path.join(run, "checkpoint_2.pt"), out_dir=os.path.join(out, "resumed"))
            assert b.iteration == 2 and b.num_envs == 256 and b.env.num_envs == 128
            rb = []
            record(b, rb)
            b.run()
            for k in keys:
                assert torch.equal(ra[2][k], rb[0][k]), k              # iteration 3's rollout, bit for bit, on every rank
            torch.testing.assert_close(flat(b), flat(a), rtol=1e-5, atol=1e-6)
            res["first_rewards"] = ra[0]["rewards"].cpu()
    torch.save(res, os.path.join(out, f"rank{rank}.pt"))


def _lines(path):
    with open(os.path.join(str(path), "training_metrics.jsonl")) as f:
        return [json.loads(ln) for ln in f]


def test_trainer_on_two_ranks(tmp_path):
    _spawn("_trainer_worker", tmp_path, timeout=900)
    r = [_load(tmp_path, k) for k in range(WORLD)]
    for name, iters in (("ippo", 3), ("cppo", 2)):
        assert len(r[0][name]["params"]) == iters
        for a, b in zip(r[0][name]["params"], r[1][name]["params"]):
            assert torch.equal(a, b), name                             # after every iteration
        lines = _lines(tmp_path / name)
        assert [ln["iteration"] for ln in lines] == list(range(1, iters + 1))
        assert all(ln["ranks"] == 2 and "eval" in ln for ln in lines)
        assert [ln["env_steps"] for ln in lines] == [i * 256 * 4 for i in range(1, iters + 1)]
        tags = ["best", "final"] + [str(i) for i in range(2 if name == "ippo" else 1, iters + 1, 2 if name == "ippo" else 1)]
        for tag in tags:
            main = torch.load(tmp_path / name / f"checkpoint_{tag}.pt", map_location="cpu", weights_only=False)
            assert main["world_size"] == 2 and main["args"]["num_envs"] == 256 and main["args"]["num_eval_envs"] == 33
            assert "env" not in main and "collector" not in main
            for k in range(WORLD):
                shard = torch.load(tmp_path / name / f"checkpoint_{tag}.rank{k}.pt", map_location="cpu", weights_only=False)
                assert shard["rank"] == k and shard["iteration"] == main["iteration"] and "env" in shard
        rets = [ln["eval"]["episode_return"]["mean"] for ln in lines]
        best = torch.load(tmp_path / name / "checkpoint_best.pt", map_location="cpu", weights_only=False)
        assert best["best_return"] == max(rets)
    # the ranks' environments draw different streams
    assert not torch.equal(r[0]["first_rewards"], r[1]["first_rewards"])
    assert len(_lines(tmp_path / "resumed")) == 1


# ------------------------------------------------------------------ 5. command line
def test_train_cli_under_torch_distributed_run(tmp_path):
    env_yaml, algo_yaml = tmp_path / "env.yaml", tmp_path / "algo.yaml"
    env_yaml.write_text(yaml.safe_dump(dict(environment=small_default())))
    from test_host_logic import IPPO
    d = copy.deepcopy(IPPO)
    d["algorithm"]["shared"].update(num_iterations=2, checkpoint_freq=1, batch_size=256 * 4, num_epochs=2, num_minibatches=2)
    algo_yaml.write_text(yaml.safe_dump(d))
    out = tmp_path / "run"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc-per-node", "2",
           os.path.join(ROOT, "tools", "train.py"), "--env-config", str(env_yaml), "--algo-config", str(algo_yaml),
           "--num-envs", "256", "--out", str(out), "--eval-envs", "32"]
    proc = subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, start_new_session=True)
    try:
        stdout, stderr = proc.communicate(timeout=900)
    finally:
        if proc.poll() is None:
            os.killpg(proc.pid, signal.SIGKILL)                        # torchrun and its ranks share the session
            proc.communicate()
    assert proc.returncode == 0, stdout + stderr
    assert stdout.count("power limit") == 1 and "2 ranks" in stdout
    assert stdout.count("iter     1") == 1 and stdout.count("iter     2") == 1
    assert [ln["iteration"] for ln in _lines(out)] == [1, 2] and all(ln["ranks"] == 2 for ln in _lines(out))
    for f in ("checkpoint_final.pt", "checkpoint_final.rank0.pt", "checkpoint_final.rank1.pt"):
        assert (out / f).exists(), f
