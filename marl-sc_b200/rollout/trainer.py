"""Training from an algorithm config: IPPO, MAPPO and CPPO on the device, with the config's learning-rate schedule, periodic
evaluation, checkpoints and resume (the reference's ``run_experiment.py --mode single``, ``ExperimentRunner.run``,
runner.py:112-214), on one GPU or data-parallel on several.

One iteration is: set the learning rate, collect ``horizon`` steps of ``num_envs`` environments (``RolloutCollector``: K1 /
K4 / K7 / K2 / K3), one ``PPOLearner.update`` (``num_epochs`` x ``num_minibatches`` K6 steps), every ``eval_interval``
iterations ``evaluate()`` on a separate environment batch, and one JSON line in ``training_metrics.jsonl``. A checkpoint
holds everything the next iteration depends on - model, optimiser, filter, generators, the collector's carried observation
and both environments' ``state_dict()`` - so a resumed run continues the same trajectory.

Under a default process group of more than one rank (``torchrun``), every rank holds ``num_envs / world`` of the training
environments and its shard of the evaluation environments, and the ranks agree on everything the single-GPU algorithm computes
over the whole batch: the gradients (``GradBuckets``), the advantage standardisation and the ``meanstd`` filter
(``RolloutCollector(process_group=...)``), the learner statistics and KL coefficient (``PPOLearner.update``), the evaluation
metrics (``EpisodeMetrics.gather``) and so the best checkpoint. A checkpoint is then a main file written by rank 0 with the
shared state plus one ``checkpoint_<tag>.rank<r>.pt`` shard per rank with that rank's environments and generators."""
from __future__ import annotations

import json
import os
import time
import warnings
from typing import Any, Callable, Dict, Optional

import numpy as np
import torch
import torch.distributed as dist

from ..config.schema import CPPOConfig, EnvironmentConfig
from ..seeds import SeedManager
from .collector import RolloutCollector, shard_envs
from .evaluate import evaluate
from .obs_filter import MeanStdFilter
from .obs_stats import compute_obs_statistics
from .policy import ActorCritic, CentralizedActorCritic, env_meta_from_algorithm_config
from .ppo import PPOLearner, lr_schedule

METRICS_FILE = "training_metrics.jsonl"
CHECKPOINT_VERSION = 1
# what a rank's checkpoint shard holds in a data-parallel run; the main file holds the rest, the same on every rank
RANK_KEYS = ("learner_gen", "collector", "env", "eval_env")


def unsupported_algorithm_fields(algo_config) -> list:
    """The fields of an algorithm config that the trainer's models cannot honour (they would otherwise be ignored)."""
    sp = algo_config.algorithm_specific
    net = sp.networks
    bad = []
    if net.shared_layers is not None:
        bad.append("networks.shared_layers")
    if net.use_mu_sigma_head:
        bad.append("networks.use_mu_sigma_head")
    for head in ("actor", "critic"):
        c = getattr(net, head).config
        for f in ("output_activation", "output_activation_mu", "output_activation_sigma"):
            if getattr(c, f) is not None:
                bad.append(f"networks.{head}.config.{f}")
    if net.critic.config.activation != net.actor.config.activation:
        bad.append("networks.critic.config.activation")
    if getattr(sp, "actor_obs_type", "local") == "global":
        bad.append("actor_obs_type")
    if sp.warmstart_weights_path is not None:
        bad.append("warmstart_weights_path")
    if sp.use_gae is False:
        bad.append("use_gae")
    return bad


def _rank_world() -> tuple:
    """(rank, world size) of the default process group; (0, 1) without one."""
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def _rank_seed(seed: int, rank: int) -> int:
    """The root seed of a rank's streams in a data-parallel run: distinct per rank, a function of ``(seed, rank)`` alone."""
    return int(np.random.SeedSequence([seed, rank]).generate_state(1, dtype=np.uint32)[0])


def shard_path(path: str, rank: int) -> str:
    """``checkpoint_<tag>.rank<r>.pt`` next to the main file ``checkpoint_<tag>.pt``."""
    root, ext = os.path.splitext(path)
    return f"{root}.rank{rank}{ext}"


def _check(env_config: EnvironmentConfig, algo_config, num_envs: int, horizon: Optional[int], num_eval_envs: int = 1,
           world: int = 1) -> int:
    """The horizon of a run, after refusing what the trainer cannot honour; touches no CUDA state."""
    bad = unsupported_algorithm_fields(algo_config)
    if bad:
        raise ValueError(f"the trainer cannot honour {bad[0]} (unsupported: {', '.join(bad)})")
    ds = env_config.components.demand_sampler.type
    if ds not in ("poisson", "empirical"):
        raise ValueError(f"the trainer draws demand on the device (poisson) or from the empirical frame, not from a '{ds}' sampler")
    if int(num_envs) < 1:
        raise ValueError("num_envs must be positive")
    if world > 1:
        # equal shards: the mean of the ranks' minibatch gradients is then the gradient of the global minibatch
        if int(num_envs) % world != 0:
            raise ValueError(f"num_envs ({num_envs}) must be a multiple of the world size ({world})")
        if int(num_eval_envs) < world:
            raise ValueError(f"num_eval_envs ({num_eval_envs}) must be at least the world size ({world})")
    if horizon is None:
        bs = algo_config.shared.batch_size
        if bs % int(num_envs) != 0:
            raise ValueError(f"batch_size ({bs}) is not a multiple of num_envs ({num_envs}): pass horizon")
        horizon = bs // int(num_envs)
    if int(horizon) < 1:
        raise ValueError("horizon must be a positive number of steps")
    return int(horizon)


class Trainer:
    """``Trainer(env_config, algo_config, num_envs, out_dir).run()`` trains for ``shared.num_iterations`` iterations of
    ``num_envs x horizon`` env steps each (``horizon`` defaults to ``batch_size / num_envs``) and writes
    ``out_dir/training_metrics.jsonl``, ``checkpoint_<iter>.pt`` every ``checkpoint_freq`` iterations,
    ``checkpoint_best.pt`` (highest mean evaluation ``episode_return``, summed over the warehouses) and
    ``checkpoint_final.pt``. ``Trainer.resume(path)`` continues from a checkpoint. Under a default process group of several
    ranks ``num_envs`` and ``num_eval_envs`` are global: ``num_envs`` must be a multiple of the world size, and every rank
    needs at least one evaluation environment."""

    def __init__(self, env_config: EnvironmentConfig, algo_config, num_envs: int, out_dir: str, seed: int = 0,
                 device=None, horizon: Optional[int] = None, num_eval_envs: Optional[int] = None,
                 env_meta: Optional[Dict[str, Any]] = None, _obs_stats=None):
        self.rank, self.world = _rank_world()
        self.num_eval_envs = int(num_eval_envs) if num_eval_envs is not None else min(int(num_envs), 1024)
        self.horizon = _check(env_config, algo_config, num_envs, horizon, self.num_eval_envs, self.world)
        self.env_config, self.algo_config = env_config, algo_config
        self.num_envs, self.seed = int(num_envs), int(seed)
        self.group = dist.group.WORLD if self.world > 1 else None
        self.out_dir = str(out_dir)
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        sh, sp = algo_config.shared, algo_config.algorithm_specific
        self.steps_per_iteration = self.num_envs * self.horizon
        self.schedule = lr_schedule(sh.learning_rate)
        self._user_meta = {k: v for k, v in (env_meta or {}).items() if k != "preprocessed_data"}
        meta = dict(env_meta or {})
        meta.update(env_meta_from_algorithm_config(algo_config))
        norm = meta["obs_normalization"]
        # environments, demand, leads, collector and learner draw per rank; the initial weights and the fixed observation
        # statistics depend on the seed alone
        seeds = SeedManager(self.seed if self.world == 1 else _rank_seed(self.seed, self.rank))
        if norm in ("meanstd_custom", "meanstd_grouped"):
            # fixed statistics, once, before the environments are built (runner.py:83-93); computed on rank 0 and broadcast
            self.obs_stats = _obs_stats
            if self.obs_stats is None and self.rank == 0:
                self.obs_stats = compute_obs_statistics(env_config, SeedManager(self.seed), mode=norm, device=self.device)
            if _obs_stats is None and self.world > 1:
                box = [self.obs_stats]
                dist.broadcast_object_list(box, src=0)
                self.obs_stats = box[0]
            meta["obs_stats"] = self.obs_stats
        else:
            self.obs_stats = None
        from ..envs import BatchedInventoryEnv
        n_train = len(shard_envs(self.num_envs, self.rank, self.world))
        n_eval = len(shard_envs(self.num_eval_envs, self.rank, self.world))
        self.env = self._make_env(BatchedInventoryEnv, n_train, seeds.get_seed_int("train"), meta, False)
        self.eval_env = self._make_env(BatchedInventoryEnv, n_eval, seeds.get_seed_int("eval"), meta, True)
        W, S, D = self.env.n_warehouses, self.env.n_skus, self.env.obs_dim
        self.central = isinstance(algo_config, CPPOConfig)
        with torch.random.fork_rng(devices=[]):
            torch.manual_seed(self.seed)                    # the initial weights depend on the seed alone
            model = (CentralizedActorCritic if self.central else ActorCritic).from_algorithm_config(algo_config, D, W, S)
        self.policy = model.to(self.device)
        col_seed, learn_seed = seeds.spawn_child_seeds("train", 2)
        self.filter_dim = W * D if self.central else D
        self.obs_filter = MeanStdFilter(self.filter_dim, self.device) if norm == "meanstd" else None
        self.collector = RolloutCollector(self.env, self.policy, self.horizon, gamma=sp.gamma, lam=sp.lam, seed=col_seed,
                                          keep_dist_inputs=bool(sp.use_kl_loss), obs_filter=self.obs_filter,
                                          process_group=self.group)
        self.learner = PPOLearner.from_algorithm_config(self.policy, algo_config, seed=learn_seed)
        self.iteration = 0
        self.best_return: Optional[float] = None
        os.makedirs(self.out_dir, exist_ok=True)
        self.metrics_path = os.path.join(self.out_dir, METRICS_FILE)
        if self.rank == 0:
            open(self.metrics_path, "w").close()

    def _make_env(self, cls, n: int, seed: int, meta: Dict[str, Any], eval_env: bool):
        with warnings.catch_warnings():
            # "meanstd" leaves the env's observations raw and asks for the running filter, which this trainer applies
            warnings.filterwarnings("ignore", message="obs_normalization='meanstd'")
            env = cls(self.env_config, n, device=self.device, seed=seed, env_meta=meta, host_samplers=False,
                      episode_metrics=eval_env)
        if self.env_config.components.demand_sampler.type == "poisson":
            env.enable_device_demand(seed)
        if env.stochastic_lead:
            env.enable_device_leads(seed + 1)
        return env

    # ------------------------------------------------------------------ training
    def lr_at(self, iteration: int) -> float:
        """Learning rate of update ``iteration`` (0-based): the schedule at the env steps sampled before it."""
        return self.schedule(iteration * self.steps_per_iteration)

    def _sync(self) -> float:
        torch.cuda.synchronize(self.device)
        return time.perf_counter()

    def train_iteration(self) -> Dict[str, Any]:
        """One iteration; returns the line it appends to ``training_metrics.jsonl``."""
        sh = self.algo_config.shared
        lr = self.lr_at(self.iteration)
        self.learner.set_lr(lr)
        t0 = self._sync()
        ro = self.collector.collect()
        reward = ro.rewards.reshape(self.horizon, self.env.num_envs, -1).sum(-1).mean()
        if self.world > 1:
            dist.all_reduce(reward, op=dist.ReduceOp.SUM)
            reward = reward / self.world
        reward = float(reward)
        t1 = self._sync()
        stats = self.learner.update(ro)
        t2 = self._sync()
        self.iteration += 1
        line: Dict[str, Any] = dict(iteration=self.iteration, env_steps=self.iteration * self.steps_per_iteration, lr=lr,
                                    learner=stats, reward_mean=reward, collect_s=t1 - t0, update_s=t2 - t1, eval_s=0.0)
        if self.world > 1:
            line["ranks"] = self.world
        if self.iteration % sh.eval_interval == 0:
            frozen = None
            if self.obs_filter is not None:
                frozen = MeanStdFilter(self.filter_dim, self.device, update=False)
                frozen.load_state_dict(self.obs_filter.state_dict())
            metrics = evaluate(self.eval_env, self.policy, sh.num_eval_episodes, obs_filter=frozen)
            if self.world > 1:
                metrics = metrics.gather(self.group)
            summary = metrics.summary()
            line["eval_s"] = self._sync() - t2
            line["eval"] = summary
        if self.rank == 0:
            with open(self.metrics_path, "a") as f:
                f.write(json.dumps(line) + "\n")
        best = "eval" in line and (self.best_return is None or line["eval"]["episode_return"]["mean"] > self.best_return)
        if best:
            self.best_return = line["eval"]["episode_return"]["mean"]
            self.save(os.path.join(self.out_dir, "checkpoint_best.pt"))
        if self.iteration % sh.checkpoint_freq == 0:
            self.save(os.path.join(self.out_dir, f"checkpoint_{self.iteration}.pt"))
        return line

    def run(self, num_iterations: Optional[int] = None, log: Optional[Callable[[Dict[str, Any]], None]] = None) -> None:
        """Train until ``num_iterations`` (default ``shared.num_iterations``) iterations are done in all, counting those
        before a resume; then write ``checkpoint_final.pt``. ``log`` receives every metrics line."""
        n = self.algo_config.shared.num_iterations if num_iterations is None else int(num_iterations)
        while self.iteration < n:
            line = self.train_iteration()
            if log is not None:
                log(line)
        self.save(os.path.join(self.out_dir, "checkpoint_final.pt"))

    # ------------------------------------------------------------------ checkpoints
    def state_dict(self) -> Dict[str, Any]:
        col = self.collector
        return dict(
            version=CHECKPOINT_VERSION, env_config=self.env_config.model_dump(), algo_config=self.algo_config.model_dump(),
            args=dict(num_envs=self.num_envs, seed=self.seed, horizon=self.horizon, num_eval_envs=self.num_eval_envs),
            env_meta=self._user_meta, obs_stats=self.obs_stats,
            policy=self.policy.state_dict(), optimizer=self.learner.opt.state_dict(),
            obs_filter=None if self.obs_filter is None else self.obs_filter.state_dict(),
            kl_coeff=self.learner.kl_coeff, learner_gen=self.learner.gen.get_state(),
            collector=dict(gen=col.gen.get_state(), obs_T=col.obs[col.T].cpu(), need_reset=col._need_reset,
                           total_steps=col.total_steps),
            env=self.env.state_dict(), eval_env=self.eval_env.state_dict(),
            iteration=self.iteration, env_steps=self.iteration * self.steps_per_iteration, best_return=self.best_return)

    def save(self, path: str) -> None:
        """One file with one process. With several ranks: every rank's shard (``shard_path``), a barrier, then rank 0's main
        file with the shared state and ``world_size``, so that a main file on disk means the checkpoint is complete."""
        sd = self.state_dict()
        if self.world == 1:
            torch.save(sd, path)
            return
        if self.rank == 0 and os.path.exists(path):
            os.remove(path)                       # a rewritten tag (checkpoint_best) is incomplete until its main file returns
        dist.barrier()
        torch.save(dict({k: sd[k] for k in RANK_KEYS}, rank=self.rank, iteration=self.iteration), shard_path(path, self.rank))
        dist.barrier()
        if self.rank == 0:
            torch.save(dict({k: v for k, v in sd.items() if k not in RANK_KEYS}, world_size=self.world), path)

    def _load(self, ck: Dict[str, Any]) -> None:
        self.policy.load_state_dict(ck["policy"])
        self.learner.opt.load_state_dict(ck["optimizer"])
        if self.obs_filter is not None:
            self.obs_filter.load_state_dict({k: v.to(self.device) for k, v in ck["obs_filter"].items()})
        self.learner.kl_coeff = float(ck["kl_coeff"])
        self.learner.gen.set_state(ck["learner_gen"])
        col, c = self.collector, ck["collector"]
        col.gen.set_state(c["gen"])
        col.obs[col.T].copy_(c["obs_T"])
        col._need_reset, col.total_steps = bool(c["need_reset"]), int(c["total_steps"])
        self.env.load_state_dict(ck["env"])
        self.eval_env.load_state_dict(ck["eval_env"])
        self.iteration, self.best_return = int(ck["iteration"]), ck["best_return"]

    @classmethod
    def resume(cls, path: str, out_dir: Optional[str] = None, env_meta: Optional[Dict[str, Any]] = None,
               device=None) -> "Trainer":
        """Rebuild a run from one of its checkpoints and continue it in ``out_dir`` (default: the checkpoint's directory),
        whose metrics file keeps the lines up to the checkpoint's iteration. An empirical run passes its ``env_meta``
        again: the demand frame is not stored. A checkpoint of a data-parallel run resumes under the same world size only,
        every rank from the main file and its own shard."""
        from ..config.loader import algorithm_config_from_dict, environment_config_from_dict
        ck = torch.load(path, map_location="cpu", weights_only=False)
        if ck.get("version") != CHECKPOINT_VERSION:
            raise ValueError(f"{path}: checkpoint version {ck.get('version')!r}, this trainer reads {CHECKPOINT_VERSION}")
        rank, world = _rank_world()
        saved = int(ck.get("world_size", 1))
        if saved != world:
            raise ValueError(f"{path} was written by a run of world size {saved}; this process group has world size {world}")
        if world > 1:
            sp = shard_path(path, rank)
            if not os.path.exists(sp):
                raise ValueError(f"{path}: the checkpoint shard of rank {rank}, {sp}, is missing")
            shard = torch.load(sp, map_location="cpu", weights_only=False)
            if shard.get("rank") != rank or shard.get("iteration") != ck["iteration"]:
                raise ValueError(f"{sp} is not rank {rank}'s shard of iteration {ck['iteration']}")
            ck.update({k: shard[k] for k in RANK_KEYS})
        out = out_dir if out_dir is not None else os.path.dirname(os.path.abspath(path))
        metrics = os.path.join(out, METRICS_FILE)
        kept = []
        if rank == 0 and os.path.exists(metrics):
            with open(metrics) as f:
                kept = [ln for ln in f if ln.strip() and json.loads(ln)["iteration"] <= ck["iteration"]]
        meta = dict(ck["env_meta"]) if env_meta is None else dict(env_meta)
        tr = cls(environment_config_from_dict(ck["env_config"]), algorithm_config_from_dict(ck["algo_config"]), out_dir=out,
                 device=device, env_meta=meta, _obs_stats=ck["obs_stats"], **ck["args"])
        tr._load(ck)
        if rank == 0:
            with open(tr.metrics_path, "w") as f:
                f.writelines(kept)
        return tr
