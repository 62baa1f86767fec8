"""Policy evaluation on the device: whole episodes of E environments with the per-episode metrics the step kernels
accumulate (``BatchedInventoryEnv(..., episode_metrics=True)``) - cost by component, units ordered / shipped / demanded /
lost and the unit fill rate, the numbers the reference's baseline runs and seed evaluations report from
``collect_step_info`` (src/environment/envs/multi_env.py:330-362). Nothing is copied to the host per step.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Callable, Dict, Optional, Union

import numpy as np
import torch
import torch.distributed as dist

from ..envs import BatchedInventoryEnv
from ..envs.batched_env import COST_METRICS, METRICS_PER_ENV, METRICS_PER_ROW, fill_rate
from .policy import ActorCritic, CentralizedActorCritic


@dataclass
class EpisodeMetrics:
    """Per-episode results, float64: ``values[name]`` is [num_episodes, E, W] for the per-warehouse metrics
    (``holding_cost``, ``penalty_cost``, ``outbound_cost``, ``inbound_cost``, ``total_cost``, ``ordered_units``,
    ``shipped_units``, ``episode_return``) and [num_episodes, E] for ``demand_units``, ``lost_units`` and ``fill_rate``."""
    values: Dict[str, torch.Tensor]

    @staticmethod
    def from_accumulators(per_episode: Dict[str, torch.Tensor]) -> "EpisodeMetrics":
        """From the stacked accumulators [num_episodes, E(, W)] of ``METRICS_PER_ROW + METRICS_PER_ENV``: adds
        ``total_cost`` and ``fill_rate``."""
        v = dict(per_episode)
        v["total_cost"] = sum(v[k] for k in COST_METRICS)
        v["fill_rate"] = fill_rate(v["demand_units"], v["lost_units"])
        return EpisodeMetrics(v)

    def __getitem__(self, name: str) -> torch.Tensor:
        return self.values[name]

    def per_env(self, name: str) -> torch.Tensor:
        """[num_episodes, E]: a per-warehouse metric summed over the warehouses; the fill rate of the environment's
        summed units."""
        x = self.values[name]
        return x if x.dim() == 2 else x.sum(-1)

    def gather(self, group=None) -> "EpisodeMetrics":
        """Every rank's metrics of ``group`` (default: the default process group) joined along the environment axis in rank
        order, on every rank; the ranks may hold different numbers of environments. One all-reduce."""
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        names = list(self.values)
        first = self.values[names[0]]
        E = first.shape[1]
        dev = first.device
        sizes = torch.zeros(world, dtype=torch.float64, device=dev)
        sizes[rank] = E
        dist.all_reduce(sizes, op=dist.ReduceOp.SUM, group=group)
        sizes = [int(n) for n in sizes.tolist()]
        off = sum(sizes[:rank])
        # [E, ...] per metric -> one [E, F] row block per rank; the other ranks' rows stay 0, so the sum is a gather
        cols = [self.values[k].movedim(1, 0).reshape(E, -1).to(torch.float64) for k in names]
        rows = torch.zeros((sum(sizes), sum(c.shape[1] for c in cols)), dtype=torch.float64, device=dev)
        rows[off:off + E] = torch.cat(cols, dim=1)
        dist.all_reduce(rows, op=dist.ReduceOp.SUM, group=group)
        out, c0 = {}, 0
        for k, c in zip(names, cols):
            v = self.values[k]
            out[k] = rows[:, c0:c0 + c.shape[1]].reshape(sum(sizes), v.shape[0], *v.shape[2:]).movedim(0, 1).to(v.dtype).contiguous()
            c0 += c.shape[1]
        return EpisodeMetrics(out)

    def summary(self) -> Dict[str, Dict[str, float]]:
        """Mean and (population) standard deviation of every metric over all environments of all episodes, one sample per
        (episode, environment) - per-warehouse metrics summed over the warehouses first."""
        out = {}
        for name in self.values:
            x = self.per_env(name).reshape(-1).to(torch.float64)
            out[name] = dict(mean=float(x.mean()), std=float(x.std(unbiased=False)) if x.numel() > 1 else 0.0)
        return out


Actor = Union[ActorCritic, CentralizedActorCritic, torch.Tensor, np.ndarray, Callable[[torch.Tensor], torch.Tensor]]


def _resolve_actor(env: BatchedInventoryEnv, actor: Actor):
    """("actor_critic", module) | ("base_stock", level tensor [W,S] or [E,W,S]) | ("callable", fn); ValueError otherwise."""
    E, W, S = env.num_envs, env.n_warehouses, env.n_skus
    if isinstance(actor, ActorCritic):
        if actor.action_dim != S or actor.local_obs_dim != env.obs_dim:
            raise ValueError(f"the ActorCritic maps {actor.local_obs_dim}-wide observations to {actor.action_dim} actions; the "
                             f"environment has {env.obs_dim} and {S}")
        return "actor_critic", actor
    if isinstance(actor, CentralizedActorCritic):
        if (actor.n_warehouses, actor.action_dim, actor.local_obs_dim) != (W, S, env.obs_dim):
            raise ValueError(f"the CentralizedActorCritic is built for {actor.n_warehouses} warehouses x {actor.action_dim} SKUs "
                             f"with {actor.local_obs_dim}-wide local observations; the environment has {W} x {S} and {env.obs_dim}")
        return "centralized", actor
    if isinstance(actor, (torch.Tensor, np.ndarray)):
        if tuple(actor.shape) not in ((W, S), (E, W, S)):
            raise ValueError(f"a base-stock level must have shape {(W, S)} or {(E, W, S)}, got {tuple(actor.shape)}")
        if env.env_config.action_space.type != "direct":
            raise ValueError("the base-stock policy assumes the direct action space")
        return "base_stock", torch.as_tensor(actor, dtype=torch.float32, device=env.device).contiguous()
    if callable(actor):
        return "callable", actor
    raise ValueError("actor must be an ActorCritic, a CentralizedActorCritic, a base-stock level [W,S] / [E,W,S] or a callable obs -> actions")


@torch.no_grad()
def evaluate(env: BatchedInventoryEnv, actor: Actor, num_episodes: int, orders_fn: Optional[Callable[[int], object]] = None,
             obs_filter=None) -> EpisodeMetrics:
    """Run ``num_episodes`` whole episodes of every environment under ``actor`` and return their metrics.

    ``actor`` is an ``ActorCritic`` (its mean action clipped to [-1, 1], the reference's ``explore=False`` path,
    src/algorithms/base.py:98-265, on the observations passed through ``obs_filter`` when given - a copy, the env's
    buffer stays raw), a ``CentralizedActorCritic`` (the same with the joint mean action [E, W*S] viewed as [E, W, S]; its
    filter normalises the [E, W*D] global state), a base-stock level [W,S] or [E,W,S] (evaluated inside the step on the compact layout, by the
    policy kernel otherwise), or a callable ``obs [E,W,obs_dim] -> actions [E,W,S]``. Demand comes from
    ``orders_fn(t)``, else from whatever the environment is set up with (device sampler, empirical frame, host samplers).
    Each episode starts with ``env.reset()``."""
    if int(num_episodes) < 1:
        raise ValueError("num_episodes must be positive")
    if not env.has_episode_metrics:
        raise ValueError("evaluate() needs an environment constructed with episode_metrics=True")
    kind, pol = _resolve_actor(env, actor)
    in_step = kind == "base_stock" and env.layout == "compact"
    act = torch.empty((env.num_envs, env.n_warehouses, env.n_skus), device=env.device) if kind == "base_stock" and not in_step else None
    episodes = {k: [] for k in METRICS_PER_ROW + METRICS_PER_ENV}
    for _ in range(int(num_episodes)):
        obs = env.reset()
        done = False
        while not done:
            orders = orders_fn(env.timestep) if orders_fn is not None else None
            if in_step:
                obs, _, done = env.step(None, orders=orders, base_stock_level=pol)
                continue
            if kind == "base_stock":
                a = env.base_stock_actions(pol, out=act)
            elif kind == "actor_critic":
                x = obs if obs_filter is None else obs_filter(obs.clone())
                a = pol.action_mean(x).clamp(-1.0, 1.0)
            elif kind == "centralized":
                # the joint mean action [E, W*S], warehouse-major; a CPPO filter normalises the [E, W*D] global state
                x = obs if obs_filter is None else obs_filter(obs.clone().view(obs.shape[0], -1)).view(obs.shape)
                a = pol.action_mean(x).clamp(-1.0, 1.0).view(obs.shape[0], env.n_warehouses, env.n_skus)
            else:
                a = pol(obs)
            obs, _, done = env.step(a.contiguous(), orders=orders)
        m = env.episode_metrics()
        for k in episodes:
            episodes[k].append(m[k].clone())
    return EpisodeMetrics.from_accumulators({k: torch.stack(v) for k, v in episodes.items()})
