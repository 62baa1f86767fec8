"""On-device rollout collection: policy forward (PyTorch) -> fused env step (CUDA) -> buffer, then the
GAE scan kernel. Replaces RLlib's EnvRunner / MultiAgentEpisode / learner-connector chain that the
reference configures (reference: src/algorithms/ippo.py:145-214, mappo.py:142-209; SURVEY.md A17-A18).

Buffers are time-major and preallocated; the env writes observations and rewards straight into them.
Environments never interact, so a multi-GPU run shards them by rank and steps them with no communication. With a
``process_group`` the collector standardises the advantages over every rank's batch and merges the ranks' observation
filter moments after each collection.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Callable, Optional, Union

import torch
import torch.distributed as dist

from ..envs import BatchedInventoryEnv, DeviceOrders
from .gae import compute_gae, standardize_, standardize_columns_
from .policy import ActorCritic, CentralizedActorCritic


@dataclass
class Rollout:
    """Shapes for an ``ActorCritic``; with a ``CentralizedActorCritic`` the agent axis goes: actions and mean_old are
    [T, E, W*S], logp / rewards (summed over the warehouses) / values / advantages / targets are [T(+1), E] and
    log_std_old is [1, W*S]."""
    obs: torch.Tensor        # [T+1, E, W, D]
    actions: torch.Tensor    # [T, E, W, S] RAW (unclipped) samples - what ``logp`` refers to; the env saw clamp(-1, 1)
    logp: torch.Tensor       # [T, E, W]
    rewards: torch.Tensor    # [T, E, W]
    values: torch.Tensor     # [T+1, E, W]
    advantages: torch.Tensor  # [T, E, W]
    targets: torch.Tensor    # [T, E, W]
    cut: torch.Tensor        # [T] uint8, 1 where an episode ended after step t
    mean_old: Optional[torch.Tensor] = None      # [T, E, W, S] behaviour-policy action means (KL term only)
    log_std_old: Optional[torch.Tensor] = None   # [n_policies, S] behaviour-policy log-std, floored (KL term only)


def shard_envs(total_envs: int, rank: int, world_size: int) -> range:
    """Contiguous env range owned by ``rank`` (SURVEY.md section 8e)."""
    base, extra = divmod(total_envs, world_size)
    start = rank * base + min(rank, extra)
    return range(start, start + base + (1 if rank < extra else 0))


class RolloutCollector:
    """Collects T steps of E environments under an ``ActorCritic`` (one sample per agent) or a
    ``CentralizedActorCritic`` (CPPO: one sample per environment - the joint action, the summed reward, one value)."""

    def __init__(self, env: BatchedInventoryEnv, policy: Union[ActorCritic, CentralizedActorCritic], horizon: int,
                 gamma: float = 0.99, lam: float = 0.95, demand_fn: Optional[Callable[[int], DeviceOrders]] = None,
                 standardize_advantages: bool = True, seed: int = 0, keep_dist_inputs: bool = False,
                 obs_filter=None, process_group=None):
        self.env, self.policy, self.T = env, policy, int(horizon)
        self.gamma, self.lam = float(gamma), float(lam)
        self.demand_fn = demand_fn            # step index -> DeviceOrders; None = env host samplers
        self.standardize = standardize_advantages
        # running MeanStdFilter (obs_normalization == "meanstd"), applied in place: per local column shared by the agents,
        # or, for the centralised policy, per global column over the [E, W*D] view
        self.obs_filter = obs_filter
        # data parallel: advantage moments all-reduced, filter buffers gathered and merged in rank order after collect()
        self.group = process_group if process_group is not None and dist.get_world_size(process_group) > 1 else None
        if self.group is not None and obs_filter is not None:
            obs_filter.track_buffer()
        E, W, S, D, dev = env.num_envs, env.n_warehouses, env.n_skus, env.obs_dim, env.device
        T = self.T
        central = isinstance(policy, CentralizedActorCritic)
        if central and obs_filter is not None and obs_filter.mean.numel() != W * D:
            raise ValueError(f"the centralised policy's observation filter normalises the global state: MeanStdFilter({W * D})")
        self._flt_shape = (E, W * D) if central else (E, W, D)
        agent = () if central else (W,)       # per-agent axis of the per-sample buffers
        act = (W * S,) if central else (W, S)
        self.obs = torch.empty((T + 1, E, W, D), device=dev)
        self.actions = torch.empty((T, E, *act), device=dev)
        self.mean_old = torch.empty((T, E, *act), device=dev) if keep_dist_inputs else None   # use_kl_loss needs it
        self.logp = torch.empty((T, E, *agent), device=dev)
        self.rewards = torch.empty((T, E, *agent), device=dev)
        # the step writes [E, W] rewards; the centralised policy's reward is their sum (CentralizedEnvWrapper.step)
        self._step_rewards = torch.empty((E, W), device=dev) if central else None
        self.values = torch.empty((T + 1, E, *agent), device=dev)
        self.cut_values = torch.zeros((T, E, *agent), device=dev)
        self.adv = torch.empty((T, E, *agent), device=dev)
        self.targets = torch.empty((T, E, *agent), device=dev)
        self.gen = torch.Generator(device=dev)
        self.gen.manual_seed(seed)
        self._need_reset = True
        self.total_steps = 0

    @torch.no_grad()
    def collect(self) -> Rollout:
        env, pol, T = self.env, self.policy, self.T
        cut_host = [0] * T
        flt = self.obs_filter
        if self._need_reset:
            env.reset(obs_out=self.obs[0])
            if flt is not None:
                flt(self.obs[0].view(self._flt_shape))
            self._need_reset = False
        else:
            self.obs[0].copy_(self.obs[T])
        any_cut = False
        for t in range(T):
            # RLlib keeps the raw Gaussian sample (and its log-prob) in the batch and clips only the copy that goes to
            # the env (clip_actions=True, reference ippo.py:183-188); the learner's ratio is then exactly 1 at the
            # behaviour parameters
            act, raw, logp, val, mean = pol.act(self.obs[t], generator=self.gen, return_raw=True)
            self.actions[t], self.logp[t], self.values[t] = raw, logp, val
            if self.mean_old is not None:
                self.mean_old[t] = mean
            orders = self.demand_fn(self.total_steps) if self.demand_fn is not None else None
            rew = self.rewards[t] if self._step_rewards is None else self._step_rewards
            _, _, truncated = env.step(act.contiguous(), orders=orders, obs_out=self.obs[t + 1], rewards_out=rew)
            if self._step_rewards is not None:
                torch.sum(rew, dim=1, out=self.rewards[t])
            if flt is not None:
                flt(self.obs[t + 1].view(self._flt_shape))
            self.total_steps += 1
            if truncated:
                # the final observation bootstraps the value target (RLlib appends it to the episode); the
                # next episode then starts from a fresh reset
                cut_host[t] = 1
                any_cut = True
                self.cut_values[t] = pol.value(self.obs[t + 1])
                env.reset(obs_out=self.obs[t + 1])
                if flt is not None:
                    flt(self.obs[t + 1].view(self._flt_shape))
        self.values[T] = pol.value(self.obs[T])
        cut = torch.tensor(cut_host, dtype=torch.uint8, device=env.device)
        compute_gae(self.rewards, self.values, self.gamma, self.lam, cut if any_cut else None,
                    self.cut_values if any_cut else None, adv_out=self.adv, targets_out=self.targets)
        if self.standardize:
            # RLlib standardises the advantages per module batch: over everything with a shared policy, per
            # warehouse column with independent policies
            if pol.n_policies == 1:
                standardize_(self.adv, self.group)
            else:
                standardize_columns_(self.adv, pol.n_policies, self.group)
        if self.group is not None and flt is not None:
            flt.sync(self.group)
        ls_old = pol.clamped_log_std().detach().reshape(pol.n_policies, -1).clone() if self.mean_old is not None else None
        return Rollout(self.obs, self.actions, self.logp, self.rewards, self.values, self.adv, self.targets, cut,
                       self.mean_old, ls_old)
