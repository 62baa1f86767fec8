"""Running mean / std observation filter for ``obs_normalization: "meanstd"``.

In the reference this mode leaves the env's observations untouched and adds RLlib's ``MeanStdFilter`` connector
in front of the module (reference: src/algorithms/ippo.py:173-176); the env itself emits raw features
(multi_env.py:700-702 only handles the fixed-statistics modes). ``MeanStdFilter`` keeps running per-feature moments
over everything sampled so far and returns ``(x - mean) / (std + 1e-8)``. This is the batched device counterpart: one
parallel-Welford merge per call (Chan et al.), statistics per observation column shared by all agents that share a
policy.
"""
from __future__ import annotations

from typing import Sequence, Tuple

import torch
import torch.distributed as dist

Moments = Tuple[torch.Tensor, torch.Tensor, torch.Tensor]      # (count, mean, M2): float64 [], [D], [D]


def chan_merge(a: Moments, b) -> Moments:
    """The moments of the union of two sample sets (Chan et al.'s pairwise update); ``b``'s count may be a number. The two
    sets must not both be empty."""
    ca, ma, qa = a
    cb, mb, qb = b
    tot = ca + cb
    delta = mb - ma
    return tot, ma + delta * (cb / tot), qa + (qb + delta * delta * (ca * cb / tot))


def merge_buffers(base: Moments, buffers: Sequence[Moments]) -> Moments:
    """``base`` merged with every buffer in turn, in the order given (rank order in a data-parallel run, so that every
    rank computes the same bits)."""
    out = base
    for b in buffers:
        out = chan_merge(out, b)
    return out


class MeanStdFilter:
    def __init__(self, obs_dim: int, device, eps: float = 1e-8, update: bool = True):
        self.count = torch.zeros((), dtype=torch.float64, device=device)
        self.mean = torch.zeros(obs_dim, dtype=torch.float64, device=device)
        self.m2 = torch.zeros(obs_dim, dtype=torch.float64, device=device)
        self.eps, self.update = eps, update
        # data-parallel runs (track_buffer): the moments at the last sync, and those added locally since
        self.synced: Moments = None
        self.buffer: Moments = None

    @torch.no_grad()
    def __call__(self, obs: torch.Tensor) -> torch.Tensor:
        """Update the running moments with ``obs [..., obs_dim]`` (when ``update``) and normalise it in place."""
        flat = obs.reshape(-1, obs.shape[-1])
        if self.update:
            n = float(flat.shape[0])
            bm = flat.mean(0, dtype=torch.float64)
            bm2 = ((flat.to(torch.float64) - bm) ** 2).sum(0)
            self.count, self.mean, self.m2 = chan_merge((self.count, self.mean, self.m2), (n, bm, bm2))
            if self.buffer is not None:
                self.buffer = chan_merge(self.buffer, (n, bm, bm2))
        std = torch.sqrt(self.m2 / torch.clamp(self.count - 1.0, min=1.0))
        flat.sub_(self.mean.to(obs.dtype)).div_((std + self.eps).to(obs.dtype))
        return obs

    def state_dict(self):
        return dict(count=self.count.clone(), mean=self.mean.clone(), m2=self.m2.clone())

    def load_state_dict(self, sd):
        self.count, self.mean, self.m2 = sd["count"].clone(), sd["mean"].clone(), sd["m2"].clone()
        if self.buffer is not None:
            self.track_buffer()

    # ------------------------------------------------------------------ data-parallel runs
    def track_buffer(self) -> None:
        """From now on keep the moments this process adds apart (``buffer``) from those of the last sync (``synced``), the
        way RLlib's ``MeanStdFilter`` keeps a buffer per env runner."""
        self.synced = (self.count.clone(), self.mean.clone(), self.m2.clone())
        self.buffer = (torch.zeros_like(self.count), torch.zeros_like(self.mean), torch.zeros_like(self.m2))

    @torch.no_grad()
    def sync(self, group=None) -> None:
        """Gather every rank's buffer ``(count, mean, M2)`` and merge them, in rank order, into the moments of the last
        sync; every rank then holds the same filter and starts an empty buffer. Needs ``track_buffer()``."""
        if self.buffer is None:
            raise RuntimeError("MeanStdFilter.sync needs track_buffer() first")
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        D = self.mean.numel()
        rows = torch.zeros((world, 2 * D + 1), dtype=torch.float64, device=self.mean.device)
        rows[rank, 0] = self.buffer[0]
        rows[rank, 1:D + 1] = self.buffer[1]
        rows[rank, D + 1:] = self.buffer[2]
        dist.all_reduce(rows, op=dist.ReduceOp.SUM, group=group)      # an all-gather: each row has one non-zero owner
        bufs = [(r[0], r[1:D + 1], r[D + 1:]) for r in rows]
        self.count, self.mean, self.m2 = merge_buffers(self.synced, bufs)
        self.track_buffer()
