"""Device GAE / value targets and advantage standardisation (csrc/gae.cu) on torch tensors.

Replaces the RLlib learner-connector step the reference configures with ``use_gae`` / ``lam`` /
``gamma`` (reference: src/algorithms/ippo.py:145-160, config_files/algorithms/ippo.yaml:18-20).
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch
import torch.distributed as dist

from .. import _capi


def _stream(t: torch.Tensor) -> int:
    return torch.cuda.current_stream(t.device).cuda_stream


def compute_gae(rewards: torch.Tensor, values: torch.Tensor, gamma: float, lam: float,
                cut: Optional[torch.Tensor] = None, cut_values: Optional[torch.Tensor] = None,
                adv_out: Optional[torch.Tensor] = None, targets_out: Optional[torch.Tensor] = None
                ) -> Tuple[torch.Tensor, torch.Tensor]:
    """rewards [T, ...], values [T+1, ...] (last row bootstraps), both float32 CUDA and time-major.
    cut: uint8 [T] on the device, non-zero where an episode ended after step t; cut_values [T, ...]
    holds V(final observation) for those steps (omit for termination semantics).
    Returns (advantages, value_targets) shaped like rewards."""
    if not rewards.is_cuda:
        raise RuntimeError("compute_gae runs on CUDA tensors only (no CPU implementation)")
    T = rewards.shape[0]
    if values.shape[0] != T + 1 or values.shape[1:] != rewards.shape[1:]:
        raise ValueError(f"values must have shape {(T + 1, *rewards.shape[1:])}, got {tuple(values.shape)}")
    if rewards.dtype != torch.float32 or values.dtype != torch.float32:
        raise ValueError("rewards and values must be float32")
    rewards, values = rewards.contiguous(), values.contiguous()
    N = rewards[0].numel()
    adv = torch.empty_like(rewards) if adv_out is None else adv_out
    tgt = torch.empty_like(rewards) if targets_out is None else targets_out
    if cut is not None:
        if cut.dtype != torch.uint8 or cut.shape != (T,) or cut.device != rewards.device:
            raise ValueError("cut must be a uint8 [T] tensor on the same device")
        if cut_values is not None:
            if cut_values.shape != rewards.shape or cut_values.dtype != torch.float32:
                raise ValueError("cut_values must be float32 with the shape of rewards")
            cut_values = cut_values.contiguous()
    elif cut_values is not None:
        raise ValueError("cut_values needs cut")
    _capi.check(_capi.lib().marlsc_gae(
        rewards.data_ptr(), values.data_ptr(), None if cut is None else cut.data_ptr(),
        None if cut_values is None else cut_values.data_ptr(), T, N, float(gamma), float(lam),
        adv.data_ptr(), tgt.data_ptr(), _stream(rewards)))
    return adv, tgt


_ws = {}


def _spans_ranks(group) -> bool:
    return group is not None and dist.get_world_size(group) > 1


def standardize_(x: torch.Tensor, group=None) -> torch.Tensor:
    """In place (x - mean) / max(1e-4, std) over all elements of a float32 CUDA tensor. With a process ``group`` of more
    than one rank the moments are those of every rank's ``x`` together: K3's moments kernel, one all-reduce of its three
    float64 sums (sum, sum of squares, count), then K3's apply kernel."""
    if not x.is_cuda or x.dtype != torch.float32 or not x.is_contiguous():
        raise ValueError("standardize_ needs a contiguous float32 CUDA tensor")
    L = _capi.lib()
    ws = _ws.get(x.device)
    if ws is None:
        ws = _ws[x.device] = torch.zeros(max(16, int(L.marlsc_standardize_workspace_bytes())), dtype=torch.uint8, device=x.device)
    if not _spans_ranks(group):
        _capi.check(L.marlsc_standardize(x.data_ptr(), x.numel(), ws.data_ptr(), _stream(x)))
        return x
    _capi.check(L.marlsc_standardize_moments(x.data_ptr(), x.numel(), ws.data_ptr(), _stream(x)))
    dist.all_reduce(ws[:24].view(torch.float64), op=dist.ReduceOp.SUM, group=group)
    _capi.check(L.marlsc_standardize_apply(x.data_ptr(), x.numel(), ws.data_ptr(), _stream(x)))
    return x


def standardize_columns_(x: torch.Tensor, n_columns: int, group=None) -> torch.Tensor:
    """In place ``(x - mean_c) / max(1e-4, std_c)`` per last-axis column c (one column per independent policy:
    RLlib standardises the advantages of every module's batch on their own). With a process ``group`` of more than one
    rank the per-column float64 sums, sums of squares and counts are all-reduced first, so every column is standardised
    over all ranks' values."""
    if x.shape[-1] != n_columns:
        raise ValueError("the last axis must be the policy axis")
    flat = x.view(-1, n_columns)
    if not _spans_ranks(group):
        mean = flat.mean(0)
        std = flat.std(0, unbiased=False).clamp_min(1e-4)
        flat.sub_(mean).div_(std)
        return x
    x64 = flat.to(torch.float64)
    m = torch.cat([x64.sum(0), (x64 * x64).sum(0), x64.new_full((n_columns,), float(flat.shape[0]))])
    dist.all_reduce(m, op=dist.ReduceOp.SUM, group=group)
    s, q, n = m.view(3, n_columns)
    mean = s / n
    std = torch.sqrt(torch.clamp(q / n - mean * mean, min=0.0)).clamp_min(1e-4)
    flat.sub_(mean.to(flat.dtype)).div_(std.to(flat.dtype))
    return x
