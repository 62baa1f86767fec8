"""Actor-critic MLPs for the rollout path (plain PyTorch: the dense contractions go to cuBLAS).

Mirrors what the reference's ``ActorCriticRLModule`` does for its shipped IPPO / MAPPO configs
(reference: src/algorithms/models/rlmodules/base.py:150-275 network setup, :192-194 observation routing,
:473-478 free log-std with floor, :514-584 forward): an MLP actor on the local observation producing the
action means, a state-independent ``log_std`` parameter clamped from below, and an MLP critic on the
local observation (IPPO) or on ``[local_i | global]`` (MAPPO, ``critic_obs_type: global``).

``parameter_sharing`` follows src/algorithms/ippo.py:106-115: with sharing every warehouse runs the same
module (and the env prepends a one-hot warehouse id, ippo.py:70); without it every warehouse owns an
independent module - here one set of stacked weights ``[W, in, out]`` evaluated with a batched GEMM, so the
W policies still run as one kernel per layer.

The centralised critic never materialises the W-times duplicated ``[local_i | global]`` vector: its first
layer is split into a local and a global block, ``W1 [local|global]^T = Wl local_i^T + Wg global^T``,
and the global term is computed once per environment.

CPPO (src/algorithms/cppo.py) is :class:`CentralizedActorCritic`: one policy over the global state and the joint action.
"""
from __future__ import annotations

import math
from typing import List, Optional, Sequence, Tuple

import torch
from torch import nn

_ACT = {"relu": nn.ReLU, "tanh": nn.Tanh, "sigmoid": nn.Sigmoid, "elu": nn.ELU, "selu": nn.SELU, "gelu": nn.GELU,
        "swish": nn.SiLU, "mish": nn.Mish, "hard_swish": nn.Hardswish, "hard_sigmoid": nn.Hardsigmoid}


def mlp(in_dim: int, hidden: Sequence[int], out_dim: int, activation: str = "relu",
        output_activation: Optional[str] = None) -> nn.Sequential:
    layers: List[nn.Module] = []
    d = in_dim
    for h in hidden:
        layers += [nn.Linear(d, h), _ACT[activation]()]
        d = h
    layers.append(nn.Linear(d, out_dim))
    if output_activation:
        layers.append(_ACT[output_activation]())
    return nn.Sequential(*layers)


class StackedLinear(nn.Module):
    """P independent ``nn.Linear(in, out)`` layers evaluated together: x ``[..., P, in]`` -> ``[..., P, out]``.
    Initialised like P separate ``nn.Linear`` modules."""

    def __init__(self, n: int, in_dim: int, out_dim: int):
        super().__init__()
        self.n, self.in_features, self.out_features = n, in_dim, out_dim
        self.weight = nn.Parameter(torch.empty(n, in_dim, out_dim))
        self.bias = nn.Parameter(torch.empty(n, 1, out_dim))
        bound = 1.0 / math.sqrt(in_dim)
        for p in range(n):
            w = torch.empty(out_dim, in_dim)
            nn.init.kaiming_uniform_(w, a=math.sqrt(5))
            self.weight.data[p] = w.t()
            nn.init.uniform_(self.bias.data[p], -bound, bound)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        lead = x.shape[:-2]
        h = x.reshape(-1, self.n, self.in_features).transpose(0, 1)          # [P, B, in]
        out = torch.baddbmm(self.bias, h, self.weight).transpose(0, 1)       # [B, P, out]
        return out.reshape(*lead, self.n, self.out_features)


def stacked_mlp(n: int, in_dim: int, hidden: Sequence[int], out_dim: int, activation: str = "relu",
                output_activation: Optional[str] = None) -> nn.Sequential:
    layers: List[nn.Module] = []
    d = in_dim
    for h in hidden:
        layers += [StackedLinear(n, d, h), _ACT[activation]()]
        d = h
    layers.append(StackedLinear(n, d, out_dim))
    if output_activation:
        layers.append(_ACT[output_activation]())
    return nn.Sequential(*layers)


def _fused_mlp1(mods, h: torch.Tensor, max_in: int = 64, max_out: int = 3) -> Optional[torch.Tensor]:
    """K7 (``marlsc_mlp1_forward``, csrc/mlp_forward.cu): a ``Linear -> ReLU|Tanh -> Linear`` head with at most ``max_in``
    inputs and ``max_out`` outputs (by default 64 and 3: the IPPO actor / critic of the small networks; the kernel takes up
    to 128 and 16) in one kernel that keeps the hidden activations in registers. Returns None when the network or the
    tensors do not qualify."""
    if len(mods) != 3 or not isinstance(mods[0], nn.Linear) or not isinstance(mods[2], nn.Linear):
        return None
    act = 0 if isinstance(mods[1], nn.ReLU) else (1 if isinstance(mods[1], nn.Tanh) else -1)
    l1, l2 = mods[0], mods[2]
    if (act < 0 or l1.bias is None or l2.bias is None or l1.in_features > max_in or l2.out_features > max_out
            or h.dtype != torch.float32
            or any(t.dtype != torch.float32 or not t.is_contiguous() for t in (l1.weight, l1.bias, l2.weight, l2.bias))):
        return None
    from .. import _capi
    h = h.contiguous()
    out = torch.empty((h.shape[0], l2.out_features), dtype=torch.float32, device=h.device)
    with torch.cuda.device(h.device):
        stream = torch.cuda.current_stream(h.device).cuda_stream
        _capi.check(_capi.lib().marlsc_mlp1_forward(h.data_ptr(), h.shape[0], l1.in_features, l1.weight.data_ptr(), l1.bias.data_ptr(),
                                                    l1.out_features, l2.weight.data_ptr(), l2.bias.data_ptr(), l2.out_features, act,
                                                    out.data_ptr(), stream))
    return out


def _linear_out_ok(m, h: torch.Tensor, max_out: int = 4) -> bool:
    """Shapes ``marlsc_linear_out_forward`` takes: a multiple of 4 inputs (<= 2048), at most ``max_out`` outputs (by
    default 4; the kernel takes up to 16)."""
    return (isinstance(m, nn.Linear) and m.bias is not None and m.out_features <= max_out and m.in_features % 4 == 0
            and 4 <= m.in_features <= 2048 and h.dtype == torch.float32 and m.weight.dtype == torch.float32
            and m.weight.is_contiguous() and m.bias.is_contiguous())


def _linear_out(h: torch.Tensor, m: nn.Linear, pre_bias: Optional[torch.Tensor] = None) -> torch.Tensor:
    from .. import _capi
    h = h.contiguous()
    out = torch.empty((h.shape[0], m.out_features), dtype=torch.float32, device=h.device)
    with torch.cuda.device(h.device):
        _capi.check(_capi.lib().marlsc_linear_out_forward(h.data_ptr(), h.shape[0], m.in_features,
                                                          pre_bias.data_ptr() if pre_bias is not None else None,
                                                          m.weight.data_ptr(), m.bias.data_ptr(), m.out_features, out.data_ptr(),
                                                          torch.cuda.current_stream(h.device).cuda_stream))
    return out


def _linear_in_ok(m, h: torch.Tensor) -> bool:
    """Shapes ``marlsc_linear_in_forward`` takes: <= 64 inputs, <= 256 units, ceil(units / 32) x padded inputs <= 128."""
    if not isinstance(m, nn.Linear) or m.bias is None or m.in_features > 64 or m.out_features > 256:
        return False
    dp = 16 if m.in_features <= 16 else (32 if m.in_features <= 32 else 64)
    upl = 1 if m.out_features <= 32 else (2 if m.out_features <= 64 else (4 if m.out_features <= 128 else 8))
    return (upl * dp <= 128 and h.dtype == torch.float32 and m.weight.dtype == torch.float32 and m.weight.is_contiguous()
            and m.bias.is_contiguous())


def forward_mlp(seq: nn.Sequential, x: torch.Tensor) -> torch.Tensor:
    """``seq(x)`` for an :func:`mlp`; without autograd on a CUDA tensor a Linear followed by ReLU runs as one
    cuBLASLt GEMM with the bias and the ReLU in its epilogue, so the hidden activations (800 MB per MLP at
    262,144 small environments) cross HBM once instead of three times - and a one-hidden-layer head with few inputs and
    outputs runs in the library's own kernel, where they do not cross HBM at all (``_fused_mlp1``)."""
    if torch.is_grad_enabled() or not x.is_cuda or not hasattr(torch, "_addmm_activation"):
        return seq(x)
    lead = x.shape[:-1]
    h = x.reshape(-1, x.shape[-1])
    mods = list(seq)
    if any(isinstance(m, StackedLinear) for m in mods):
        return seq(x)
    fused = _fused_mlp1(mods, h)
    if fused is not None:
        return fused.reshape(*lead, fused.shape[-1])
    i = 0
    while i < len(mods):
        m = mods[i]
        if i == 0 and _linear_in_ok(m, h):
            # K7a: the input layer (few inputs, up to 256 units) with its activation (csrc/mlp_forward.cu)
            nxt = mods[1] if len(mods) > 1 else None
            act = 0 if isinstance(nxt, nn.ReLU) else (1 if isinstance(nxt, nn.Tanh) else 2)
            from .. import _capi
            h = h.contiguous()
            out = torch.empty((h.shape[0], m.out_features), dtype=torch.float32, device=h.device)
            with torch.cuda.device(h.device):
                _capi.check(_capi.lib().marlsc_linear_in_forward(h.data_ptr(), h.shape[0], m.in_features, m.weight.data_ptr(),
                                                                 m.bias.data_ptr(), m.out_features, act, out.data_ptr(),
                                                                 torch.cuda.current_stream(h.device).cuda_stream))
            h = out
            i += 1 if act == 2 else 2
        elif (isinstance(m, nn.Linear) and m.bias is not None and i + 2 == len(mods) - 1 and isinstance(mods[i + 1], nn.ReLU)
              and _linear_out_ok(mods[i + 2], h) and m.out_features == mods[i + 2].in_features and m.bias.is_contiguous()):
            # last hidden layer + output layer: a plain product, then K7b applies this layer's bias and ReLU on the way in
            # (the library's "fused" bias + ReLU epilogue is a second pass over the activations for fp32)
            h = _linear_out(torch.mm(h, m.weight.t()), mods[i + 2], pre_bias=m.bias)
            i += 3
        elif isinstance(m, nn.Linear) and m.bias is not None and i + 1 < len(mods) and isinstance(mods[i + 1], nn.ReLU):
            h = torch._addmm_activation(m.bias, h, m.weight.t())
            i += 2
        elif isinstance(m, nn.Linear) and i == len(mods) - 1 and _linear_out_ok(m, h):
            h = _linear_out(h, m)                                  # K7b: the output layer in one pass over the activations
            i += 1
        else:
            h = m(h)
            i += 1
    return h.reshape(*lead, h.shape[-1])


class ActorCritic(nn.Module):
    def __init__(self, local_obs_dim: int, n_warehouses: int, action_dim: int, actor_hidden: Sequence[int] = (256,),
                 critic_hidden: Sequence[int] = (256,), activation: str = "relu", critic_obs_type: str = "local",
                 logstd_init: float = 0.0, logstd_floor: float = -2.0, parameter_sharing: bool = True):
        super().__init__()
        self.local_obs_dim, self.n_warehouses, self.action_dim = local_obs_dim, n_warehouses, action_dim
        self.critic_obs_type = critic_obs_type
        self.logstd_floor = float(logstd_floor)
        self.parameter_sharing = bool(parameter_sharing)
        self.n_policies = 1 if self.parameter_sharing else n_warehouses
        crit_in = local_obs_dim * (1 + n_warehouses) if critic_obs_type == "global" else local_obs_dim
        if self.parameter_sharing:
            self.actor = mlp(local_obs_dim, actor_hidden, action_dim, activation)
            self.log_std = nn.Parameter(torch.full((action_dim,), float(logstd_init)))
            self.critic = mlp(crit_in, critic_hidden, 1, activation)
        else:
            W = n_warehouses
            self.actor = stacked_mlp(W, local_obs_dim, actor_hidden, action_dim, activation)
            self.log_std = nn.Parameter(torch.full((W, action_dim), float(logstd_init)))
            self.critic = stacked_mlp(W, crit_in, critic_hidden, 1, activation)

    @classmethod
    def from_algorithm_config(cls, algo_config, local_obs_dim: int, n_warehouses: int, action_dim: int) -> "ActorCritic":
        """``local_obs_dim`` must include the one-hot warehouse id when ``parameter_sharing`` is on: the reference
        turns ``include_warehouse_id`` on with it (ippo.py:70, mappo.py:67) - build the env with
        ``env_meta_from_algorithm_config(algo_config)``. A CPPO config is rejected: its model is
        :class:`CentralizedActorCritic`."""
        from ..config.schema import CPPOConfig
        if isinstance(algo_config, CPPOConfig):
            raise ValueError("a CPPO config describes one centralised policy over the joint action: build it with "
                             "CentralizedActorCritic.from_algorithm_config")
        sp = algo_config.algorithm_specific
        net = sp.networks
        return cls(local_obs_dim, n_warehouses, action_dim, actor_hidden=net.actor.config.hidden_sizes,
                   critic_hidden=net.critic.config.hidden_sizes, activation=net.actor.config.activation,
                   critic_obs_type=getattr(sp, "critic_obs_type", "local"), logstd_init=sp.logstd_init,
                   logstd_floor=sp.logstd_floor, parameter_sharing=bool(getattr(sp, "parameter_sharing", False)))

    # obs: [E, W, D] local observations (flattened over W this is the global state)
    def action_mean(self, obs: torch.Tensor) -> torch.Tensor:
        return forward_mlp(self.actor, obs)

    def clamped_log_std(self) -> torch.Tensor:
        return torch.clamp(self.log_std, min=self.logstd_floor)

    def std(self) -> torch.Tensor:
        return self.clamped_log_std().exp()

    def value(self, obs: torch.Tensor) -> torch.Tensor:
        if self.critic_obs_type != "global":
            return forward_mlp(self.critic, obs).squeeze(-1)
        E, W, D = obs.shape
        first = self.critic[0]
        if self.parameter_sharing and not torch.is_grad_enabled() and obs.is_cuda and _linear_in_ok(first, obs):
            # rollouts: [local | global] rows written once (E x W x (D + W D) floats), then the whole critic through the
            # library's own layer kernels
            xcat = torch.cat([obs, obs.reshape(E, 1, W * D).expand(E, W, W * D)], dim=-1)
            return forward_mlp(self.critic, xcat).squeeze(-1)
        if self.parameter_sharing:
            wl, wg = first.weight[:, :D], first.weight[:, D:]
            h = obs @ wl.t() + (obs.reshape(E, W * D) @ wg.t()).unsqueeze(1) + first.bias
        else:
            wl, wg = first.weight[:, :D], first.weight[:, D:]                      # [W, D, H], [W, W*D, H]
            h = torch.baddbmm(first.bias, obs.transpose(0, 1), wl)                   # [W, E, H]
            h = (h + torch.einsum("eg,wgh->weh", obs.reshape(E, W * D), wg)).transpose(0, 1)
        return forward_mlp(self.critic[1:], h).squeeze(-1)

    def act(self, obs: torch.Tensor, generator: Optional[torch.Generator] = None, deterministic: bool = False,
            return_raw: bool = False):
        """``(clipped action in [-1,1], log-prob of the unclipped sample, value)`` - RLlib samples the diagonal
        Gaussian, stores the RAW sample and its log-prob in the batch and clips only the copy it sends to the env
        (``clip_actions=True``, ippo.py:183-188). ``return_raw=True`` returns
        ``(clipped, raw, logp, value, mean)`` so that a collector can store what the log-prob refers to."""
        mean = self.action_mean(obs)
        std = self.std()
        if deterministic:
            raw = mean
        else:
            raw = mean + std * torch.randn(mean.shape, device=mean.device, dtype=mean.dtype, generator=generator)
        logp = self.log_prob(mean, raw)
        clipped = raw.clamp(-1.0, 1.0)
        if return_raw:
            return clipped, raw, logp, self.value(obs), mean
        return clipped, logp, self.value(obs)

    def log_prob(self, mean: torch.Tensor, raw_action: torch.Tensor) -> torch.Tensor:
        log_std = self.clamped_log_std()
        z = (raw_action - mean) / log_std.exp()
        return (-0.5 * z * z - log_std - 0.9189385332046727).sum(-1)

    def entropy(self) -> torch.Tensor:
        """Sum over policies of the per-policy Gaussian entropy (state independent)."""
        return (self.clamped_log_std() + 1.4189385332046727).sum()


# K7 runs a centralised one-hidden-layer head up to this many inputs (the kernel takes 128)
_CENTRAL_K7_MAX_IN = 128


def _mlp1_smem_bytes(in_dim: int, hidden: int, out_dim: int) -> int:
    """Shared memory K7 needs for a head (csrc/mlp_forward.cu): hidden x (padded inputs + 4) floats for the narrow form
    (<= 64 inputs, <= 3 outputs), hidden x (padded inputs + padded outputs + 4) for the wide one."""
    if in_dim <= 64 and out_dim <= 3:
        dp = 16 if in_dim <= 16 else (32 if in_dim <= 32 else 64)
        return hidden * (dp + 4) * 4
    dp = 16 if in_dim <= 16 else (32 if in_dim <= 32 else (64 if in_dim <= 64 else 128))
    nop = 4 if out_dim <= 4 else (8 if out_dim <= 8 else 16)
    return hidden * (dp + nop + 4) * 4


def _central_forward(seq: nn.Sequential, x: torch.Tensor) -> torch.Tensor:
    """``seq(x)`` for the :func:`mlp` heads of :class:`CentralizedActorCritic`, x ``[B, W*D]``. Without autograd on a CUDA
    tensor a one-hidden-layer head runs in K7 (up to ``_CENTRAL_K7_MAX_IN`` inputs and 16 outputs, when its hidden layer's
    weights fit the device's shared memory); any other head runs its hidden layers through the library GEMMs - the last one
    as a plain product whose bias and ReLU K7b applies on the way in - and its output layer through K7b (up to 16
    outputs)."""
    if torch.is_grad_enabled() or not x.is_cuda or not hasattr(torch, "_addmm_activation"):
        return seq(x)
    mods = list(seq)
    if (len(mods) == 3 and isinstance(mods[0], nn.Linear) and isinstance(mods[2], nn.Linear)
            and _mlp1_smem_bytes(mods[0].in_features, mods[0].out_features, mods[2].out_features)
            <= torch.cuda.get_device_properties(x.device).shared_memory_per_block_optin):
        fused = _fused_mlp1(mods, x, max_in=_CENTRAL_K7_MAX_IN, max_out=16)
        if fused is not None:
            return fused
    return _central_layers(mods, x)


def _central_layers(mods, x: torch.Tensor) -> torch.Tensor:
    """The layer-by-layer rollout forward of :func:`_central_forward`: library GEMMs for the hidden layers (the last one a
    plain product whose bias and ReLU K7b applies on the way in), K7b for the output layer."""
    h, i, last = x, 0, mods[-1]
    while i < len(mods) - 1:
        m = mods[i]
        if isinstance(m, nn.Linear) and m.bias is not None and isinstance(mods[i + 1], nn.ReLU):
            if i + 2 == len(mods) - 1 and _linear_out_ok(last, h, max_out=16) and m.bias.is_contiguous():
                return _linear_out(torch.mm(h, m.weight.t()), last, pre_bias=m.bias)
            h = torch._addmm_activation(m.bias, h, m.weight.t())
            i += 2
        else:
            h = m(h)
            i += 1
    return _linear_out(h, last) if _linear_out_ok(last, h, max_out=16) else last(h)


class CentralizedActorCritic(nn.Module):
    """CPPO's model (reference: src/algorithms/cppo.py, RLlib single-agent PPO on ``CentralizedEnvWrapper``): one actor
    MLP from the global state ``obs.reshape(B, W*D)`` to the joint action means ``[W*S]``, a free ``log_std [W*S]`` clamped
    from below, and one critic MLP from the global state to the value.

    The joint action is warehouse-major: entry ``w*S + s`` is warehouse w, SKU s (``CentralizedEnvWrapper._split_action``),
    so ``[..., W*S]`` viewed as ``[..., W, S]`` is what the batched env takes. The interface is ActorCritic's, for the
    collector, the learner and ``evaluate()``, with one policy and one log-prob and value per environment."""

    n_policies = 1

    def __init__(self, local_obs_dim: int, n_warehouses: int, action_dim: int, actor_hidden: Sequence[int] = (256,),
                 critic_hidden: Sequence[int] = (256,), activation: str = "relu", logstd_init: float = 0.0,
                 logstd_floor: float = -2.0):
        super().__init__()
        self.local_obs_dim, self.n_warehouses, self.action_dim = local_obs_dim, n_warehouses, action_dim
        self.global_obs_dim = n_warehouses * local_obs_dim
        self.joint_action_dim = n_warehouses * action_dim
        self.logstd_floor = float(logstd_floor)
        self.actor = mlp(self.global_obs_dim, actor_hidden, self.joint_action_dim, activation)
        self.log_std = nn.Parameter(torch.full((self.joint_action_dim,), float(logstd_init)))
        self.critic = mlp(self.global_obs_dim, critic_hidden, 1, activation)

    @classmethod
    def from_algorithm_config(cls, algo_config, local_obs_dim: int, n_warehouses: int,
                              action_dim: int) -> "CentralizedActorCritic":
        """From a CPPO config (``config_files/algorithms/cppo.yaml``); ``action_dim`` is the SKU count per warehouse. The
        env carries no warehouse id (``env_meta_from_algorithm_config`` of a CPPO config)."""
        from ..config.schema import CPPOConfig
        if not isinstance(algo_config, CPPOConfig):
            raise ValueError("CentralizedActorCritic is CPPO's model: IPPO and MAPPO configs build an ActorCritic")
        sp = algo_config.algorithm_specific
        net = sp.networks
        return cls(local_obs_dim, n_warehouses, action_dim, actor_hidden=net.actor.config.hidden_sizes,
                   critic_hidden=net.critic.config.hidden_sizes, activation=net.actor.config.activation,
                   logstd_init=sp.logstd_init, logstd_floor=sp.logstd_floor)

    def _head(self, seq: nn.Sequential, obs: torch.Tensor) -> torch.Tensor:
        if tuple(obs.shape[-2:]) != (self.n_warehouses, self.local_obs_dim):
            raise ValueError(f"obs must be [..., {self.n_warehouses}, {self.local_obs_dim}], got {tuple(obs.shape)}")
        lead = obs.shape[:-2]
        out = _central_forward(seq, obs.reshape(-1, self.global_obs_dim))
        return out.reshape(*lead, out.shape[-1])

    # obs: [B, W, D] local observations, flattened over W to the global state
    def action_mean(self, obs: torch.Tensor) -> torch.Tensor:
        """Joint action means [B, W*S]."""
        return self._head(self.actor, obs)

    def value(self, obs: torch.Tensor) -> torch.Tensor:
        """[B]."""
        return self._head(self.critic, obs).squeeze(-1)

    def act(self, obs: torch.Tensor, generator: Optional[torch.Generator] = None, deterministic: bool = False,
            return_raw: bool = False):
        """As ``ActorCritic.act``: ``(clipped [B, W, S], logp [B], value [B])``, or with ``return_raw=True``
        ``(clipped [B, W, S], raw [B, W*S], logp [B], value [B], mean [B, W*S])``."""
        mean = self.action_mean(obs)
        if deterministic:
            raw = mean
        else:
            raw = mean + self.std() * torch.randn(mean.shape, device=mean.device, dtype=mean.dtype, generator=generator)
        logp = self.log_prob(mean, raw)
        clipped = raw.clamp(-1.0, 1.0).view(*mean.shape[:-1], self.n_warehouses, self.action_dim)
        if return_raw:
            return clipped, raw, logp, self.value(obs), mean
        return clipped, logp, self.value(obs)

    # the diagonal Gaussian over the joint action: the same functions as ActorCritic's single shared policy
    clamped_log_std = ActorCritic.clamped_log_std
    std = ActorCritic.std
    log_prob = ActorCritic.log_prob
    entropy = ActorCritic.entropy


def env_meta_from_algorithm_config(algo_config) -> dict:
    """The ``env_meta`` keys the reference's algorithm wrappers derive from the algorithm config
    (ippo.py:68-73, 121-142): parameter sharing switches the one-hot warehouse id on. CPPO has no parameter sharing, so
    no warehouse id."""
    sp = algo_config.algorithm_specific
    meta = {"obs_normalization": getattr(sp, "obs_normalization", "off")}
    if getattr(sp, "parameter_sharing", False):
        meta["include_warehouse_id"] = True
    return meta
