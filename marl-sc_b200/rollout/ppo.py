"""PPO learner for the collected rollouts (clipped surrogate, clipped value loss, entropy bonus, optional KL
penalty), data-parallel across GPUs: each rank learns on its own env shard and the gradients are summed with
NCCL all-reduces issued per parameter bucket while the backward pass is still running - the only collective of the
whole path (SURVEY.md section 8e).

Reference wiring this replaces (RLlib's PPOTorchLearner as configured by the reference): hyper-parameters
src/algorithms/ippo.py:145-160 / mappo.py:142-157 (``num_epochs``, ``minibatch_size = batch_size //
num_minibatches``, ``shuffle_batch_per_epoch=True``, ``use_kl_loss``, ``grad_clip``), per-policy modules
ippo.py:106-115, hysteretic weighting src/algorithms/learners/hysteretic_learner.py:39-42."""
from __future__ import annotations

from typing import Callable, Dict, List, Optional, Sequence, Union

import torch
import torch.distributed as dist

from .. import _capi
from .collector import Rollout
from .policy import ActorCritic, CentralizedActorCritic


def lr_schedule(value: Union[float, Sequence[Sequence[float]]]) -> Callable[[int], float]:
    """The learning rate as a function of lifetime env steps, for the config's ``learning_rate``: a scalar is constant; a
    list of ``[timestep, lr]`` points is interpolated linearly between the points and held at the last value after the last
    point (RLlib's piecewise schedule, which the reference's learner steps with the lifetime count of sampled env steps)."""
    if isinstance(value, (int, float)):
        return lambda t: float(value)
    pts = [(float(t), float(lr)) for t, lr in value]

    def at(t: int) -> float:
        t = float(t)
        if t <= pts[0][0]:
            return pts[0][1]
        for (t0, v0), (t1, v1) in zip(pts, pts[1:]):
            if t < t1:
                return v0 + (t - t0) / (t1 - t0) * (v1 - v0)
        return pts[-1][1]
    return at


class _FusedPPOObjective(torch.autograd.Function):
    """Clipped surrogate + clipped value loss (+ KL penalty) through K6 (``marlsc_ppo_loss``): one kernel computes the
    loss terms and the gradients with respect to the action means, ``log_std`` and the values; backward only scales them."""

    @staticmethod
    def forward(ctx, mean, log_std, value, actions, logp_old, adv, targets, mean_old, log_std_old, floor, clip, vf_clip,
                vf_coeff, beta, kl_coeff):
        S = mean.shape[-1]
        P = 1 if log_std.dim() == 1 else log_std.shape[0]
        mean_c, value_c = mean.contiguous(), value.contiguous()
        n = value_c.numel()
        if mean_c.numel() != n * S or mean_c.dtype != torch.float32 or not mean_c.is_cuda:
            raise ValueError("mean must be a float32 CUDA tensor [..., S] matching value [...]")
        args = [t.detach().to(torch.float32).contiguous() for t in (actions, logp_old, adv, targets)]
        if args[0].numel() != n * S or any(a.numel() != n for a in args[1:]):
            raise ValueError("actions / logp_old / adv / targets do not match the minibatch shape")
        if P > 1 and mean.shape[-2] != P:
            raise ValueError("with independent policies the axis before the action axis must be the warehouse axis")
        ls = log_std.detach().contiguous()
        use_kl = mean_old is not None
        mo = mean_old.detach().to(torch.float32).contiguous() if use_kl else None
        lo = log_std_old.detach().to(torch.float32).contiguous() if use_kl else None
        g_mean = torch.empty_like(mean_c)
        g_value = torch.empty_like(value_c)
        sums = torch.empty((P, 3 + S), dtype=torch.float64, device=mean.device)
        _capi.check(_capi.lib().marlsc_ppo_loss(
            mean_c.data_ptr(), args[0].data_ptr(), ls.data_ptr(), P, float(floor), args[1].data_ptr(), args[2].data_ptr(),
            value_c.data_ptr(), args[3].data_ptr(), None if mo is None else mo.data_ptr(), None if lo is None else lo.data_ptr(),
            float(kl_coeff), n, S, float(clip), float(vf_clip), float(vf_coeff), -1.0 if beta is None else float(beta),
            g_mean.data_ptr(), g_value.data_ptr(), sums.data_ptr(), torch.cuda.current_stream(mean.device).cuda_stream))
        # clamp(min=floor) passes the gradient where it does not bind
        g_ls = (sums[:, 3:].reshape(ls.shape) * (ls >= floor)).to(torch.float32)
        ctx.save_for_backward(g_mean, g_ls, g_value)
        ctx.shapes = (mean.shape, value.shape)
        per = float(P) / n                                            # every policy averages over its own samples
        policy = (-sums[:, 0].sum() * per).to(torch.float32)
        vf = (sums[:, 1].sum() * per).to(torch.float32)
        kl = (sums[:, 2].sum() * per).to(torch.float32)
        return policy + vf_coeff * vf + kl_coeff * kl, policy, vf, kl

    @staticmethod
    def backward(ctx, g, _gp, _gv, _gk):
        g_mean, g_ls, g_value = ctx.saved_tensors
        return (g_mean.reshape(ctx.shapes[0]) * g, g_ls * g, g_value.reshape(ctx.shapes[1]) * g) + (None,) * 12


class GradBuckets:
    """Flat gradient buckets with the parameters' ``.grad`` as views into them (no copies), all-reduced
    asynchronously as soon as the backward pass has produced every gradient of a bucket - the overlap DDP gives,
    without wrapping the module. Buckets are filled in reverse registration order (the order backward produces them)."""

    def __init__(self, params: List[torch.nn.Parameter], bucket_bytes: int = 1 << 20):
        self.params = params
        self.buckets: List[torch.Tensor] = []
        self._members: List[List[torch.nn.Parameter]] = []
        self._bucket_of: Dict[int, int] = {}
        self._views: Dict[int, torch.Tensor] = {}
        self._ready: List[int] = []
        self._work: List = []
        self.bytes_reduced = 0
        cur: List[torch.nn.Parameter] = []
        size = 0
        for p in reversed(params):
            if cur and (size + p.numel()) * p.element_size() > bucket_bytes:
                self._close(cur)
                cur, size = [], 0
            cur.append(p)
            size += p.numel()
        if cur:
            self._close(cur)
        for p in params:
            p.register_post_accumulate_grad_hook(self._on_grad)

    def _close(self, members: List[torch.nn.Parameter]) -> None:
        flat = torch.zeros(sum(p.numel() for p in members), dtype=members[0].dtype, device=members[0].device)
        off = 0
        for p in members:
            self._views[id(p)] = flat[off:off + p.numel()].view_as(p)
            p.grad = self._views[id(p)]
            off += p.numel()
            self._bucket_of[id(p)] = len(self.buckets)
        self.buckets.append(flat)
        self._members.append(members)
        self._ready.append(0)

    @staticmethod
    def _distributed() -> bool:
        return dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1

    def zero(self) -> None:
        for b in self.buckets:
            b.zero_()
        for p in self.params:                      # somebody may have replaced .grad (zero_grad(set_to_none=True))
            if p.grad is not self._views[id(p)]:
                p.grad = self._views[id(p)]
        self._ready = [0] * len(self.buckets)
        self._work = []

    def _on_grad(self, p: torch.nn.Parameter) -> None:
        b = self._bucket_of[id(p)]
        self._ready[b] += 1
        if self._ready[b] == len(self._members[b]) and self._distributed():
            self._work.append(dist.all_reduce(self.buckets[b], op=dist.ReduceOp.SUM, async_op=True))
            self.bytes_reduced += self.buckets[b].numel() * self.buckets[b].element_size()

    def finish(self) -> None:
        """Wait for the outstanding all-reduces and turn the sums into means."""
        if not self._distributed():
            return
        # parameters that received no gradient this step still have to take part in the collective
        for b, n in enumerate(self._ready):
            if n < len(self._members[b]):
                self._work.append(dist.all_reduce(self.buckets[b], op=dist.ReduceOp.SUM, async_op=True))
                self.bytes_reduced += self.buckets[b].numel() * self.buckets[b].element_size()
        for w in self._work:
            w.wait()
        inv = 1.0 / dist.get_world_size()
        for b in self.buckets:
            b.mul_(inv)
        self._work = []


class PPOLearner:
    def __init__(self, policy: Union[ActorCritic, CentralizedActorCritic], lr: float = 5e-4, clip_param: float = 0.2, vf_clip_param: float = 10.0,
                 vf_loss_coeff: float = 1.0, entropy_coeff: float = 0.01, grad_clip: Optional[float] = None,
                 hysteretic_beta: Optional[float] = None, fused_loss: Optional[bool] = None, use_kl_loss: bool = False,
                 kl_coeff: float = 0.2, kl_target: float = 0.01, num_epochs: int = 1, num_minibatches: int = 1,
                 bucket_bytes: int = 1 << 20, seed: int = 0):
        self.policy = policy
        # K6 on CUDA parameters unless asked otherwise; loss_reference() keeps the plain PyTorch form
        self.fused = next(policy.parameters()).is_cuda if fused_loss is None else bool(fused_loss)
        if self.fused and policy.log_std.shape[-1] > 512:
            # a centralised policy's joint action (W*S) can outgrow K6's shared-memory tables
            raise ValueError(f"the fused PPO loss (K6) takes at most 512 action dimensions per policy, this policy has "
                             f"{policy.log_std.shape[-1]}: pass fused_loss=False for the PyTorch objective")
        self.opt = torch.optim.Adam(policy.parameters(), lr=lr)
        self.clip, self.vf_clip, self.vf_coeff, self.ent_coeff = clip_param, vf_clip_param, vf_loss_coeff, entropy_coeff
        self.grad_clip, self.beta = grad_clip, hysteretic_beta
        # RLlib PPO defaults: kl_coeff 0.2, kl_target 0.01, adapted after every update (x1.5 above 2 target, x0.5 below half)
        self.use_kl, self.kl_coeff, self.kl_target = bool(use_kl_loss), float(kl_coeff), float(kl_target)
        self.num_epochs, self.num_minibatches = int(num_epochs), int(num_minibatches)
        self.params = [p for p in policy.parameters() if p.requires_grad]
        self.buckets = GradBuckets(self.params, bucket_bytes)
        dev = self.params[0].device
        self.gen = torch.Generator(device=dev)
        self.gen.manual_seed(seed)

    @classmethod
    def from_algorithm_config(cls, policy: Union[ActorCritic, CentralizedActorCritic], algo_config, **kw) -> "PPOLearner":
        sp, sh = algo_config.algorithm_specific, algo_config.shared
        lr = sh.learning_rate if isinstance(sh.learning_rate, (int, float)) else sh.learning_rate[0][1]
        return cls(policy, lr=lr, clip_param=sp.clip_param, vf_clip_param=sp.vf_clip_param, vf_loss_coeff=sp.vf_loss_coeff,
                   entropy_coeff=sp.entropy_coeff, grad_clip=sp.grad_clip, hysteretic_beta=getattr(sp, "hysteretic_beta", None),
                   use_kl_loss=bool(getattr(sp, "use_kl_loss", False)), num_epochs=sh.num_epochs,
                   num_minibatches=sh.num_minibatches, **kw)

    def set_lr(self, lr: float) -> None:
        """Learning rate of the following updates (a schedule sets it before every update, see ``lr_schedule``)."""
        for g in self.opt.param_groups:
            g["lr"] = float(lr)

    # ------------------------------------------------------------------ objective
    def loss(self, obs, actions, logp_old, adv, targets, mean_old=None, log_std_old=None) -> Dict[str, torch.Tensor]:
        if not self.fused:
            return self.loss_reference(obs, actions, logp_old, adv, targets, mean_old, log_std_old)
        pol = self.policy
        kl_on = self.use_kl and mean_old is not None
        partial, policy, vf, kl = _FusedPPOObjective.apply(
            pol.action_mean(obs), pol.log_std, pol.value(obs), actions, logp_old, adv, targets, mean_old if kl_on else None,
            log_std_old if kl_on else None, pol.logstd_floor, self.clip, self.vf_clip, self.vf_coeff, self.beta,
            self.kl_coeff if kl_on else 0.0)
        ent = pol.entropy()
        return dict(total=partial - self.ent_coeff * ent, policy=policy.detach(), vf=vf.detach(), entropy=ent, kl=kl.detach())

    def loss_reference(self, obs, actions, logp_old, adv, targets, mean_old=None, log_std_old=None) -> Dict[str, torch.Tensor]:
        """The same objective in plain PyTorch (autograd): the numerical reference of K6. Per-policy means summed over
        the policies (one policy with parameter sharing)."""
        pol = self.policy
        P = pol.n_policies
        mean = pol.action_mean(obs)
        logp = pol.log_prob(mean, actions)
        ratio = (logp - logp_old).exp()
        if self.beta is not None:
            adv = torch.where(adv < 0, adv * self.beta, adv)
        surr = torch.minimum(ratio * adv, ratio.clamp(1 - self.clip, 1 + self.clip) * adv)
        v = pol.value(obs)
        vf = torch.clamp((v - targets) ** 2, max=self.vf_clip)
        ent = pol.entropy()
        red = (lambda x: x.mean()) if P == 1 else (lambda x: x.reshape(-1, P).mean(0).sum())
        kl = torch.zeros((), device=mean.device)
        if self.use_kl and mean_old is not None:
            ls_new = pol.clamped_log_std()
            ls_old = log_std_old.reshape(ls_new.shape)
            klv = (ls_new - ls_old + (torch.exp(2 * ls_old) + (mean_old - mean) ** 2) / (2 * torch.exp(2 * ls_new)) - 0.5).sum(-1)
            kl = red(klv)
        total = -red(surr) + self.vf_coeff * red(vf) - self.ent_coeff * ent + (self.kl_coeff * kl if self.use_kl else 0.0)
        return dict(total=total, policy=-red(surr), vf=red(vf), entropy=ent, kl=kl.detach())

    # ------------------------------------------------------------------ gradient step
    def all_reduce_grads(self) -> int:
        """Bytes all-reduced so far (the collectives themselves run from the backward hooks, see GradBuckets)."""
        return self.buckets.bytes_reduced

    def _clip(self) -> None:
        """``grad_clip`` by global norm per policy module, as RLlib applies it per module."""
        pol = self.policy
        if pol.n_policies == 1:
            torch.nn.utils.clip_grad_norm_(self.params, self.grad_clip)
            return
        P = pol.n_policies
        sq = torch.zeros(P, device=self.params[0].device)
        for p in self.params:
            sq += p.grad.reshape(P, -1).pow(2).sum(1)
        scale = torch.clamp(self.grad_clip / (sq.sqrt() + 1e-6), max=1.0)
        for p in self.params:
            p.grad.mul_(scale.view(P, *([1] * (p.dim() - 1))))

    def step_on(self, obs, actions, logp_old, adv, targets, mean_old=None, log_std_old=None) -> Dict[str, torch.Tensor]:
        self.buckets.zero()
        out = self.loss(obs, actions, logp_old, adv, targets, mean_old, log_std_old)
        out["total"].backward()          # bucket all-reduces start from the hooks while backward runs
        self.buckets.finish()
        if self.grad_clip:
            self._clip()
        self.opt.step()
        return out

    def minibatch_step(self, ro: Rollout, t_slice: slice, e_slice: slice) -> Dict[str, float]:
        obs = ro.obs[t_slice, e_slice].flatten(0, 1)           # [B, W, D]
        mo = ro.mean_old[t_slice, e_slice].flatten(0, 1) if (self.use_kl and ro.mean_old is not None) else None
        out = self.step_on(obs, ro.actions[t_slice, e_slice].flatten(0, 1), ro.logp[t_slice, e_slice].flatten(0, 1),
                           ro.advantages[t_slice, e_slice].flatten(0, 1), ro.targets[t_slice, e_slice].flatten(0, 1),
                           mo, ro.log_std_old)
        return {k: float(v.detach()) for k, v in out.items()}

    def update(self, ro: Rollout, num_epochs: Optional[int] = None, num_minibatches: Optional[int] = None,
               shuffle: bool = True, max_minibatches: Optional[int] = None) -> Dict[str, float]:
        """One learner update on a rollout: ``num_epochs`` passes, each over a fresh on-device permutation of the
        (timestep, environment) samples cut into ``num_minibatches`` minibatches (reference ippo.py:149-152:
        ``minibatch_size = batch_size // num_minibatches``, ``shuffle_batch_per_epoch=True``). All agents of a sample
        stay together, so a minibatch is ``[B, W, ...]``. Adapts the KL coefficient afterwards when ``use_kl_loss``."""
        E_ = ro.rewards.shape[1]
        T = ro.rewards.shape[0]
        n = T * E_
        epochs = self.num_epochs if num_epochs is None else int(num_epochs)
        nmb = self.num_minibatches if num_minibatches is None else int(num_minibatches)
        mb = max(1, n // nmb)
        dev = ro.rewards.device
        flat = lambda x: x[:T].reshape(n, *x.shape[2:])                                       # noqa: E731
        obs, act, logp, adv, tgt = flat(ro.obs), flat(ro.actions), flat(ro.logp), flat(ro.advantages), flat(ro.targets)
        kl_on = self.use_kl and ro.mean_old is not None
        mo = flat(ro.mean_old) if kl_on else None
        sums: Dict[str, torch.Tensor] = {}
        steps = 0
        for _ in range(epochs):
            perm = torch.randperm(n, device=dev, generator=self.gen) if shuffle else torch.arange(n, device=dev)
            for k in range(nmb):
                idx = perm[k * mb:(k + 1) * mb]
                out = self.step_on(obs.index_select(0, idx), act.index_select(0, idx), logp.index_select(0, idx),
                                   adv.index_select(0, idx), tgt.index_select(0, idx),
                                   mo.index_select(0, idx) if kl_on else None, ro.log_std_old)
                for name, v in out.items():
                    sums[name] = sums.get(name, 0) + v.detach()
                steps += 1
                if max_minibatches is not None and steps >= max_minibatches:
                    break
            if max_minibatches is not None and steps >= max_minibatches:
                break
        res = {name: float(v) / steps for name, v in sums.items()}      # one device->host read per metric
        if kl_on:
            if res["kl"] > 2.0 * self.kl_target:
                self.kl_coeff *= 1.5
            elif res["kl"] < 0.5 * self.kl_target:
                self.kl_coeff *= 0.5
        res["minibatches"] = steps
        res["kl_coeff"] = self.kl_coeff
        return res
