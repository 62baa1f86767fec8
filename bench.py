#!/usr/bin/env python
"""bench.py - agent-steps/s of the hot path (env step K1 + GAE scan K2) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload large|small]
                    [--dump-outputs DIR]

One bench "step" is one rollout segment: SEG env steps of all E environments (one marlsc_env_step call each =
four launches of the split step K1a-K1d, or one fused launch; plus a reset launch when an episode ends) followed
by one K2 launch over the segment's
[SEG, E, W] rewards/values. agent-steps per bench step = E * W * SEG. Workload (default): BASELINE.json
configs[2], the large network (10 warehouses x 100 SKUs x 50 regions, lead times 1..10) with 65,536
envs per GPU - the config the 1e9 agent-steps/s target is quoted on. Environments are independent,
so N GPUs run N shards with no communication on the path (weak scaling).

Printed JSON (rank 0): the driver's contract plus
  roofline     - K1 achieved HBM GB/s (algorithmic bytes / CUDA-event time of the step's launches) against
                 MEASURED_PEAKS.json, plus every launch of the step on its own (kernels[])
  cpu_baseline - the CPU oracle port (oracle/inventory_oracle.py + gae_oracle.py) on a bounded sample
  e2e          - same metric through the host-buffer C-ABI call (marlsc_env_step_host): pinned host
                 actions/demand copied in, rewards (and the segment's advantages/targets) copied out
  clocks       - nvidia-smi SM clock / throttle reasons sampled during the timed region
`--impl reference` times the reference's CPU algorithm (the oracle port; the reference is pure Python and
cannot be compiled into oracle/_ref) on all host cores for the same metric and config.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "agent_steps_per_sec_env_step_plus_gae"
UNIT = "agent-steps/s"
SEG = 20                # env steps per rollout segment (episode_length 100 = 5 segments)
GAMMA, LAM = 0.99, 0.95
ACTION_RANGE = (-1.0, -0.5)   # direct action space, max 40: mean order 5/cell/step = mean demand


# --------------------------------------------------------------------------------------- workloads
def workload(name: str):
    from golden.scenarios import large_network, small_default
    if name == "large":
        env = large_network()
        return env, dict(workload="large_network_10wh_100sku_50reg_lead1-10 (BASELINE configs[2])",
                         envs_per_gpu=65536, mean_orders_per_env_step=50.0)
    env = small_default()
    return env, dict(workload="env_symmetric_3WH2SKU (BASELINE configs[1] shape)", envs_per_gpu=4096,
                     mean_orders_per_env_step=12.0)


def base_stock_levels(env_dict, spec, z):
    """S[w,k] = L*E[D] + z*sqrt(L*E[D]) (reference run_baselines.py:188-196), with E[D] summed over the
    regions a warehouse serves first (its cheapest-priority regions) so that it also makes sense when
    there are more regions than warehouses; for R == W symmetric configs this is the home region."""
    import numpy as np
    p = env_dict["components"]["demand_sampler"]["params"]
    W, S, R = env_dict["n_warehouses"], env_dict["n_skus"], env_dict["n_regions"]
    lam_o, prob = np.asarray(p["lambda_orders"], float), np.asarray(p["probability_skus"], float)
    lam_q = np.asarray(p["lambda_quantity"], float)
    out_var = spec.tables["out_var"]
    first = np.argsort(out_var, axis=0, kind="stable")[0]            # cheapest warehouse per region
    ed = np.zeros((W, S))
    for r in range(R):
        ed[first[r]] += lam_o[r] * prob[r] * lam_q[r]
    lead = spec.tables["expected_lead"].astype(float)
    return lead * ed + z * np.sqrt(lead * ed)


def record_base_stock_actions(env, env_dict, demand, z):
    import numpy as np
    import torch
    dev = env.device
    level = torch.from_numpy(base_stock_levels(env_dict, env.spec, z)).to(dev)
    maxq = torch.tensor(env_dict["action_space"]["params"]["max_order_quantities"], dtype=torch.float64, device=dev)
    actions = []
    env.reset()
    for t in range(len(demand)):
        qty = torch.clamp(level - env.inventory.to(torch.float64) - env.pending_matrix().to(torch.float64), min=0.0)
        qty = torch.minimum(qty, maxq)
        act = (2.0 * qty / maxq - 1.0).to(torch.float32)
        actions.append(act)
        env.step(act, orders=demand[t])
    torch.cuda.synchronize()
    return actions


def algorithmic_bytes_per_env_step(W, S, L, obs_dim, mean_orders, qty_bytes=1, layout="wide", mean_lines=0.0):
    """SURVEY.md section 8d, evaluated with the actual dtype sizes of the layout in use (as 8d requires for narrower state).
    reads: actions + inventory + pipeline (L planes) + history (sum + oldest) + demand
    writes: inventory + new pipeline slot + history (2) + obs 4*W*obs_dim + rewards 4W + trunc 1
    wide:    int32 state, dense demand rows + region id            -> 4WS(L+8) + orders (S+2) + ...
    compact: uint16 stock/history, uint8 ring, 2-byte demand lines -> WS(4 + 2*2 + L + 1 + 4*2) + 2 lines + 4 + ..."""
    tail = 4 * W * obs_dim + 4 * W + 1
    if layout == "compact":
        return W * S * (4 + 4 + L + 1 + 8) + 2 * mean_lines + 4 + tail
    return 4 * W * S * (L + 8) + mean_orders * (S * qty_bytes + 2) + tail


# --------------------------------------------------------------------------------------- --dump-outputs
DUMP_BYTES = 60 << 20    # what --dump-outputs writes stays under 64 MB in all


def dump_outputs(out_dir, arrays, n_envs):
    """Write the timed path's outputs as ``out_dir/<name>.npy`` (float32, float64 stays float64) so that two builds can be
    compared output for output. ``arrays`` maps a name to (device tensor, axis of the environment index). When the whole
    batch does not fit DUMP_BYTES, the same environments are kept in every array: a fixed seeded sample, identical from
    run to run."""
    import numpy as np
    import torch
    wide = {name: t.dtype == torch.float64 for name, (t, _) in arrays.items()}
    per_env = sum(t.numel() // n_envs * (8 if wide[name] else 4) for name, (t, _) in arrays.items())
    k = min(n_envs, DUMP_BYTES // per_env)
    if k == 0:
        raise ValueError(f"--dump-outputs: one environment's outputs ({per_env} bytes) exceed the {DUMP_BYTES}-byte cap")
    idx = np.arange(n_envs) if k == n_envs else np.sort(np.random.default_rng(0).choice(n_envs, k, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, (t, axis) in arrays.items():
        sel = t.index_select(axis, torch.from_numpy(idx).to(t.device))
        np.save(os.path.join(out_dir, name + ".npy"), sel.to(torch.float64 if wide[name] else torch.float32).cpu().numpy())
    print(f"dump-outputs: {', '.join(arrays)} of {k} of {n_envs} environments -> {out_dir}", file=sys.stderr, flush=True)


# --------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock and throttle reasons of one GPU during the timed region: NVML polled from a thread every 20 ms (first
    sample taken synchronously in start(), last in stop(), so even a 100 ms region has samples); `nvidia-smi -lms` as the
    fallback when the NVML binding is missing."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None
        self.nvml, self.handle, self.stop_flag, self.thread = None, None, threading.Event(), None
        self.sm, self.mx, self.reasons = [], [], set()

    def _nvml_sample(self):
        n, h = self.nvml, self.handle
        self.sm.append(float(n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM)))
        self.mx.append(float(n.nvmlDeviceGetMaxClockInfo(h, n.NVML_CLOCK_SM)))
        try:
            get = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
            bits = int(get(h))
        except Exception:
            return
        for name, const in (("hw_slowdown", "HwSlowdown"), ("hw_thermal_slowdown", "HwThermalSlowdown"),
                            ("sw_thermal_slowdown", "SwThermalSlowdown"), ("sw_power_cap", "SwPowerCap")):
            mask = getattr(n, "nvmlClocksEventReason" + const, None) or getattr(n, "nvmlClocksThrottleReason" + const, 0)
            if bits & int(mask):
                self.reasons.add(name)

    def _nvml_loop(self):
        while not self.stop_flag.wait(0.02):
            try:
                self._nvml_sample()
            except Exception:
                return

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml, self.handle = pynvml, pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self._nvml_sample()
            self.thread = threading.Thread(target=self._nvml_loop, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.nvml is not None:
            self.stop_flag.set()
            if self.thread is not None:
                self.thread.join(timeout=1.0)
            try:
                self._nvml_sample()
            except Exception:
                pass
            if not self.sm:
                return None
            return dict(sm_mhz=statistics.median(self.sm), sm_max_mhz=max(self.mx), reasons=sorted(self.reasons),
                        samples=len(self.sm), source="nvml")
        if self.proc is None:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for name, val in zip(self.NAMES, r[3:7]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        if not sm:
            return None
        return dict(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm), source="nvidia-smi")


# --------------------------------------------------------------------------------------- synthetic data (device)
def synth_demand(env_dict, E, steps, device, seed):
    """Per step CSR orders drawn on the device with the reference sampler's distribution
    (demand_sampler.py:105-163): Poisson order counts per region, Bernoulli SKU masks,
    max(1, Poisson) quantities. Synthetic input generation, outside every timed region."""
    import torch
    from marlsc_b200.envs import DeviceOrders
    p = env_dict["components"]["demand_sampler"]["params"]
    R, S = env_dict["n_regions"], env_dict["n_skus"]
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    lam_o = torch.tensor(p["lambda_orders"], dtype=torch.float32, device=device)
    prob = torch.tensor(p["probability_skus"], dtype=torch.float32, device=device)
    lam_q = torch.tensor(p["lambda_quantity"], dtype=torch.float32, device=device)
    out = []
    for _ in range(steps):
        counts = torch.poisson(lam_o.expand(E, R).contiguous(), generator=g).to(torch.int64)
        offsets = torch.zeros(E + 1, dtype=torch.int32, device=device)
        offsets[1:] = counts.sum(1).cumsum(0).to(torch.int32)
        region = torch.repeat_interleave(torch.arange(R, device=device).repeat(E), counts.reshape(-1))
        n = int(region.numel())
        mask = torch.rand((n, S), device=device, generator=g) < prob[region][:, None]
        qty = torch.clamp(torch.poisson(lam_q[region], generator=g), min=1.0, max=255.0)
        rows = (qty * mask).to(torch.uint8)
        pad = (-(n * S)) % 16 + (16 if n == 0 else 0)
        flat = torch.cat([rows.reshape(-1), torch.zeros(pad, dtype=torch.uint8, device=device)])
        out.append(DeviceOrders(offsets, region.to(torch.int16) if n else torch.zeros(1, dtype=torch.int16, device=device), flat, n))
    return out


# --------------------------------------------------------------------------------------- CPU port timing
def _cpu_worker(args):
    env_dict, n_envs, steps, seed = args
    import numpy as np
    from marlsc_b200.config import environment_config_from_dict
    from marlsc_b200.context import create_environment_context
    from marlsc_b200.registry import get_demand_sampler
    from oracle.gae_oracle import gae_targets
    from oracle.inventory_oracle import OracleEnv
    d = dict(env_dict)
    d["allow_region_mismatch"] = True
    cfg = environment_config_from_dict(d)
    W, S = cfg.n_warehouses, cfg.n_skus
    rng = np.random.default_rng(seed)
    init = np.full((W, S), 60)
    envs, demand = [], []
    for i in range(n_envs):
        smp = get_demand_sampler(cfg, context=create_environment_context(cfg))
        smp.reset(np.random.default_rng(seed * 1000 + i))
        demand.append([[(o.region_id, o.sku_demands) for o in smp.sample(t)] for t in range(steps)])
        o = OracleEnv(env_dict)
        o.reset(init)
        envs.append(o)
    acts = rng.uniform(ACTION_RANGE[0], ACTION_RANGE[1], (n_envs, steps, W, S)).astype(np.float32)
    vals = rng.normal(-30, 5, (steps + 1, n_envs * W)).astype(np.float32)
    t0 = time.perf_counter()
    rew = np.zeros((steps, n_envs, W), np.float32)
    for i, o in enumerate(envs):
        for t in range(steps):
            rew[t, i] = o.step(acts[i, t], demand[i][t])["rewards"]
    gae_targets(rew.reshape(steps, -1), vals, GAMMA, LAM)
    return time.perf_counter() - t0, n_envs * W * steps


def _ref_worker(args):
    """The reference's own InventoryEnvironment (the checkout at MARLSC_REFERENCE_ROOT, or its copy in oracle/_ref) under the
    base-stock heuristic with its own Poisson demand sampler: the same segment the GPU arm times, on one host core."""
    env_dict, n_envs, steps, seed, z = args
    import numpy as np
    from oracle import ref_harness as H
    from oracle.gae_oracle import gae_targets
    large = env_dict["n_regions"] != env_dict["n_warehouses"]
    cfg = H.env_config_from_dict(env_dict, allow_region_mismatch=large)
    W, S, R = env_dict["n_warehouses"], env_dict["n_skus"], env_dict["n_regions"]
    p = env_dict["components"]["demand_sampler"]["params"]
    lam_o, prob = np.broadcast_to(np.asarray(p["lambda_orders"], float), (R,)), np.broadcast_to(np.asarray(p["probability_skus"], float), (R,))
    lam_q = np.broadcast_to(np.asarray(p["lambda_quantity"], float), (R, S))
    out_var = np.asarray(env_dict["cost_structure"]["shipment_cost"]["outbound_variable"], float)
    first = np.argsort(out_var, axis=0, kind="stable")[0]
    ed = np.zeros((W, S))
    for r in range(R):
        ed[first[r]] += lam_o[r] * prob[r] * lam_q[r]
    lead = np.asarray(env_dict["components"]["lead_time_sampler"]["params"]["expected_lead_times"], float)
    level = lead * ed + z * np.sqrt(lead * ed)
    envs = [H.make_env(cfg, seed=H.derive_env_seed(seed, 0, i)) for i in range(n_envs)]
    for e in envs:
        e.reset()
    vals = np.random.default_rng(seed).normal(-30, 5, (steps + 1, n_envs * W)).astype(np.float32)
    t0 = time.perf_counter()
    rew = np.zeros((steps, n_envs, W), np.float32)
    for i, e in enumerate(envs):
        for t in range(steps):
            act = H.base_stock_policy(e, level)
            _, r, _, _, _ = e.step({a: act[k] for k, a in enumerate(e.agents)})
            rew[t, i] = [r[a] for a in e.agents]
    gae_targets(rew.reshape(steps, -1), vals, GAMMA, LAM)
    return time.perf_counter() - t0, n_envs * W * steps


def cpu_port(env_dict, n_envs_per_worker, steps, workers, kind="port", z=2.0):
    import multiprocessing as mp
    if kind == "reference":
        from oracle import ref_harness as H
        os.environ.update(H.STABLE_SORT_ENV)               # inherited by the workers: stable argsort ties (SURVEY 7.2-1)
        fn, jobs = _ref_worker, [(env_dict, n_envs_per_worker, steps, 17 + k, z) for k in range(workers)]
    else:
        fn, jobs = _cpu_worker, [(env_dict, n_envs_per_worker, steps, 17 + k) for k in range(workers)]
    t0 = time.perf_counter()
    if workers == 1:
        res = [fn(jobs[0])]
    else:
        with mp.get_context("spawn").Pool(workers) as pool:
            res = pool.map(fn, jobs)
    wall = time.perf_counter() - t0
    agent_steps = sum(r[1] for r in res)
    busy = max(r[0] for r in res)
    return agent_steps / busy, agent_steps, wall


def reference_kind():
    """"reference" when the reference's own env can be imported here (oracle/_ref made by oracle/make_ref.py, or the
    checkout at MARLSC_REFERENCE_ROOT), else "port" (oracle/inventory_oracle.py)."""
    try:
        from oracle import ref_harness as H
        return "reference" if H.available() else "port"
    except Exception:
        return "port"


# --------------------------------------------------------------------------------------- reference arm
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    env_dict, cfg = workload(args.workload)
    large = args.workload == "large"
    cores = os.cpu_count() or 1
    workers = max(1, min(cores, 64))
    kind = reference_kind()
    # per worker and bench step: the GPU arm's segment (SEG env steps) of a few environments - a few seconds of host work
    n_env = (2 if large else 16) if kind == "reference" else (4 if large else 32)
    seg = SEG
    values = []
    for _ in range(args.warmup):
        cpu_port(env_dict, n_env, seg, workers, kind, args.z)
    t0 = time.perf_counter()
    total = 0
    for _ in range(args.steps):
        v, n, _ = cpu_port(env_dict, n_env, seg, workers, kind, args.z)
        values.append(v)
        total += n
    wall = time.perf_counter() - t0
    value = statistics.mean(values)
    what = ("the reference's own InventoryEnvironment (unmodified copy under oracle/_ref), its own Poisson demand sampler, "
            "base-stock heuristic z=%g" % args.z) if kind == "reference" else "the CPU oracle port (oracle/inventory_oracle.py), pre-sampled demand"
    sample = f"{workers} processes x {n_env} envs x {seg} env steps + NumPy GAE per bench step; {what}"
    line = dict(impl="reference", metric=METRIC, value=value, unit=UNIT, n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=1e3 * wall / max(1, args.steps), higher_is_better=True, scaling="weak", vs_baseline=None,
                dtype="f64", data="synthetic", config=dict(cfg, segment_env_steps=seg, gamma=GAMMA, lam=LAM,
                                                           actions=f"base-stock heuristic z={args.z}"),
                cpu_baseline=dict(value=value, unit=UNIT, cores=workers, kind=kind, sample=sample),
                e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0,
                note=("timed: the reference's own Python env step + a NumPy GAE restatement (RLlib, which owns GAE in the "
                      "reference, is not installable here)") if kind == "reference" else
                     "oracle/_ref is missing (run oracle/make_ref.py with MARLSC_REFERENCE_ROOT set to a marl-sc checkout): "
                     "timed the CPU oracle port")
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------- host placement
def bind_to_gpu_cpus(index: int):
    """Pin this process to the CPU cores NVML reports as local to GPU ``index`` (same NUMA node / PCIe root). Pinned host
    buffers are placed by first touch, so the end-to-end arm's staging memory ends up next to the GPU it feeds: eight ranks
    streaming from one socket's memory was what held round 1's 8-GPU end-to-end number at 0.42 of linear."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        n_cpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (n_cpu + 63) // 64)
        cpus = [64 * i + b for i, wd in enumerate(words) for b in range(64) if (wd >> b) & 1 and 64 * i + b < n_cpu]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return dict(cpus=len(cpus), first=cpus[0], last=cpus[-1])
    except Exception as ex:                          # no NVML, restricted cpuset: keep the default placement
        return dict(error=str(ex)[:80])
    return None


# --------------------------------------------------------------------------------------- learner collective
def learner_allreduce_record(dev, world, rank, minibatch_envs=8192):
    """The only collective of the path (SURVEY 8e): one MAPPO-sized PPO minibatch - actor [14->256->256->2], centralised
    critic [56->64->64->1] (reference config_files/algorithms/mappo.yaml:43-55, wiring src/algorithms/mappo.py:142-157) -
    forward + backward with the gradients all-reduced over NCCL from the backward hooks (rollout/ppo.py GradBuckets), timed
    with CUDA events on every rank (max over ranks), and the bare all-reduce of the same flat buffer for its bus bandwidth."""
    import torch
    import torch.distributed as dist
    from marlsc_b200.rollout import ActorCritic, PPOLearner
    torch.manual_seed(0)
    W, D, S = 3, 14, 2
    pol = ActorCritic(D, W, S, actor_hidden=(256, 256), critic_hidden=(64, 64), critic_obs_type="global", logstd_init=-1.2,
                      logstd_floor=-3.5).to(dev)
    learner = PPOLearner(pol, lr=5e-4, grad_clip=5.0, use_kl_loss=True)
    B = minibatch_envs
    g = torch.Generator(device=dev).manual_seed(rank)
    obs = torch.randn((B, W, D), device=dev, generator=g)
    with torch.no_grad():
        mean = pol.action_mean(obs)
        act = mean + 0.3 * torch.randn(mean.shape, device=dev, generator=g)
        logp = pol.log_prob(mean, act)
    adv, tgt = torch.randn((B, W), device=dev, generator=g), torch.randn((B, W), device=dev, generator=g)
    ls_old = pol.clamped_log_std().detach().reshape(1, S).clone()

    def step():
        learner.step_on(obs, act, logp, adv, tgt, mean, ls_old)

    def timed(fn, n):
        torch.cuda.synchronize()
        dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        torch.cuda.synchronize()
        t = torch.tensor([a.elapsed_time(b) / n], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for _ in range(5):
        step()
    ms_step = timed(step, 20)
    n_par = sum(p.numel() for p in learner.params)
    flat = torch.zeros(n_par, device=dev)
    for _ in range(5):
        dist.all_reduce(flat)
    ms_ar = timed(lambda: dist.all_reduce(flat), 50)
    nbytes = n_par * 4
    big = torch.zeros(64 << 20, device=dev)                       # 256 MB: what the links sustain
    for _ in range(3):
        dist.all_reduce(big)
    ms_big = timed(lambda: dist.all_reduce(big), 10)
    bus = lambda b, ms: 2.0 * (world - 1) / world * b / (ms * 1e-3) / 1e9     # noqa: E731  (ring all-reduce bus bandwidth)
    return dict(ranks=world, parameters=n_par, bytes=nbytes, buckets=len(learner.buckets.buckets),
                minibatch_agent_samples=B * W, ms_minibatch_step_with_allreduce=ms_step, ms_allreduce_alone=ms_ar,
                learner_agent_samples_per_s=world * B * W / (ms_step * 1e-3),
                busbw_gbs_gradient_allreduce=bus(nbytes, ms_ar), busbw_gbs_256mb_allreduce=bus(big.numel() * 4, ms_big),
                note="gradient all-reduce of a 0.3 MB buffer is latency-bound; the 256 MB figure shows the NVLink/NVSwitch "
                     "bandwidth NCCL reaches on this box; no collective runs on the step / GAE path")


# --------------------------------------------------------------------------------------- our arm
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    import marlsc_b200  # noqa: F401
    from marlsc_b200 import _capi
    from marlsc_b200.config import environment_config_from_dict
    from marlsc_b200.envs import BatchedInventoryEnv
    from marlsc_b200.rollout import compute_gae

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_cpus(local)                   # pinned staging buffers then live next to this rank's GPU
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    env_dict, cfg_desc = workload(args.workload)
    d = dict(env_dict)
    d["allow_region_mismatch"] = True
    cfg = environment_config_from_dict(d)
    E = args.envs or cfg_desc["envs_per_gpu"]
    W, S = cfg.n_warehouses, cfg.n_skus
    env = BatchedInventoryEnv(cfg, E, device=dev, host_samplers=False, team_size=args.team, fused_kernel=args.fused,
                              layout=args.layout)
    L = _capi.lib()
    compact = env.layout == "compact"

    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    n_in = args.distinct_steps if args.policy == "uniform" else cfg.episode_length
    demand = synth_demand(env_dict, E, n_in, dev, 99 + rank)
    mean_orders = float(np.mean([dm.n_orders for dm in demand])) / E
    dense_demand = demand
    mean_lines = 0.0
    if compact:
        # the compact layout's native demand format: sparse lines, converted once on the device (outside every timed region)
        demand = []
        for dm in dense_demand:
            demand.append(env.lines_from_orders(dm))
        mean_lines = float(np.mean([dm.n_lines for dm in demand])) / E
        spot_dense = dense_demand[:SEG]                # the oracle spot check replays the first segment
        dense_demand = dense_demand[:4]
        torch.cuda.empty_cache()
    else:
        spot_dense = dense_demand[:SEG]
    if args.policy == "uniform":
        lo, hi = ACTION_RANGE
        actions = [(torch.rand((E, W, S), device=dev, generator=gen) * (hi - lo) + lo) for _ in range(n_in)]
    else:
        # Pre-sampled actions of the reference's heuristic base-stock baseline (BASELINE configs[0];
        # reference run_baselines.py:133-207): one untimed recording episode on the same demand, then
        # the timed passes replay demand + actions, so every timed episode is the same trajectory.
        actions = record_base_stock_actions(env, env_dict, demand, args.z)
    values = torch.randn((SEG + 1, E, W), device=dev, generator=gen) * 5 - 30
    rewards = torch.empty((SEG, E, W), device=dev)
    adv = torch.empty_like(rewards)
    tgt = torch.empty_like(rewards)
    obs_buf = [torch.empty_like(env.obs), torch.empty_like(env.obs)]
    k1_events = []
    k2_events = []

    def segment(time_k1: bool, counter: list):
        for i in range(SEG):
            if env.timestep >= env.episode_length or counter[0] == 0:
                env.reset(obs_out=obs_buf[0])
            j = env.timestep % n_in if args.policy == "base_stock" else counter[0] % n_in
            if time_k1:
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
            env.step(actions[j], orders=demand[j], obs_out=obs_buf[counter[0] & 1], rewards_out=rewards[i])
            if time_k1:
                b.record()
                k1_events.append((a, b))
            counter[0] += 1
        if time_k1:
            ga, gb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ga.record()
        compute_gae(rewards, values, GAMMA, LAM, adv_out=adv, targets_out=tgt)
        if time_k1:
            gb.record()
            k2_events.append((ga, gb))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    counter = [0]
    for _ in range(args.warmup):
        segment(False, counter)
    barrier()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    launches0 = L.marlsc_launch_count()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(args.steps):
        segment(True, counter)
    stop.record()
    barrier()
    elapsed_ms = start.elapsed_time(stop)
    launches = L.marlsc_launch_count() - launches0
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # the last timed segment: its rewards, GAE advantages / targets and the observations of its last env step
        dump_outputs(args.dump_outputs, dict(observations=(obs_buf[(counter[0] - 1) & 1], 0), rewards=(rewards, 1),
                                             advantages=(adv, 1), targets=(tgt, 1)), E)
    # per-launch durations of the step's kernels: a separate short pass with the library's own CUDA events
    # around each launch (marlsc_env_set_timing); each step is read back before the next one starts
    per_launch = []
    if rank == 0:
        env.set_timing(True)
        for i in range(12):
            if env.timestep >= env.episode_length:
                env.reset(obs_out=obs_buf[0])
            j = env.timestep % n_in if args.policy == "base_stock" else i % n_in
            env.step(actions[j], orders=demand[j], obs_out=obs_buf[i & 1], rewards_out=rewards[i % SEG])
            per_launch.append(env.last_step_timing())
        env.set_timing(False)
        per_launch = per_launch[2:]
    k1_ms = [a.elapsed_time(b) for a, b in k1_events]
    k2_ms = [a.elapsed_time(b) for a, b in k2_events]
    if world > 1:
        tmax = torch.tensor([elapsed_ms], device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        elapsed_ms = float(tmax.item())
    agent_steps = E * W * SEG * args.steps * world
    value = agent_steps / (elapsed_ms * 1e-3)

    # ---- end to end through the host-buffer C-ABI call (marlsc_env_rollout_host) -----------------
    e2e = None
    e2e_obs = None
    if not args.no_e2e:
        from marlsc_b200.envs import HostRollout
        n_host = min(n_in, 4)
        h_rew = torch.empty((SEG, E, W)).pin_memory()
        h_val = values.cpu().pin_memory()
        h_adv, h_tgt = torch.empty((SEG, E, W)).pin_memory(), torch.empty((SEG, E, W)).pin_memory()
        idx = [i % n_host for i in range(SEG)]
        if compact:
            # the compact layout's host-facing inputs: integer order quantities (uint8, the rescaled action) and sparse
            # demand lines - 2.3x fewer bytes over PCIe than float actions + dense order rows
            maxq = torch.tensor(env_dict["action_space"]["params"]["max_order_quantities"], dtype=torch.float64, device=dev)
            h_act = [torch.round((a.to(torch.float64) + 1.0) * 0.5 * maxq).clamp_(0, 255).to(torch.uint8).cpu().pin_memory()
                     for a in actions[:n_host]]
            h_off = [dm.offsets.cpu().pin_memory() for dm in demand[:n_host]]
            h_lines = [dm.lines.cpu().pin_memory() for dm in demand[:n_host]]
            h_n = [dm.n_rounds for dm in demand[:n_host]]
            hr = HostRollout(env, max_rounds_per_step=max(h_n))
            seg_in = ([h_act[i] for i in idx], [h_off[i] for i in idx], [h_lines[i] for i in idx], [h_n[i] for i in idx])
            run = hr.run_lines
            h2d_seg = sum(h_act[i].numel() + h_off[i].numel() * 4 + h_n[i] * 64 for i in idx) + h_val.numel() * 4
            api = ("marlsc_env_rollout_host (pinned host uint8 order quantities + sparse demand lines in per env step, copies "
                   "overlapped with the step kernels, rewards out) + marlsc_gae (host values in, advantages/targets out)")
        else:
            h_act = [a.cpu().pin_memory() for a in actions[:n_host]]
            h_off = [dm.offsets.cpu().pin_memory() for dm in dense_demand[:n_host]]
            h_reg = [dm.region.cpu().pin_memory() for dm in dense_demand[:n_host]]
            h_qty = [dm.qty.cpu().pin_memory() for dm in dense_demand[:n_host]]
            h_n = [dm.n_orders for dm in dense_demand[:n_host]]
            hr = HostRollout(env, max(h_n))
            seg_in = ([h_act[i] for i in idx], [h_off[i] for i in idx], [h_reg[i] for i in idx], [h_qty[i] for i in idx],
                      [h_n[i] for i in idx])
            run = hr.run
            h2d_seg = sum(h_act[i].numel() * 4 + h_off[i].numel() * 4 + h_n[i] * (2 + S) for i in idx) + h_val.numel() * 4
            api = ("marlsc_env_rollout_host (pinned host actions+orders in per env step, copies overlapped with the "
                   "step kernels, rewards out) + marlsc_gae (host values in, advantages/targets out)")
        d2h_seg = SEG * E * W * 4 + 2 * h_adv.numel() * 4

        def host_segment(obs_host=None):
            if env.timestep + SEG > env.episode_length:
                env.reset(obs_out=obs_buf[0])
            run(*seg_in, h_rew, rewards, obs_host=obs_host)          # SEG steps: host actions+demand in, rewards out
            values.copy_(h_val, non_blocking=True)
            compute_gae(rewards, values, GAMMA, LAM, adv_out=adv, targets_out=tgt)
            h_adv.copy_(adv, non_blocking=True)
            h_tgt.copy_(tgt, non_blocking=True)
            torch.cuda.synchronize()

        def timed(fn, n):
            barrier()
            t0 = time.perf_counter()
            for _ in range(n):
                fn()
            barrier()
            dt = time.perf_counter() - t0
            if world > 1:
                tm = torch.tensor([dt], device=dev)
                dist.all_reduce(tm, op=dist.ReduceOp.MAX)
                dt = float(tm.item())
            return dt

        e2e_steps = max(1, min(args.steps, 3))
        host_segment()
        launches_e2e0 = L.marlsc_launch_count()
        dt = timed(host_segment, e2e_steps)
        e2e = dict(value=E * W * SEG * e2e_steps * world / dt, unit=UNIT, h2d_bytes_per_step=int(h2d_seg),
                   d2h_bytes_per_step=int(d2h_seg), ms_per_step=1e3 * dt / e2e_steps,
                   h2d_gbs_per_gpu=h2d_seg * e2e_steps / dt / 1e9, api=api, host_cpu_binding=numa,
                   segments=e2e_steps, gpu_launches=int(L.marlsc_launch_count() - launches_e2e0))
        # the same with every step's observations copied back to the host (what a host-side policy would need):
        # 4*W*obs_dim bytes per env step device->host, PCIe-bound by construction
        try:
            h_obs = [torch.empty((E, W, env.obs_dim)).pin_memory() for _ in range(2)]
            obs_list = [h_obs[i & 1] for i in range(SEG)]
            dt = timed(lambda: host_segment(obs_list), 1)
            e2e_obs = dict(value=E * W * SEG * world / dt, unit=UNIT, ms_per_step=1e3 * dt,
                           d2h_bytes_per_step=int(d2h_seg + SEG * E * W * env.obs_dim * 4),
                           d2h_gbs_per_gpu=(d2h_seg + SEG * E * W * env.obs_dim * 4) / dt / 1e9,
                           note="rewards AND observations [E,W,obs_dim] float32 copied to pinned host memory every env step")
            del h_obs
        except RuntimeError as ex:                                   # pinned allocation of 2 x 3.1 GB refused
            e2e_obs = dict(unavailable=str(ex)[:120])

    # ---- parity spot check on the benchmarked trajectory itself (outside every timed region) -------------------
    # 8 strided environments of this rank's batch, the first SEG steps of the replayed episode: the same demand and
    # actions through the CPU oracle, compared with what the timed kernels compute at this batch size
    spot = None
    if rank == 0 and not args.no_spot_check:
        from oracle.inventory_oracle import OracleEnv
        picks = sorted(set(int(x) for x in np.linspace(0, E - 1, 8)))
        env.reset(obs_out=obs_buf[0])
        orcs = {i: OracleEnv(env_dict) for i in picks}
        init = env.inventory[picks].cpu().numpy()
        for k, i in enumerate(picks):
            orcs[i].reset(init[k])
        ok, worst = True, 0.0
        for t in range(min(SEG, len(spot_dense))):
            env.step(actions[t], orders=demand[t], obs_out=obs_buf[0], rewards_out=rewards[0])
            dm = spot_dense[t]
            off = dm.offsets.cpu().numpy()
            inv_d, rew_d, obs_d, act_h = (env.inventory[picks].cpu().numpy(), rewards[0][picks].cpu().numpy(),
                                          obs_buf[0][picks].cpu().numpy(), actions[t][picks].cpu().numpy())
            for k, i in enumerate(picks):
                a, b = int(off[i]), int(off[i + 1])
                reg = dm.region[a:b].cpu().numpy()
                q = dm.qty[a * S:b * S].cpu().numpy().reshape(b - a, S)
                out = orcs[i].step(act_h[k], [(int(reg[j]), q[j].astype(float)) for j in range(b - a)])
                ok = ok and np.array_equal(inv_d[k], out["inventory"])
                err = max(float(np.max(np.abs(rew_d[k] - out["rewards"]) / (np.abs(out["rewards"]) + 1e-6))),
                          float(np.max(np.abs(obs_d[k] - out["obs_local"]) / (np.abs(out["obs_local"]) + 1.0))))
                worst = max(worst, err)
        ok = ok and worst < 1e-5
        spot = dict(envs=len(picks), steps=min(SEG, len(spot_dense)), ok=bool(ok), max_rel_err=worst,
                    what="inventory exact, rewards / observations relative error vs oracle/inventory_oracle.py on strided "
                         "environments of the timed batch (same demand, same actions)")
        env.reset(obs_out=obs_buf[0])

    # ---- everything on the device: demand sampler (K4) -> env step with the base-stock heuristic inside -----------
    on_device = None
    if args.workload == "large" and not args.no_e2e:
        from marlsc_b200.rollout import base_stock_levels
        env.enable_device_demand(seed=5 + rank)
        lvl = torch.from_numpy(base_stock_levels(env, args.z, serve="cheapest")).float().to(dev)
        act_buf = torch.empty((E, W, S), device=dev)

        def device_segment():
            for i in range(SEG):
                if env.timestep >= env.episode_length:
                    env.reset(obs_out=obs_buf[0])
                if compact:                            # K4 writes lines, K1a' evaluates the heuristic itself
                    env.step(None, obs_out=obs_buf[i & 1], rewards_out=rewards[i], base_stock_level=lvl)
                else:
                    env.base_stock_actions(lvl, out=act_buf)
                    env.step(act_buf, obs_out=obs_buf[i & 1], rewards_out=rewards[i])
            compute_gae(rewards, values, GAMMA, LAM, adv_out=adv, targets_out=tgt)

        env.reset(obs_out=obs_buf[0])
        for _ in range(2):
            device_segment()
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(3):
            device_segment()
        b.record()
        barrier()
        ms = a.elapsed_time(b)
        if world > 1:
            tmx = torch.tensor([ms], device=dev)
            dist.all_reduce(tmx, op=dist.ReduceOp.MAX)
            ms = float(tmx.item())
        on_device = dict(value=E * W * SEG * 3 * world / (ms * 1e-3), unit=UNIT, ms_per_step=ms / 3,
                         pipeline=("per env step: marlsc_demand_sample_lines (K4, writes the sparse lines the step consumes) -> "
                                   "marlsc_env_step with base_stock_level (the heuristic evaluated inside K1a'); no host input at all"
                                   if compact else
                                   "per env step: marlsc_policy_base_stock (K5) -> marlsc_demand_sample (K4) -> marlsc_env_step (K1); "
                                   "no host input at all"), demand_overflow=env.demand_overflowed())

    # ---- launch-bound shapes: the whole episode (reset + T steps) as one CUDA graph (rollout/graph.py) ------------------
    graphed = None
    if args.workload == "small" and rank == 0:
        from marlsc_b200.rollout import GraphedEpisode
        Tg = min(cfg.episode_length, len(actions), len(demand))
        ep = GraphedEpisode(env, torch.stack(actions[:Tg]), demand[:Tg])
        for _ in range(3):
            ep.replay()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(20):
            ep.replay()
        b.record()
        torch.cuda.synchronize()
        us = a.elapsed_time(b) * 1e3 / (20 * (Tg + 1))
        graphed = dict(us_per_env_step=us, value=E * W * Tg * 20 / (a.elapsed_time(b) * 1e-3), unit=UNIT, steps_per_graph=Tg,
                       note="reset + T steps of the replayed episode captured in one CUDA graph: no Python, ctypes or launch "
                            "latency between the kernels (the eager loop above pays ~100 us of host time per step)")
        env.reset(obs_out=obs_buf[0])

    # ---- the path's only collective: the learner's gradient all-reduce (multi-GPU runs) -----------------------------
    learner_ar = None
    if world > 1:
        learner_ar = learner_allreduce_record(dev, world, rank)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (K1) ------------------------------------------------------
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = json.load(open(peaks_path))["hbm_gbs"], "MEASURED_PEAKS.json hbm_gbs (measured)"
    else:
        peak, peak_src = 6650.0, "B200_PROFILING.md fallback"
    b_env = algorithmic_bytes_per_env_step(W, S, env.max_expected_lead_time, env.obs_dim, mean_orders,
                                           layout=env.layout, mean_lines=mean_lines)
    k1_avg_ms = statistics.mean(k1_ms)
    achieved = b_env * E / (k1_avg_ms * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "k1_traffic.json")
    if os.path.exists(tpath):
        try:
            tj = json.load(open(tpath))
            if tj.get("envs") == E and tj.get("workload") == args.workload and tj.get("layout", "wide") == env.layout:
                traffic = tj.get("dram_bytes_per_launch")
        except Exception:
            pass
    n_launch = len(per_launch[0]) if per_launch else 0
    split = n_launch == 4
    kernels = []
    if per_launch:
        ms = [statistics.mean(x[i] for x in per_launch) for i in range(n_launch)]
        WS, Lmax, od = W * S, env.max_expected_lead_time, env.obs_dim
        if split and compact:
            # the compact split step (csrc/env_compact.cu): bytes each launch needs per env step with the layout's element
            # sizes; inventory and the home-demand plane pass through HBM between the kernels
            parts = [("compact_place_kernel (K1a')", WS * (4 + 2 + 2 + Lmax + 1 + 2) + 4 * W * Lmax * S + 8 * W, "hbm"),
                     ("compact_alloc_kernel (K1b')", WS * (2 + 2) + 2 * mean_lines + 4 + 8 * W, "issue"),
                     ("compact_feature_kernel (K1c')", WS * (2 + 2 + 2) + 4 * W * (od - Lmax * S) + 20 * W + 1, "hbm"),
                     ("(K1d: rewards are written by K1c' with agent-scope rewards)", 0, "-")]
        elif split:
            # algorithmic bytes per env step of each launch (int32 state, fp32 obs), including what the split itself adds
            # (inventory and the home-demand plane pass through HBM between the kernels)
            parts = [("env_place_kernel (K1a)", 4 * WS * (2 * Lmax + 6), "hbm"),
                     ("env_alloc_warp_kernel (K1b)", 8 * WS + mean_orders * (S + 2) + 8 * W, "issue"),
                     ("env_feature_kernel (K1c)", 4 * WS * 7 + 4 * W * (od - Lmax * S) + 8 * W, "hbm"),
                     ("env_reward_kernel (K1d)", 20 * W + 1, "latency")]
        elif compact:
            parts = [("env_step_compact_kernel (fused K1, csrc/env_compact.cu)", b_env, "hbm")]
        else:
            parts = [("env_step_kernel (fused K1)", b_env, "hbm")]
        for (name, b, bound), t_ms in zip(parts, ms):
            if b == 0:
                continue
            kernels.append(dict(kernel=name, ms_per_launch=t_ms, bound=bound, algorithmic_bytes_per_env_step=b,
                                achieved=b * E / (t_ms * 1e-3) / 1e9, frac=b * E / (t_ms * 1e-3) / 1e9 / peak))
    roofline = dict(bound="hbm",
                    kernel=("env step K1 = compact_place + compact_alloc + compact_feature launches over the compact layout "
                            "(csrc/env_compact.cu)" if (split and compact)
                            else "env step K1 = place + allocate + features + rewards launches (csrc/env_split.cuh)" if split
                            else "env_step_compact_kernel (K1, one fused launch per env step, csrc/env_compact.cu)" if compact
                            else "env_step_kernel (K1)"),
                    achieved=achieved, peak=peak, unit="GB/s", frac=achieved / peak,
                    traffic=traffic, peak_source=peak_src, algorithmic_bytes_per_env_step=b_env, k1_ms_per_launch=k1_avg_ms,
                    k1_share_of_step=sum(k1_ms) / elapsed_ms, launches_per_env_step=n_launch, kernels=kernels,
                    note=("achieved = SURVEY 8d algorithmic bytes of one env step x envs / time of the step's launches; "
                          "kernels[] gives every launch with its own bytes (K1b is issue-bound, not HBM-bound)") if split else None)

    # K2 (GAE scan): reads rewards [T,N] + values [T+1,N], writes advantages + targets [T,N]; small working set
    # (L2 resident at this size), reported for completeness
    gae_bytes = 4.0 * E * W * (4 * SEG + 1)
    k2_avg = statistics.mean(k2_ms)
    roofline_gae = dict(bound="hbm", kernel="gae_kernel (K2)", achieved=gae_bytes / (k2_avg * 1e-3) / 1e9, peak=peak, unit="GB/s",
                        frac=gae_bytes / (k2_avg * 1e-3) / 1e9 / peak, k2_ms_per_launch=k2_avg, bytes_per_launch=gae_bytes,
                        note="%.0f MB per launch: fits the 126 MB L2 only partly" % (gae_bytes / 1e6))

    # ---- CPU baseline on a bounded sample, one core: the reference itself (oracle/_ref) when present, else the port ----
    cpu = None
    if not args.no_cpu:
        large = args.workload == "large"
        kind = reference_kind()
        if kind == "reference":
            n_env, seg = (24, SEG) if large else (128, 100)  # ~15 s of single-core work
        else:
            n_env, seg = (48, 100) if large else (256, 100)
        v, n, wall = cpu_port(env_dict, n_env, seg, 1, kind, args.z)
        src = ("the reference's own InventoryEnvironment (oracle/_ref, unmodified copy) under the base-stock heuristic"
               if kind == "reference" else "oracle/inventory_oracle.py")
        cpu = dict(value=v, unit=UNIT, cores=1, kind=kind,
                   sample=f"{n_env} envs x {seg} env steps + NumPy GAE, {src}, 1 process, {wall:.1f}s")
        if kind == "reference" and large:                   # the port's number as a second key (round-1 baseline)
            v2, _, wall2 = cpu_port(env_dict, 24, SEG, 1, "port")
            cpu["port_value"] = v2
            cpu["port_sample"] = f"24 envs x {SEG} env steps, oracle/inventory_oracle.py, 1 process, {wall2:.1f}s"

    line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=args.warmup,
                ms_per_step=elapsed_ms / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None,
                dtype=("uint16 stock+history, uint8 ring / fp32 obs+GAE / fp64 cost sums" if compact
                       else "int32 state / fp32 obs+GAE / fp64 cost sums"), data="synthetic",
                config=dict(cfg_desc, envs_per_gpu=E, segment_env_steps=SEG, gamma=GAMMA, lam=LAM, team_size=env.team_size,
                            mean_orders_per_env_step=mean_orders, layout=env.layout,
                            demand_format=(f"sparse lines, {mean_lines:.0f} per env step (2 bytes each)" if compact
                                           else "dense order rows (S + 2 bytes per order)"),
                            actions=(f"pre-sampled base-stock heuristic z={args.z} (recorded once, replayed)" if args.policy == "base_stock"
                                     else f"uniform{ACTION_RANGE}"),
                            l2="inputs larger than L2 (per-step state+obs far exceeds 126 MB)" if args.workload == "large"
                            else "small working set; L2 resident (launch-latency bound)",
                            distinct_input_steps=n_in),
                roofline=roofline, roofline_gae=roofline_gae, cpu_baseline=cpu, e2e=e2e, e2e_with_observations=e2e_obs,
                on_device_pipeline=on_device, cuda_graph_episode=graphed, parity_spot_check=spot, learner_allreduce=learner_ar, gpu_launches=int(launches), clocks=clk)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_rollout(args):
    """BASELINE configs[3]/[4]: full on-device rollout on the small env - PyTorch MLP policy/critic forward,
    fused env step, rollout buffer, GAE scan (+ one PPO minibatch step with the NCCL gradient all-reduce for
    MAPPO). Demand is drawn on the device (K4). A bench step = one rollout of T = episode length."""
    import torch
    import torch.distributed as dist

    import marlsc_b200  # noqa: F401
    from golden.scenarios import small_default
    from marlsc_b200 import _capi
    from marlsc_b200.config import environment_config_from_dict
    from marlsc_b200.envs import BatchedInventoryEnv
    from marlsc_b200.rollout import ActorCritic, PPOLearner, RolloutCollector

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    mappo = args.workload == "mappo"
    total = 1048576 if mappo else 262144
    E = args.envs or (total // world if mappo else total)          # MAPPO: 1M envs sharded; IPPO: 262k per GPU
    cfg = environment_config_from_dict(small_default())
    env = BatchedInventoryEnv(cfg, E, device=dev, host_samplers=False, device_demand=True, demand_seed=1 + rank,
                              env_meta=dict(include_warehouse_id=True))
    torch.manual_seed(0)
    pol = ActorCritic(env.obs_dim, 3, 2, actor_hidden=(256, 256) if mappo else (256,), critic_hidden=(64, 64) if mappo else (256,),
                      critic_obs_type="global" if mappo else "local", logstd_init=-1.2, logstd_floor=-3.5).to(dev)
    T = cfg.episode_length
    col = RolloutCollector(env, pol, T, gamma=GAMMA, lam=LAM, seed=rank)
    learner = PPOLearner(pol, lr=5e-4, grad_clip=5.0)
    L = _capi.lib()

    def step():
        ro = col.collect()
        if mappo:
            learner.minibatch_step(ro, slice(0, 1), slice(0, min(E, 65536)))   # one minibatch, grads all-reduced
        return ro

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(max(1, args.warmup)):
        step()
    barrier()
    l0 = L.marlsc_launch_count()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(args.steps):
        ro = step()
    b.record()
    barrier()
    ms = a.elapsed_time(b)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {name: (getattr(ro, name), 1) for name in
                                         ("obs", "actions", "logp", "rewards", "values", "advantages", "targets")}, E)
    if world > 1:
        tm = torch.tensor([ms], device=dev)
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        ms = float(tm.item())
    # the learner's minibatch step on its own (MAPPO): forward + K6 + backward with the bucketed all-reduce, max over ranks
    learner_rec = None
    if mappo:
        sl = (slice(0, 1), slice(0, min(E, 65536)))
        for _ in range(3):
            learner.minibatch_step(ro, *sl)
        barrier()
        la, lb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        bytes0 = learner.all_reduce_grads()
        la.record()
        for _ in range(10):
            learner.minibatch_step(ro, *sl)
        lb.record()
        barrier()
        lms = la.elapsed_time(lb) / 10
        if world > 1:
            tl = torch.tensor([lms], device=dev)
            dist.all_reduce(tl, op=dist.ReduceOp.MAX)
            lms = float(tl.item())
        learner_rec = dict(ms_minibatch_step=lms, minibatch_agent_samples=min(E, 65536) * 3,
                           allreduce_bytes_per_step=(learner.all_reduce_grads() - bytes0) // 10,
                           buckets=len(learner.buckets.buckets), ranks=world)
    # K1 at this shape: the library's own events around the step's launches
    k1 = None
    if rank == 0:
        env.set_timing(True)
        obs_t, times = col.obs[0], []
        env.reset(obs_out=obs_t)
        act0 = torch.zeros((E, 3, 2), device=dev)
        for _ in range(8):
            env.step(act0, obs_out=obs_t, rewards_out=col.rewards[0])
            times.append(sum(env.last_step_timing()))
        env.set_timing(False)
        k1_ms = statistics.mean(times[2:])
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        peak = json.load(open(peaks_path))["hbm_gbs"] if os.path.exists(peaks_path) else 6650.0
        b_env = algorithmic_bytes_per_env_step(3, 2, env.max_expected_lead_time, env.obs_dim, 0.0)   # demand drawn on the device
        k1 = dict(bound="hbm", kernel="env_step_kernel (K1, thread per environment)", k1_ms_per_launch=k1_ms,
                  algorithmic_bytes_per_env_step=b_env, achieved=b_env * E / (k1_ms * 1e-3) / 1e9, peak=peak, unit="GB/s",
                  frac=b_env * E / (k1_ms * 1e-3) / 1e9 / peak, traffic=None,
                  note="the step of this shape is one part of the rollout next to the MLP forwards (K7 for one-hidden-layer heads, library GEMMs otherwise) and the demand sampler")
    if rank == 0:
        value = E * 3 * T * args.steps * world / (ms * 1e-3)
        r_host = ro.rewards.mean().item()                       # device->host read of the rollout's result
        print(json.dumps(dict(
            roofline=k1, learner_allreduce=learner_rec,
            e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=4,
                     note="the whole rollout runs on the device (policy, demand, env, buffer, GAE); the only host traffic is "
                          "the 4-byte mean reward read back per rollout"),
            metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=args.warmup, ms_per_step=ms / args.steps,
            higher_is_better=True, scaling="strong" if mappo else "weak", vs_baseline=None, dtype="int32 state / fp32 obs, MLPs, GAE",
            data="synthetic", gpu_launches=int(L.marlsc_launch_count() - l0),
            config=dict(workload=("MAPPO centralised critic, 1,048,576 envs sharded (BASELINE configs[4])" if mappo else
                                  "IPPO rollout, 262,144 envs per GPU (BASELINE configs[3])"),
                        envs_per_gpu=E, horizon=T, env="env_symmetric_3WH2SKU + warehouse id", demand="device Poisson sampler (K4)",
                        policy="PyTorch MLP actor/critic forward every step", learner="one PPO minibatch, NCCL grad all-reduce" if mappo else None,
                        mean_reward=r_host))), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="large", choices=["large", "small", "ippo", "mappo"])
    ap.add_argument("--envs", type=int, default=0, help="envs per GPU (default: the workload's)")
    ap.add_argument("--team", type=int, default=0, help="threads per env (0 = auto)")
    ap.add_argument("--fused", action="store_true", help="keep the step in the single fused kernel (comparison)")
    ap.add_argument("--layout", default=None, choices=["wide", "compact"], help="state layout (default: compact where the config qualifies)")
    ap.add_argument("--distinct-steps", type=int, default=8, help="uniform policy: distinct pre-sampled input steps cycled through")
    ap.add_argument("--policy", default="base_stock", choices=["base_stock", "uniform"],
                    help="pre-sampled actions: recorded base-stock heuristic (default) or uniform noise")
    ap.add_argument("--z", type=float, default=2.0, help="base-stock safety factor")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-spot-check", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (at most 64 MB; a fixed sample of "
                         "environments when the batch is larger; with several GPUs, rank 0's environments)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU path (--impl ours)")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.workload in ("ippo", "mappo"):
        if args.impl == "reference":
            args.workload = "small"
            run_reference(args)
        else:
            run_rollout(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
