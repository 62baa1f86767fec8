#!/usr/bin/env python3
"""Where the time of a CPPO rollout step goes on the GPU, and whether the head kernels beat the library GEMMs.

    python tools/cppo_timing.py [--envs 262144] [--reps 20] [--repeats 5] [--out FILE]

For the small config (3 warehouses x 2 SKUs: global state 33 floats, joint action 6) and a 3 x 5 variant of it (78 and 15),
with device-drawn demand and a CentralizedActorCritic whose heads have one hidden layer of 256 ([W*D -> 256 -> W*S] /
[W*D -> 256 -> 1]) or two ([W*D -> 256 -> 256 -> ...]), the ms per rollout step of
  * the actor and the critic forward: the routed rollout path (K7 for one hidden layer; library GEMMs + K7b for two), the
    layer-by-layer path (library GEMMs + K7b, what a head not routed to K7 runs) and the plain nn.Sequential (library
    GEMMs, bias and ReLU as separate passes), alternated --repeats times in this process, each the mean over --reps calls
    between CUDA events; the median is reported, and the largest difference from the nn.Sequential's output;
  * the env step (--reps steps, resets outside the timed window) and GAE over a 100-step rollout of the E environments,
    per step.
Inputs: a fresh observation batch of E x W*D floats (34 / 82 MB at 262,144 environments), re-read every call. Prints one
JSON object with the device name and its power limit.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def _gpu() -> dict:
    import torch
    out = dict(device=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()
        out["power_limit_and_max_sm_clock"] = q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        out["power_limit_and_max_sm_clock"] = "unknown"
    return out


def _config(n_skus: int):
    """small_default, or the same network with every per-SKU list widened to n_skus."""
    from golden.scenarios import small_default
    from marlsc_b200.config import environment_config_from_dict
    d = small_default()
    if n_skus != 2:
        S, c = n_skus, d["cost_structure"]
        d["n_skus"] = S
        d["action_space"]["params"]["max_order_quantities"] = [40] * S
        d["initial_inventory"]["params"]["values"] = [[60] * S for _ in range(3)]
        c["penalty_cost"], c["sku_weights"] = [5] * S, [1.0] * S
        c["shipment_cost"]["inbound_fixed"] = [[0] * S for _ in range(3)]
        c["shipment_cost"]["inbound_variable"] = [[1.0] * S for _ in range(3)]
        p = d["components"]
        p["demand_sampler"]["params"]["lambda_quantity"] = [[5] * S for _ in range(3)]
        p["lead_time_sampler"]["params"]["expected_lead_times"] = [[3] * S for _ in range(3)]
    return environment_config_from_dict(d)


def _time(fn, reps: int) -> float:
    import torch
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def _heads(pol, x, reps: int, repeats: int) -> dict:
    """For the actor and the critic, alternated: the rollout forward as routed (``routed_ms``), the layer-by-layer path a
    head takes when it is not routed to K7 (library GEMM + K7b, ``gemm_k7b_ms``; for a deeper head this is the routed path)
    and the plain nn.Sequential (``sequential_ms``)."""
    import torch
    from marlsc_b200.rollout.policy import _central_layers
    out = {}
    flat = x.reshape(x.shape[0], -1)
    for name, seq in (("actor", pol.actor), ("critic", pol.critic)):
        arms = dict(routed_ms=lambda: pol._head(seq, x), gemm_k7b_ms=lambda: _central_layers(list(seq), flat),
                    sequential_ms=lambda: seq(flat))
        with torch.no_grad():
            want = seq(flat)
            diff = {k.replace("_ms", "_max_abs_diff"): float((f() - want).abs().max()) for k, f in arms.items() if k != "sequential_ms"}
            for f in arms.values():                     # warm-up: module loads, library heuristics
                _time(f, 3)
            times = {k: [] for k in arms}
            for _ in range(repeats):
                for k, f in arms.items():
                    times[k].append(_time(f, reps))
        out[name] = dict({k: round(statistics.median(v), 4) for k, v in times.items()}, **diff)
    return out


def _env_step_ms(env, reps: int) -> float:
    import torch
    act = torch.zeros((env.num_envs, env.n_warehouses, env.n_skus), device=env.device)
    env.reset()
    for _ in range(3):
        env.step(act)
    total, done = 0.0, 0
    while done < reps:
        n = min(reps - done, env.episode_length - env.timestep)
        if n == 0:
            env.reset()
            continue
        total += _time(lambda: env.step(act), n) * n
        done += n
    return total / reps


def _gae_ms(E: int, reps: int) -> float:
    import torch
    from marlsc_b200.rollout import compute_gae
    T = 100
    r = torch.randn((T, E), device="cuda:0")
    v = torch.randn((T + 1, E), device="cuda:0")
    adv, tgt = torch.empty_like(r), torch.empty_like(r)
    compute_gae(r, v, 0.99, 0.95, adv_out=adv, targets_out=tgt)
    return _time(lambda: compute_gae(r, v, 0.99, 0.95, adv_out=adv, targets_out=tgt), reps) / T


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--envs", type=int, default=262144)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("cppo_timing.py measures on a CUDA device; none is visible")
    import marlsc_b200  # noqa: F401
    from marlsc_b200.envs import BatchedInventoryEnv
    from marlsc_b200.rollout import CentralizedActorCritic
    torch.backends.cuda.matmul.allow_tf32 = False
    res = dict(gpu=_gpu(), envs=args.envs, reps=args.reps, repeats=args.repeats, configs={})
    for S in (2, 5):
        cfg = _config(S)
        env = BatchedInventoryEnv(cfg, args.envs, device="cuda:0", host_samplers=False, device_demand=True, demand_seed=1, seed=1)
        W, D = env.n_warehouses, env.obs_dim
        torch.manual_seed(0)
        x = env.reset().clone()
        row = dict(global_obs=W * D, joint_action=W * S, env_step_ms=round(_env_step_ms(env, args.reps), 4),
                   gae_ms_per_step=round(_gae_ms(args.envs, args.reps), 4), heads={})
        for hidden in ((256,), (256, 256)):
            pol = CentralizedActorCritic(D, W, S, actor_hidden=hidden, critic_hidden=hidden).cuda()
            row["heads"]["x".join(map(str, hidden))] = _heads(pol, x, args.reps, args.repeats)
            del pol
        res["configs"][f"{W}x{S}"] = row
        env.close()
        del env, x
        torch.cuda.empty_cache()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
