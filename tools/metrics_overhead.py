#!/usr/bin/env python3
"""What per-episode metrics (BatchedInventoryEnv(episode_metrics=True)) cost on the GPU.

    python tools/metrics_overhead.py [--steps 200] [--repeats 5] [--eval-envs 65536] [--eval-episodes 100] [--out FILE]

Step time with metrics off and on, measured with CUDA events over --steps steps after a warm-up, the two arms alternated
--repeats times in one process (median reported):
  * the large config (10 warehouses x 100 SKUs x 50 regions) at 65,536 environments, COMPACT layout, device-drawn demand
    lines (the draw is inside the timed step) and a fixed random action tensor;
  * the small config (3 x 2 x 3) at 4,096 and 262,144 environments, WIDE layout, device-drawn demand. With metrics on, a
    WIDE step runs the generic kernel with its diagnostic outputs and one fold launch.
Then a base-stock (z = 2) evaluation of the large config through rollout.evaluate: --eval-episodes episodes of
--eval-envs environments, in environment-episodes per second (host clock around the whole run, ended by a device
synchronise). Prints one JSON object with the device name and its power limit.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

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


def _make(cfg, E, metrics, layout=None):
    from marlsc_b200.envs import BatchedInventoryEnv
    return BatchedInventoryEnv(cfg, E, device="cuda:0", host_samplers=False, device_demand=True, demand_seed=1, seed=1,
                               layout=layout, episode_metrics=metrics)


def _time_steps(env, act, steps) -> float:
    """ms per step over `steps` steps (resets in between are outside the timed window)."""
    import torch
    total, done_steps = 0.0, 0
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    while done_steps < steps:
        n = min(steps - done_steps, env.episode_length - env.timestep)
        if n == 0:
            env.reset()
            continue
        start.record()
        for _ in range(n):
            env.step(act)
        stop.record()
        stop.synchronize()
        total += start.elapsed_time(stop)
        done_steps += n
    return total / steps


def step_overhead(cfg, E, layout, steps, repeats) -> dict:
    import torch
    envs = {m: _make(cfg, E, m, layout) for m in (False, True)}
    W, S = envs[False].n_warehouses, envs[False].n_skus
    act = torch.rand((E, W, S), device="cuda:0", generator=torch.Generator(device="cuda:0").manual_seed(0)) * 2 - 1
    for env in envs.values():
        env.reset()
        _time_steps(env, act, min(steps, 20))           # warm-up: module loads, line buffers, first launches
    times = {False: [], True: []}
    for _ in range(repeats):
        for m in (False, True):
            times[m].append(_time_steps(envs[m], act, steps))
    res = dict(num_envs=E, layout=envs[False].layout, steps=steps, repeats=repeats,
               off_ms=statistics.median(times[False]), on_ms=statistics.median(times[True]),
               off_ms_all=times[False], on_ms_all=times[True])
    res["ratio"] = res["on_ms"] / res["off_ms"]
    for env in envs.values():
        env.close()
    return res


def evaluation_rate(cfg, E, episodes) -> dict:
    import torch
    from marlsc_b200.rollout import base_stock_levels, evaluate
    env = _make(cfg, E, True)
    level = base_stock_levels(env, 2.0)
    evaluate(env, level, 1)                               # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = evaluate(env, level, episodes)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    s = res.summary()
    out = dict(num_envs=E, layout=env.layout, episodes=episodes, episode_length=env.episode_length, seconds=dt,
               env_episodes_per_s=E * episodes / dt, mean_episode_return=s["episode_return"]["mean"],
               mean_fill_rate=s["fill_rate"]["mean"], mean_total_cost=s["total_cost"]["mean"])
    env.close()
    return out


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--eval-envs", type=int, default=65536)
    ap.add_argument("--eval-episodes", type=int, default=100)
    ap.add_argument("--out", default=None, help="also write the JSON here")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("metrics_overhead.py measures on a CUDA device; none is available")
    import __graft_entry__  # noqa: F401  (puts the package on the path)
    from golden.scenarios import large_network, small_default
    from marlsc_b200.config import environment_config_from_dict
    large = environment_config_from_dict(dict(large_network(), allow_region_mismatch=True))
    small = environment_config_from_dict(small_default())
    res = dict(gpu=_gpu(), step=[step_overhead(large, 65536, None, a.steps, a.repeats),
                                 step_overhead(small, 4096, None, a.steps, a.repeats),
                                 step_overhead(small, 262144, None, a.steps, a.repeats)],
               evaluation=evaluation_rate(large, a.eval_envs, a.eval_episodes))
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
