#!/usr/bin/env python3
"""Train IPPO, MAPPO or CPPO on one GPU from the reference's YAML files.

    python tools/train.py --env-config ENV.yaml --algo-config ALGO.yaml --num-envs 4096 --out runs/x
                          [--seed 0] [--horizon T] [--eval-envs N] [--resume CHECKPOINT]

One iteration collects --num-envs x horizon env steps (horizon defaults to batch_size / num-envs) and runs one PPO update;
see marlsc_b200.rollout.Trainer. Writes training_metrics.jsonl and checkpoint_*.pt under --out and prints, per iteration,
the phase times (host clock, each ending in a device synchronise) after a header with the card name and power limit.
With --resume the run continues from a checkpoint (--env-config / --algo-config / --num-envs are then taken from it).
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _gpu() -> str:
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30).stdout.strip().splitlines()
        power = q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return f"{name}, power limit {power}"


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--env-config")
    ap.add_argument("--algo-config")
    ap.add_argument("--num-envs", type=int)
    ap.add_argument("--out", required=True)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--horizon", type=int, default=None)
    ap.add_argument("--eval-envs", type=int, default=None)
    ap.add_argument("--resume", default=None, help="checkpoint to continue from")
    args = ap.parse_args(argv)
    if args.resume is None and (args.env_config is None or args.algo_config is None or args.num_envs is None):
        ap.error("--env-config, --algo-config and --num-envs are required unless --resume is given")
    import torch
    if not torch.cuda.is_available():
        sys.exit("train.py trains on a CUDA device; none is visible")
    import marlsc_b200  # noqa: F401
    from marlsc_b200.config import load_algorithm_config, load_environment_config
    from marlsc_b200.rollout import Trainer
    if args.resume is not None:
        tr = Trainer.resume(args.resume, out_dir=args.out)
    else:
        tr = Trainer(load_environment_config(args.env_config), load_algorithm_config(args.algo_config), args.num_envs, args.out,
                     seed=args.seed, horizon=args.horizon, num_eval_envs=args.eval_envs)
    print(f"# {_gpu()}; {tr.algo_config.name}, {tr.num_envs} envs x horizon {tr.horizon}, "
          f"{tr.algo_config.shared.num_epochs} epochs x {tr.algo_config.shared.num_minibatches} minibatches", flush=True)

    def log(line) -> None:
        ev = line.get("eval")
        cost = f"  eval total_cost {ev['total_cost']['mean']:.2f}" if ev else ""
        print(f"iter {line['iteration']:5d}  env_steps {line['env_steps']}  lr {line['lr']:.3g}  reward {line['reward_mean']:.4f}  "
              f"collect {line['collect_s']:.3f}s  update {line['update_s']:.3f}s  eval {line['eval_s']:.3f}s{cost}", flush=True)

    tr.run(log=log)
    return 0


if __name__ == "__main__":
    sys.exit(main())
