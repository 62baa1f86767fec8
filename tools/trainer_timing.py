#!/usr/bin/env python3
"""Where the time of a training iteration goes: collect, learner update and evaluation of ``marlsc_b200.rollout.Trainer``.

    python tools/trainer_timing.py [--envs 4096 262144] [--horizon 25] [--iterations 3] [--per-gpu] [--out FILE]
    torchrun --nproc-per-node N tools/trainer_timing.py ...      (data-parallel: --envs are global, or per GPU with --per-gpu)

IPPO (parameter sharing, local critic) and MAPPO (global critic) on the small config (3 warehouses x 2 SKUs), device
demand, the hyper-parameters of the reference's IPPO / MAPPO configs (256-unit heads, meanstd_custom, num_epochs 20,
num_minibatches 10, lr 5e-4), one evaluation episode of min(envs, 1024) environments per iteration. Each phase is host-clock time
ending in a device synchronise, as the trainer logs it; the first iteration is reported apart (module loads, library
heuristics) and the rest as medians. Prints one JSON object with the device name and its power limit. Under torchrun the
phases are rank 0's (each ends in a device synchronise, and the collectives inside the collect and the update hold the ranks
together), and every row records whether the ranks' parameters were bit-identical at the end of the run.
"""
from __future__ import annotations

import argparse
import copy
import json
import os
import statistics
import sys
import tempfile

ALGO = dict(
    shared=dict(num_iterations=3, checkpoint_freq=3, batch_size=8000, num_epochs=20, num_minibatches=10, learning_rate=5e-4),
    algorithm_specific=dict(use_gae=True, lam=0.95, gamma=0.99, clip_param=0.1, vf_clip_param=800.0, logstd_init=-1.15,
                            logstd_floor=-3.5, obs_normalization="meanstd_custom", parameter_sharing=True,
                            networks=dict(shared_layers=None, use_mu_sigma_head=False,
                                          actor=dict(type="mlp", config=dict(hidden_sizes=[256], activation="relu")),
                                          critic=dict(type="mlp", config=dict(hidden_sizes=[256], activation="relu")))))

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--envs", type=int, nargs="+", default=[4096, 262144])
    ap.add_argument("--horizon", type=int, default=25)
    ap.add_argument("--iterations", type=int, default=3)
    ap.add_argument("--per-gpu", action="store_true", help="--envs per GPU (weak scaling) instead of global")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("trainer_timing.py measures on a CUDA device; none is visible")
    import torch.distributed as dist
    from train import init_distributed
    rank, world = init_distributed()
    try:
        _measure(args, rank, world)
    finally:
        if world > 1:
            dist.destroy_process_group()


def _params_identical(policy, world: int) -> bool:
    """Whether every rank holds the same parameters, bit for bit (true with one rank)."""
    import torch
    import torch.distributed as dist
    if world == 1:
        return True
    flat = torch.cat([p.detach().reshape(-1) for p in policy.parameters()])
    lo, hi = flat.clone(), flat.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    return bool(torch.equal(lo, hi))


def _measure(args, rank: int, world: int) -> None:
    import torch
    import marlsc_b200  # noqa: F401
    from cppo_timing import _gpu
    from golden.scenarios import small_default
    from marlsc_b200.config import algorithm_config_from_dict, environment_config_from_dict
    from marlsc_b200.rollout import Trainer
    env_cfg = environment_config_from_dict(small_default())
    res = dict(gpu=_gpu(), ranks=world, config="small_default (3 WH x 2 SKU)", horizon=args.horizon,
               iterations=args.iterations, runs=[])
    for name in ("ippo", "mappo"):
        d = dict(copy.deepcopy(ALGO), name=name)
        d["shared"].update(num_iterations=args.iterations, checkpoint_freq=args.iterations)
        algo = algorithm_config_from_dict(d)
        for E in args.envs:
            E = E * world if args.per_gpu else E
            with tempfile.TemporaryDirectory() as out:
                # every rank writes its checkpoint shards into the same directory
                box = [out]
                if world > 1:
                    torch.distributed.broadcast_object_list(box, src=0)
                tr = Trainer(env_cfg, algo, E, box[0], horizon=args.horizon)
                lines = []
                tr.run(log=lines.append)
                same = _params_identical(tr.policy, world)
                if world > 1:
                    torch.distributed.barrier()          # rank 0 removes the directory after every rank is done with it
            rest = lines[1:] or lines
            med = {k: statistics.median(ln[k] for ln in rest) for k in ("collect_s", "update_s", "eval_s")}
            total = sum(med.values())
            row = dict(algorithm=name, ranks=world, envs=E, envs_per_rank=E // world, env_steps_per_iteration=E * args.horizon,
                       minibatches=lines[0]["learner"]["minibatches"], first_iteration_s={k: round(lines[0][k], 4) for k in med},
                       median_s={k: round(v, 4) for k, v in med.items()},
                       share={k: round(v / total, 4) for k, v in med.items()},
                       env_steps_per_s=round(E * args.horizon / total, 1), params_identical_across_ranks=same)
            res["runs"].append(row)
            if rank == 0:
                print(json.dumps(row), flush=True)
            del tr
            torch.cuda.empty_cache()
    if rank != 0:
        return
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
