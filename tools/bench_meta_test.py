#!/usr/bin/env python
"""Meta-testing measurements (DESIGN.md section 10), printed as one JSON line:

  * toued_optimal_return on 512 levels of all_shortlife, tabular and mazes at the mode's max_rollout_len: mean time of
    one call over repeated calls (CUDA events, after a warm-up call) and levels/s;
  * the wall time and env-steps/s of a 512-agent all_shortlife meta-test (250 updates, eval_interval 25) and of a
    512-agent mazes meta-test (2500 updates, eval_interval 250), host clock around meta_test() ended by a device
    synchronise; env-steps are the training and evaluation rollout steps the run enqueued (_lib.ENV_STEPS).

The card's name and power limit come from a read-only nvidia-smi query in the same run.

    python tools/bench_meta_test.py [--agents 512] [--reps 20]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from to_ued_b200 import _lib  # noqa: E402
from to_ued_b200.util import prng  # noqa: E402
from to_ued_b200.experiments.parse_args import parse_args  # noqa: E402


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [s.strip() for s in out.split(",")]
    return {"gpu": name, "power_limit": power}


def time_optimal_return(mode, n, reps):
    from to_ued_b200.environments.gridworld import configs as grid_conf
    from to_ued_b200.environments.gridworld.gridworld import GridWorld
    from to_ued_b200.environments.gridworld.levelgen import generate_levels
    kw, horizon = grid_conf.get_env_spec(mode)
    env = GridWorld(**kw)
    packed = generate_levels(prng.split(prng.PRNGKey(1), n), mode, device="cuda")
    opt = env.optimal_return(packed, horizon)                  # warm-up (module load, shared-memory attribute)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        env.optimal_return(packed, horizon)
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / reps
    return {"mode": mode, "levels": n, "horizon": horizon, "ms": round(ms, 4), "levels_per_s": round(n / ms * 1e3, 1),
            "mean_optimal": float(opt.mean())}


def time_meta_test(mode, n, num_updates, eval_interval, eval_workers=64):
    from to_ued_b200.environments.level_sampler import LevelSampler
    from to_ued_b200.meta.meta_test import meta_test
    from to_ued_b200.models.lpg import LPG
    args = parse_args(["--env_mode", mode])
    sampler = LevelSampler(args)
    lpg_rng, rng = prng.split(prng.PRNGKey(0), 2)
    lpg = LPG().init(lpg_rng, device="cuda")
    meta_test(rng, lpg, False, sampler, n, 2, 1, eval_workers)             # warm-up: every kernel once
    torch.cuda.synchronize()
    _lib.reset_counters()
    t0 = time.perf_counter()
    curve, pts, opt, _ = meta_test(rng, lpg, False, sampler, n, num_updates, eval_interval, eval_workers)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    steps = int(_lib.ENV_STEPS[0])
    keep = opt > 1e-6
    return {"mode": mode, "agents": n, "num_updates": num_updates, "eval_interval": eval_interval,
            "eval_workers": eval_workers, "env_workers": args.env_workers, "wall_s": round(wall, 3), "env_steps": steps,
            "env_steps_per_s": round(steps / wall, 1), "final_mean_return": float(curve[-1].mean()),
            "final_mean_normalised": float((curve[-1][keep] / opt[keep]).mean()) if keep.any() else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--agents", type=int, default=512)
    ap.add_argument("--reps", type=int, default=20)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "bench_meta_test.py needs a CUDA device"
    out = dict(gpu_info())
    out["optimal_return"] = [time_optimal_return(m, a.agents, a.reps) for m in ("all_shortlife", "tabular", "mazes")]
    out["meta_test"] = [time_meta_test("all_shortlife", a.agents, 250, 25), time_meta_test("mazes", a.agents, 2500, 250)]
    print(json.dumps(out))


if __name__ == "__main__":
    main()
