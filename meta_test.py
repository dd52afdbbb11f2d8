"""Meta-testing entry point: train fresh agents with a frozen LPG on levels of a test mode and report their returns,
raw and normalised by each level's optimal return (to_ued_b200/meta/meta_test.py).

    python meta_test.py --checkpoint runs/<run>/checkpoints/checkpoint_<step>.npz --env_mode mazes \\
        --num_agents 512 [--num_updates N] [--eval_interval 250] [--eval_workers 64] [--out result.json] [--seed 0]

The meta-test flags are parsed first; every other flag goes to the training parser (experiments/parse_args.py), so the
reference flags keep their meaning (``--env_mode``, ``--env_workers``, ``--train_rollout_len``, ``--seed``,
``--lifetime_conditioning``, ``--lpg_agent_target_coeff`` ...) and unknown flags still raise.

A checkpoint written by ``train.py --log`` is meta-tested at its LPG parameters; an ES checkpoint (``es_state/mean``
present) at its ES mean, which is the result of ES training (the ES path never refreshes ``params``).  Without
``--checkpoint`` the freshly initialised LPG of ``--seed`` is meta-tested: the untrained baseline.  Keys:
``lpg_rng, test_rng = split(PRNGKey(seed), 2)``; ``lpg_rng`` initialises that baseline LPG, ``test_rng`` is the key
of ``meta_test``.  The result is one JSON document on stdout, or in ``--out``.  Single GPU."""
import argparse
import json
import os
import sys

import numpy as np


def parse_meta_test_args(cmd_args):
    """-> (meta-test flags, training args).  Raises ValueError on unknown flags (parse_args)."""
    p = argparse.ArgumentParser(description="Meta-test a trained LPG", allow_abbrev=False)
    p.add_argument("--checkpoint", type=str, default=None, help="checkpoint_<step>.npz written by train.py --log")
    p.add_argument("--num_agents", type=int, default=512, help="Number of test agents (one level each)")
    p.add_argument("--num_updates", type=int, default=None,
                   help="Agent updates per agent (default: the mode's maximum lifetime)")
    p.add_argument("--eval_interval", type=int, default=250, help="Agent updates between evaluations")
    p.add_argument("--eval_workers", type=int, default=64, help="Evaluation workers per agent")
    p.add_argument("--out", type=str, default=None, help="Write the JSON result here instead of stdout")
    meta, rest = p.parse_known_args(cmd_args)
    from to_ued_b200.experiments.parse_args import parse_args
    return meta, parse_args(rest)


def load_lpg_params(path: str, lifetime_conditioning: bool) -> np.ndarray:
    """Flat f32 LPG parameters of a checkpoint: the ES mean of an ES checkpoint, ``params`` otherwise.  Raises
    ValueError when the count does not match the model that ``lifetime_conditioning`` selects (host only)."""
    from to_ued_b200.models.lpg import LPG
    with np.load(path) as z:
        key = "es_state/mean" if "es_state/mean" in z.files else "params"
        vec = np.asarray(z[key], np.float32).reshape(-1)
    expected = LPG(lifetime_conditioning=bool(lifetime_conditioning)).size
    if vec.size != expected:
        raise ValueError(f"{path}: '{key}' holds {vec.size} LPG parameters, but the model selected by "
                         f"--lifetime_conditioning={bool(lifetime_conditioning)} has {expected}")
    return vec


def run_meta_test(meta, args) -> dict:
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        raise RuntimeError("meta_test.py runs on a single GPU; multi-GPU sharding of the test agents is not implemented")
    lpg = None
    if meta.checkpoint is not None:
        lpg = load_lpg_params(meta.checkpoint, args.lifetime_conditioning)      # before any GPU work
    from to_ued_b200.util import prng
    from to_ued_b200.environments.level_sampler import LevelSampler
    from to_ued_b200.meta.meta_test import meta_test, summarize
    from to_ued_b200.models.lpg import LPG
    lpg_rng, test_rng = prng.split(prng.PRNGKey(args.seed), 2)
    if lpg is None:
        lpg = LPG(lifetime_conditioning=args.lifetime_conditioning).init(lpg_rng, device="cpu").numpy()
    sampler = LevelSampler(args)
    curve, points, optimal, agents = meta_test(
        test_rng, lpg, args.lifetime_conditioning, sampler, meta.num_agents, meta.num_updates, meta.eval_interval,
        meta.eval_workers, agent_target_coeff=args.lpg_agent_target_coeff)
    config = {"checkpoint": meta.checkpoint, "env_name": args.env_name, "env_mode": args.env_mode,
              "num_agents": meta.num_agents, "num_updates": int(points[-1]), "eval_interval": meta.eval_interval,
              "eval_workers": meta.eval_workers, "env_workers": args.env_workers,
              "train_rollout_len": args.train_rollout_len, "max_rollout_len": sampler.max_rollout_len,
              "lifetime_conditioning": bool(args.lifetime_conditioning),
              "lpg_agent_target_coeff": args.lpg_agent_target_coeff, "seed": args.seed}
    return {"config": config, **summarize(curve, points, optimal, agents.level.lifetime)}


def main(cmd_args=sys.argv[1:]):
    meta, args = parse_meta_test_args(cmd_args)
    result = run_meta_test(meta, args)
    text = json.dumps(result)
    if meta.out:
        with open(meta.out, "w") as f:
            f.write(text + "\n")
    else:
        print(text)
    return result


if __name__ == "__main__":
    main()
