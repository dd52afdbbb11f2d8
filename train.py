"""LPG / GROOVE meta-training entry point (reference train.py:14-82), B200-native.

Same flags as the reference (experiments/parse_args.py).  Differences: the outer loop is a Python
loop over meta-steps that enqueues CUDA work (the reference jit-compiles one lax.scan); --train_steps
is honoured (the reference hard-codes 10, Q1); with torchrun, agents are sharded over ranks."""
import os
import sys

import numpy as np
import torch

from to_ued_b200.util import prng
from to_ued_b200.environments.level_sampler import LevelSampler
from to_ued_b200.experiments.parse_args import parse_args
from to_ued_b200.meta.meta import create_lpg_train_state, make_lpg_train_step


def _init_distributed():
    if "RANK" in os.environ and int(os.environ.get("WORLD_SIZE", "1")) > 1:
        import torch.distributed as dist
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
        dist.init_process_group("nccl")
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def make_train(args, rank=0, world=1):
    if args.num_agents % world != 0:
        raise ValueError(f"num_agents ({args.num_agents}) must be divisible by the number of GPUs ({world})")
    n_local = args.num_agents // world

    def _train_fn(rng):
        # --- Initialize LPG and level sampler ---  (train.py:17-21)
        rng, lpg_rng, buffer_rng = prng.split(rng, 3)
        train_state = create_lpg_train_state(lpg_rng, args)
        level_sampler = LevelSampler(args)
        level_buffer = level_sampler.initialize_buffer(buffer_rng)
        # --- Initialize agents and value critics --- (the sampler derives the keys of the global batch and creates
        #     this rank's slice; the level buffer is replicated and stays identical on every rank)
        require_value_critic = not args.use_es
        rng, _rng = prng.split(rng, 2)
        level_buffer, agent_states, value_critic_states = level_sampler.initial_sample(
            _rng, level_buffer, args.num_agents, require_value_critic)
        assert len(agent_states.level) == n_local
        lpg_train_step_fn = make_lpg_train_step(args, level_sampler)
        history = []
        for _ in range(args.train_steps):          # Q1: the reference runs a fixed 10 steps
            rng, _rng = prng.split(rng, 2)
            train_state, agent_states, value_critic_states, metrics = lpg_train_step_fn(
                rng=_rng, lpg_train_state=train_state, agent_states=agent_states,
                value_critic_states=value_critic_states)
            rng, _rng = prng.split(rng, 2)
            level_buffer, agent_states, value_critic_states = level_sampler.sample(
                _rng, level_buffer, agent_states, value_critic_states)
            history.append(metrics)
        _GRAPHED.append(lpg_train_step_fn)
        return history, train_state, level_buffer

    return _train_fn


_GRAPHED = []      # step functions created by make_train (released before the process group is torn down)


def _shard(agents, vcs, rank, n_local):
    """Rank ``rank``'s slice [rank * n_local, (rank + 1) * n_local) of a batch of agents (utility for callers that
    build the global batch themselves; ``LevelSampler.initial_sample`` creates the local slice directly)."""
    from to_ued_b200.util.data import Level
    from to_ued_b200.environments.gridworld.gridworld import EnvState
    sl = slice(rank * n_local, (rank + 1) * n_local)
    lv = agents.level
    level = Level(lv.env_params[sl], lv.lifetime[sl], lv.buffer_id[sl], lv.packed[sl].contiguous())
    a, c = agents.actor_state, agents.critic_state
    out = agents.replace(actor_state=a.replace(params=a.params[sl].contiguous(), step=a.step[sl].contiguous()),
                         critic_state=c.replace(params=c.params[sl].contiguous(), step=c.step[sl].contiguous()),
                         level=level, env_obs=agents.env_obs[sl].contiguous(),
                         env_state=EnvState(agents.env_state.packed[sl].contiguous(), agents.env_state.max_n_objs),
                         host_step=None if agents.host_step is None else agents.host_step[sl])
    if vcs is not None:
        vcs = vcs.replace(params=vcs.params[sl].contiguous(), step=vcs.step[sl].contiguous())
    return out, vcs


def _to_float(m):
    from to_ued_b200.experiments.logging import to_host
    return to_host(m)


def run_training_experiment(args):
    rank, world = _init_distributed()
    if args.log and rank == 0:                       # train.py:63-64 (local run directory instead of WandB)
        from to_ued_b200.experiments.logging import init_logger
        print(f"[to_ued_b200] --log: run directory {init_logger(args)}")
    train_fn = make_train(args, rank, world)
    metrics, train_state, level_buffer = train_fn(prng.PRNGKey(args.seed))
    torch.cuda.synchronize()
    from to_ued_b200.meta.train import reverse_status
    status = int(reverse_status())
    if status:
        print(f"[to_ued_b200] warning (rank {rank}): the tensor-core reverse pass reported status {status:#x} "
              "(1: inf / NaN cotangent, 2: fp16 operand saturated or not finite); some meta-gradients may be wrong. "
              "TOUED_GRU_PRECISION=fp32 runs the exact-fp32 reverse pass.", file=sys.stderr)
    if rank == 0:
        print([_to_float(m) for m in metrics])
        if args.log:                                 # train.py:68-69
            from to_ued_b200.experiments.logging import log_results
            print("[to_ued_b200] checkpoints:", log_results(args, metrics, train_state, level_buffer))
    if world > 1:
        from to_ued_b200.util import dist as udist
        udist.shutdown(*_GRAPHED)
    return metrics, train_state, level_buffer


def main(cmd_args=sys.argv[1:]):
    args = parse_args(cmd_args)
    return run_training_experiment(args)


if __name__ == "__main__":
    main()
