"""Meta-testing: train fresh tabular agents from scratch with a frozen LPG on held-out levels and score them against the
optimal return of each level (the evaluation protocol of LPG / GROOVE; the reference announces a meta-testing script
but has none).

``meta_test`` samples ``num_agents`` levels from the test mode's generator, creates one agent per level, trains every
agent with the frozen LPG for ``num_updates`` agent updates (default: the mode's maximum lifetime; on ``*randlife``
modes the lifetime mask of the agent update turns updates past a level's lifetime into no-ops) and evaluates the
agents at update 0, after every ``eval_interval`` updates and at the end.  Each level's return is normalised by
``GridWorld.optimal_return`` over the same horizon (the mode's ``max_rollout_len``, as in ``eval_agent``).

Key plumbing (fixed; the tests rely on it)::

    rng = the key passed to meta_test (meta_test.py at the repository root passes split(PRNGKey(seed), 2)[1];
          split(PRNGKey(seed), 2)[0] initialises the LPG when no checkpoint is given)
    level_rng, agent_rng, train_rng, eval_rng = split(rng, 4)
    levels        = level_sampler._sample_random_levels(level_rng, num_agents)     (one key per level: split(level_rng, N))
    agents        = level_sampler._create_agent(split(agent_rng, N), levels)
    train key i   = split(train_rng, N)[i]; update u of agent i uses link u of its ``rng, _rng = split(rng)`` chain
                    (what train_lpg_agent does with K = num_updates in one call; the segments continue the chain)
    eval key p, i = link p of the chain of split(eval_rng, N)[i]; eval point p calls eval_agent with it

so training does not depend on ``eval_interval`` or ``eval_workers``, and the evaluations do not perturb training.

The loop enqueues device work only: one non-recording ``Tape`` (two table slots, no saved activations) is reused by
every segment, the evaluation results go into a device tensor, and the host reads the curve and the optimal returns
back once, at the end."""
from __future__ import annotations

from types import SimpleNamespace

import numpy as np
import torch

from ..util import prng
from ..agents.lpg_agent import Tape, train_lpg_agent
from ..agents.agents import eval_agent

OPTIMAL_EPS = 1e-6          # levels whose optimal return is <= this are excluded from the normalised score


def split_keys(rng, num_agents: int) -> dict:
    """The documented key plumbing of ``meta_test``: host uint32 keys."""
    level_rng, agent_rng, train_rng, eval_rng = prng.split(np.asarray(rng, np.uint32), 4)
    return {"level": level_rng, "agent": prng.split(agent_rng, num_agents),
            "train": prng.split(train_rng, num_agents), "eval": prng.split(eval_rng, num_agents)}


def create_test_agents(keys: dict, level_sampler, num_agents: int):
    """Fresh agents on fresh levels of the sampler's mode (``split_keys(rng, num_agents)``)."""
    levels = level_sampler._sample_random_levels(keys["level"], num_agents)
    return level_sampler._create_agent(keys["agent"], levels)


def eval_points(num_updates: int, eval_interval: int) -> np.ndarray:
    """Update counts at which the agents are evaluated: 0, every ``eval_interval`` updates, and ``num_updates``."""
    if eval_interval <= 0:
        raise ValueError(f"eval_interval must be positive, got {eval_interval}")
    return np.unique(np.r_[np.arange(0, num_updates, eval_interval), num_updates]).astype(np.int64)


def meta_test(rng, lpg_params, lifetime_conditioning: bool, level_sampler, num_agents: int, num_updates=None,
              eval_interval: int = 250, eval_workers: int = 64, agent_target_coeff: float = 0.5):
    """Train ``num_agents`` fresh agents with the frozen LPG ``lpg_params`` (flat f32 vector, host or device) on levels
    of ``level_sampler``'s mode.  Returns ``(curve f32[P, N], eval_updates int[P], optimal f64[N], final AgentState)``:
    ``curve[p, i]`` is agent i's ``eval_agent`` return (``eval_workers`` workers, first episode, horizon
    ``max_rollout_len``) after ``eval_updates[p]`` updates; ``optimal[i]`` the optimal return of its level over the
    same horizon.  ``curve`` and ``optimal`` are host numpy arrays."""
    from ..models.lpg import LPG
    ro = level_sampler.rollout_manager
    env = ro.env
    dev = level_sampler.device
    K = int(level_sampler.max_lifetime if num_updates is None else num_updates)
    if K < 0:
        raise ValueError(f"num_updates must be >= 0, got {K}")
    model = LPG(lifetime_conditioning=bool(lifetime_conditioning))
    lpg = torch.as_tensor(lpg_params, dtype=torch.float32).to(dev).contiguous()
    if lpg.numel() != model.size:
        raise ValueError(f"LPG parameter vector has {lpg.numel()} entries, the model has {model.size}")
    lpg_state = SimpleNamespace(params=lpg, model=model)

    keys = split_keys(rng, num_agents)
    agents = create_test_agents(keys, level_sampler, num_agents)
    points = eval_points(K, eval_interval)
    N, W = agents.env_state.packed.shape
    eval_keys = prng.chain_device(prng.to_device(keys["eval"], dev), len(points))     # [P, N, 2]
    curve = torch.empty((len(points), N), dtype=torch.float32, device=dev)
    optimal = env.optimal_return(agents.level.packed, ro.eval_rollout_len)

    def _eval(p):
        curve[p] = eval_agent(eval_keys[p], ro, agents.level.packed, agents.actor_state, eval_workers)

    _eval(0)
    # a non-recording tape's buffers do not depend on its number of updates: one tape serves every segment
    seg_max = int(np.diff(points).max()) if len(points) > 1 else 1
    tape = Tape(N, W, ro.train_rollout_len, env.obs_dim, seg_max, dev, keep_gates=False)
    carry = prng.to_device(keys["train"], dev)
    for p in range(1, len(points)):
        seg = int(points[p] - points[p - 1])
        _, nxt = prng.chain_device(carry, seg, want_carry=True)       # where the chain stands after this segment
        agents, _, _ = train_lpg_agent(carry, lpg_state, agents, ro, seg, agent_target_coeff, tape=tape)
        carry = nxt
        _eval(p)
    host = torch.cat([curve.double().reshape(-1), optimal]).cpu().numpy()    # the one read-back
    return host[:curve.numel()].reshape(curve.shape).astype(np.float32), points, host[curve.numel():], agents


def summarize(curve, eval_updates, optimal, lifetimes=None) -> dict:
    """Scores of a meta-test: per eval point the mean / min / max return and the mean normalised score
    return / optimal over the levels with optimal > OPTIMAL_EPS (the others are counted as excluded)."""
    curve, optimal = np.asarray(curve, np.float64), np.asarray(optimal, np.float64)
    keep = optimal > OPTIMAL_EPS
    norm = curve[:, keep] / optimal[keep]
    out = {
        "eval": [{"update": int(u), "mean_return": float(c.mean()), "min_return": float(c.min()),
                  "max_return": float(c.max()),
                  "mean_normalised_score": float(n.mean()) if keep.any() else None}
                 for u, c, n in zip(eval_updates, curve, norm)],
        "mean_optimal_return": float(optimal.mean()),
        "num_excluded_levels": int((~keep).sum()),
        "levels": {"optimal": optimal.tolist(), "final_return": curve[-1].tolist()},
    }
    if lifetimes is not None:
        out["levels"]["lifetime"] = np.asarray(lifetimes).astype(int).tolist()
    return out
