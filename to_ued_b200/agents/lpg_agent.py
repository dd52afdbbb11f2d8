"""LPG-driven agent training (reference agents/lpg_agent.py:13-140), batched over agents and
executed by the CUDA kernels in csrc/{rollout,lpg_forward,agent_update}.cu.

``train_lpg_agent`` keeps the reference's signature and return value (agent_state, rollouts,
metrics); when a ``Tape`` is passed it additionally records what the meta-gradient needs
(per-update tables, trajectories, LPG activations) so that meta/train.py can run the hand-written
backward pass where the reference calls ``jax.grad``."""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Any, List, Optional

import numpy as np
import torch

from .. import _lib
from ..util import prng
from ..util.data import AgentState, Transition


@dataclass
class LPGAgentMetrics:
    """agents/lpg_agent.py:13-28; fields are f32[N] tensors (mean over the K updates)."""
    policy_l2: Any
    policy_entropy: Any
    critic_loss: Any
    critic_l2: Any
    critic_entropy: Any

    def as_dict(self):
        return {"policy_l2": self.policy_l2, "policy_entropy": self.policy_entropy,
                "critic_loss": self.critic_loss, "critic_l2": self.critic_l2,
                "critic_entropy": self.critic_entropy}


class Tape:
    """Device buffers of K agent updates (allocated once and reused).

    ``keep_gates=True`` (meta-gradient path) records everything the reverse pass needs: K+1 table
    versions, K+1 rollouts and the LPG activations of all K updates.  ``keep_gates=False`` (ES / plain
    agent training, no reverse pass) keeps ring buffers only: 2 table slots and 1 slot for everything
    else, so K can be the full agent lifetime."""

    def __init__(self, n_agents, n_workers, rollout_len, obs_dim, num_updates, device, keep_gates=True,
                 precision=None, per_agent_params=False):
        import to_ued_b200
        N, W, L, D, K = n_agents, n_workers, rollout_len, obs_dim, num_updates
        R, dev = N * W, device
        f32, u8, i32 = torch.float32, torch.uint8, torch.int32
        self.N, self.W, self.L, self.D, self.K, self.R = N, W, L, D, K, R
        self.record = bool(keep_gates)
        kt = K + 1 if self.record else 2            # table slots
        kr = K + 1 if self.record else 1            # rollout slots (K train + 1 eval)
        ka = K if self.record else 1                # activation slots
        self.kt, self.kr, self.ka = kt, kr, ka
        self.actor = torch.empty((kt, N, D, 8), dtype=f32, device=dev)
        self.critic = torch.empty((kt, N, D, 8), dtype=f32, device=dev)
        self.obs = torch.empty((kr, N, L + 1, W), dtype=i32, device=dev)
        self.action = torch.empty((kr, N, L, W), dtype=u8, device=dev)
        self.reward = torch.empty((kr, N, L, W), dtype=f32, device=dev)
        self.done = torch.empty((kr, N, L, W), dtype=u8, device=dev)
        self.sorted_tok = torch.empty((kr, N, L * W), dtype=torch.int16, device=dev)
        self.precision = precision or to_ued_b200.GRU_PRECISION
        self.x = torch.empty((ka, L, R, 8), dtype=f32, device=dev)
        self.ximg = None
        if self.precision == "tc":
            f16 = torch.float16
            Rp = (R + 63) // 64 * 64
            R32 = (R + 31) // 32 * 32                         # RB32 layout pads rows to blocks of 32
            # h16 (h_t for the reverse pass) only on recording tapes: inference never reads it
            self.h16 = torch.empty((ka, L, R32, 256), dtype=f16, device=dev) if self.record and not per_agent_params else None
            self.fac = torch.empty((ka, 4, L, R32, 256), dtype=f16, device=dev) if self.record else None
            # bf16 token-tile images (rows >= R of a partial 64-token block stay zero)
            self.hpimg = torch.zeros((ka, L * Rp * 256 * 2), dtype=torch.uint8, device=dev) if self.record else None
            self.ximg = torch.zeros((ka, L * Rp * 128), dtype=torch.uint8, device=dev) if self.record else None
            # 16 pass images of 26 KiB per LPG parameter set (one set, or one per agent on the ES path)
            self.wh_img = torch.zeros((N if per_agent_params else 1) * 16 * 26624 // 2, dtype=f16, device=dev)
            self.h = self.gates = None
        else:
            self.h = torch.empty((ka, L, R, 256), dtype=f32, device=dev)
            self.gates = torch.empty((ka, 4, L, R, 256), dtype=f32, device=dev) if self.record else None
        self.pi_hat = torch.empty((ka, L, R), dtype=f32, device=dev)
        self.y_hat = torch.empty((ka, L, R, 8), dtype=f32, device=dev)
        self.scalars = torch.empty((ka, N, 8), dtype=f32, device=dev)
        self.scal_sum = torch.zeros((N, 8), dtype=f32, device=dev)
        self.step_in = torch.empty((ka, N), dtype=i32, device=dev)
        self.ep_return = torch.empty((N, W), dtype=f32, device=dev)
        # run-sum scratch of toued_agent_update (one launch at a time per tape: the updates of a tape are sequential)
        self.agent_scratch = torch.empty(_lib.lib().toued_agent_scratch_floats(N, W, L, D), dtype=f32, device=dev)

    def ti(self, k):       # table slot of theta_k
        return k if self.record else (k & 1)

    def ri(self, k):       # rollout slot
        return k if self.record else 0

    def ai(self, k):       # activation slot
        return k if self.record else 0

    def transition(self, k) -> Transition:
        r = self.ri(k)
        return Transition(self.obs[r], self.action[r], self.reward[r], self.done[r])


_SORT_STREAMS = {}


def _sort_stream(cur):
    """One side stream per chain stream (created on first use)."""
    key = (cur.device.index, cur.cuda_stream)
    st = _SORT_STREAMS.get(key)
    if st is None:
        st = _SORT_STREAMS[key] = torch.cuda.Stream(device=cur.device)
    return st


def _mark(label):
    """Fine-grained device timeline (tools/phase_timeline.py FINE=1): an event on the current stream; no-op in production."""
    import to_ued_b200
    if to_ued_b200.PHASE_EVENTS is not None and getattr(to_ued_b200, "PHASE_FINE", False):
        e = torch.cuda.Event(enable_timing=True)
        e.record(torch.cuda.current_stream())
        to_ued_b200.PHASE_EVENTS.append((label, -2, e))


def lpg_agent_train_step(k, tape: Tape, levels, step, lpg_params, lifetime_conditioning, agent_target_coeff,
                         lr_actor, lr_critic, max_grad_norm, lpg_stride=0):
    """agents/lpg_agent.py:31-85 for update ``k`` of the tape: reads theta_k / phi_k and the k-th rollout,
    writes theta_{k+1} / phi_{k+1}, the LPG activations and the per-agent scalars."""
    N, W, L, D = tape.N, tape.W, tape.L, tape.D
    s = _lib.stream_ptr()
    p = _lib.ptr
    r, a, t0, t1 = tape.ri(k), tape.ai(k), tape.ti(k), tape.ti(k + 1)
    # the token sort is only needed by the agent update: it runs on a side stream next to the LPG forward
    import to_ued_b200
    cur = torch.cuda.current_stream()
    side = _sort_stream(cur) if to_ued_b200.SIDE_STREAMS else cur
    ev_roll, ev_sort = torch.cuda.Event(), torch.cuda.Event()
    ev_roll.record(cur)
    with torch.cuda.stream(side):
        side.wait_event(ev_roll)
        _lib.call("toued_sort_tokens", p(tape.obs[r]), p(tape.sorted_tok[r]), N, W, L, _lib.stream_ptr())
        # the dense copy theta_k -> theta_{k+1} (the update changes only touched rows) depends on nothing but theta_k:
        # it rides on the side stream next to the LPG forward instead of heading the agent-update kernel
        precopied = bool(to_ued_b200.SIDE_STREAMS)
        if precopied:
            tape.actor[t1].copy_(tape.actor[t0])
            tape.critic[t1].copy_(tape.critic[t0])
        ev_sort.record(side)
    _mark("rollout")
    tape.step_in[a].copy_(step)
    _lib.call("toued_lpg_prepare", p(tape.obs[r]), p(tape.action[r]), p(tape.reward[r]), p(tape.done[r]),
              p(tape.actor[t0]), p(tape.critic[t0]), p(lpg_params), p(step), p(levels), p(tape.x[a]),
              p(tape.ximg[a]) if tape.ximg is not None else None,
              N, W, L, D, int(lifetime_conditioning), int(lpg_stride), s)
    if lpg_stride and tape.precision == "tc":
        # per-candidate parameters on the tensor cores: one CTA and one set of pass images per agent
        _lib.call("toued_gru_forward_tc_multi", p(tape.x[a]), p(tape.done[r]), p(lpg_params), p(tape.wh_img),
                  p(tape.pi_hat[a]), p(tape.y_hat[a]), N, W, L, int(lifetime_conditioning), int(lpg_stride), s)
    elif lpg_stride or tape.precision != "tc":
        # exact-fp32 kernel (also the default per-candidate-parameter path of ES: one CTA per agent)
        _lib.call("toued_gru_forward", p(tape.x[a]), p(tape.done[r]), p(lpg_params), p(tape.h[a]),
                  p(tape.gates[a]) if tape.gates is not None else None, p(tape.pi_hat[a]), p(tape.y_hat[a]),
                  N, W, L, int(lifetime_conditioning), int(lpg_stride), s)
    else:
        _lib.call("toued_gru_forward_tc", p(tape.x[a]), p(tape.done[r]), p(lpg_params), p(tape.wh_img),
                  p(tape.h16[a]) if tape.h16 is not None else None, p(tape.fac[a]) if tape.fac is not None else None,
                  p(tape.hpimg[a]) if tape.hpimg is not None else None, p(tape.pi_hat[a]), p(tape.y_hat[a]),
                  N, W, L, int(lifetime_conditioning), s)
    _mark("gru_fwd")
    cur.wait_event(ev_sort)
    _mark("sort_wait")
    _lib.call("toued_agent_update", p(tape.obs[r]), p(tape.action[r]), p(tape.sorted_tok[r]), p(tape.pi_hat[a]),
              p(tape.y_hat[a]), p(tape.actor[t0]), p(tape.critic[t0]), p(tape.actor[t1]), p(tape.critic[t1]),
              p(levels), p(step), p(tape.scalars[a]), N, W, L, D, float(lr_actor), float(lr_critic),
              float(max_grad_norm), float(agent_target_coeff), int(precopied), p(tape.agent_scratch), s)
    tape.scal_sum += tape.scalars[a]
    _mark("update")


def train_lpg_agent_steps(rng, lpg_train_state, agent_state: AgentState, rollout_manager, num_train_steps: int,
                          agent_target_coeff: float, tape: Optional[Tape] = None, lpg_stride: int = 0):
    """``train_lpg_agent`` as a generator: yields after the set-up and after every update (nothing is yielded but
    control), returns the result tuple.  Lets a caller that drives several agent chunks on different CUDA streams
    enqueue their updates round-robin; every resumption must happen under the chunk's own stream context."""
    env = rollout_manager.env
    actor, critic = agent_state.actor_state, agent_state.critic_state
    N, W = agent_state.env_state.packed.shape
    L, K = rollout_manager.train_rollout_len, num_train_steps
    dev = actor.params.device
    if tape is None:
        import to_ued_b200
        tape = Tape(N, W, L, env.obs_dim, K, dev, keep_gates=False,
                    precision=to_ued_b200.ES_PRECISION if lpg_stride else None, per_agent_params=bool(lpg_stride))
    levels = agent_state.level.packed
    step = actor.step.clone()
    state = agent_state.env_state.packed.clone()
    tape.actor[0].copy_(actor.params)
    tape.critic[0].copy_(critic.params)
    tape.scal_sum.zero_()
    keys_d = prng.chain_device(prng.to_device(rng, dev), K)   # lpg_agent.py:104-105, derived on the device
    p = _lib.ptr
    lpg = lpg_train_state.params if hasattr(lpg_train_state, "params") else lpg_train_state
    cond = lpg_train_state.model.lifetime_conditioning if hasattr(lpg_train_state, "model") else False
    if tape.precision == "tc" and not lpg_stride:             # recurrent matrix -> fp16 SW128 pass images
        _lib.call("toued_pack_wh_forward", p(lpg), p(tape.wh_img), int(cond), _lib.stream_ptr())
    elif tape.precision == "tc":                              # ... one set of images per candidate
        _lib.call("toued_pack_wh_forward_multi", p(lpg), p(tape.wh_img), int(cond), N, int(lpg_stride), _lib.stream_ptr())
    yield
    for k in range(K):
        r = tape.ri(k)
        _lib.call("toued_rollout", p(levels), p(keys_d[k]), p(tape.actor[tape.ti(k)]), None, p(state), p(tape.obs[r]),
                  p(tape.action[r]), p(tape.reward[r]), p(tape.done[r]), None, N, W, L, env.obs_dim,
                  env.max_grid_size, env.max_n_objs, 0, _lib.stream_ptr())
        lpg_agent_train_step(k, tape, levels, step, lpg, cond, agent_target_coeff, actor.learning_rate,
                             critic.learning_rate, actor.max_grad_norm, lpg_stride=lpg_stride)
        yield
    sc = tape.scal_sum / K                                    # lpg_agent.py:140 mean over updates
    metrics = LPGAgentMetrics(policy_l2=sc[:, 4], policy_entropy=sc[:, 6], critic_loss=sc[:, 3],
                              critic_l2=sc[:, 5], critic_entropy=sc[:, 7])
    from ..environments.gridworld.gridworld import EnvState
    new_agent = agent_state.replace(
        actor_state=actor.replace(params=tape.actor[tape.ti(K)].clone(), step=step),
        critic_state=critic.replace(params=tape.critic[tape.ti(K)].clone(), step=step.clone()),
        env_obs=tape.obs[tape.ri(K - 1)][:, -1].clone(), env_state=EnvState(state, env.max_n_objs))
    rollouts = [tape.transition(k) for k in range(K)] if tape.record else [tape.transition(K - 1)]
    return new_agent, rollouts, metrics


def train_lpg_agent(rng, lpg_train_state, agent_state: AgentState, rollout_manager, num_train_steps: int,
                    agent_target_coeff: float, tape: Optional[Tape] = None, lpg_stride: int = 0):
    """agents/lpg_agent.py:88-140, batched: rng uint32[N, 2].
    Returns (agent_state, rollouts (list of Transition; all K only when the tape records), LPGAgentMetrics
    of f32[N]).  ``lpg_stride`` != 0: ``lpg_train_state`` holds one parameter vector per agent."""
    gen = train_lpg_agent_steps(rng, lpg_train_state, agent_state, rollout_manager, num_train_steps,
                                agent_target_coeff, tape=tape, lpg_stride=lpg_stride)
    while True:
        try:
            next(gen)
        except StopIteration as done:
            return done.value
