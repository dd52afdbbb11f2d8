"""LPG meta-optimisation steps (reference meta/train.py:14-227) on the B200 kernels.

``lpg_meta_grad_train_step`` keeps the reference's keyword signature.  Where the reference takes
``jax.grad`` of the unrolled inner loop, this runs the hand-written reverse pass:

    forward  (per update k)  rollout -> sort tokens -> LPG inputs -> GRU + heads -> agent update
    eval rollout with theta_K -> meta loss (GAE with the frozen value critic, Q2; LPG loss, Q16) -> lam_K
    backward (k = K-1 .. 0)  agent adjoint (HVPs through clip/SGD/mask) -> d pi_hat, d y_hat
                             -> GRU BPTT -> token-split weight-gradient partials
    reduce partials -> (all-reduce over ranks) -> Adam

Agents are the data-parallel axis: with torch.distributed initialised, every rank holds
``num_agents / world_size`` agents and the flat LPG gradient plus the metric sums are all-reduced
(one NCCL call each); ``num_mini_batches`` (a memory device in the reference, util/jax.py:25-41)
splits the local agents into sequential chunks whose partial sums accumulate, giving identical
results."""
from __future__ import annotations

from typing import Any, Optional

import numpy as np
import torch

from .. import _lib
from ..util import prng
from ..util.data import AgentState, LpgHyperparams
from ..agents.lpg_agent import Tape, train_lpg_agent, train_lpg_agent_steps
from ..agents.agents import eval_agent
from ..environments.gridworld.gridworld import EnvState


class LPGTrainState:
    """flax TrainState of the LPG network: flat params + Adam state (+ the model description)."""

    def __init__(self, model, params, tx, opt_state=None, step=0):
        self.model, self.params, self.tx = model, params, tx
        self.opt_state = tx.init(params) if opt_state is None else opt_state
        self.step = step

    def replace(self, **kw):
        d = dict(model=self.model, params=self.params, tx=self.tx, opt_state=self.opt_state, step=self.step)
        d.update(kw)
        return LPGTrainState(**d)


class MetaGradWorkspace:
    """All device buffers of one meta-gradient step for a chunk of agents (allocated once)."""

    def __init__(self, n_agents, n_workers, rollout_len, obs_dim, num_updates, n_params, device):
        N, W, L, K = n_agents, n_workers, rollout_len, num_updates
        R = N * W
        f32 = torch.float32
        self.tape = Tape(N, W, L, obs_dim, K, device, keep_gates=True)
        # cotangent buffers are double-buffered over the update index: the agent adjoint of update k-1 and the
        # embedding gradient of update k run on side streams next to the tensor-core kernels of update k / k-1
        self.d_pi_hat2 = [torch.empty((L, R), dtype=f32, device=device) for _ in range(2)]
        self.d_y_hat2 = [torch.empty((L, R, 8), dtype=f32, device=device) for _ in range(2)]
        self.dx2 = [torch.empty((L, R, 2), dtype=f32, device=device) for _ in range(2)]
        self.d_pi_hat, self.d_y_hat, self.dx = self.d_pi_hat2[0], self.d_y_hat2[0], self.dx2[0]
        self.dl2 = [torch.empty((L, R, 8), dtype=f32, device=device) for _ in range(2)]
        self.dl = self.dl2[0]
        self.lam = torch.empty((N, obs_dim, 8), dtype=f32, device=device)
        self.mu = torch.empty((N, obs_dim, 8), dtype=f32, device=device)
        self.whT = torch.empty((768, 256), dtype=f32, device=device)
        self.partials = torch.empty(_lib.lib().toued_lpg_wgrad_workspace_floats(), dtype=f32, device=device)
        self.loss_scal = torch.empty((N, 2), dtype=f32, device=device)
        # run-sum scratch of toued_agent_backward (its launches of one chunk are sequential on the agent stream)
        self.ab_scratch = torch.empty(_lib.lib().toued_agent_scratch_floats(N, W, L, obs_dim), dtype=f32, device=device)
        if self.tape.precision == "tc":
            Rp = (R + 63) // 64 * 64
            self.whb_img = torch.empty(256 * 768, dtype=torch.float16, device=device)
            # {max |cotangent|, status bits} of every update's reverse launch (scaled fp16 operands, csrc/tc.cuh;
            # include/toued.h toued_cotangent_max): the status words are sticky, read by reverse_status()
            self.cotmax = torch.zeros((K, 2), dtype=torch.int32, device=device)
            # fp16 token-tile image of S * (dar, daz, dhn, dan): 16 column groups of 64
            # (double-buffered over the update index like the cotangents: the weight-gradient GEMMs of update k run on
            #  their own stream next to the BPTT of update k-1)
            self.dgimg2 = [torch.zeros(L * Rp * 1024 * 2, dtype=torch.uint8, device=device) for _ in range(2)]
            self.dgimg = self.dgimg2[0]
        self.off_small = _lib.lib().toued_lpg_wgrad_workspace_offset(1)
        self.key = (N, W, L, obs_dim, K, n_params, str(device))


_WS_CACHE = {}
_STREAMS = {}


def _workspace(n, w, L, D, K, P, device, slot=0) -> MetaGradWorkspace:
    import to_ued_b200
    key = (n, w, L, D, K, P, str(device), to_ued_b200.GRU_PRECISION)
    if _WS_CACHE and next(iter(_WS_CACHE))[:-1] != key:
        _WS_CACHE.clear()
    ws = _WS_CACHE.get(key + (slot,))
    if ws is None:
        ws = _WS_CACHE[key + (slot,)] = MetaGradWorkspace(n, w, L, D, K, P, device)
    return ws


def reverse_status(reset=False):
    """OR of the status words of the tensor-core reverse passes run since the workspaces were created (or last reset):
    an int32 device tensor, 0 when every meta-gradient came out clean.  Bit TOUED_STATUS_NONFINITE_COT (1): a cotangent
    was inf / NaN; bit TOUED_STATUS_FP16_RANGE (2): an fp16 operand of the reverse pass saturated or was not finite, so
    the meta-gradient may be wrong (include/toued.h).  Only the tensor-core path (GRU_PRECISION "tc") sets bits.  No
    host synchronisation unless the caller reads the value."""
    st = torch.zeros((), dtype=torch.int32, device="cuda")
    for ws in _WS_CACHE.values():
        if getattr(ws, "cotmax", None) is not None:
            for w in ws.cotmax[:, 1]:
                st = st | w
            if reset:
                ws.cotmax[:, 1].zero_()
    return st


def _eval_stream(device):
    key = ("eval", str(device))
    if key not in _STREAMS:
        _STREAMS[key] = [torch.cuda.Stream(device=device)]
    return _STREAMS[key][0]


def _side_streams(device, n):
    key = str(device)
    lst = _STREAMS.setdefault(key, [])
    while len(lst) < n:
        lst.append(torch.cuda.Stream(device=device))
    return lst[:n]


def _world():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        return dist.get_world_size(), dist
    return 1, None


def lpg_meta_grad_train_step(rng, lpg_train_state: LPGTrainState, agent_states: AgentState, value_critic_states,
                             rollout_manager, num_mini_batches: int, gamma: float, gae_lambda: float,
                             lpg_hypers: LpgHyperparams, *, outer_product_quirk: bool = True,
                             global_agent_offset: int = 0, global_num_agents: Optional[int] = None,
                             eval_workers: int = 4, return_grad: bool = False, num_streams: Optional[int] = None,
                             _static: Optional[dict] = None):
    """Update a batch of agents with LPG, then update LPG with the regularised final agent loss
    (meta/train.py:14-130).  rng: the step key (uint32[2], or an int32[1, 2] device tensor).  Returns
    (lpg_train_state, agent_states, value_critic_states, metrics).

    ``_static`` (used by meta/graph.py when the step is captured into a CUDA graph): the per-agent outputs are written
    into the given buffers (which may be the input buffers: every chunk reads its slice before it writes it), Adam runs
    in place on the LPG parameters with its update count in device memory, and the metric vector is returned as one
    tensor -- nothing in the enqueued work then depends on host state."""
    env = rollout_manager.env
    actor, critic = agent_states.actor_state, agent_states.critic_state
    N, W = agent_states.env_state.packed.shape
    L, K, D = rollout_manager.train_rollout_len, lpg_hypers.num_agent_updates, env.obs_dim
    dev = actor.params.device
    world, dist = _world()
    n_global = global_num_agents if global_num_agents is not None else N * world
    if dist is not None and global_num_agents is None:
        global_agent_offset = dist.get_rank() * N
    model = lpg_train_state.model
    cond = int(model.lifetime_conditioning)
    lpg = lpg_train_state.params
    P = lpg.numel()
    p, s = _lib.ptr, _lib.stream_ptr()

    # ---- keys: split(rng, n_global)[local slice], then the per-agent chain of meta/train.py:40-110
    #      derived on the device (csrc/prng.cu); the only host input of the step is the 8-byte key
    rngs = prng.split_device(prng.to_device(rng, dev), n_global, global_agent_offset, N)[0]
    r_train, r_eval, r_evalagent = prng.chain_device(rngs, 3)

    if N % num_mini_batches != 0:
        raise ValueError(f"local agents ({N}) must be divisible by num_mini_batches ({num_mini_batches})")
    nb = N // num_mini_batches
    # Mini-batches are independent chains of kernels: run up to `num_streams` of them concurrently on side
    # streams (each with its own workspace) so that one chain's latency-bound kernels and wave tails overlap
    # with another chain's GEMMs.  Results are identical to the sequential order (partials are per workspace).
    import to_ued_b200
    if num_streams is None:
        num_streams = to_ued_b200.NUM_STREAMS
    S = max(1, min(int(num_streams), num_mini_batches))
    wss = [_workspace(nb, W, L, D, K, P, dev, slot=i) for i in range(S)]
    main = torch.cuda.current_stream()
    streams = [main] if S == 1 else _side_streams(dev, S)
    tc = wss[0].tape.precision == "tc"
    gscale = 1.0 / n_global
    bK = [c / K for c in (lpg_hypers.policy_entropy_coeff, lpg_hypers.target_entropy_coeff,
                          lpg_hypers.policy_l2_coeff, lpg_hypers.target_l2_coeff)]
    if _static is not None:
        new_actor, new_critic, new_step, new_state, new_obs = _static["out"]
    else:
        new_actor = torch.empty_like(actor.params)
        new_critic = torch.empty_like(critic.params)
        new_step = torch.empty_like(actor.step)
        new_state = torch.empty_like(agent_states.env_state.packed)
        new_obs = torch.empty_like(agent_states.env_obs)
    msums = [torch.zeros(8, dtype=torch.float32, device=dev) for _ in range(S)]
    returns = torch.empty(N, dtype=torch.float32, device=dev)
    ready = torch.cuda.Event()
    ready.record(main)

    def _phase(label, chunk, stream):                            # tools/phase_timeline.py; no-op in production
        if to_ued_b200.PHASE_EVENTS is not None:
            e = torch.cuda.Event(enable_timing=True)
            e.record(stream)
            to_ued_b200.PHASE_EVENTS.append((label, chunk, e))
    _phase("start", -1, main)
    eval_done = [None] * S
    eval_stream = _side_streams(dev, S + 1)[S] if S > 1 else _eval_stream(dev)
    # per chunk: a stream for the agent adjoints and one for the embedding gradients of the reverse pass
    pool = _side_streams(dev, 5 * S + 1)
    ab_streams, em_streams = pool[S + 1:2 * S + 1], pool[2 * S + 1:3 * S + 1]
    ev_streams = [eval_stream] + pool[3 * S + 1:4 * S]          # one evaluation stream per chunk
    wg_streams = pool[4 * S + 1:5 * S + 1]                      # weight-gradient GEMMs of the tensor-core reverse pass
    if not to_ued_b200.SIDE_STREAMS:                            # per-kernel timing mode: everything on the chunk's stream
        ab_streams = em_streams = ev_streams = wg_streams = list(streams)
    evs = {}

    # The host enqueues the chains of a group of S mini-batches round-robin, one agent update at a time (forward:
    # k = 0..K-1, reverse: k = K-1..0), so every stream has work from the start of the step and the chains finish
    # together (enqueueing one mini-batch's whole chain before the next would leave the other streams idle for
    # the first milliseconds and alone for the last).
    ctx, gens = {}, {}

    def forward_begin(mb):
        slot = mb % S
        ws, tape = wss[slot], wss[slot].tape
        with torch.cuda.stream(streams[slot]):
            if S > 1 and mb < S:
                streams[slot].wait_event(ready)
            if eval_done[slot] is not None:           # the previous chunk on this workspace is still being evaluated
                streams[slot].wait_event(eval_done[slot])
            sl = slice(mb * nb, (mb + 1) * nb)
            sub = AgentState(actor.replace(params=actor.params[sl], step=actor.step[sl]),
                             critic.replace(params=critic.params[sl], step=critic.step[sl]),
                             _sub_level(agent_states.level, sl), agent_states.env_obs[sl],
                             EnvState(agent_states.env_state.packed[sl], env.max_n_objs))
            levels = sub.level.packed
            # ---- K agent updates (forward, taped): set-up now, the updates are driven by forward_step ----
            gens[mb] = (train_lpg_agent_steps(r_train[sl], lpg_train_state, sub, rollout_manager, K,
                                              lpg_hypers.agent_target_coeff, tape=tape), sl, levels)
            next(gens[mb][0])

    def forward_step(mb):
        with torch.cuda.stream(streams[mb % S]):
            try:
                next(gens[mb][0])
            except StopIteration as fin:
                gens[mb] = (fin.value,) + gens[mb][1:]
            _phase("update", mb, streams[mb % S])

    def forward_end(mb):
        slot = mb % S
        ws, tape = wss[slot], wss[slot].tape
        res, sl, levels = gens.pop(mb)
        with torch.cuda.stream(streams[slot]):
            s = _lib.stream_ptr()
            if not isinstance(res, tuple):                   # run the generator to its return value
                try:
                    while True:
                        next(res)
                except StopIteration as fin:
                    res = fin.value
            sub2, _, am = res
            # ---- rollout the updated agent (meta/train.py:46-58) ----
            state = sub2.env_state.packed
            _lib.call("toued_rollout", p(levels), p(r_eval[sl]), p(tape.actor[K]), None, p(state), p(tape.obs[K]),
                      p(tape.action[K]), p(tape.reward[K]), p(tape.done[K]), None, nb, W, L, D,
                      env.max_grid_size, env.max_n_objs, 0, s)
            _lib.call("toued_sort_tokens", p(tape.obs[K]), p(tape.sorted_tok[K]), nb, W, L, s)
            # ---- evaluate agent return: 4 workers, metric only (meta/train.py:109-117, Q11).  A long, thin
            #      kernel (max_rollout_len sequential steps): it runs on its own stream next to the reverse pass.
            fwd_done = torch.cuda.Event()
            fwd_done.record(streams[slot])
            _phase("forward", mb, streams[slot])
            with torch.cuda.stream(ev_streams[slot]):
                ev_streams[slot].wait_event(fwd_done)
                returns[sl] = eval_agent(r_evalagent[sl], rollout_manager, levels, tape.actor[K], eval_workers)
                eval_done[slot] = torch.cuda.Event()
                eval_done[slot].record(ev_streams[slot])
            ctx[mb] = (sl, sub2, state, am, levels)

    def backward_begin(mb):
        slot = mb % S
        ws, tape = wss[slot], wss[slot].tape
        sl = ctx[mb][0]
        with torch.cuda.stream(streams[slot]):
            s = _lib.stream_ptr()
            if mb < S:                                  # recurrent matrix in the reverse pass's operand layout
                if tc:
                    _lib.call("toued_pack_wh_backward", p(lpg), p(ws.whb_img), s)
                else:
                    _lib.call("toued_transpose_wh", p(lpg), p(ws.whT), s)
            # ---- value "update" (Q2) + advantage + LPG loss + lam_K (meta/train.py:60-100) ----
            vparams = value_critic_states.params[sl]
            _lib.call("toued_meta_loss", p(tape.obs[K]), p(tape.action[K]), p(tape.reward[K]), p(tape.done[K]),
                      p(tape.sorted_tok[K]), p(vparams), p(tape.actor[K]), p(ws.lam), p(ws.mu), p(ws.loss_scal),
                      nb, W, L, D, vparams.shape[-1], float(gamma), float(gae_lambda), float(gscale),
                      int(outer_product_quirk), s)
            evs[mb] = {"ml": torch.cuda.Event(), "ab": {}, "bwd": {}, "wg": {}, "em": {}}
            evs[mb]["ml"].record(streams[slot])

    def _agent_backward(ws, tape, k, buf, s):
        _lib.call("toued_agent_backward", p(tape.obs[k]), p(tape.action[k]), p(tape.sorted_tok[k]),
                  p(tape.pi_hat[k]), p(tape.y_hat[k]), p(tape.actor[k]), p(tape.critic[k]),
                  p(tape.actor[k + 1]), p(tape.critic[k + 1]), p(tape.scalars[k]), p(ws.lam), p(ws.mu),
                  p(ws.d_pi_hat2[buf]), p(ws.d_y_hat2[buf]), nb, W, L, D, float(actor.learning_rate),
                  float(critic.learning_rate), float(actor.max_grad_norm),
                  float(lpg_hypers.agent_target_coeff), *[float(b) for b in bK], float(gscale), p(ws.ab_scratch), s)

    def backward_step(mb, k):
        """Reverse pass of update k.  Tensor-core path: three streams per chunk --
             agent stream : agent adjoint (HVPs through clip/SGD) of update k        -> d pi_hat / d y_hat [k & 1]
             chain stream : GRU BPTT, weight-gradient GEMMs of update k              (back to back over k)
             embed stream : embedding-MLP gradient of update k                       (reads dx [k & 1])
           so the latency-bound per-agent kernels run beside the tensor-core kernels of the neighbouring update
           instead of between them."""
        slot = mb % S
        ws, tape = wss[slot], wss[slot].tape
        first = (mb < S and k == K - 1)                 # first use of this workspace's partial buffers
        if not tc:
            with torch.cuda.stream(streams[slot]):
                s = _lib.stream_ptr()
                _agent_backward(ws, tape, k, 0, s)
                _lib.call("toued_gru_backward", p(tape.done[k]), p(lpg), p(ws.whT), p(tape.h[k]), p(tape.gates[k]),
                          p(tape.y_hat[k]), p(ws.d_pi_hat), p(ws.d_y_hat), p(ws.dl), p(ws.dx), nb, W, L, cond, s)
                _lib.call("toued_lpg_wgrad", p(tape.obs[k]), p(tape.done[k]), p(tape.critic[k]), p(lpg), p(tape.x[k]),
                          p(tape.h[k]), p(tape.gates[k]), p(ws.d_pi_hat), p(ws.dl), p(ws.dx), p(ws.partials),
                          nb, W, L, D, cond, 0 if first else 1, s)
            return
        ev, buf = evs[mb], k & 1
        for d in ("ab", "bwd", "wg", "em"):
            ev[d][k] = torch.cuda.Event()
        with torch.cuda.stream(ab_streams[slot]):
            st = ab_streams[slot]
            if k == K - 1:
                st.wait_event(ev["ml"])
            if k + 2 <= K - 1:
                st.wait_event(ev["wg"][k + 2])              # the cotangent buffer is free again
            _agent_backward(ws, tape, k, buf, _lib.stream_ptr())
            _lib.call("toued_cotangent_max", p(ws.d_pi_hat2[buf]), p(ws.d_y_hat2[buf]), nb, W, L, p(ws.cotmax[k]),
                      _lib.stream_ptr())
            ev["ab"][k].record(st)
        with torch.cuda.stream(streams[slot]):
            st = streams[slot]
            s = _lib.stream_ptr()
            st.wait_event(ev["ab"][k])
            if k + 2 <= K - 1:
                st.wait_event(ev["em"][k + 2])              # dx [k & 1] has been consumed
                st.wait_event(ev["wg"][k + 2])              # ... and so have the dG image and dl [k & 1]
            _lib.call("toued_gru_backward_tc", p(tape.done[k]), p(lpg), p(ws.whb_img), p(tape.h16[k]),
                      p(tape.fac[k]), p(tape.y_hat[k]), p(ws.d_pi_hat2[buf]), p(ws.d_y_hat2[buf]), p(ws.dgimg2[buf]), p(ws.dl2[buf]),
                      p(ws.dx2[buf]), p(ws.cotmax[k]), nb, W, L, cond, s)
            ev["bwd"][k].record(st)
            _phase(f"bwd{k}", mb, st)
        with torch.cuda.stream(wg_streams[slot]):
            st = wg_streams[slot]
            st.wait_event(ev["bwd"][k])
            _lib.call("toued_lpg_wgrad_tc", p(tape.hpimg[k]), p(ws.dgimg2[buf]), p(tape.ximg[k]), p(tape.h16[k]),
                      p(ws.d_pi_hat2[buf]), p(ws.dl2[buf]), p(ws.partials), p(ws.partials[ws.off_small:]),
                      p(ws.cotmax[k]), nb, W, L, 0 if first else 1, _lib.stream_ptr())
            ev["wg"][k].record(st)
            _phase(f"wgrad{k}", mb, st)
        with torch.cuda.stream(em_streams[slot]):
            st = em_streams[slot]
            st.wait_event(ev["bwd"][k])
            _lib.call("toued_lpg_wgrad_embed", p(tape.obs[k]), p(tape.done[k]), p(tape.critic[k]), p(lpg),
                      p(ws.dx2[buf]), p(ws.partials), p(ws.cotmax[k]), nb, W, L, D, cond, 0 if first else 1,
                      _lib.stream_ptr())
            ev["em"][k].record(st)

    def backward_end(mb):
        slot = mb % S
        ws, tape, msum = wss[slot], wss[slot].tape, msums[slot]
        sl, sub2, state, am, levels = ctx.pop(mb)
        with torch.cuda.stream(streams[slot]):
            ev = evs.pop(mb)
            if ev["em"]:
                streams[slot].wait_event(ev["em"][0])          # joins the embed stream (the agent stream is already joined)
                streams[slot].wait_event(ev["wg"][0])          # ... and the weight-gradient stream
            # ---- metrics (sums over agents; divided by n_global after the all-reduce) ----
            lpg_loss, value_loss = ws.loss_scal[:, 0], ws.loss_scal[:, 1]
            reg = (lpg_loss - lpg_hypers.policy_entropy_coeff * am.policy_entropy + lpg_hypers.policy_l2_coeff * am.policy_l2
                   - lpg_hypers.target_entropy_coeff * am.critic_entropy + lpg_hypers.target_l2_coeff * am.critic_l2)
            msum[:7] += torch.stack([lpg_loss.sum(), reg.sum(), value_loss.sum(), am.policy_l2.sum(),
                                     am.policy_entropy.sum(), am.critic_loss.sum(), am.critic_l2.sum()])
            msum[7] += am.critic_entropy.sum()
            new_actor[sl] = sub2.actor_state.params
            new_critic[sl] = sub2.critic_state.params
            new_step[sl] = sub2.actor_state.step
            new_state[sl] = state
            new_obs[sl] = tape.obs[K][:, -1]
            _phase("reverse_end", mb, streams[slot])

    for g0 in range(0, num_mini_batches, S):
        group = range(g0, min(num_mini_batches, g0 + S))
        for mb in group:                                 # first update right behind each chunk's set-up: the GPU
            forward_begin(mb)                            # gets its first rollout as early as possible
            forward_step(mb)
        for k in range(1, K):
            for mb in group:
                forward_step(mb)
        for mb in group:
            forward_end(mb)
        for mb in group:
            backward_begin(mb)
        for k in reversed(range(K)):
            for mb in group:
                backward_step(mb, k)
        for mb in group:
            backward_end(mb)
    for st in ([] if S == 1 else list(streams)) + ev_streams:
        ev = torch.cuda.Event()
        ev.record(st)
        main.wait_event(ev)
    s = _lib.stream_ptr()
    msum = msums[0] if S == 1 else torch.stack(msums).sum(0)

    grad = torch.empty(P, dtype=torch.float32, device=dev)
    L_ = _lib.lib()
    n_wh, n_sm = (L_.toued_wgrad_tc_splits(), L_.toued_wgrad_tc_small_splits()) if tc else \
        (L_.toued_lpg_wgrad_splits(0), L_.toued_lpg_wgrad_splits(1))
    _lib.call("toued_reduce_partials", p(wss[0].partials), p(grad), cond, n_wh, n_sm, s)
    for ws in wss[1:min(S, num_mini_batches)]:
        g2 = torch.empty_like(grad)
        _lib.call("toued_reduce_partials", p(ws.partials), p(g2), cond, n_wh, n_sm, s)
        grad += g2
    # one collective for the gradient AND the 9 metric sums: they travel in the same buffer
    red = torch.cat([grad, msum, returns.sum().view(1)])
    if dist is not None:
        dist.all_reduce(red)                      # sum of per-rank (1/n_global)-scaled sums = mean
    grad, mvec = red[:P], red[P:] / n_global
    # ---- Adam on the LPG parameters (meta/train.py:129) ----
    if _static is not None:
        ost = lpg_train_state.opt_state
        lpg_train_state.tx.update_dev_(lpg, grad, ost["mu"], ost["nu"], _static["count_dev"])
        new_lpg = lpg_train_state
    else:
        new_params = lpg.clone()
        opt_state = lpg_train_state.tx.update_(new_params, grad, {**lpg_train_state.opt_state,
                                                                  "mu": lpg_train_state.opt_state["mu"].clone(),
                                                                  "nu": lpg_train_state.opt_state["nu"].clone()})
        new_lpg = lpg_train_state.replace(params=new_params, opt_state=opt_state, step=lpg_train_state.step + 1)
    agent_out = agent_states.replace(
        actor_state=actor.replace(params=new_actor, step=new_step),
        critic_state=critic.replace(params=new_critic, step=new_step if _static is not None else new_step.clone()),
        env_obs=new_obs, env_state=EnvState(new_state, env.max_n_objs),
        host_step=_advance_host_step(agent_states.host_step, agent_states.level.lifetime, K))
    # value critic: parameters untouched (Q2); its step counter advances K + 1 per meta-step
    if _static is not None:
        value_critic_states.step.add_(K + 1)
        value_out = value_critic_states
    else:
        value_out = value_critic_states.replace(step=value_critic_states.step + (K + 1))
    metrics = {
        "lpg_loss": mvec[0], "reg_lpg_loss": mvec[1], "value_loss": mvec[2],
        "lpg_agent": {"policy_l2": mvec[3], "policy_entropy": mvec[4], "critic_loss": mvec[5],
                      "critic_l2": mvec[6], "critic_entropy": mvec[7]},
        "lpg_agent_return": mvec[8],
    }
    if return_grad:
        metrics["_grad"] = grad
    if _static is not None:
        metrics["_mvec"] = mvec
    _phase("end", -1, main)
    return new_lpg, agent_out, value_out, metrics


def _advance_host_step(step, lifetime, k):
    """K masked updates: step <- step + 1 while step + 1 <= lifetime (lpg_agent.py:78-82)."""
    if step is None:
        return None
    return np.minimum(step + k, np.maximum(step, lifetime)).astype(np.int32)


def _sub_level(level, sl):
    from ..util.data import Level
    return Level(level.env_params, level.lifetime[sl], level.buffer_id[sl], level.packed[sl])
