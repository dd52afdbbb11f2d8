"""Vectorised numpy restatement of the optimal-return DP (test infrastructure, beside oracle/): the loop DP
``oracle.gridworld.optimal_return`` restated over a batch of levels with the operations, and their order, of
csrc/optimal_return.cu.  tests/test_09_optimal_return_cpu.py holds it against the loop DP; the GPU tests hold the
kernel against it."""
import numpy as np

from oracle.gridworld import EnvParams, GridWorld


def optimal_return_batch(env: GridWorld, p: EnvParams, max_rollout_len: int) -> np.ndarray:
    """``optimal_return`` for every level of ``p`` at once: f64[N].  The same DP, restated with numpy over the
    level axis and factorised the way csrc/optimal_return.cu computes it (the kernel performs these operations in
    this order, each rounded once):

      E[n, m] = expected V_{t+1}[n, m'] over the respawns, as a subset transform: for object i = 0..n_objs-1, at
                masks with bit i clear (object absent: respawns w.p. p) E <- p * E[bit i = 1] + (1 - p) * E[bit i = 0],
                at masks with bit i set E <- E[bit i = 0] if object i sits on cell n (collected) else E[bit i = 1];
      V_t[c, m] = max_a  r(coll) + E[nxt, m] * (1 - p_term(coll)),  coll = m & objs(nxt), r / p_term summed in
                object order; wall cells 0.

    A level's episode is capped at H' = min(max_rollout_len, max_steps) steps: V = T^H'(0) at (start_pos, all
    objects present)."""
    N, G2, O = len(p), env.max_grid_size ** 2, env.max_n_objs
    nm = 1 << O
    g = p.grid_size.astype(np.int64)
    n_objs = p.n_objs.astype(np.int64)
    r_obj = env._take_type(p.obj_rewards, p.obj_ids).astype(np.float64)
    p_t = env._take_type(p.obj_p_terminate, p.obj_ids).astype(np.float64)
    p_r = env._take_type(p.obj_p_respawn, p.obj_ids).astype(np.float64)
    live = np.arange(O)[None, :] < n_objs[:, None]                                    # [N, O]
    cell = np.arange(G2)
    in_grid = cell[None, :] < (g * g)[:, None]                                         # [N, G2]
    # objects on each cell (bit mask), next cell of every (cell, action)
    objs = np.zeros((N, G2), np.int64)
    for i in range(O):
        objs |= ((p.static_obj_poss[:, i:i + 1] == cell[None, :]) & live[:, i:i + 1]).astype(np.int64) << i
    pos = np.broadcast_to(np.where(in_grid, cell[None, :], 0), (N, G2)).astype(np.int32)
    nxt = np.stack([env._get_next_pos(pos, np.full((N, G2), a), p) for a in range(5)], 0).astype(np.int64)
    # reward / termination probability of every collected subset, summed in object order
    r_sub = np.zeros((N, nm)); pt_sub = np.zeros((N, nm))
    masks = np.arange(nm)
    for i in range(O):
        has = ((masks >> i) & 1).astype(bool)[None, :] & live[:, i:i + 1]
        r_sub = np.where(has, r_sub + r_obj[:, i:i + 1], r_sub)
        pt_sub = np.where(has, pt_sub + p_t[:, i:i + 1], pt_sub)
    walls = np.asarray(p.walls, bool) | ~in_grid
    horizon = np.minimum(int(max_rollout_len), p.max_steps_in_episode.astype(np.int64))
    ni = np.arange(N)[:, None, None]
    v = np.zeros((N, G2, nm))
    for t in range(int(horizon.max()) if N else 0):
        e = v.copy()
        for i in range(O):
            b = 1 << i
            lo = masks[(masks & b) == 0]
            e0, e1 = e[:, :, lo], e[:, :, lo | b]
            pi = p_r[:, i, None, None]
            new_lo = pi * e1 + (1.0 - pi) * e0
            new_hi = np.where(((objs >> i) & 1).astype(bool)[:, :, None], e0, e1)
            act = live[:, i, None, None]
            e[:, :, lo] = np.where(act, new_lo, e0)
            e[:, :, lo | b] = np.where(act, new_hi, e1)
        best = None
        for a in range(5):
            n = nxt[a][:, :, None]                                                     # [N, G2, 1]
            coll = masks[None, None, :] & objs[np.arange(N)[:, None], nxt[a]][:, :, None]
            val = r_sub[ni, coll] + e[ni, n, masks[None, None, :]] * (1.0 - pt_sub[ni, coll])
            best = val if best is None else np.maximum(best, val)
        best = np.where(walls[:, :, None], 0.0, best)
        v = np.where((t < horizon)[:, None, None], best, v)
    start = p.start_pos.astype(np.int64)
    full = (1 << n_objs) - 1
    return v[np.arange(N), start, full]
