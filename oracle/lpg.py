"""LPG network oracle (torch, CPU, differentiable).  TEST INFRASTRUCTURE — see oracle/__init__.py.

Restates models/lpg.py:11-96 (``LPGGRU``, ``LPG``) and models/common.py:6-18 (``MLP``) with
flax==0.6.11 ``Dense`` / ``GRUCell`` semantics [3P-recall]:

    r  = sigmoid(x W_ir + b_ir + h W_hr)
    z  = sigmoid(x W_iz + b_iz + h W_hz)
    n  = tanh   (x W_in + b_in + r * (h W_hn + b_hn))
    h' = (1 - z) * n + z * h

Deviation Q5 (SURVEY.md §2.1): the reference passes ``features=len(gru_state)`` (the *batch*
size) to GRUCell; the evident intent — hidden = lpg_gru_width — is what is implemented.
Q6 is reproduced: the conditioning inputs are the raw ``step`` and ``lifetime`` cast to float.

Parameters are one flat vector (the layout the CUDA kernels use, to_ued_b200/models/lpg.py):
    Wh[H,3H] Wi[X,3H] bi[3H] bhn[H] w_pi[H] W_y[H,Y] b_y[Y] | e_w0[Y,E] e_b0[E] e_w1[E] e_b1[1] | b_pi[1]
gate order (r, z, n) along the 3H axis.
"""
from __future__ import annotations

import numpy as np
import torch


class LPGLayout:
    def __init__(self, embedding_net_width=16, gru_width=256, target_width=8, lifetime_conditioning=False):
        self.E, self.H, self.Y = embedding_net_width, gru_width, target_width
        self.X = 7 if lifetime_conditioning else 5
        self.lifetime_conditioning = lifetime_conditioning
        E, H, Y, X = self.E, self.H, self.Y, self.X
        self.shapes = [("Wh", (H, 3 * H)), ("Wi", (X, 3 * H)), ("bi", (3 * H,)), ("bhn", (H,)), ("w_pi", (H,)),
                       ("W_y", (H, Y)), ("b_y", (Y,)), ("e_w0", (Y, E)), ("e_b0", (E,)), ("e_w1", (E,)),
                       ("e_b1", (1,)), ("b_pi", (1,))]
        self.offsets, off = {}, 0
        for name, shp in self.shapes:
            n = int(np.prod(shp))
            self.offsets[name] = (off, n, shp)
            off += n
        self.size = off

    def unpack(self, flat):
        return {name: flat[o:o + n].reshape(shp) for name, (o, n, shp) in self.offsets.items()}


def _trunc_normal(rs, shape, std):
    """flax lecun_normal: truncated normal on [-2, 2] scaled by std / 0.87962566"""
    v = rs.randn(*shape)
    bad = np.abs(v) > 2
    while bad.any():
        v[bad] = rs.randn(int(bad.sum()))
        bad = np.abs(v) > 2
    return v * std / 0.87962566103423978


def init_lpg_params(layout: LPGLayout, seed: int = 0) -> np.ndarray:
    """Random init with flax's default *distributions* (lecun-normal Dense kernels, zero biases,
    orthogonal recurrent kernels); the draw itself is numpy's, not jax's (init is an input of the
    hot path, not part of it)."""
    rs = np.random.RandomState(seed)
    E, H, Y, X = layout.E, layout.H, layout.Y, layout.X
    p = {
        "e_w0": _trunc_normal(rs, (Y, E), Y ** -0.5), "e_b0": np.zeros(E),
        "e_w1": _trunc_normal(rs, (E,), E ** -0.5), "e_b1": np.zeros(1),
        "Wi": _trunc_normal(rs, (X, 3 * H), X ** -0.5), "bi": np.zeros(3 * H),
        "Wh": np.concatenate([np.linalg.qr(rs.randn(H, H))[0] for _ in range(3)], axis=1), "bhn": np.zeros(H),
        "w_pi": _trunc_normal(rs, (H,), H ** -0.5), "b_pi": np.zeros(1),
        "W_y": _trunc_normal(rs, (H, Y), H ** -0.5), "b_y": np.zeros(Y),
    }
    return np.concatenate([p[name].reshape(-1) for name, _ in layout.shapes]).astype(np.float32)


def lpg_forward(layout: LPGLayout, flat, r, d, pi, yt, yt1, step, lifetime, hidden=None):
    """models/lpg.py:48-85.  r, d, pi: [B, L]; yt, yt1: [B, L, Y]; step, lifetime: [B] (per
    sequence).  Returns pi_hat [B, L], y_hat [B, L, Y].  ``hidden`` (a list, optional) receives the
    hidden states h_t [B, H] in time order, e.g. to read their gradients."""
    P = layout.unpack(flat)
    H = layout.H
    dt = flat.dtype
    d = d.to(dt)

    def embed(y):                                           # MLP([E, 1]), models/common.py:6-18
        return torch.relu(y @ P["e_w0"] + P["e_b0"]) @ P["e_w1"] + P["e_b1"]

    pyt = embed(yt)
    pyt1 = embed(yt1) * (1.0 - d)                           # lpg.py:69
    cols = [r.to(dt), d, pi, pyt, pyt1]
    if layout.lifetime_conditioning:                        # lpg.py:70-75 (raw values, Q6)
        cols += [step.to(dt)[:, None].expand_as(d), lifetime.to(dt)[:, None].expand_as(d)]
    x = torch.stack(cols, dim=-1)                           # [B, L, X]
    gi = x @ P["Wi"] + P["bi"]                              # [B, L, 3H]
    B, L = d.shape
    h = torch.zeros(B, H, dtype=dt)
    outs = [None] * L
    for t in reversed(range(L)):                            # LPGGRU: reverse scan, lpg.py:14-30
        h = h * (1.0 - d[:, t:t + 1])                       # reset at terminal states
        gh = h @ P["Wh"]
        rg = torch.sigmoid(gi[:, t, :H] + gh[:, :H])
        zg = torch.sigmoid(gi[:, t, H:2 * H] + gh[:, H:2 * H])
        ng = torch.tanh(gi[:, t, 2 * H:] + rg * (gh[:, 2 * H:] + P["bhn"]))
        h = (1.0 - zg) * ng + zg * h
        outs[t] = h
    if hidden is not None:
        hidden.extend(outs)
    y = torch.relu(torch.stack(outs, dim=1))                # [B, L, H]
    pi_hat = y @ P["w_pi"] + P["b_pi"]                      # Dense(1), squeezed
    y_hat = torch.softmax(y @ P["W_y"] + P["b_y"], dim=-1)
    return pi_hat, y_hat
