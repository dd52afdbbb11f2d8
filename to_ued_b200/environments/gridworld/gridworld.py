"""Gridworld environment of the LPG paper, B200-native.

Mirrors the reference's ``environments/gridworld/gridworld.py`` interface (``EnvParams``,
``EnvState``, ``GridWorld.reset/step/default_params/num_actions/observation_space``) but every
transition runs in the CUDA kernels of ``to_ued_b200/csrc/rollout.cu``.  Differences in
*representation* (not behaviour):

  * everything is batched: ``EnvParams`` fields have a leading agent axis ``[N]`` (host numpy),
    ``EnvState`` holds ``[N, W]`` environments on the GPU in one packed int32 each;
  * an observation is the packed pair ``row | time << 16`` (``obs[row] = 1``,
    ``obs[D-1] = 0.001 * time``, reference gridworld.py:184-205); ``GridWorld.dense_obs``
    materialises the reference's f32[D] vector on demand;
  * only ``tabular=True`` environments are implemented (every in-scope env_mode is tabular).
"""
from __future__ import annotations

from dataclasses import dataclass, fields
from typing import Optional, Tuple

import numpy as np
import torch

from .. import _shapes
from ... import _lib

LEVEL_BYTES = 192
_LEVEL_DTYPE = np.dtype([
    ("max_steps", "<i4"), ("grid_size", "<i4"), ("start_pos", "<i4"), ("n_objs", "<i4"),
    ("lifetime", "<i4"), ("buffer_id", "<i4"), ("_pad0", "<i4", (2,)),
    ("obj_pos", "<i4", (8,)), ("obj_reward", "<f4", (8,)), ("obj_p_term", "<f4", (8,)),
    ("obj_p_resp", "<f4", (8,)), ("walls", "<u4", (8,)),
])
assert _LEVEL_DTYPE.itemsize == LEVEL_BYTES


@dataclass
class EnvParams:
    """Reference gridworld.py:22-35, batched over a leading agent axis (host numpy arrays)."""
    max_steps_in_episode: np.ndarray
    random_respawn: np.ndarray
    auto_collect: np.ndarray
    grid_size: np.ndarray
    walls: np.ndarray
    start_pos: np.ndarray
    n_objs: np.ndarray
    obj_ids: np.ndarray
    static_obj_poss: np.ndarray
    obj_rewards: np.ndarray
    obj_p_terminate: np.ndarray
    obj_p_respawn: np.ndarray

    def __len__(self):
        return int(np.asarray(self.grid_size).shape[0])

    def __getitem__(self, ids) -> "EnvParams":
        return EnvParams(**{f.name: np.asarray(getattr(self, f.name))[ids] for f in fields(self)})

    def where(self, mask, other: "EnvParams") -> "EnvParams":
        """tree_map(jnp.where(mask, self, other)) over the agent axis."""
        out = {}
        for f in fields(self):
            a, b = np.asarray(getattr(self, f.name)), np.asarray(getattr(other, f.name))
            m = np.asarray(mask).reshape((-1,) + (1,) * (a.ndim - 1))
            out[f.name] = np.where(m, a, b)
        return EnvParams(**out)

    @staticmethod
    def concat(parts) -> "EnvParams":
        return EnvParams(**{f.name: np.concatenate([np.asarray(getattr(p, f.name)) for p in parts])
                            for f in fields(EnvParams)})


def pack_levels(params: EnvParams, lifetime=None, buffer_id=None) -> np.ndarray:
    """EnvParams (+ Level.lifetime / buffer_id) -> LevelRec[N] (structured numpy array).

    The per-type tables are gathered with ``obj_ids`` here, once per level, instead of on every
    step (reference gridworld.py:87,115,122 ``jnp.take(params.obj_X, params.obj_ids)``; negative
    padding ids wrap like jnp.take)."""
    n = len(params)
    rec = np.zeros(n, _LEVEL_DTYPE)
    rec["max_steps"] = params.max_steps_in_episode
    rec["grid_size"] = params.grid_size
    rec["start_pos"] = params.start_pos
    rec["n_objs"] = params.n_objs
    rec["lifetime"] = 0 if lifetime is None else lifetime
    rec["buffer_id"] = 0 if buffer_id is None else np.asarray(buffer_id).astype(np.int32)
    ids = np.asarray(params.obj_ids, np.int64)
    O = ids.shape[1]
    if O > 5:
        raise ValueError(f"max_n_objs={O} > 5 is not supported by the kernels")
    T = np.asarray(params.obj_rewards).shape[1]
    wrapped = np.clip(np.where(ids < 0, ids + T, ids), 0, T - 1)
    rec["obj_pos"][:, :O] = params.static_obj_poss
    rec["obj_pos"][:, O:] = -1
    for dst, src in (("obj_reward", params.obj_rewards), ("obj_p_term", params.obj_p_terminate),
                     ("obj_p_resp", params.obj_p_respawn)):
        rec[dst][:, :O] = np.take_along_axis(np.asarray(src, np.float32), wrapped, axis=1)
    walls = np.asarray(params.walls, bool)
    G2 = walls.shape[1]
    if G2 > 255:
        raise ValueError("max_grid_size**2 must be <= 255")
    padded = np.zeros((n, 256), bool)
    padded[:, :G2] = walls
    rec["walls"] = np.packbits(padded, axis=1, bitorder="little").view("<u4")
    return rec


def levels_to_device(rec: np.ndarray, device="cuda") -> torch.Tensor:
    t = torch.from_numpy(rec.view(np.uint8).reshape(len(rec), LEVEL_BYTES))
    _lib.h2d(t)
    return t.pin_memory().to(device, non_blocking=True) if torch.cuda.is_available() else t


class EnvState:
    """Reference gridworld.py:12-18 over ``[N, W]`` environments.  ``packed`` is the device tensor
    the kernels use (pos | exists << 8 | time << 16); the reference fields are views of it."""

    def __init__(self, packed: torch.Tensor, max_n_objs: int):
        self.packed = packed
        self.max_n_objs = max_n_objs

    @property
    def time(self):
        return (self.packed >> 16) & 0xFFFF

    @property
    def pos(self):
        return self.packed & 0xFF

    @property
    def obj_existss(self):
        bits = (self.packed >> 8) & 0xFF
        return ((bits.unsqueeze(-1) >> torch.arange(self.max_n_objs, device=bits.device)) & 1).bool()

    @property
    def early_term(self):
        return torch.zeros_like(self.packed, dtype=torch.bool)

    def clone(self):
        return EnvState(self.packed.clone(), self.max_n_objs)


class Box:
    def __init__(self, low, high, shape, dtype=np.float32):
        self.low, self.high, self.shape, self.dtype = low, high, shape, dtype


class Discrete:
    def __init__(self, n):
        self.n = n
        self.shape = ()


class GridWorld:
    """Reference gridworld.py:38-51.  gymnax-style API over batched levels."""

    def __init__(self, max_grid_size: int = 11, max_n_objs: int = 4, max_n_obj_types: int = 3,
                 tabular: bool = True):
        if not tabular:
            raise NotImplementedError("only tabular gridworlds are implemented on the B200 path")
        self.max_grid_size = max_grid_size
        self.max_n_objs = max_n_objs
        self.max_n_obj_types = max_n_obj_types
        self.tabular = tabular

    @property
    def default_params(self) -> EnvParams:
        """gridworld.py:54-70 (a batch of one level)."""
        g = 11
        return EnvParams(
            max_steps_in_episode=np.array([500], np.int32), random_respawn=np.array([False]),
            auto_collect=np.array([True]), grid_size=np.array([g], np.int32),
            walls=np.zeros((1, g * g), bool), start_pos=np.array([0], np.int32),
            n_objs=np.array([4], np.int32), obj_ids=np.array([[0, 0, 1, 2]], np.int32),
            static_obj_poss=np.array([[1 * g + 3, 3 * g + 7, 8 * g + 7, 9 * g + 2]], np.int32),
            obj_rewards=np.array([[1.0, -1.0, -1.0]], np.float32),
            obj_p_terminate=np.array([[0.0, 0.5, 0.0]], np.float32),
            obj_p_respawn=np.array([[0.05, 0.1, 0.5]], np.float32))

    @property
    def name(self) -> str:
        return "GridWorld-v0"

    @property
    def num_actions(self) -> int:
        return 5

    @property
    def obs_dim(self) -> int:
        return _shapes.obs_dim(self.max_grid_size, self.max_n_objs)

    def action_space(self, params: Optional[EnvParams] = None) -> Discrete:
        return Discrete(5)

    def observation_space(self, params: EnvParams) -> Box:
        return Box(0.0, float(np.max(params.max_steps_in_episode) - 1), (self.obs_dim,))

    # -- gymnax API ------------------------------------------------------------------------
    def _levels(self, params):
        if isinstance(params, torch.Tensor):
            return params
        return levels_to_device(pack_levels(params))

    def reset(self, key, params, num_workers: int = 1) -> Tuple[torch.Tensor, EnvState]:
        """``reset(key, params) -> (obs, state)`` for ``num_workers`` envs per level.  ``key`` is
        accepted for signature parity; tabular resets are deterministic (gridworld.py:163-165)."""
        lv = self._levels(params)
        n = lv.shape[0]
        st = torch.empty((n, num_workers), dtype=torch.int32, device=lv.device)
        obs = torch.empty_like(st)
        _lib.call("toued_env_reset", _lib.ptr(lv), _lib.ptr(st), _lib.ptr(obs), n, num_workers,
                  self.max_grid_size, _lib.stream_ptr())
        return obs, EnvState(st, self.max_n_objs)

    def step(self, key, state: EnvState, action, params):
        """``step(key, state, action, params) -> (obs, state, reward, done, info)`` with gymnax
        auto-reset.  key: uint32[N, W, 2] (numpy or tensor); action: int[N, W]."""
        lv = self._levels(params)
        n, w = state.packed.shape
        dev = lv.device
        keys = torch.as_tensor(np.ascontiguousarray(key).view(np.int32) if isinstance(key, np.ndarray) else key,
                               device=dev).contiguous().view(torch.int32)
        act = torch.as_tensor(action, device=dev).to(torch.int32).contiguous()
        st = state.packed.clone()
        obs = torch.empty_like(st)
        rew = torch.empty((n, w), dtype=torch.float32, device=dev)
        done = torch.empty((n, w), dtype=torch.uint8, device=dev)
        _lib.call("toued_env_step", _lib.ptr(lv), _lib.ptr(keys), _lib.ptr(act), _lib.ptr(st), _lib.ptr(obs),
                  _lib.ptr(rew), _lib.ptr(done), n, w, self.max_grid_size, self.max_n_objs, _lib.stream_ptr())
        return obs, EnvState(st, self.max_n_objs), rew, done.bool(), {}

    def optimal_return(self, levels, max_rollout_len: int) -> torch.Tensor:
        """Reference gridworld.py:253-323, batched: the optimal expected undiscounted first-episode return of every
        level over ``max_rollout_len`` steps (each level's ``max_steps_in_episode`` caps its episode), an upper bound
        on what any policy's evaluation (``eval_agent`` with the same horizon) can reach in expectation.  ``levels``:
        ``EnvParams`` or packed device records ``[N, 192]``.  Returns a device f64 tensor ``[N]`` (the exact DP of
        csrc/optimal_return.cu; no host synchronisation)."""
        lv = self._levels(levels)
        n = lv.shape[0]
        out = torch.empty(n, dtype=torch.float64, device=lv.device)
        _lib.call("toued_optimal_return", _lib.ptr(lv), n, int(max_rollout_len), self.max_grid_size, self.max_n_objs,
                  _lib.ptr(out), _lib.stream_ptr())
        return out

    def dense_obs(self, obs: torch.Tensor) -> torch.Tensor:
        """packed obs -> the reference's f32[..., D] observation (gridworld.py:184-199)."""
        idx = (obs & 0xFFFF).long()
        t = ((obs >> 16) & 0xFFFF).float() * 0.001
        out = torch.zeros(obs.shape + (self.obs_dim,), dtype=torch.float32, device=obs.device)
        out.scatter_(-1, idx.unsqueeze(-1), 1.0)
        out[..., -1] = t
        return out

    def __eq__(self, other):
        if not isinstance(other, GridWorld):
            return NotImplemented
        return (self.max_grid_size, self.max_n_objs, self.max_n_obj_types, self.tabular) == \
               (other.max_grid_size, other.max_n_objs, other.max_n_obj_types, other.tabular)

    def __hash__(self):
        return hash((self.max_grid_size, self.max_n_objs, self.max_n_obj_types, self.tabular))


registered_envs = ["GridWorld-v0"]
