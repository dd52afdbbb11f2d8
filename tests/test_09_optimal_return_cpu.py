"""The vectorised optimal-return DP (tests/optimal_return_np.py::optimal_return_batch, the numpy twin of
csrc/optimal_return.cu) against the loop DP it restates, hand-derived known answers, and the checkpoint check of
meta_test.py.  No GPU."""
import os

import numpy as np
import pytest

from oracle import configs, prng
from oracle.gridworld import EnvParams, GridWorld, optimal_return
from optimal_return_np import optimal_return_batch


def _close(a, b, rel):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    assert np.all(np.abs(a - b) <= rel * np.maximum(np.abs(b), 1.0)), (a, b)


def _generated(mode, n, seed):
    p, _ = configs.reset_env_params(prng.split(prng.PRNGKey(seed), n), mode)
    kw, _ = configs.get_env_spec(mode)
    return GridWorld(**kw), p


@pytest.mark.parametrize("mode,seed,horizon", [("debug", 0, 30), ("debug", 1, 7), ("small", 2, 30), ("small", 3, 12)])
def test_batch_matches_loop_on_generated_levels(mode, seed, horizon):
    env, p = _generated(mode, 6, seed)
    got = optimal_return_batch(env, p, horizon)
    want = [optimal_return(env, p, horizon, agent=i) for i in range(len(p))]
    _close(got, want, 1e-12)


def test_generated_levels_cover_walls_negative_rewards_and_respawn():
    """The 24 levels above include walls, negative rewards and p_respawn > 0 (so the comparison exercises them)."""
    walls = neg = resp = 0
    for mode, seed in (("debug", 0), ("debug", 1), ("small", 2), ("small", 3)):
        env, p = _generated(mode, 6, seed)
        r = env._take_type(p.obj_rewards, p.obj_ids)
        pr = env._take_type(p.obj_p_respawn, p.obj_ids)
        live = np.arange(env.max_n_objs)[None, :] < p.n_objs[:, None]
        walls += int(p.walls.any(1).sum())
        neg += int(((r < 0) & live).any(1).sum())
        resp += int(((pr > 0) & live).any(1).sum())
    assert walls > 0 and neg > 0 and resp > 0, (walls, neg, resp)


def one_object_level(g, d, reward, p_term, p_resp, max_steps, extra_objs=0):
    """Wall-free g x g grid, start at cell 0, one object at cell d of the first row (plus ``extra_objs`` padding
    slots); a batch of one level."""
    O = 1 + extra_objs
    return GridWorld(max_grid_size=g, max_n_objs=O, max_n_obj_types=1), EnvParams(
        max_steps_in_episode=np.array([max_steps], np.int32), random_respawn=np.array([False]),
        auto_collect=np.array([True]), grid_size=np.array([g], np.int32), walls=np.zeros((1, g * g), bool),
        start_pos=np.array([0], np.int32), n_objs=np.array([1], np.int32),
        obj_ids=np.array([[0] + [-1] * extra_objs], np.int32),
        static_obj_poss=np.array([[d] + [g * g - 1] * extra_objs], np.int32),
        obj_rewards=np.array([[reward]], np.float32), obj_p_terminate=np.array([[p_term]], np.float32),
        obj_p_respawn=np.array([[p_resp]], np.float32))


def known_answer(d, reward, p_term, p_resp, hp):
    """Optimal return of ``one_object_level`` with H' = min(max_steps, horizon) (p_term, p_resp in {0, 1})."""
    if reward <= 0 or d > hp:
        return 0.0
    if p_term == 1.0:
        return float(reward)                               # collected once at step d, the episode ends
    if p_resp == 1.0:
        return float(reward) * ((hp - d) // 2 + 1)      # absent for one step after each collection, then back
    return float(reward)


KNOWN = [  # g, d, reward, p_term, p_resp, max_steps, horizon
    (5, 3, 1.0, 1.0, 0.0, 50, 10), (5, 3, 1.0, 1.0, 0.0, 2, 10), (5, 4, 2.5, 1.0, 0.5, 50, 4),
    (5, 4, 2.5, 1.0, 0.5, 50, 3), (6, 2, 1.0, 0.0, 1.0, 50, 11), (6, 2, 1.0, 0.0, 1.0, 9, 30),
    (6, 5, 0.5, 0.0, 1.0, 40, 25), (4, 1, 1.0, 0.0, 1.0, 20, 20), (5, 2, -1.0, 1.0, 0.0, 20, 20),
    (5, 2, -1.0, 0.0, 1.0, 20, 20), (5, 3, 1.0, 0.0, 1.0, 3, 30), (5, 3, 1.0, 0.0, 1.0, 2, 30),
]


@pytest.mark.parametrize("g,d,reward,p_term,p_resp,max_steps,horizon", KNOWN)
@pytest.mark.parametrize("extra_objs", [0, 2])
def test_known_answers(g, d, reward, p_term, p_resp, max_steps, horizon, extra_objs):
    env, p = one_object_level(g, d, reward, p_term, p_resp, max_steps, extra_objs)
    want = known_answer(d, reward, p_term, p_resp, min(max_steps, horizon))
    assert optimal_return_batch(env, p, horizon)[0] == pytest.approx(want, rel=1e-12, abs=1e-12)
    assert optimal_return(env, p, horizon) == pytest.approx(want, rel=1e-12, abs=1e-12)


def test_several_objects_on_one_cell_are_collected_together():
    """Two objects on the same cell: one step collects both (rewards and termination probabilities add up)."""
    g = 4
    env = GridWorld(max_grid_size=g, max_n_objs=2, max_n_obj_types=2)
    p = EnvParams(max_steps_in_episode=np.array([20], np.int32), random_respawn=np.array([False]),
                  auto_collect=np.array([True]), grid_size=np.array([g], np.int32), walls=np.zeros((1, g * g), bool),
                  start_pos=np.array([0], np.int32), n_objs=np.array([2], np.int32), obj_ids=np.array([[0, 1]], np.int32),
                  static_obj_poss=np.array([[2, 2]], np.int32), obj_rewards=np.array([[1.0, 0.5]], np.float32),
                  obj_p_terminate=np.array([[0.25, 0.5]], np.float32), obj_p_respawn=np.array([[0.3, 0.0]], np.float32))
    for h in (1, 2, 5, 12):
        _close(optimal_return_batch(env, p, h), [optimal_return(env, p, h)], 1e-12)
    assert optimal_return_batch(env, p, 2)[0] == pytest.approx(1.5)


def test_batch_mixes_levels_of_different_shapes():
    """A level's value does not depend on the other levels of the batch."""
    env, p = _generated("small", 8, 5)
    whole = optimal_return_batch(env, p, 20)
    for i in range(len(p)):
        assert optimal_return_batch(env, p.index([i]), 20)[0] == whole[i]


def test_meta_test_rejects_mismatched_checkpoint_before_cuda(tmp_path, monkeypatch):
    import meta_test as mt
    from to_ued_b200 import _lib

    def _no_gpu(*a, **k):
        raise AssertionError("meta_test.py touched the CUDA library before checking the checkpoint")
    monkeypatch.setattr(_lib, "lib", _no_gpu)
    monkeypatch.setattr(_lib, "call", _no_gpu)
    ck = os.path.join(tmp_path, "checkpoint_2.npz")
    np.savez(ck, params=np.zeros(203946, np.float32), step=np.asarray(2))
    with pytest.raises(ValueError, match=r"203946.*205482"):
        mt.main(["--checkpoint", ck, "--env_mode", "small", "--num_agents", "8", "--lifetime_conditioning"])
    es = os.path.join(tmp_path, "checkpoint_3.npz")
    np.savez(es, params=np.zeros(205482, np.float32), **{"es_state/mean": np.zeros(203946 + 1, np.float32)})
    with pytest.raises(ValueError, match=r"es_state/mean.*203947.*205482"):
        mt.main(["--checkpoint", es, "--env_mode", "small", "--lifetime_conditioning"])
    with pytest.raises(ValueError, match="Unknown args"):
        mt.main(["--checkpoint", ck, "--no_such_flag", "1"])
    assert mt.load_lpg_params(ck, False).shape == (203946,)
