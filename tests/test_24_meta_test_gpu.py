"""Meta-testing on the B200: the optimal-return kernel (csrc/optimal_return.cu) against its numpy twin, its
reproducibility, the DP as an upper bound on trained agents' returns, the inference-only GRU forward without h16, and
the meta-test driver (to_ued_b200/meta/meta_test.py) and entry point (meta_test.py) against direct calls."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import configs, prng
from oracle.gridworld import GridWorld as OGrid
from optimal_return_np import optimal_return_batch
from oracle.maze_data import MAZE_WALL_MASKS
from test_09_optimal_return_cpu import KNOWN, known_answer, one_object_level

pytestmark = pytest.mark.gpu


def _product(env_o, p_o):
    from to_ued_b200.environments.gridworld.gridworld import EnvParams, GridWorld
    env = GridWorld(env_o.max_grid_size, env_o.max_n_objs, env_o.max_n_obj_types)
    return env, EnvParams(**{k: getattr(p_o, k) for k in p_o.__dataclass_fields__})


def _assert_matches(got, want):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    assert np.all(np.abs(got - want) <= 1e-9 * np.maximum(np.abs(want), 1.0)), (got, want)


def _kernel(env_o, p_o, horizon):
    env, p = _product(env_o, p_o)
    out = env.optimal_return(p, horizon)
    assert out.dtype == torch.float64 and out.is_cuda
    return out.cpu().numpy()


def _levels(mode, n, seed):
    p, _ = configs.reset_env_params(prng.split(prng.PRNGKey(seed), n), mode)
    kw, ep = configs.get_env_spec(mode)
    return OGrid(**kw), p, ep


def test_kernel_known_answers(built_lib):
    for g, d, r, pt, pr, ms, h in KNOWN:
        for extra in (0, 2):
            env, p = one_object_level(g, d, r, pt, pr, ms, extra)
            got = _kernel(env, p, h)
            _assert_matches(got, optimal_return_batch(env, p, h))
            _assert_matches(got, [known_answer(d, r, pt, pr, min(ms, h))])


@pytest.mark.parametrize("modes,n,horizon", [
    (("all_shortlife",), 8, 750),
    (tuple(MAZE_WALL_MASKS), 1, 50),
    (("dense", "longer", "long_dense"), 1, 2000),
])
def test_kernel_matches_numpy_dp(built_lib, modes, n, horizon):
    for i, mode in enumerate(modes):
        env, p, _ = _levels(mode, n, 11 + i)
        _assert_matches(_kernel(env, p, horizon), optimal_return_batch(env, p, horizon))


def test_kernel_is_bitwise_reproducible_and_batch_independent(built_lib):
    from to_ued_b200.environments.gridworld.levelgen import generate_levels
    from to_ued_b200.environments.gridworld.gridworld import GridWorld
    kw, ep = configs.get_env_spec("all_shortlife")
    env = GridWorld(**kw)
    packed = generate_levels(prng.split(prng.PRNGKey(7), 512), "all_shortlife", device="cuda")
    a = env.optimal_return(packed, ep)
    b = env.optimal_return(packed, ep)
    assert torch.equal(a, b)
    for i in (0, 1, 77, 300, 511):
        alone = env.optimal_return(packed[i:i + 1].contiguous(), ep)
        assert torch.equal(alone, a[i:i + 1]), i
    assert bool((a >= 0).all()) and bool(torch.isfinite(a).all())


def test_kernel_rejects_unsupported_sizes(built_lib):
    from to_ued_b200 import _lib
    from to_ued_b200.environments.gridworld.gridworld import GridWorld
    out = torch.empty(1, dtype=torch.float64, device="cuda")
    lv = torch.zeros((1, 192), dtype=torch.uint8, device="cuda")
    with pytest.raises(_lib.TouedError, match="max_n_objs"):
        _lib.call("toued_optimal_return", _lib.ptr(lv), 1, 10, 5, 6, _lib.ptr(out), _lib.stream_ptr())
    with pytest.raises(_lib.TouedError, match="max_grid_size"):
        _lib.call("toued_optimal_return", _lib.ptr(lv), 1, 10, 16, 3, _lib.ptr(out), _lib.stream_ptr())
    assert GridWorld(4, 2, 2).optimal_return(lv[:0], 10).shape == (0,)


# ---------------------------------------------------------------------------------------------- meta-test driver
def _sampler(mode="small", extra=()):
    from to_ued_b200.environments.level_sampler import LevelSampler
    from to_ued_b200.experiments.parse_args import parse_args
    return LevelSampler(parse_args(["--env_mode", mode, "--num_agents", "8", "--num_mini_batches", "1", *extra]))


def _lpg(seed=0, cond=False):
    from to_ued_b200.models.lpg import LPG
    return LPG(lifetime_conditioning=cond).init(prng.split(prng.PRNGKey(seed), 2)[0], device="cuda")


RNG = prng.split(prng.PRNGKey(0), 2)[1]


def test_upper_bound_holds_for_trained_agents(built_lib):
    from to_ued_b200.meta.meta_test import meta_test
    sampler = _sampler()
    curve, pts, opt, agents = meta_test(RNG, _lpg(), False, sampler, 8, 40, 20, 64)
    ro = sampler.rollout_manager
    obs, st = ro.batch_reset(None, agents.level.packed, 64)
    keys = prng.split(prng.PRNGKey(99), 8)
    _, _, _, ret = ro.batch_rollout(keys, agents.actor_state, agents.level.packed, obs, st, eval=True,
                                    want_trajectory=False)
    ret = ret.double().cpu().numpy()
    mean, se = ret.mean(1), ret.std(1, ddof=1) / np.sqrt(ret.shape[1])
    assert np.all(mean <= opt + 5 * se + 1e-5), (mean, opt, se)
    assert pts.tolist() == [0, 20, 40] and curve.shape == (3, 8) and np.isfinite(curve).all()


def test_gru_forward_tc_without_h16_is_bitwise_equal(built_lib):
    from helpers import Case
    from to_ued_b200 import _lib
    from to_ued_b200.agents.lpg_agent import Tape
    c = Case("all_shortlife", n=3, seed=4, table_scale=0.3)
    ag, ro = c.agent_state()
    lpg = torch.from_numpy(c.lpg).cuda()
    p, s = _lib.ptr, _lib.stream_ptr()
    traj, _, _, _ = ro.batch_rollout(c.keys, ag.actor_state, ag.level.packed, ag.env_obs, ag.env_state)
    tape = Tape(c.n, c.w, c.L, c.D, 1, "cuda", precision="tc")
    tape.obs[0].copy_(traj.obs); tape.action[0].copy_(traj.action)
    tape.reward[0].copy_(traj.reward); tape.done[0].copy_(traj.done)
    _lib.call("toued_lpg_prepare", p(tape.obs[0]), p(tape.action[0]), p(tape.reward[0]), p(tape.done[0]),
              p(ag.actor_state.params), p(ag.critic_state.params), p(lpg), p(ag.actor_state.step), p(ag.level.packed),
              p(tape.x[0]), None, c.n, c.w, c.L, c.D, 0, 0, s)
    _lib.call("toued_pack_wh_forward", p(lpg), p(tape.wh_img), 0, s)
    outs = []
    for h16, fac, hp in ((None, None, None), (tape.h16[0], None, None), (tape.h16[0], tape.fac[0], tape.hpimg[0])):
        tape.pi_hat.fill_(float("nan")); tape.y_hat.fill_(float("nan"))
        _lib.call("toued_gru_forward_tc", p(tape.x[0]), p(tape.done[0]), p(lpg), p(tape.wh_img), p(h16), p(fac), p(hp),
                  p(tape.pi_hat[0]), p(tape.y_hat[0]), c.n, c.w, c.L, 0, s)
        outs.append((tape.pi_hat[0].clone(), tape.y_hat[0].clone()))
    for pi, y in outs[1:]:
        assert torch.equal(pi, outs[0][0]) and torch.equal(y, outs[0][1])
    assert bool(torch.isfinite(outs[0][0]).all())
    with pytest.raises(_lib.TouedError, match="h16"):        # the reverse-pass buffers still need h16
        _lib.call("toued_gru_forward_tc", p(tape.x[0]), p(tape.done[0]), p(lpg), p(tape.wh_img), None, p(tape.fac[0]),
                  None, p(tape.pi_hat[0]), p(tape.y_hat[0]), c.n, c.w, c.L, 0, s)
    inference = Tape(c.n, c.w, c.L, c.D, 5, "cuda", keep_gates=False, precision="tc")
    assert inference.h16 is None and inference.fac is None and inference.hpimg is None


def test_meta_test_training_matches_recording_tape_and_ignores_eval_interval(built_lib):
    from types import SimpleNamespace
    from to_ued_b200.agents.agents import eval_agent
    from to_ued_b200.agents.lpg_agent import Tape, train_lpg_agent
    from to_ued_b200.meta.meta_test import meta_test, split_keys, create_test_agents
    from to_ued_b200.models.lpg import LPG
    from to_ued_b200.util import prng as dprng
    sampler = _sampler()
    ro, env, K, N = sampler.rollout_manager, sampler.env, 40, 8
    lpg = _lpg()
    c1, p1, o1, a1 = meta_test(RNG, lpg, False, sampler, N, K, K, 64)
    c7, p7, o7, a7 = meta_test(RNG, lpg, False, sampler, N, K, 7, 64)
    assert p1.tolist() == [0, 40] and p7.tolist() == [0, 7, 14, 21, 28, 35, 40]
    # recording tape (keep_gates=True, writes h16 and the other reverse-pass buffers), one call with K updates
    keys = split_keys(RNG, N)
    fresh = create_test_agents(keys, sampler, N)
    tape = Tape(N, sampler.env_workers, ro.train_rollout_len, env.obs_dim, K, "cuda", keep_gates=True)
    ref, _, _ = train_lpg_agent(keys["train"], SimpleNamespace(params=lpg, model=LPG()), fresh, ro, K, 0.5, tape=tape)
    for a in (a1, a7):
        assert torch.equal(a.actor_state.params, ref.actor_state.params)
        assert torch.equal(a.critic_state.params, ref.critic_state.params)
        assert torch.equal(a.actor_state.step, ref.actor_state.step)
        assert torch.equal(a.critic_state.step, ref.critic_state.step)
        assert torch.equal(a.env_state.packed, ref.env_state.packed)
    assert int(ref.actor_state.step.min()) == K            # small: lifetime 250 > 40, every update counted
    # curve points 0 and last: eval_agent with the documented eval keys
    ev = dprng.chain_device(dprng.to_device(keys["eval"], "cuda"), len(p7))
    first = eval_agent(ev[0], ro, fresh.level.packed, fresh.actor_state, 64)       # (train_lpg_agent left it as is)
    last = eval_agent(ev[len(p7) - 1], ro, ref.level.packed, ref.actor_state, 64)
    assert np.array_equal(c7[0], first.cpu().numpy()) and np.array_equal(c1[0], c7[0])
    assert np.array_equal(c7[-1], last.cpu().numpy())
    assert np.array_equal(o1, o7)
    _assert_matches(o1, sampler.env.optimal_return(fresh.level.packed, ro.eval_rollout_len).cpu().numpy())


def test_meta_test_randlife_stops_at_lifetime(built_lib):
    from to_ued_b200.meta.meta_test import meta_test
    sampler = _sampler("all_vrandlife")
    _, pts, _, agents = meta_test(RNG, _lpg(), False, sampler, 8, 30, 15, 16)
    life = np.asarray(agents.level.lifetime)
    assert np.array_equal(agents.actor_state.step.cpu().numpy(), np.minimum(life, 30))


def _train_and_checkpoint(tmp_path, monkeypatch, group, extra=()):
    import train
    monkeypatch.setenv("TOUED_LOG_DIR", str(tmp_path))
    train.main(["--env_mode", "small", "--num_agents", "8", "--num_mini_batches", "1", "--train_steps", "2", "--log",
                "--wandb_group", group, *extra])
    run = [d for d in os.listdir(tmp_path) if d.startswith(group + "-")][0]
    return os.path.join(tmp_path, run, "checkpoints", "checkpoint_2.npz")


MT_ARGS = ["--env_mode", "small", "--num_agents", "8", "--num_updates", "30", "--eval_interval", "10"]


def test_meta_test_entry_point_end_to_end(built_lib, tmp_path, monkeypatch):
    import meta_test as entry
    ck = _train_and_checkpoint(tmp_path, monkeypatch, "mg")
    outs = []
    for i in range(2):
        f = os.path.join(tmp_path, f"r{i}.json")
        entry.main(["--checkpoint", ck, *MT_ARGS, "--out", f])
        outs.append(open(f).read())
    assert outs[0] == outs[1]
    r = json.loads(outs[0])
    assert set(r) == {"config", "eval", "mean_optimal_return", "num_excluded_levels", "levels"}
    assert r["config"]["checkpoint"] == ck and r["config"]["num_updates"] == 30 and r["config"]["env_mode"] == "small"
    assert [e["update"] for e in r["eval"]] == [0, 10, 20, 30]
    for e in r["eval"]:
        assert set(e) == {"update", "mean_return", "min_return", "max_return", "mean_normalised_score"}
        assert e["min_return"] <= e["mean_return"] <= e["max_return"]
    assert set(r["levels"]) == {"optimal", "final_return", "lifetime"}
    assert all(len(v) == 8 for v in r["levels"].values())
    assert 0 <= r["num_excluded_levels"] <= 8


def test_meta_test_es_checkpoint_uses_es_mean(built_lib, tmp_path, monkeypatch, capsys):
    import meta_test as entry
    from to_ued_b200.meta.meta_test import meta_test, summarize
    ck = _train_and_checkpoint(tmp_path, monkeypatch, "es", ["--use_es", "--lifetime_conditioning"])
    z = np.load(ck)
    mean = z["es_state/mean"]
    assert mean.shape == (205482,) and np.abs(mean).max() > 0            # ES moved its mean; params stay the init
    capsys.readouterr()
    r = entry.main(["--checkpoint", ck, *MT_ARGS, "--lifetime_conditioning"])
    printed = json.loads(capsys.readouterr().out)
    assert printed == json.loads(json.dumps(r))
    sampler = _sampler(extra=["--lifetime_conditioning"])
    curve, pts, opt, _ = meta_test(RNG, mean, True, sampler, 8, 30, 10, 64)
    direct = summarize(curve, pts, opt)
    assert r["eval"] == direct["eval"] and r["levels"]["final_return"] == direct["levels"]["final_return"]
    assert r["levels"]["optimal"] == direct["levels"]["optimal"]
    with pytest.raises(ValueError, match="205482.*203946"):
        entry.main(["--checkpoint", ck, *MT_ARGS])
