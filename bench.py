#!/usr/bin/env python
"""Benchmark of the LPG meta-training hot path (BASELINE.json metric: gridworld agent env-steps/s
including the LPG update, and meta-steps/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--config lpg_all_shortlife|tabular8|groove_mazes|talpg_es|double_oracle] [--scaling strong|weak]
                    [--dump-outputs DIR]

Default config = BASELINE configs[1]: LPG meta-gradient, env_mode all_shortlife, 512 agents x 64 workers x 20 steps x
K = 5 updates.  A "step" is one full iteration of the reference's train loop (train.py:32-52): the meta-step
(lpg_meta_grad_train_step or lpg_es_train_step) + level_sampler.sample.  Prints ONE JSON line (rank 0).

Scaling over N GPUs: ``strong`` (default) shards the 512 agents of the north-star workload over the ranks (SURVEY.md
section 8e: 64 agents per GPU at N = 8); the line additionally carries a ``weak_scaling`` object (512 agents PER GPU)
measured in the same run.  ``value`` counts the env-steps actually simulated by the enqueued rollouts (all ranks) in the
timed region, divided by the max-over-ranks device time.

--impl reference times the CPU restatement of the reference (oracle/, torch CPU + numpy; the JAX reference itself cannot
be installed in this image) on a bounded sample of the same workload.

--dump-outputs DIR writes, after the timed steps, what the last timed step returned to its caller (LPG train state,
agents, value critics, level buffer(s), metrics; rank 0's share) as DIR/<name>.npy, so that two builds can be compared
output for output: the inputs are seeded, so the same arguments give the same inputs on every run.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CPU_SAMPLE_AGENTS = 8

# BASELINE.json `configs`, in order; `agents` is the GLOBAL meta-batch
CONFIGS = {
    "tabular8": dict(baseline=0, agents=8, kind="metagrad", env_mode="tabular",
                     flags=["--env_mode", "tabular"],
                     what="LPG meta-training, env_mode=tabular, num_agents=8, num_mini_batches=1 (BASELINE configs[0])"),
    "lpg_all_shortlife": dict(baseline=1, agents=512, kind="metagrad", env_mode="all_shortlife",
                              flags=["--env_mode", "all_shortlife"],
                              what="LPG meta-gradient step (train.py loop body), env_mode=all_shortlife, 512 agents "
                                   "(BASELINE configs[1])"),
    "groove_mazes": dict(baseline=2, agents=512, kind="metagrad", env_mode="mazes",
                         flags=["--env_mode", "mazes", "--score_function", "alg_regret", "--buffer_size", "2048"],
                         what="GROOVE: LPG + PLR with score_function=alg_regret on env_mode=mazes, 512 agents, buffer 2048 "
                              "(BASELINE configs[2])"),
    "talpg_es": dict(baseline=3, agents=512, kind="es", env_mode="all_vrandlife",
                     flags=["--env_mode", "all_vrandlife", "--use_es", "--lifetime_conditioning"],
                     what="TA-LPG: ES with antithetic task sampling, lifetime conditioning, env_mode=all_vrandlife, "
                          "population 1024 (BASELINE configs[3])"),
    "double_oracle": dict(baseline=4, agents=32, kind="do", env_mode="mazes",
                          flags=["--env_mode", "mazes", "--score_function", "alg_regret", "--buffer_size", "6", "-br", "16",
                                 "--train_steps", "5"],
                          what="train_do.py double-oracle / Nash level sampler on mazes: one outer iteration = meta-step + "
                               "train/eval best responses + payoff matrix + Nash solve, buffer 6 (BASELINE configs[4])"),
}
DEFAULT_CONFIG = "lpg_all_shortlife"


# ------------------------------------------------------------------------------------------------
def cpu_reference_step(n_agents, env_mode, seed=0, threads=None):
    """One meta-gradient step of the CPU oracle on n_agents agents of env_mode; returns (seconds, env-steps)."""
    import numpy as np
    import torch
    from oracle import prng, configs
    from oracle.gridworld import GridWorld
    from oracle.rollout import RolloutWrapper
    from oracle.lpg import LPGLayout, init_lpg_params
    from oracle.agents import AgentTables
    from oracle.meta import lpg_meta_grad_train_step, Adam
    if threads:
        torch.set_num_threads(threads)
    kw, ep = configs.get_env_spec(env_mode)
    env = GridWorld(**kw)
    ro = RolloutWrapper(env, 20, ep)
    keys = prng.split(prng.PRNGKey(seed), n_agents)
    p, life = configs.reset_env_params(keys, env_mode)
    D = env.obs_dim
    rs = np.random.RandomState(seed)
    f = lambda c: torch.tensor((rs.randn(n_agents, D, c) / np.sqrt(D)).astype(np.float32))
    ag = AgentTables(f(5), f(8), torch.zeros(n_agents, dtype=torch.long))
    value = f(1)
    lay = LPGLayout()
    flat = torch.tensor(init_lpg_params(lay, seed))
    adam = Adam(lay.size, 1e-4)
    s0 = ro.batch_reset(None, p, 64)
    t0 = time.perf_counter()
    out = lpg_meta_grad_train_step(prng.PRNGKey(seed + 1), lay, flat, ag, value, ro, p, s0, life)
    adam.step(flat, out["grad"])
    dt = time.perf_counter() - t0
    return dt, n_agents * (5 * 64 * 20 + 64 * 20 + 4 * ep)


def run_reference(a):
    """Reference arm: the CPU restatement on the host cores (rank 0 only)."""
    import torch
    if int(os.environ.get("RANK", "0")) != 0:
        return
    cfg = CONFIGS[a.config]
    torch.set_num_threads(os.cpu_count() or 1)          # torchrun pins OMP_NUM_THREADS=1; use every host core
    cores = torch.get_num_threads()
    n = min(CPU_SAMPLE_AGENTS, cfg["agents"])
    for _ in range(a.warmup):
        cpu_reference_step(2, cfg["env_mode"])
    times, steps = [], 0
    for i in range(a.steps):
        dt, steps = cpu_reference_step(n, cfg["env_mode"], seed=i)
        times.append(dt)
    per_step = sum(times) / len(times)
    val = steps / per_step
    sample = (f"{n} of {cfg['agents']} agents, one LPG meta-gradient step on env_mode={cfg['env_mode']} each step "
              "(oracle: torch CPU + numpy restatement of the reference, not JAX)")
    if cfg["kind"] != "metagrad":
        sample += "; the inner loop shared with this config (rollout + LPG agent update), not its ES / double-oracle outer logic"
    line = {
        "impl": "reference", "metric": "gridworld agent env-steps/sec incl. LPG update", "value": val,
        "unit": "env-steps/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": per_step * 1e3, "higher_is_better": True, "scaling": a.scaling, "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": cfg["what"] + " -- CPU restatement of the reference (not JAX)", "name": a.config,
                   "agents": n, "env_workers": 64, "train_rollout_len": 20, "num_agent_updates": 5},
        "meta_steps_per_s": 1.0 / per_step * n / cfg["agents"],
        "cpu_baseline": {"value": val, "unit": "env-steps/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                self.rows.append([c.strip() for c in out.strip().split(",")])
            except Exception:
                pass
            time.sleep(0.05)

    def summary(self):
        import statistics
        sm = [float(r[0]) for r in self.rows if len(r) >= 8 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) < 8:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


def _flat_metrics(metrics):
    out = []
    for k, v in metrics.items():
        if k.startswith("_"):
            continue
        if isinstance(v, dict):
            out += [vv for vv in v.values()]
        else:
            out.append(v)
    return out


class Workload:
    """One BASELINE config on this rank: builds the state and exposes one_step() = the train-loop body."""

    def __init__(self, name, n_global, world, cuda_graph=None, mini_batches=None):
        import torch
        from to_ued_b200.util import prng
        from to_ued_b200.experiments.parse_args import parse_args
        from to_ued_b200.meta.meta import create_lpg_train_state, make_lpg_train_step
        self.cfg = cfg = CONFIGS[name]
        self.name, self.n_global, self.world = name, n_global, world
        self.n_local = n_global // world
        pop_local = self.n_local * (2 if cfg["kind"] == "es" else 1)
        if mini_batches is None:
            # chunks only pay when every chunk still fills the GPU with 128-row tiles (DESIGN.md section 7)
            mini_batches = int(os.environ.get("TOUED_BENCH_MINI_BATCHES", "2" if self.n_local >= 512 and cfg["kind"] == "metagrad" else "1"))
        self.mini_batches = mini_batches
        self.args = args = parse_args(cfg["flags"] + ["--num_agents", str(n_global), "--num_mini_batches", str(mini_batches)])
        self.prng = prng
        rng = prng.PRNGKey(args.seed)
        if cfg["kind"] == "do":
            self._init_do(rng)
            return
        from to_ued_b200.environments.level_sampler import LevelSampler
        rng, lpg_rng, buffer_rng = prng.split(rng, 3)
        self.train_state = create_lpg_train_state(lpg_rng, args)
        self.sampler = LevelSampler(args)
        self.buf = self.sampler.initialize_buffer(buffer_rng)
        rng, _rng = prng.split(rng, 2)
        self.buf, self.agents, self.vcs = self.sampler.initial_sample(_rng, self.buf, n_global, not args.use_es)
        self.step_fn = make_lpg_train_step(args, self.sampler, cuda_graph=cuda_graph)
        self.eager_fn = make_lpg_train_step(args, self.sampler, cuda_graph=False) if cfg["kind"] == "metagrad" else self.step_fn
        self.rng = rng
        self.metrics = None
        self.meta_steps = 0

    # ---- double oracle: one outer iteration of train_do.py:30-71 ----
    def _init_do(self, rng):
        import torch
        import train_do
        from to_ued_b200.environments.nash_sampler import NashSampler
        from to_ued_b200.meta.meta import create_lpg_train_state, make_lpg_train_step
        args, prng = self.args, self.prng
        B = args.buffer_size
        self.train_nash = torch.zeros(B, device="cuda"); self.train_nash[0] = 1
        self.eval_nash = torch.zeros(B, device="cuda"); self.eval_nash[0] = 1
        self.sampler = NashSampler(args)
        rng, buffer_rng, train_rng = prng.split(rng, 3)
        self.train_buffer, self.eval_buffer = self.sampler.initialize_buffers(buffer_rng)
        self.train_state = create_lpg_train_state(train_rng, args)
        self.step_fn = make_lpg_train_step(args, self.sampler, cuda_graph=False)
        self.eager_fn = self.step_fn
        self.rng, self.t, self._write = rng, 1, train_do._write_level
        self.metrics = None
        self.meta_steps = 0

    def _one_step_do(self):
        prng, s, args = self.prng, self.sampler, self.args
        t = 1 + (self.t - 1) % (args.buffer_size - 1)
        self.rng, _rng = prng.split(self.rng, 2)
        agents, vcs = s.get_training_levels(_rng, self.train_buffer, self.train_nash, create_value_critic=True)
        self.rng, _rng = prng.split(self.rng, 2)
        self.train_state, agents, vcs, metrics = self.step_fn(rng=_rng, lpg_train_state=self.train_state,
                                                              agent_states=agents, value_critic_states=vcs)
        self.rng, k1, k2, k3 = prng.split(self.rng, 4)
        new_train = s.get_train_br(k1, self.train_state, self.eval_nash, self.eval_buffer)
        new_eval, _ = s.get_eval_br(k2, self.train_state)
        self.train_buffer = self._write(self.train_buffer, t, new_train)
        self.eval_buffer = self._write(self.eval_buffer, t, new_eval)
        self.train_nash, self.eval_nash, _ = s.compute_nash(k3, self.train_state, self.train_buffer, self.eval_buffer)
        self.t += 1
        self.metrics = metrics
        self.meta_steps += 1

    def one_step(self, fn=None, **kw):
        if self.cfg["kind"] == "do":
            return self._one_step_do()
        prng = self.prng
        self.rng, _rng = prng.split(self.rng, 2)
        self.train_state, self.agents, self.vcs, self.metrics = (fn or self.step_fn)(
            rng=_rng, lpg_train_state=self.train_state, agent_states=self.agents, value_critic_states=self.vcs, **kw)
        self.rng, _rng = prng.split(self.rng, 2)
        self.buf, self.agents, self.vcs = self.sampler.sample(_rng, self.buf, self.agents, self.vcs)
        self.meta_steps += 1

    def pending_recreation(self):
        a = self.agents
        return self.cfg["kind"] != "do" and a.host_step is not None and bool((a.host_step >= a.level.lifetime).any())


def _barrier(world):
    import torch
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


def _allmax(vals, world):
    import torch
    t = torch.tensor(vals, dtype=torch.float64, device="cuda")
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(x) for x in t]


def _allsum(vals, world):
    import torch
    t = torch.tensor(vals, dtype=torch.float64, device="cuda")
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(t)
    return [float(x) for x in t]


def timed_device(wl, steps, world):
    """K steps, device-timed, inputs resident, no host reads of results: (ms, env-steps of all ranks, launches)."""
    import torch
    from to_ued_b200 import _lib
    _barrier(world)
    _lib.reset_counters(profile=False)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        wl.one_step()
    e1.record()
    _barrier(world)
    ms = _allmax([e0.elapsed_time(e1)], world)[0]
    env_steps = _allsum([_lib.ENV_STEPS[0]], world)[0]
    return ms, env_steps, _lib.kernel_launches()


def timed_e2e(wl, steps, world):
    """K steps end to end through the public API: host key in, the step's result scalars read back every step."""
    import torch
    from to_ued_b200 import _lib
    _barrier(world)
    _lib.reset_counters(profile=False)
    t0 = time.perf_counter()
    d2h = 0
    for _ in range(steps):
        wl.one_step()
        flat = _flat_metrics(wl.metrics)
        host = torch.stack([f.reshape(()) if hasattr(f, "reshape") else torch.tensor(float(f)) for f in flat]).cpu()   # ONE D2H read
        d2h = host.numel() * host.element_size()
    _barrier(world)
    ms = _allmax([(time.perf_counter() - t0) * 1e3], world)[0]
    env_steps = _allsum([_lib.ENV_STEPS[0]], world)[0]
    return ms, env_steps, _lib.H2D_BYTES[0] / steps, d2h


DUMP_BUDGET = 64 << 20     # bytes of all dumped arrays together
DUMP_SAMPLE = 1 << 20      # an output with more elements is dumped as a fixed, seeded sample of this many


def output_arrays(wl):
    """name -> array of what the last one_step() returned to its caller (rank 0's share of the agents)."""
    from to_ued_b200.experiments.logging import _buffer_arrays, _train_state_arrays, to_host
    out = {}

    def put(prefix, tree):
        for k, v in tree.items():
            if isinstance(v, dict):
                put(f"{prefix}.{k}", v)
            else:
                out[f"{prefix}.{k.replace('/', '.')}"] = v

    put("train_state", _train_state_arrays(wl.train_state))
    put("metrics", to_host(wl.metrics))
    if wl.cfg["kind"] == "do":
        put("train_buffer", _buffer_arrays(wl.train_buffer))
        put("eval_buffer", _buffer_arrays(wl.eval_buffer))
        out["train_nash"], out["eval_nash"] = wl.train_nash, wl.eval_nash
        return out
    if wl.buf is not None:                   # domain randomisation keeps no level buffer
        put("level_buffer", _buffer_arrays(wl.buf))
    ag = wl.agents
    for name, ts in (("agents.actor", ag.actor_state), ("agents.critic", ag.critic_state), ("value_critics", wl.vcs)):
        if ts is not None:                   # ES steps return no value critics
            out[f"{name}.kernel"], out[f"{name}.step"] = ts.kernel, ts.step
    out["agents.env_obs"], out["agents.env_state"] = ag.env_obs, ag.env_state.packed
    out["agents.level.lifetime"], out["agents.level.buffer_id"] = ag.level.lifetime, ag.level.buffer_id
    return out


def dump_outputs(arrays, directory):
    """Write every array as <directory>/<name>.npy: floats as float32 (float64 stays float64), integers and booleans as
    float64 (exact to 2**53).  An array of more than DUMP_SAMPLE elements is written flat, as the elements at DUMP_SAMPLE
    indices drawn with a fixed seed (the same indices for the same size)."""
    import numpy as np
    import torch
    host = {}
    for name, a in arrays.items():
        if isinstance(a, torch.Tensor):
            a = (a.float() if a.dtype in (torch.float16, torch.bfloat16) else a).detach().cpu().numpy()
        a = np.asarray(a)
        a = a.astype(np.float32 if a.dtype.kind == "f" and a.dtype != np.float64 else np.float64)
        if a.size > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(0).choice(a.size, DUMP_SAMPLE, replace=False))
            a = a.reshape(-1)[idx]
        host[name] = a
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_BUDGET:
        raise SystemExit(f"--dump-outputs: {total} bytes of outputs exceed the {DUMP_BUDGET}-byte budget")
    os.makedirs(directory, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def run_ours(a):
    import torch
    import torch.distributed as dist
    import to_ued_b200
    from to_ued_b200 import _lib

    cfg = CONFIGS[a.config]
    precision = to_ued_b200.GRU_PRECISION
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if (a.agents or cfg["agents"]) % world != 0 and a.scaling == "strong":
        raise SystemExit(f"config {a.config}: {a.agents or cfg['agents']} agents do not split over {world} GPUs")
    base_agents = a.agents or cfg["agents"]
    n_global = base_agents if a.scaling == "strong" else base_agents * world
    wl = Workload(a.config, n_global, world)
    for _ in range(a.warmup):
        wl.one_step()
    _barrier(world)

    # ---- timed region 1: device-timed throughput ----
    clocks = ClockSampler(local) if rank == 0 else None
    if clocks:
        clocks.start()
    dev_ms, env_steps, launches = timed_device(wl, a.steps, world)
    # ---- timed region 2: end to end through the public API ----
    e2e_ms, e2e_env_steps, h2d, d2h = timed_e2e(wl, a.steps, world)
    if clocks:
        clocks.stop_flag = True
        clocks.join(timeout=2)
    # the graphed step returns views of its static buffers, which the untimed steps below overwrite
    if a.dump_outputs and rank == 0:
        dump_outputs(output_arrays(wl), a.dump_outputs)

    # ---- per-kernel CUDA-event times for the roofline / shares: eager enqueue (no graph), the mini-batches one after the
    #      other on one stream and no side streams, so that every launch is timed without a concurrent neighbour ----
    PROF_STEPS = 2
    prof, prof_kw = {}, ({"num_streams": 1} if cfg["kind"] == "metagrad" else {})
    if cfg["kind"] in ("metagrad", "es"):
        to_ued_b200.SIDE_STREAMS = False
        wl.one_step(wl.eager_fn, **prof_kw)
        _barrier(world)
        _lib.reset_counters(profile=True)
        for _ in range(PROF_STEPS):
            wl.one_step(wl.eager_fn, **prof_kw)
        _barrier(world)
        prof = _lib.profile_ms()
        _lib.reset_counters(profile=False)
        to_ued_b200.SIDE_STREAMS = True

    # ---- the step that re-creates agents (lifetime reached): run on until the sampler has to act, time that call and the
    #      step after it (which re-uploads the re-created agents into the graph's static buffers) ----
    recreate = None
    if cfg["kind"] == "metagrad" and a.config == DEFAULT_CONFIG:
        prng = wl.prng
        for _ in range(60):
            wl.rng, _rng = prng.split(wl.rng, 2)
            wl.train_state, wl.agents, wl.vcs, wl.metrics = wl.step_fn(rng=_rng, lpg_train_state=wl.train_state,
                                                                       agent_states=wl.agents, value_critic_states=wl.vcs)
            wl.meta_steps += 1
            pending = wl.pending_recreation()
            wl.rng, _rng = prng.split(wl.rng, 2)
            if pending:
                n_term = int((wl.agents.host_step >= wl.agents.level.lifetime).sum())
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                wl.buf, wl.agents, wl.vcs = wl.sampler.sample(_rng, wl.buf, wl.agents, wl.vcs)
                torch.cuda.synchronize()
                t1 = time.perf_counter()
                wl.one_step()
                torch.cuda.synchronize()
                t2 = time.perf_counter()
                r = _allmax([(t1 - t0) * 1e3, (t2 - t1) * 1e3], world)
                recreate = {"at_meta_step": wl.meta_steps, "agents_recreated_on_rank0": n_term, "sample_ms": r[0],
                            "next_step_ms": r[1],
                            "note": "level_sampler.sample with terminated agents (new levels drawn on the host, tables "
                                    "re-initialised and envs reset on the device), host-timed with a synchronize on both sides"}
                break
            wl.buf, wl.agents, wl.vcs = wl.sampler.sample(_rng, wl.buf, wl.agents, wl.vcs)

    # ---- same-precision number: the exact-fp32 SIMT GRU path on the same workload (N = 1 only) ----
    fp32_path = None
    if world == 1 and cfg["kind"] == "metagrad" and precision == "tc" and a.config == DEFAULT_CONFIG and not a.no_fp32:
        to_ued_b200.GRU_PRECISION = "fp32"
        w32 = Workload(a.config, n_global, world, cuda_graph=False)
        for _ in range(2):
            w32.one_step()
        ms32, steps32, _ = timed_device(w32, 3, world)
        fp32_path = {"ms_per_step": ms32 / 3, "value": steps32 / (ms32 * 1e-3), "unit": "env-steps/s", "steps": 3,
                     "note": "TOUED_GRU_PRECISION=fp32: exact-fp32 SIMT GRU kernels (the reference's arithmetic type), eager enqueue"}
        del w32
        to_ued_b200.GRU_PRECISION = precision
        from to_ued_b200.meta.train import _WS_CACHE
        _WS_CACHE.clear()
        torch.cuda.empty_cache()

    # ---- the other scaling mode, measured in the same run (N > 1, default config) ----
    other = None
    if world > 1 and a.config == DEFAULT_CONFIG and not a.no_other_scaling:
        if hasattr(wl.step_fn, "release"):
            wl.step_fn.release()
        from to_ued_b200.meta.train import _WS_CACHE
        _WS_CACHE.clear()
        torch.cuda.empty_cache()
        n_other = base_agents * world if a.scaling == "strong" else base_agents
        wo = Workload(a.config, n_other, world)
        for _ in range(a.warmup):
            wo.one_step()
        oms, osteps, _ = timed_device(wo, a.steps, world)
        other = {"scaling": "weak" if a.scaling == "strong" else "strong", "global_agents": n_other,
                 "agents_per_gpu": n_other // world, "ms_per_step": oms / a.steps, "value": osteps / (oms * 1e-3),
                 "unit": "env-steps/s", "meta_steps_per_s": 1e3 / (oms / a.steps)}

    def _shutdown():
        from to_ued_b200.util import dist as udist
        udist.shutdown(*[w.step_fn for w in (wl,) if hasattr(w, "step_fn")], *([wo.step_fn] if other else []))
    if rank != 0:
        _shutdown()
        return
    ms_per_step = dev_ms / a.steps
    value = env_steps / (dev_ms * 1e-3)
    e2e_val = e2e_env_steps / (e2e_ms * 1e-3)
    args = wl.args
    K, W, L = args.num_agent_updates, args.env_workers, args.train_rollout_len

    # ---- roofline of the dominant kernel (live CUDA-event times of the per-kernel pass) ----
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    per_launch_agents = max(1, wl.n_local * (2 if cfg["kind"] == "es" else 1) // wl.mini_batches)
    tokens = per_launch_agents * W * L
    fl_fwd = 403968.0 if args.lifetime_conditioning else 400896.0
    flops = {   # algorithmic FLOPs per launch (DESIGN.md section 5)
        "toued_gru_forward": tokens * fl_fwd, "toued_gru_forward_tc": tokens * fl_fwd, "toued_gru_forward_tc_multi": tokens * fl_fwd,
        "toued_gru_backward": per_launch_agents * W * (L - 1) * 2.0 * 768 * 256 + tokens * 2.0 * 256 * 9,
        "toued_gru_backward_tc": per_launch_agents * W * (L - 1) * 2.0 * 768 * 256 + tokens * 2.0 * 256 * 9,
        "toued_lpg_wgrad": tokens * (2.0 * 256 * 768 + 2.0 * 8 * 768 + 2.0 * 256 * 9),
        "toued_lpg_wgrad_tc": tokens * (2.0 * 256 * 768 + 2.0 * 8 * 768 + 2.0 * 256 * 9),
    }
    hbm_bytes = {"toued_gru_forward_tc": tokens * BYTES_PER_TOKEN["toued_gru_forward_tc"],
                 "toued_gru_backward_tc": tokens * BYTES_PER_TOKEN["toued_gru_backward_tc"],
                 "toued_lpg_wgrad_tc": tokens * BYTES_PER_TOKEN["toued_lpg_wgrad_tc"]}
    total_prof = sum(ms for _, ms in prof.values()) or 1.0
    shares = {k: {"calls": c, "ms_per_step": ms / PROF_STEPS, "share": ms / total_prof} for k, (c, ms) in prof.items()}
    roofline = None
    cand = [k for k in prof if k in flops]
    if cand:
        dom = max(cand, key=lambda k: prof[k][1])
        calls, ms = prof[dom]
        achieved = flops[dom] / (ms / calls * 1e-3) / 1e12
        peak = peaks.get("bf16_tflops_sustained", 1400.0)
        traffic = None
        try:
            ncu = json.load(open(os.path.join(ROOT, "profiles", NCU_SUMMARY)))
            traffic = ncu["kernels"][dom]["dram_bytes_per_token"] * tokens
        except Exception:
            pass
        roofline = {"kernel": dom, "bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                    "frac": achieved / peak, "traffic": traffic, "agents_per_launch": per_launch_agents,
                    "ms_per_launch": ms / calls,
                    "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (of measured)" if peaks else "fallback 1400 (of fallback)",
                    "note": ("tcgen05 path (fp16/bf16 operands, fp32 accumulate in TMEM)" if precision == "tc" else
                             "exact-fp32 SIMT GRU path") + "; FLOPs = algorithmic GRU/head/weight-gradient FLOPs per launch"}
        if dom in hbm_bytes:
            gbs = hbm_bytes[dom] / (ms / calls * 1e-3) / 1e9
            roofline["hbm"] = {"achieved": gbs, "peak": peaks.get("hbm_gbs", 6556.8), "unit": "GB/s",
                               "frac": gbs / peaks.get("hbm_gbs", 6556.8),
                               "note": "algorithmic activation bytes of the same kernel (DESIGN.md section 3)"}
    elif "toued_rollout" in prof or "toued_a2c_train" in prof:
        dom = "toued_a2c_train" if "toued_a2c_train" in prof else "toued_rollout"
        calls, ms = prof[dom]
        gbs = 10.2 * (env_steps / a.steps / world) / max(ms / PROF_STEPS * 1e-3, 1e-9) / 1e9
        roofline = {"kernel": dom, "bound": "hbm", "achieved": gbs, "peak": peaks.get("hbm_gbs", 6556.8), "unit": "GB/s",
                    "frac": gbs / peaks.get("hbm_gbs", 6556.8), "traffic": None,
                    "note": "10.2 B written per env-step (DESIGN.md section 3); issue/latency-bound, see DESIGN.md section 7"}

    if roofline is None:
        gbs = 10.2 * (env_steps / world) / (dev_ms * 1e-3) / 1e9
        roofline = {"kernel": "rollout kernels over the whole step", "bound": "hbm", "achieved": gbs,
                    "peak": peaks.get("hbm_gbs", 6556.8), "unit": "GB/s", "frac": gbs / peaks.get("hbm_gbs", 6556.8), "traffic": None,
                    "note": "no per-kernel pass for this config: 10.2 B written per env-step (DESIGN.md section 3) over the step time"}

    # ---- CPU baseline on a bounded sample (rank 0, N=1 only) ----
    cpu = None
    if world == 1:
        n = min(CPU_SAMPLE_AGENTS, cfg["agents"])
        dt, steps_cpu = cpu_reference_step(n, cfg["env_mode"])
        cpu = {"value": steps_cpu / dt, "unit": "env-steps/s", "cores": torch.get_num_threads(), "kind": "port",
               "sample": f"one LPG meta-gradient step of {n} of the {cfg['agents']} agents on env_mode={cfg['env_mode']} ({dt:.1f} s); "
                         "CPU restatement of the reference (torch CPU + numpy), not JAX"}
    graph = bool(getattr(wl.step_fn, "graph", None) is not None) if hasattr(wl, "step_fn") else to_ued_b200.CUDA_GRAPH
    line = {
        "metric": "gridworld agent env-steps/sec incl. LPG update", "value": value, "unit": "env-steps/s",
        "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": a.scaling, "vs_baseline": None,
        "dtype": ("f16/bf16 operands, f32 accumulate (GRU); f32 elsewhere" if precision == "tc" else "f32"), "data": "synthetic",
        "config": {"workload": f"{cfg['what']}: {n_global} agents over {world} GPU(s) = {wl.n_local} per GPU x {W} workers x {L} steps"
                               + (f" x K={K} updates" if cfg["kind"] != "es" else " x lifetime updates per candidate")
                               + f", num_mini_batches={wl.mini_batches}"
                               + (" (run concurrently on CUDA streams; the reference README uses 16 sequential mini-batches as a "
                                  "memory device, results identical)" if wl.mini_batches > 1 else ""),
                   "name": a.config, "gru_precision": precision, "agents_per_gpu": wl.n_local, "global_agents": n_global,
                   "env_steps_per_meta_step": env_steps / a.steps, "cuda_graph": graph,
                   "l2_policy": "working set per step exceeds L2 (activations of one update > 2 GB); no explicit flush"},
        "meta_steps_per_s": 1e3 / ms_per_step,
        "e2e": {"value": e2e_val, "unit": "env-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_ms / a.steps},
        "gpu_launches": launches, "roofline": roofline, "kernel_shares": shares,
        "clocks": clocks.summary() if clocks else None,
    }
    if cpu:
        line["cpu_baseline"] = cpu
    if fp32_path:
        line["fp32_path"] = fp32_path
    if recreate:
        line["recreate"] = recreate
    if other:
        line[other["scaling"] + "_scaling"] = other
    print(json.dumps(line), flush=True)
    _shutdown()


# algorithmic HBM bytes per token of the tensor-core kernels (DESIGN.md section 3: fp16 gate planes + h, bf16 dG / h' images)
BYTES_PER_TOKEN = {"toued_gru_forward_tc": 32.0 + 4 * 512 + 512 + 512 + 36,
                   "toued_gru_backward_tc": 4 * 512 + 512 + 72 + 2048 + 40.0,
                   "toued_lpg_wgrad_tc": 2048 + 512 + 512 + 128 + 36.0}
NCU_SUMMARY = "r02_ncu_summary.json"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default=DEFAULT_CONFIG, choices=sorted(CONFIGS))
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--agents", type=int, default=0, help="override the config's global number of agents (experiments: "
                    "e.g. 64 = the per-GPU load of the 8-GPU strong-scaling run)")
    ap.add_argument("--no-fp32", dest="no_fp32", action="store_true", help="skip the exact-fp32 path measurement")
    ap.add_argument("--no-other-scaling", dest="no_other_scaling", action="store_true",
                    help="N > 1: skip the second (weak / strong) measurement")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR",
                    help="after the timed steps, write the last timed step's outputs as DIR/<name>.npy (--impl ours; "
                         "bench_outputs/ is git-ignored for this)")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
