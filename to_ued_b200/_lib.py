"""ctypes binding of libtoued.so (the C ABI in include/toued.h).

There is no CPU fallback: importing this module without the built library, or calling an op
without a CUDA device, raises.  Build with ``python -m to_ued_b200.csrc.build`` (or
``__graft_entry__.build()``)."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# TOUED_LIB_VARIANT selects a diagnostic build of the same sources (csrc/build.py::build(variant=...)), e.g. the
# schedule-fuzz library used by tests/test_90_full_size_gpu.py; production always loads libtoued.so
_VARIANT = os.environ.get("TOUED_LIB_VARIANT", "")
LIB_PATH = os.path.join(_HERE, f"libtoued_{_VARIANT}.so" if _VARIANT else "libtoued.so")

_lib = None


class TouedError(RuntimeError):
    pass


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise TouedError(
                f"{LIB_PATH} is missing: the CUDA extension is not built. "
                "Run `python -m to_ued_b200.csrc.build` (there is no CPU fallback).")
        _lib = C.CDLL(LIB_PATH)
        _declare(_lib)
    return _lib


_P, _I, _F = C.c_void_p, C.c_int, C.c_float

# name -> argtypes; every function returns int except the two below
SIGNATURES = {
    "toued_rollout": [_P] * 10 + [_I] * 7 + [_P],
    "toued_env_step": [_P] * 7 + [_I] * 4 + [_P],
    "toued_env_reset": [_P] * 3 + [_I] * 3 + [_P],
    "toued_sort_tokens": [_P] * 2 + [_I] * 3 + [_P],
    "toued_lpg_prepare": [_P] * 11 + [_I] * 6 + [_P],
    "toued_gru_forward": [_P] * 7 + [_I] * 5 + [_P],
    "toued_agent_update": [_P] * 12 + [_I] * 4 + [_F] * 4 + [_I, _P, _P],
    "toued_agent_scratch_floats": [_I] * 4,
    "toued_meta_loss": [_P] * 10 + [_I] * 5 + [_F] * 3 + [_I, _P],
    "toued_agent_backward": [_P] * 14 + [_I] * 4 + [_F] * 9 + [_P, _P],
    "toued_transpose_wh": [_P] * 3,
    "toued_gru_backward": [_P] * 10 + [_I] * 4 + [_P],
    "toued_lpg_wgrad_workspace_floats": [],
    "toued_lpg_wgrad": [_P] * 11 + [_I] * 6 + [_P],
    "toued_reduce_partials": [_P, _P, _I, _I, _I, _P],
    "toued_lpg_wgrad_splits": [_I],
    "toued_lpg_wgrad_workspace_offset": [_I],
    "toued_lpg_wgrad_embed": [_P] * 7 + [_I] * 6 + [_P],
    "toued_cotangent_max": [_P, _P, _I, _I, _I, _P, _P],
    "toued_pack_wh_backward": [_P] * 3,
    "toued_gru_backward_tc": [_P] * 12 + [_I] * 4 + [_P],
    "toued_wgrad_tc_splits": [],
    "toued_wgrad_tc_small_splits": [],
    "toued_lpg_wgrad_tc": [_P] * 9 + [_I] * 4 + [_P],
    "toued_adam": [_P] * 4 + [_I, _I] + [_F] * 4 + [_P],
    "toued_adam_dev": [_P] * 5 + [_I] + [_F] * 4 + [_P],
    "toued_sgd_clip": [_P] * 3 + [_I, _F, _F, _P],
    "toued_get_nash": [_P] * 5 + [_I] * 4 + [_F, _P],
    "toued_projection_simplex": [_P, _I, _I, _P],
    "toued_es_ask": [_P, _P, _F, _P, _I, _I, _I, _P],
    "toued_es_tell": [_P] * 5 + [_I, _I, _I] + [_F] * 5 + [_I, _F, _P],
    "toued_es_ask_shard": [_P, _P, _F, _P, _I, _I, _I, _I, _I, _P],
    "toued_es_grad_partial": [_P] * 4 + [_I, _I, _I, _F, _P],
    "toued_es_adam": [_P] * 4 + [_I, _I] + [_F] * 5 + [_I, _F, _P],
    "toued_a2c_update": [_P] * 12 + [_I] * 4 + [_F] * 6 + [_I, _P],
    "toued_a2c_train": [_P] * 15 + [_I] * 7 + [_F] * 6 + [_I, _P],
    "toued_init_tables": [_P] * 3 + [_I] * 3 + [_P],
    "toued_masked_reset": [_P] * 5 + [_I] * 3 + [_P],
    "toued_generate_levels_desc_bytes": [],
    "toued_generate_levels": [_P] * 5 + [_I, _P],
    "toued_plr_reset_lowest": [_P] * 3 + [_I, _I, _P, _P],
    "toued_plr_select": [C.c_uint32, C.c_uint32] + [_P] * 3 + [_I] + [_P] * 3 + [_I, _F, _F, _I, _P, _P],
    "toued_tc_gemm_test": [_P] * 5,
    "toued_tc_gemm_mixed_test": [_P] * 5,
    "toued_tc_gemm_mn_test": [_P] * 4 + [_I] * 3 + [_P],
    "toued_tc_gemm_mn2_test": [_P] * 5,
    "toued_tc_gemm_mn_x16_test": [_P] * 6,
    "toued_pack_wh_forward": [_P, _P, _I, _P],
    "toued_pack_wh_forward_multi": [_P, _P, _I, _I, _I, _P],
    "toued_gru_forward_tc_multi": [_P] * 6 + [_I] * 5 + [_P],
    "toued_host_iota_bits": [_P, _I, _I, _P],
    "toued_key_split": [_P, _I, _I, _I, _I, _P, _P],
    "toued_key_chain": [_P, _I, _I, _P, _P, _P],
    "toued_gru_forward_tc": [_P] * 9 + [_I] * 4 + [_P],
    "toued_optimal_return": [_P] + [_I] * 4 + [_P, _P],
}


def _declare(l):
    l.toued_last_error.restype = C.c_char_p
    l.toued_last_error.argtypes = []
    l.toued_version.restype = _I
    l.toued_version.argtypes = []
    for name, args in SIGNATURES.items():
        fn = getattr(l, name)
        fn.restype = _I
        fn.argtypes = args


def ptr(t):
    """device pointer of a torch tensor (None -> NULL).  Refuses CPU tensors: no fallback."""
    if t is None:
        return None
    if not t.is_cuda:
        raise TouedError("to_ued_b200 ops need CUDA tensors (there is no CPU fallback)")
    if not t.is_contiguous():
        raise TouedError("to_ued_b200 ops need contiguous tensors")
    return t.data_ptr()


def stream_ptr():
    import torch
    return torch.cuda.current_stream().cuda_stream


# kernels launched by one call of each entry point (for the bench's gpu_launches count)
KERNELS_PER_CALL = {"toued_adam_dev": 2, "toued_sgd_clip": 2, "toued_lpg_wgrad": 3, "toued_init_tables": 2, "toued_lpg_wgrad_tc": 2, "toued_pack_wh_forward": 2, "toued_pack_wh_forward_multi": 2}
LAUNCHES = {}          # entry point -> number of calls since reset_counters()
GRAPH_KERNELS = [0]    # kernels launched by CUDA-graph replays since reset_counters() (meta/graph.py)
ENV_STEPS = [0]        # gridworld env-steps simulated by the enqueued rollouts since reset_counters() (bench.py's metric)
PROFILE = None         # when a dict: entry point -> list of (start, end) CUDA events


H2D_BYTES = [0]        # bytes of host->device copies made by the package since reset_counters()


def h2d(t):
    """Count a host tensor / array about to be copied to the device; returns it unchanged."""
    H2D_BYTES[0] += int(t.numel() * t.element_size()) if hasattr(t, "element_size") else int(t.nbytes)
    return t


def reset_counters(profile=False):
    global PROFILE
    H2D_BYTES[0] = 0
    GRAPH_KERNELS[0] = 0
    ENV_STEPS[0] = 0
    LAUNCHES.clear()
    PROFILE = {} if profile else None


def kernel_launches():
    return sum(n * KERNELS_PER_CALL.get(k, 1) for k, n in LAUNCHES.items()) + GRAPH_KERNELS[0]


def profile_ms():
    """entry point -> (calls, total ms); call after torch.cuda.synchronize()."""
    return {k: (len(v), sum(a.elapsed_time(b) for a, b in v)) for k, v in (PROFILE or {}).items()}


def call(name, *args):
    LAUNCHES[name] = LAUNCHES.get(name, 0) + 1
    if name == "toued_rollout":                      # (.., n_agents, n_workers, rollout_len, ..) at 10..12
        ENV_STEPS[0] += args[10] * args[11] * args[12]
    elif name == "toued_a2c_train":                  # (.., num_updates, n_agents, n_workers, rollout_len, ..) at 15..18
        ENV_STEPS[0] += args[15] * args[16] * args[17] * args[18]
    if PROFILE is not None:
        import torch
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        rc = getattr(lib(), name)(*args)
        b.record()
        PROFILE.setdefault(name, []).append((a, b))
    else:
        rc = getattr(lib(), name)(*args)
    if rc != 0:
        raise TouedError(f"{name} failed ({rc}): {lib().toued_last_error().decode()}")
