// Device-side gridworld transition (reference environments/gridworld/gridworld.py:72-211 for
// tabular levels, plus gymnax==0.0.6 Environment.step auto-reset [3P-recall]).
// Shared by the fused rollout kernel and the single-step gymnax-style entry points.
#pragma once
#include "common.cuh"

struct EnvRegs { int pos, exists, time; };   // EnvState in registers

__device__ __forceinline__ EnvRegs env_reset(const LevelRec& lev) {       // gridworld.py:157-182
    EnvRegs s; s.pos = lev.start_pos; s.exists = (1 << lev.n_objs) - 1; s.time = 0; return s;
}

__device__ __forceinline__ int obs_row(const EnvRegs& s, int G2) {        // gridworld.py:201-205
    return s.pos + G2 * s.exists;
}

// Random inputs of one env.step(key): derived from the key only, never from the state, so the
// caller can compute them ahead of the dynamics.
template <int O>
struct StepRand { float u_term; float u_resp[O]; };

template <int O>
__device__ __forceinline__ StepRand<O> env_step_rand(Key k_env) {
    StepRand<O> r;
    const Key k_step = split2_first(k_env);          // gymnax: key, key_reset = split(key)
    Key k_term, k_resp;
    split3_first_two(k_step, k_term, k_resp);        // gridworld.py:76 (obj_key dead when tabular)
    r.u_term = uniform_scalar(k_term);               // gridworld.py:116
#pragma unroll
    for (int i = 0; i < O; ++i) r.u_resp[i] = bits_to_unit(bits_elem(k_resp, O, i));   // :88
    return r;
}

// _get_next_pos (gridworld.py:138-146) on its own: the same clamping and wall test as the first block of
// env_step_apply, for callers that enumerate moves instead of simulating them (csrc/optimal_return.cu).
__device__ __forceinline__ int env_next_pos(const LevelRec& lev, int pos, int a) {
    const int gsz = lev.grid_size;
    const int col = pos % gsz;
    int step = 0;
    if (a == 0 && pos >= gsz) step = -gsz;
    else if (a == 1 && pos < gsz * (gsz - 1)) step = gsz;
    else if (a == 2 && col != 0) step = -1;
    else if (a == 3 && col != gsz - 1) step = 1;
    const int nxt = pos + step;
    const bool blocked = (lev.walls[nxt >> 5] >> (nxt & 31)) & 1u;
    return blocked ? pos : nxt;
}

// One auto-resetting transition.  Returns reward; sets done.
template <int O>
__device__ __forceinline__ float env_step_apply(const LevelRec& lev, const StepRand<O>& rnd, int a,
                                                EnvRegs& s, bool& done) {
    const int gsz = lev.grid_size;
    {   // _get_next_pos, gridworld.py:138-146
        const int col = s.pos % gsz;
        int step = 0;
        if (a == 0 && s.pos >= gsz) step = -gsz;
        else if (a == 1 && s.pos < gsz * (gsz - 1)) step = gsz;
        else if (a == 2 && col != 0) step = -1;
        else if (a == 3 && col != gsz - 1) step = 1;
        const int nxt = s.pos + step;
        const bool blocked = (lev.walls[nxt >> 5] >> (nxt & 31)) & 1u;
        s.pos = blocked ? s.pos : nxt;
    }
    const int full_mask = (1 << lev.n_objs) - 1;
    int collected = 0, respawn = 0;
    float p_term = 0.0f, rew = 0.0f;
#pragma unroll
    for (int i = 0; i < O; ++i) {
        const bool c = ((s.exists >> i) & 1) && (lev.obj_pos[i] == s.pos);          // :83-84
        collected |= (c ? 1 : 0) << i;
        respawn |= (rnd.u_resp[i] < lev.obj_p_resp[i] ? 1 : 0) << i;                // :87-88
        const float cf = c ? 1.0f : 0.0f;
        p_term = __fadd_rn(p_term, __fmul_rn(lev.obj_p_term[i], cf));               // :115-116
        rew = __fadd_rn(rew, __fmul_rn(lev.obj_reward[i], cf));                     // :122-123
    }
    s.exists = (s.exists | respawn) & ~collected & full_mask;                       // :89,108,111-112
    const bool term = rnd.u_term < p_term;           // early_term is never carried (auto-reset)
    s.time += 1;
    done = (s.time >= lev.max_steps) || term;        // :207-211
    if (done) s = env_reset(lev);                    // gymnax auto-reset
    return rew;
}
