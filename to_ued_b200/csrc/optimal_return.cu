// Optimal expected first-episode return of tabular gridworld levels: the exact finite-horizon DP of the reference's
// optimal_return (environments/gridworld/gridworld.py:253-323, restated in oracle/gridworld.py::optimal_return) over
// the level's MDP with state (cell, exists mask), in fp64.  Used to normalise meta-test returns (meta/meta_test.py).
//
// One CTA per level.  Each thread owns fixed (cell, mask) items and keeps their values V_{t+1} in registers.  A DP step
// t = H'-1 .. 0 (H' = min(horizon, max_steps); time >= max_steps is terminal) is two phases:
//   1. E[n][m] = expected V_{t+1}[n][m'] after the agent stepped onto cell n holding mask m: every object i absent in m
//      respawns with probability p_resp[i] independently, an object present in m stays present unless it sits on n
//      (collected: its bit goes to 0 and it cannot respawn in the same step).  The expectation factorises over objects,
//      so it is a subset transform over the mask bits: one warp-shuffle butterfly per object (the nm = 2^n_objs masks
//      of a cell are consecutive lanes of one warp), instead of a sum over all successor masks.
//   2. V_t[c][m] = max_a  r(coll) + E[nxt][m] * (1 - p_term(coll)),  nxt = _get_next_pos(c, a),  coll = m & objs(nxt)
//      (any number of objects may be collected at once: r / p_term are tabulated per collected subset, in object order).
// The only shared array is E (cells x nm doubles, <= 255 x 32 x 8 B = 65 KB).  Every value is computed by one thread with
// individually rounded fp64 operations in a fixed order, so the result is bitwise reproducible and independent of the
// batch size and of the level's position in the batch; tests/optimal_return_np.py::optimal_return_batch performs the same
// operations in numpy.
#include "gridworld.cuh"
#include "../../include/toued.h"

#define OR_THREADS 512
#define OR_ITEMS 16               // ceil(255 cells x 32 masks / 512 threads)

__global__ void __launch_bounds__(OR_THREADS)
optimal_return_kernel(const LevelRec* __restrict__ levels, int horizon, int max_cells, int max_objs,
                      double* __restrict__ out) {
    extern __shared__ double sE[];                    // [cells][nm]
    __shared__ LevelRec lev;
    __shared__ double s_r[32], s_pt[32];              // reward / termination probability of each collected subset
    __shared__ double s_p[TOUED_MAX_OBJS], s_q[TOUED_MAX_OBJS];   // p_resp, 1 - p_resp
    __shared__ uint8_t s_obj[256];                    // mask of the objects placed on each cell
    __shared__ uint8_t s_nxt[256 * TOUED_NUM_ACTIONS];
    const int tid = threadIdx.x;
    if (tid == 0) lev = levels[blockIdx.x];
    __syncthreads();
    const int g = lev.grid_size, cells = g * g, no = lev.n_objs;
    if (no < 0 || no > max_objs || g <= 0 || cells > max_cells) {   // malformed record: NaN, not a fault
        if (tid == 0) out[blockIdx.x] = __longlong_as_double(0x7ff8000000000000ll);
        return;
    }
    const int nm = 1 << no, total = cells * nm;
    const int H = min(horizon, lev.max_steps);
    for (int c = tid; c < cells; c += OR_THREADS) {
        int b = 0;
        for (int i = 0; i < no; ++i) b |= (lev.obj_pos[i] == c ? 1 : 0) << i;
        s_obj[c] = (uint8_t)b;
        for (int a = 0; a < TOUED_NUM_ACTIONS; ++a) s_nxt[c * TOUED_NUM_ACTIONS + a] = (uint8_t)env_next_pos(lev, c, a);
    }
    if (tid < nm) {
        double r = 0.0, pt = 0.0;
        for (int i = 0; i < no; ++i)
            if ((tid >> i) & 1) {
                r = __dadd_rn(r, (double)lev.obj_reward[i]);
                pt = __dadd_rn(pt, (double)lev.obj_p_term[i]);
            }
        s_r[tid] = r;
        s_pt[tid] = pt;
    }
    if (tid < no) {
        s_p[tid] = (double)lev.obj_p_resp[tid];
        s_q[tid] = __dsub_rn(1.0, (double)lev.obj_p_resp[tid]);
    }
    __syncthreads();

    double v[OR_ITEMS];
#pragma unroll
    for (int j = 0; j < OR_ITEMS; ++j) v[j] = 0.0;
    for (int t = 0; t < H; ++t) {
        // ---- phase 1: respawn expectation of V_{t+1} per (next cell, mask)
#pragma unroll
        for (int j = 0; j < OR_ITEMS; ++j) {
            if (j * OR_THREADS >= total) break;                   // block-uniform: whole warps stay together
            const int item = j * OR_THREADS + tid;
            const bool live = item < total;
            const int m = item & (nm - 1);
            const int ob = live ? s_obj[item >> no] : 0;
            double e = v[j];
            for (int i = 0; i < no; ++i) {
                const double part = __shfl_xor_sync(0xffffffffu, e, 1 << i);
                if ((m >> i) & 1) e = ((ob >> i) & 1) ? part : e;                     // kept (1) or collected (0)
                else e = __dadd_rn(__dmul_rn(s_p[i], part), __dmul_rn(s_q[i], e));  // absent: respawns w.p. p
            }
            if (live) sE[item] = e;
        }
        __syncthreads();
        // ---- phase 2: Bellman maximum over the five actions
#pragma unroll
        for (int j = 0; j < OR_ITEMS; ++j) {
            if (j * OR_THREADS >= total) break;
            const int item = j * OR_THREADS + tid;
            if (item >= total) continue;
            const int c = item >> no, m = item & (nm - 1);
            if ((lev.walls[c >> 5] >> (c & 31)) & 1u) { v[j] = 0.0; continue; }
            double best = 0.0;
#pragma unroll
            for (int a = 0; a < TOUED_NUM_ACTIONS; ++a) {
                const int n = s_nxt[c * TOUED_NUM_ACTIONS + a];
                const int col = m & s_obj[n];
                const double val = __dadd_rn(s_r[col], __dmul_rn(sE[n * nm + m], __dsub_rn(1.0, s_pt[col])));
                best = a == 0 ? val : fmax(best, val);
            }
            v[j] = best;
        }
        __syncthreads();
    }
    const int target = lev.start_pos * nm + (nm - 1);             // (start_pos, all n_objs objects present)
#pragma unroll
    for (int j = 0; j < OR_ITEMS; ++j)
        if (j * OR_THREADS + tid == target) out[blockIdx.x] = v[j];
}

extern "C" int toued_optimal_return(const void* levels, int n_levels, int horizon, int max_grid_size, int max_n_objs,
                                    double* out, void* stream) {
    TOUED_CHECK(n_levels >= 0 && horizon >= 0, "toued_optimal_return: n_levels=%d, horizon=%d", n_levels, horizon);
    TOUED_CHECK(max_n_objs >= 0 && max_n_objs <= 5, "toued_optimal_return: max_n_objs=%d > 5", max_n_objs);
    TOUED_CHECK(max_grid_size > 0 && max_grid_size * max_grid_size <= 255,
                "toued_optimal_return: max_grid_size^2=%d > 255", max_grid_size * max_grid_size);
    if (n_levels == 0) return 0;
    const int max_cells = max_grid_size * max_grid_size;
    const size_t smem = sizeof(double) * (size_t)max_cells << max_n_objs;
    TOUED_CUDA(cudaFuncSetAttribute(optimal_return_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    optimal_return_kernel<<<n_levels, OR_THREADS, smem, (cudaStream_t)stream>>>((const LevelRec*)levels, horizon,
                                                                               max_cells, max_n_objs, out);
    TOUED_LAUNCH_CHECK();
    return 0;
}
