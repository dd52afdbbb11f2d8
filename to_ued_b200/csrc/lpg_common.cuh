// LPG network parameter layout + small math helpers shared by the LPG forward/backward kernels.
// Flat parameter vector (same order as oracle/lpg.py::LPGLayout and to_ued_b200/models/lpg.py):
//   Wh[H][3H] Wi[X][3H] bi[3H] bhn[H] w_pi[H] W_y[H][Y] b_y[Y] | e_w0[Y][E] e_b0[E] e_w1[E] e_b1[1] | b_pi[1]
// with H = 256 (lpg_gru_width), Y = 8 (lpg_target_width), E = 16 (lpg_embedding_net_width),
// X = 5 (or 7 with lifetime conditioning); gate order (r, z, n) along 3H.
// Reference: models/lpg.py:39-85, flax GRUCell gate equations [3P-recall].
#pragma once
#include "common.cuh"

constexpr int LPG_H = 256;
constexpr int LPG_Y = 8;
constexpr int LPG_E = 16;
constexpr int LPG_G = 3 * LPG_H;   // 768 gate columns
constexpr int LPG_XP = 8;          // LPG input row padded to 8 floats: [r d pi pyt pyt1 (step life|0 0) 1]

struct LpgOffsets {
    int e_w0, e_b0, e_w1, e_b1, Wi, bi, Wh, bhn, w_pi, b_pi, W_y, b_y, total;
};
__host__ __device__ inline LpgOffsets lpg_offsets(int X) {
    LpgOffsets o; int p = 0;
    o.Wh = p; p += LPG_H * LPG_G;      // every block up to e_b1 starts on a 16-byte boundary
    o.Wi = p; p += X * LPG_G;
    o.bi = p; p += LPG_G;
    o.bhn = p; p += LPG_H;
    o.w_pi = p; p += LPG_H;
    o.W_y = p; p += LPG_H * LPG_Y;
    o.b_y = p; p += LPG_Y;
    o.e_w0 = p; p += LPG_Y * LPG_E;    // e_w0 e_b0 e_w1 e_b1 stay contiguous (embedding MLP)
    o.e_b0 = p; p += LPG_E;
    o.e_w1 = p; p += LPG_E;
    o.e_b1 = p; p += 1;
    o.b_pi = p; p += 1;
    o.total = p;
    return o;
}

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + __expf(-x)); }
__device__ __forceinline__ float tanhf_(float x) {
    // tanh(x) = 1 - 2 / (exp(2x) + 1); accurate to ~2 ulp with the fast exp, saturates cleanly
    const float e = __expf(2.0f * x);
    return 1.0f - 2.0f / (e + 1.0f);
}

// fast variants for the tensor-core epilogues (MUFU.EX2 + MUFU.RCP, ~2 ulp): the operands there are
// fp16/bf16-rounded anyway
// straight MUFU sequences (ex2.approx / rcp.approx, ~1e-7 absolute error, no slow-path range fix-ups:
// 2^(+big) = inf -> rcp = 0, 2^(-big) = 0 -> rcp(1) = 1, which are the correct saturated values)
__device__ __forceinline__ float ex2_approx(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcp_approx(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
// single-MUFU versions (tanh.approx.f32, max relative error 2^-11 -- the precision of the fp16 hidden state)
__device__ __forceinline__ float tanh_mufu(float x) { float y; asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float sigmoid_mufu(float x) { return fmaf(0.5f, tanh_mufu(0.5f * x), 0.5f); }
__device__ __forceinline__ float sigmoid_fast(float x) { return rcp_approx(1.0f + ex2_approx(-1.4426950408889634f * x)); }
__device__ __forceinline__ float tanh_fast(float x) { return fmaf(2.0f, rcp_approx(1.0f + ex2_approx(-2.8853900817779268f * x)), -1.0f); }

// min / max that return NaN when an operand is NaN (fminf / fmaxf return the other operand): one FMNMX, like fminf,
// and the same result on non-NaN operands.  A NaN pre-activation then reaches pi_hat / y_hat instead of turning finite.
__device__ __forceinline__ float fmin_nan(float a, float b) { float r; asm("min.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ float fmax_nan(float a, float b) { float r; asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ float fmax3_nan(float a, float b, float c) {
    float r; asm("max.NaN.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c)); return r;
}

// softmax over C values (true expf; float path, tolerance-checked)
template <int C>
__device__ __forceinline__ void softmax_c(const float (&z)[C], float (&p)[C]) {
    float m = z[0];
#pragma unroll
    for (int j = 1; j < C; ++j) m = fmaxf(m, z[j]);
    float s = 0.0f;
#pragma unroll
    for (int j = 0; j < C; ++j) { p[j] = __expf(z[j] - m); s += p[j]; }
    const float inv = 1.0f / s;
#pragma unroll
    for (int j = 0; j < C; ++j) p[j] *= inv;
}

// logits of a padded [D][8] table at a packed observation: W[row] + 0.001 * time * W[D-1]
// (plain loads: the table may have been written earlier in the same kernel)
template <int C>
__device__ __forceinline__ void tab_logits8(const float* table, int D, int32_t ob, float (&z)[C]) {
    const float tf = 0.001f * (float)ob_time(ob);
    const float4* row = reinterpret_cast<const float4*>(table + (size_t)ob_idx(ob) * 8);
    const float4* last = reinterpret_cast<const float4*>(table + (size_t)(D - 1) * 8);
    float r[8], l[8];
    const float4 a0 = row[0], a1 = row[1], b0 = last[0], b1 = last[1];
    r[0] = a0.x; r[1] = a0.y; r[2] = a0.z; r[3] = a0.w; r[4] = a1.x; r[5] = a1.y; r[6] = a1.z; r[7] = a1.w;
    l[0] = b0.x; l[1] = b0.y; l[2] = b0.z; l[3] = b0.w; l[4] = b1.x; l[5] = b1.y; l[6] = b1.z; l[7] = b1.w;
#pragma unroll
    for (int j = 0; j < C; ++j) z[j] = r[j] + tf * l[j];
}

// deterministic block-wide sum (fixed tree): every thread gets the total.  `red` >= 32 floats.
__device__ __forceinline__ float block_sum(float v, float* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    float t = (lane < nw) ? red[lane] : 0.0f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    return t;
}
