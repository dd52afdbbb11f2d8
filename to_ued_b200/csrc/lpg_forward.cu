// LPG forward pass for one agent update (reference agents/lpg_agent.py:46-59 + models/lpg.py:48-85):
//
//   toued_sort_tokens   per-agent stable sort of the T = W*L trajectory tokens by table row, so that
//                       every later row-scatter (gradients, adjoints) is a deterministic segmented sum
//   toued_lpg_prepare   actor / critic row gathers + softmax, selected-action probability, the
//                       embedding MLP on y_t / y_{t+1}, and the LPG input row x = [r d pi pyt pyt1 ..]
//   toued_gru_forward   reverse GRU over the L steps for R = N*W sequences + relu + the two heads
//                       (pi_hat, y_hat = softmax).  Exact-fp32 SIMT version: a CTA owns 64 sequences,
//                       keeps their hidden state in shared memory across all L steps and streams the
//                       256x768 recurrent matrix from L2 in double-buffered cp.async chunks.
//
// Layouts: trajectory tensors are [n][t][w]; LPG tensors are time-major [t][row], row = n*W + w.
#include "lpg_common.cuh"
#include "tc.cuh"
#include "../../include/toued.h"

// ------------------------------------------------------------------------------------------------
// token sort: key = row << 12 | token  (token = t*W + w < 4096; keys are unique, so the order is that of a stable
// sort by row).  Bitonic network over P2 = 256 * E keys, thread t holding keys [t*E, (t+1)*E) in registers:
// exchange distances below E stay in registers, distances below 32 E go through warp shuffles, and only the few
// cross-warp distances go through shared memory (6 of the 66 stages at P2 = 2048).
template <int E>
__device__ __forceinline__ void sort_cmpx(uint32_t& mine, uint32_t other, bool keep_min) {
    const uint32_t lo = min(mine, other), hi = max(mine, other);
    mine = keep_min ? lo : hi;
}

template <int E>
__global__ void __launch_bounds__(256)
sort_tokens_reg_kernel(const int32_t* __restrict__ obs, uint16_t* __restrict__ sorted_tok, int W, int L, int T) {
    constexpr int P2 = 256 * E;
    __shared__ uint32_t xch[P2];
    const int n = blockIdx.x, tid = threadIdx.x, base = tid * E;
    const int32_t* ob = obs + (size_t)n * (L + 1) * W;      // [L+1][W]; token (t,w) -> ob[t*W+w]
    uint32_t v[E];
#pragma unroll
    for (int e = 0; e < E; ++e) {
        const int i = base + e;
        v[e] = i < T ? ((uint32_t)ob_idx(ob[i]) << 12) | (uint32_t)i : 0xFFFFFFFFu;
    }
    for (int k = 2; k <= P2; k <<= 1) {
        for (int j = k >> 1; j >= 32 * E; j >>= 1) {         // partner in another warp: through shared memory
#pragma unroll
            for (int e = 0; e < E; ++e) xch[base + e] = v[e];
            __syncthreads();
#pragma unroll
            for (int e = 0; e < E; ++e) {
                const int i = base + e;
                sort_cmpx<E>(v[e], xch[i ^ j], ((i & j) == 0) == ((i & k) == 0));
            }
            __syncthreads();
        }
        for (int j = min(k >> 1, 16 * E); j >= E; j >>= 1) {    // partner in another lane of this warp
            const int lane_mask = j / E;
#pragma unroll
            for (int e = 0; e < E; ++e) {
                const int i = base + e;
                const uint32_t other = __shfl_xor_sync(0xffffffffu, v[e], lane_mask);
                sort_cmpx<E>(v[e], other, ((i & j) == 0) == ((i & k) == 0));
            }
        }
#pragma unroll
        for (int j = E / 2; j > 0; j >>= 1) {                   // partner in this thread's registers
            if (j < k) {
#pragma unroll
                for (int e = 0; e < E; ++e) {
                    if ((e & j) == 0) {
                        const bool up = ((base + e) & k) == 0;
                        const uint32_t a = v[e], b = v[e | j];
                        const uint32_t lo = min(a, b), hi = max(a, b);
                        v[e] = up ? lo : hi;
                        v[e | j] = up ? hi : lo;
                    }
                }
            }
        }
    }
#pragma unroll
    for (int e = 0; e < E; ++e)
        if (base + e < T) sorted_tok[(size_t)n * T + base + e] = (uint16_t)(v[e] & 0xFFFu);
}

// small problems (P2 < 512): plain shared-memory bitonic network
__global__ void __launch_bounds__(256)
sort_tokens_kernel(const int32_t* __restrict__ obs, uint16_t* __restrict__ sorted_tok,
                   int W, int L, int T, int P2) {
    extern __shared__ uint32_t keys[];
    const int n = blockIdx.x;
    const int32_t* ob = obs + (size_t)n * (L + 1) * W;
    for (int i = threadIdx.x; i < P2; i += blockDim.x)
        keys[i] = i < T ? ((uint32_t)ob_idx(ob[i]) << 12) | (uint32_t)i : 0xFFFFFFFFu;
    __syncthreads();
    for (int k = 2; k <= P2; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < P2; i += blockDim.x) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const uint32_t a = keys[i], b = keys[ixj];
                    const bool up = (i & k) == 0;
                    if ((a > b) == up) { keys[i] = b; keys[ixj] = a; }
                }
            }
            __syncthreads();
        }
    }
    for (int i = threadIdx.x; i < T; i += blockDim.x)
        sorted_tok[(size_t)n * T + i] = (uint16_t)(keys[i] & 0xFFFu);
}

extern "C" int toued_sort_tokens(const int32_t* obs, uint16_t* sorted_tok, int n_agents, int n_workers,
                                 int rollout_len, void* stream) {
    const int T = n_workers * rollout_len;
    TOUED_CHECK(T > 0 && T <= 4096, "toued_sort_tokens: W*L=%d must be in 1..4096", T);
    int P2 = 1; while (P2 < T) P2 <<= 1;
    cudaStream_t st = (cudaStream_t)stream;
    switch (P2) {
        case 512:  sort_tokens_reg_kernel<2><<<n_agents, 256, 0, st>>>(obs, sorted_tok, n_workers, rollout_len, T); break;
        case 1024: sort_tokens_reg_kernel<4><<<n_agents, 256, 0, st>>>(obs, sorted_tok, n_workers, rollout_len, T); break;
        case 2048: sort_tokens_reg_kernel<8><<<n_agents, 256, 0, st>>>(obs, sorted_tok, n_workers, rollout_len, T); break;
        case 4096: sort_tokens_reg_kernel<16><<<n_agents, 256, 0, st>>>(obs, sorted_tok, n_workers, rollout_len, T); break;
        default:   sort_tokens_kernel<<<n_agents, 256, P2 * sizeof(uint32_t), st>>>(obs, sorted_tok, n_workers, rollout_len, T, P2);
    }
    TOUED_LAUNCH_CHECK();
    return 0;
}

// ------------------------------------------------------------------------------------------------
// LPG inputs.  One thread per token (n, t, w).
// both applications of the embedding MLP (y_t and y_{t+1}) in one pass over the weights: every weight is read once
// and nothing has to stay in registers between the two (a two-call version keeps all 161 weights live: 198 registers,
// one CTA per SM).  Per output the operation order is that of a single application.
__device__ __forceinline__ void embed_mlp2(const float (&y0)[LPG_Y], const float (&y1)[LPG_Y],
                                           const float* __restrict__ sp, float& out0, float& out1) {
    // sp: e_w0[Y][E] e_b0[E] e_w1[E] e_b1[1]
    out0 = out1 = sp[LPG_Y * LPG_E + LPG_E + LPG_E];
#pragma unroll 4
    for (int e = 0; e < LPG_E; ++e) {
        float a0 = sp[LPG_Y * LPG_E + e], a1 = a0;
#pragma unroll
        for (int i = 0; i < LPG_Y; ++i) {
            const float wgt = sp[i * LPG_E + e];
            a0 = fmaf(y0[i], wgt, a0);
            a1 = fmaf(y1[i], wgt, a1);
        }
        const float w1 = sp[LPG_Y * LPG_E + LPG_E + e];
        out0 = fmaf(fmax_nan(a0, 0.0f), w1, out0);             // relu that keeps NaN (fmaxf would drop it)
        out1 = fmaf(fmax_nan(a1, 0.0f), w1, out1);
    }
}

__global__ void __launch_bounds__(256, 4)
lpg_prepare_kernel(const int32_t* __restrict__ obs, const uint8_t* __restrict__ action,
                   const float* __restrict__ reward, const uint8_t* __restrict__ done,
                   const float* __restrict__ actor, const float* __restrict__ critic,
                   const float* __restrict__ lpg, const int32_t* __restrict__ step,
                   const LevelRec* __restrict__ levels, float* __restrict__ x, unsigned char* __restrict__ ximg,
                   int n_agents, int W, int L, int D, int cond, int emb_off, int lpg_stride) {
    __shared__ float sp_s[LPG_Y * LPG_E + LPG_E + LPG_E + 1];
    if (lpg_stride == 0) {
        for (int i = threadIdx.x; i < LPG_Y * LPG_E + 2 * LPG_E + 1; i += blockDim.x) sp_s[i] = lpg[emb_off + i];
        __syncthreads();
    }
    const size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t total = (size_t)n_agents * L * W;
    if (g >= total) return;
    const int w = (int)(g % W);
    const int t = (int)((g / W) % L);
    const int n = (int)(g / ((size_t)W * L));
    // per-agent LPG parameters (ES candidates): read the embedding MLP straight from global / L2
    const float* sp = lpg_stride ? lpg + (size_t)n * lpg_stride + emb_off : sp_s;
    const int32_t ob = obs[((size_t)n * (L + 1) + t) * W + w];
    const int32_t ob1 = obs[((size_t)n * (L + 1) + t + 1) * W + w];
    const float* at = actor + (size_t)n * D * 8;
    const float* ct = critic + (size_t)n * D * 8;
    float z[TOUED_NUM_ACTIONS], p[TOUED_NUM_ACTIONS];
    tab_logits8<TOUED_NUM_ACTIONS>(at, D, ob, z);
    softmax_c<TOUED_NUM_ACTIONS>(z, p);
    const int a = action[g];
    float pa = p[0];
#pragma unroll
    for (int j = 1; j < TOUED_NUM_ACTIONS; ++j) pa = (a == j) ? p[j] : pa;
    float zy[LPG_Y], y0[LPG_Y], y1[LPG_Y];
    tab_logits8<LPG_Y>(ct, D, ob, zy);
    softmax_c<LPG_Y>(zy, y0);
    tab_logits8<LPG_Y>(ct, D, ob1, zy);
    softmax_c<LPG_Y>(zy, y1);
    const float d = done[g] ? 1.0f : 0.0f;
    float pyt, pyt1;
    embed_mlp2(y0, y1, sp, pyt, pyt1);
    pyt1 *= (1.0f - d);                                             // lpg.py:69
    const size_t row = (size_t)n * W + w;
    float4* xo = reinterpret_cast<float4*>(x + ((size_t)t * n_agents * W + row) * LPG_XP);
    xo[0] = make_float4(reward[g], d, pa + 1e-8f, pyt);             // lpg_agent.py:41-43 (pi + 1e-8)
    const float4 v1 = make_float4(pyt1, cond ? (float)step[n] : 0.0f, cond ? (float)levels[n].lifetime : 0.0f, 1.0f);
    xo[1] = v1;
    if (ximg) {      // fp16 token-tile image (one 64-column group, columns 8..63 stay zero) for the weight-gradient GEMM
        const size_t Rp = ((size_t)n_agents * W + 63) & ~(size_t)63;
        __half2 b0 = __floats2half2_rn(reward[g], d), b1 = __floats2half2_rn(pa + 1e-8f, pyt);
        __half2 b2 = __floats2half2_rn(v1.x, v1.y), b3 = __floats2half2_rn(v1.z, v1.w);
        uint4 pk;
        pk.x = *reinterpret_cast<uint32_t*>(&b0); pk.y = *reinterpret_cast<uint32_t*>(&b1);
        pk.z = *reinterpret_cast<uint32_t*>(&b2); pk.w = *reinterpret_cast<uint32_t*>(&b3);
        *reinterpret_cast<uint4*>(ximg + tile_img_offset((size_t)t * Rp + row, 1, 0)) = pk;
    }
}

extern "C" int toued_lpg_prepare(const int32_t* obs, const uint8_t* action, const float* reward,
                                 const uint8_t* done, const float* actor, const float* critic,
                                 const float* lpg_params, const int32_t* step, const void* levels,
                                 float* x, void* ximg, int n_agents, int n_workers, int rollout_len, int obs_dim,
                                 int lifetime_conditioning, int lpg_stride, void* stream) {
    const size_t total = (size_t)n_agents * rollout_len * n_workers;
    TOUED_CHECK(total > 0, "toued_lpg_prepare: empty problem");
    lpg_prepare_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        obs, action, reward, done, actor, critic, lpg_params, step, (const LevelRec*)levels, x, (unsigned char*)ximg,
        n_agents, n_workers, rollout_len, obs_dim, lifetime_conditioning,
        lpg_offsets(lifetime_conditioning ? 7 : 5).e_w0, lpg_stride);
    TOUED_LAUNCH_CHECK();
    return 0;
}

// ------------------------------------------------------------------------------------------------
// GRU forward (SIMT fp32).  CTA = 64 rows, 256 threads.  Per timestep: gates = h' @ Wh in four
// passes of 64 hidden units (x3 gates); thread tile = 4 rows x 4 units x 3 gates.
constexpr int GF_TM = 64;          // rows per CTA
constexpr int GF_KC = 16;          // k-chunk of Wh staged in smem
constexpr int GF_HS = LPG_H + 4;   // padded row stride of the hidden-state tiles

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem)), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N)); }

template <int X>
__global__ void __launch_bounds__(256, 1)
gru_forward_kernel(const float* __restrict__ x, const uint8_t* __restrict__ done,
                   const float* __restrict__ lpg_base, float* __restrict__ h_out, float* __restrict__ gates,
                   float* __restrict__ pi_hat, float* __restrict__ y_hat, int R, int L, int W, int lpg_stride) {
    // per-agent LPG parameters (ES candidates): the CTA's 64 rows belong to one agent (W % 64 == 0)
    const float* lpg = lpg_base + (size_t)((blockIdx.x * 64) / W) * lpg_stride;
    extern __shared__ __align__(16) float sm[];
    float* hA = sm;                                  // [64][GF_HS] h' (masked carry)
    float* hB = hA + GF_TM * GF_HS;                  // [64][GF_HS] new h
    float* Bs = hB + GF_TM * GF_HS;                  // [2][KC][192]
    float* sWi = Bs + 2 * GF_KC * 192;               // [X][768]
    float* sbi = sWi + X * LPG_G;                    // [768]
    float* sbhn = sbi + LPG_G;                       // [256]
    float* swp = sbhn + LPG_H;                       // [256]
    float* sWy = swp + LPG_H;                        // [256][8]
    float* sx = sWy + LPG_H * LPG_Y;                 // [64][8]
    __shared__ float sdone[GF_TM];
    const LpgOffsets o = lpg_offsets(X);
    const float* Wh = lpg + o.Wh;
    const int tid = threadIdx.x;
    const int row0 = blockIdx.x * GF_TM;
    const int nrows = min(GF_TM, R - row0);

    for (int i = tid; i < X * LPG_G; i += 256) sWi[i] = lpg[o.Wi + i];
    for (int i = tid; i < LPG_G; i += 256) sbi[i] = lpg[o.bi + i];
    for (int i = tid; i < LPG_H; i += 256) { sbhn[i] = lpg[o.bhn + i]; swp[i] = lpg[o.w_pi + i]; }
    for (int i = tid; i < LPG_H * LPG_Y; i += 256) sWy[i] = lpg[o.W_y + i];
    for (int i = tid; i < GF_TM * GF_HS; i += 256) hB[i] = 0.0f;
    const float b_pi = lpg[o.b_pi];
    float b_y[LPG_Y];
#pragma unroll
    for (int i = 0; i < LPG_Y; ++i) b_y[i] = lpg[o.b_y + i];
    __syncthreads();

    const int rg = tid >> 4;       // 0..15 -> rows rg*4 .. rg*4+3
    const int jg = tid & 15;       // 0..15 -> units jg*4 .. jg*4+3 within the pass

    for (int t = L - 1; t >= 0; --t) {
        // ---- stage x_t, done_t; carry h' = done ? 0 : h_{t+1}  (lpg.py:27-28) ----
        { float* tmp = hA; hA = hB; hB = tmp; }
        if (tid < GF_TM) {
            const int r = row0 + tid;
            sdone[tid] = (tid < nrows && done[((size_t)(r / W) * L + t) * W + (r % W)]) ? 1.0f : 0.0f;
        }
        for (int i = tid; i < GF_TM * 2; i += 256) {
            const int r = i >> 1;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (r < nrows) v = reinterpret_cast<const float4*>(x + ((size_t)t * R + row0 + r) * LPG_XP)[i & 1];
            reinterpret_cast<float4*>(sx + r * LPG_XP)[i & 1] = v;
        }
        __syncthreads();
        for (int i = tid; i < GF_TM * 64; i += 256) {            // zero the carry of finished sequences
            const int r = i >> 6;
            if (sdone[r] != 0.0f) reinterpret_cast<float4*>(hA + r * GF_HS)[i & 63] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        __syncthreads();

        for (int jb = 0; jb < 4; ++jb) {
            float acc[4][4][3];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) { acc[i][j][0] = 0.f; acc[i][j][1] = 0.f; acc[i][j][2] = 0.f; }
            // chunk loader: [KC][3 gates][64 cols] = KC*48 float4, 3 per thread
            auto load_chunk = [&](int buf, int k0) {
#pragma unroll
                for (int q = 0; q < 3; ++q) {
                    const int f = tid + q * 256;             // float4 index 0..767
                    const int kk = f / 48, rem = f % 48, gte = rem >> 4, c4 = rem & 15;
                    cp_async16(Bs + (buf * GF_KC + kk) * 192 + gte * 64 + c4 * 4,
                               Wh + (size_t)(k0 + kk) * LPG_G + gte * LPG_H + jb * 64 + c4 * 4);
                }
                cp_async_commit();
            };
            load_chunk(0, 0);
            for (int kc = 0; kc < LPG_H / GF_KC; ++kc) {
                if (kc + 1 < LPG_H / GF_KC) { load_chunk((kc + 1) & 1, (kc + 1) * GF_KC); cp_async_wait<1>(); }
                else cp_async_wait<0>();
                __syncthreads();
                const float* bs = Bs + (kc & 1) * GF_KC * 192;
#pragma unroll
                for (int k4 = 0; k4 < GF_KC; k4 += 4) {
                    float4 a[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        a[i] = *reinterpret_cast<const float4*>(hA + (rg * 4 + i) * GF_HS + kc * GF_KC + k4);
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk) {
                        float4 b[3];
#pragma unroll
                        for (int gte = 0; gte < 3; ++gte)
                            b[gte] = *reinterpret_cast<const float4*>(bs + (k4 + kk) * 192 + gte * 64 + jg * 4);
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const float av = kk == 0 ? a[i].x : kk == 1 ? a[i].y : kk == 2 ? a[i].z : a[i].w;
#pragma unroll
                            for (int gte = 0; gte < 3; ++gte) {
                                acc[i][0][gte] = fmaf(av, b[gte].x, acc[i][0][gte]);
                                acc[i][1][gte] = fmaf(av, b[gte].y, acc[i][1][gte]);
                                acc[i][2][gte] = fmaf(av, b[gte].z, acc[i][2][gte]);
                                acc[i][3][gte] = fmaf(av, b[gte].w, acc[i][3][gte]);
                            }
                        }
                    }
                }
                __syncthreads();
            }
            // ---- gate epilogue for (4 rows) x (4 units) ----
            const int j0 = jb * 64 + jg * 4;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int rl = rg * 4 + i;
                float xr[X];
#pragma unroll
                for (int q = 0; q < X; ++q) xr[q] = sx[rl * LPG_XP + q];
                float hn4[4], r4[4], z4[4], n4[4], hv[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int u = j0 + j;
                    float gr = sbi[u], gz = sbi[LPG_H + u], gn = sbi[2 * LPG_H + u];
#pragma unroll
                    for (int q = 0; q < X; ++q) {
                        gr = fmaf(xr[q], sWi[q * LPG_G + u], gr);
                        gz = fmaf(xr[q], sWi[q * LPG_G + LPG_H + u], gz);
                        gn = fmaf(xr[q], sWi[q * LPG_G + 2 * LPG_H + u], gn);
                    }
                    const float rr = sigmoidf_(gr + acc[i][j][0]);
                    const float zz = sigmoidf_(gz + acc[i][j][1]);
                    const float hn = acc[i][j][2] + sbhn[u];
                    const float nn = tanhf_(gn + rr * hn);
                    const float hp = hA[rl * GF_HS + u];
                    r4[j] = rr; z4[j] = zz; n4[j] = nn; hn4[j] = hn;
                    hv[j] = (1.0f - zz) * nn + zz * hp;
                }
                *reinterpret_cast<float4*>(hB + rl * GF_HS + j0) = make_float4(hv[0], hv[1], hv[2], hv[3]);
                if (rl < nrows) {
                    const size_t base = ((size_t)t * R + row0 + rl) * LPG_H + j0;
                    *reinterpret_cast<float4*>(h_out + base) = make_float4(hv[0], hv[1], hv[2], hv[3]);
                    if (gates) {
                        const size_t gs = (size_t)L * R * LPG_H;
                        *reinterpret_cast<float4*>(gates + base) = make_float4(r4[0], r4[1], r4[2], r4[3]);
                        *reinterpret_cast<float4*>(gates + gs + base) = make_float4(z4[0], z4[1], z4[2], z4[3]);
                        *reinterpret_cast<float4*>(gates + 2 * gs + base) = make_float4(n4[0], n4[1], n4[2], n4[3]);
                        *reinterpret_cast<float4*>(gates + 3 * gs + base) = make_float4(hn4[0], hn4[1], hn4[2], hn4[3]);
                    }
                }
            }
        }
        __syncthreads();
        // ---- heads on relu(h_t): pi_hat = Dense(1), y_hat = softmax(Dense(8))  (lpg.py:80-84) ----
        {
            const int rl = tid >> 2, part = tid & 3;
            float hacc[1 + LPG_Y];
#pragma unroll
            for (int c = 0; c < 1 + LPG_Y; ++c) hacc[c] = 0.0f;
            for (int k = part * 64; k < part * 64 + 64; ++k) {
                const float yv = fmax_nan(hB[rl * GF_HS + k], 0.0f);     // relu that keeps NaN
                hacc[0] = fmaf(yv, swp[k], hacc[0]);
#pragma unroll
                for (int c = 0; c < LPG_Y; ++c) hacc[1 + c] = fmaf(yv, sWy[k * LPG_Y + c], hacc[1 + c]);
            }
#pragma unroll
            for (int c = 0; c < 1 + LPG_Y; ++c) {
                hacc[c] += __shfl_xor_sync(0xffffffffu, hacc[c], 1);
                hacc[c] += __shfl_xor_sync(0xffffffffu, hacc[c], 2);
            }
            if (part == 0 && rl < nrows) {
                const size_t tok = (size_t)t * R + row0 + rl;
                pi_hat[tok] = hacc[0] + b_pi;
                float zl[LPG_Y], pr[LPG_Y];
#pragma unroll
                for (int c = 0; c < LPG_Y; ++c) zl[c] = hacc[1 + c] + b_y[c];
                softmax_c<LPG_Y>(zl, pr);
                float4* yo = reinterpret_cast<float4*>(y_hat + tok * LPG_Y);
                yo[0] = make_float4(pr[0], pr[1], pr[2], pr[3]);
                yo[1] = make_float4(pr[4], pr[5], pr[6], pr[7]);
            }
        }
        // (the swap at the top of the next iteration turns hB into the carry)
    }
}

static size_t gru_fwd_smem(int X) {
    return sizeof(float) * (2 * GF_TM * GF_HS + 2 * GF_KC * 192 + X * LPG_G + LPG_G + 2 * LPG_H +
                            LPG_H * LPG_Y + GF_TM * LPG_XP);
}

extern "C" int toued_gru_forward(const float* x, const uint8_t* done, const float* lpg_params, float* h_out,
                                 float* gates, float* pi_hat, float* y_hat, int n_agents, int n_workers,
                                 int rollout_len, int lifetime_conditioning, int lpg_stride, void* stream) {
    const int R = n_agents * n_workers;
    TOUED_CHECK(R > 0 && rollout_len > 0, "toued_gru_forward: empty problem");
    TOUED_CHECK(lpg_stride == 0 || n_workers % 64 == 0, "toued_gru_forward: per-agent parameters need n_workers %% 64 == 0");
    const int blocks = (R + GF_TM - 1) / GF_TM;
    cudaStream_t st = (cudaStream_t)stream;
    if (lifetime_conditioning) {
        const size_t smem = gru_fwd_smem(7);
        TOUED_CUDA(cudaFuncSetAttribute(gru_forward_kernel<7>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        gru_forward_kernel<7><<<blocks, 256, smem, st>>>(x, done, lpg_params, h_out, gates, pi_hat, y_hat, R, rollout_len, n_workers, lpg_stride);
    } else {
        const size_t smem = gru_fwd_smem(5);
        TOUED_CUDA(cudaFuncSetAttribute(gru_forward_kernel<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        gru_forward_kernel<5><<<blocks, 256, smem, st>>>(x, done, lpg_params, h_out, gates, pi_hat, y_hat, R, rollout_len, n_workers, lpg_stride);
    }
    TOUED_LAUNCH_CHECK();
    return 0;
}
