// LPG backward pass: given the cotangents d_pi_hat, d_y_hat of one agent update (produced by
// toued_agent_backward), back-propagate through the heads, the reverse GRU and the embedding MLP
// and accumulate the gradient of the flat LPG parameter vector.  This is the part of
// jax.grad(_train_agent) (meta/train.py:121-128) that flows through models/lpg.py:48-85.
// The LPG inputs (r, d, pi, y_t, y_{t+1}) are stop_gradient'ed (lpg_agent.py:54-56): the only
// input cotangents needed are those of pyt / pyt1, which reach the embedding-MLP parameters.
//
//   toued_gru_backward   BPTT over the L steps (forward in time: the scan is reversed), exact fp32:
//                        dh' = dGh @ Wh^T per step with the carry in shared memory; overwrites the
//                        saved gate activations (r, z, n, hn) with (dar, daz, dan, dhn) in place; emits
//                        the head-softmax logit cotangents dl and d pyt / d pyt1.
//   toued_lpg_wgrad      parameter gradients as token-split partial sums (deterministic):
//                        dWh = h'^T dGh (tiled SGEMM), dWi/dbi/dbhn/heads (streaming), embedding MLP.
//   toued_reduce_partials  grad[p] (+)= sum_s partial[s][p]
//   toued_adam           optax.scale_by_adam -> scale(lr) -> scale(-1)  (models/optim.py:12-17, Q9)
//   toued_sgd_clip       optax.clip_by_global_norm -> scale(lr) -> scale(-1)  (models/optim.py:6-11, --lpg_opt SGD)
#include "lpg_common.cuh"
#include "tc.cuh"
#include "../../include/toued.h"

__device__ __forceinline__ void cp_async16z(void* smem, const void* gmem, bool valid) {
    const int sz = valid ? 16 : 0;                      // src-size 0 -> zero fill
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(smem)), "l"(gmem), "r"(sz));
}
__device__ __forceinline__ void cp_commit() { asm volatile("cp.async.commit_group;"); }
template <int N> __device__ __forceinline__ void cp_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N)); }

// ------------------------------------------------------------------------------------------------
__global__ void transpose_wh_kernel(const float* __restrict__ Wh, float* __restrict__ WhT) {
    __shared__ float tile[32][33];
    const int c0 = blockIdx.x * 32, j0 = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += 8) tile[r][threadIdx.x] = Wh[(size_t)(j0 + r) * LPG_G + c0 + threadIdx.x];
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += 8) WhT[(size_t)(c0 + r) * LPG_H + j0 + threadIdx.x] = tile[threadIdx.x][r];
}

// ------------------------------------------------------------------------------------------------
constexpr int GB_TM = 64;
constexpr int GB_KC = 16;
constexpr int GB_CS = LPG_H + 4;
constexpr int GB_AS = GB_KC + 4;

__global__ void __launch_bounds__(256, 1)
gru_backward_kernel(const uint8_t* __restrict__ done, const float* __restrict__ lpg, int X,
                    const float* __restrict__ WhT, const float* __restrict__ h, float* gates,
                    const float* __restrict__ y_hat, const float* __restrict__ d_pi_hat,
                    const float* __restrict__ d_y_hat, float* __restrict__ dl_out,
                    float* __restrict__ dx, int R, int L, int W) {
    extern __shared__ __align__(16) float sm[];
    float* C = sm;                                  // [64][GB_CS]  carry, then dh * z
    float* As = C + GB_TM * GB_CS;                  // [2][64][GB_AS]
    float* Bs = As + 2 * GB_TM * GB_AS;             // [2][KC][256]
    float* swp = Bs + 2 * GB_KC * LPG_H;            // [256]
    float* sWy = swp + LPG_H;                       // [256][8]
    float* sWi = sWy + LPG_H * LPG_Y;               // [2][768]  rows 3 (pyt) and 4 (pyt1) of Wi
    __shared__ float snd[GB_TM];
    const LpgOffsets o = lpg_offsets(X);
    const int tid = threadIdx.x;
    const int row0 = blockIdx.x * GB_TM;
    const int nrows = min(GB_TM, R - row0);
    const size_t gs = (size_t)L * R * LPG_H;        // stride between the 4 gate planes

    for (int i = tid; i < LPG_H; i += 256) swp[i] = lpg[o.w_pi + i];
    for (int i = tid; i < LPG_H * LPG_Y; i += 256) sWy[i] = lpg[o.W_y + i];
    for (int i = tid; i < 2 * LPG_G; i += 256) sWi[i] = lpg[o.Wi + 3 * LPG_G + i];
    for (int i = tid; i < GB_TM * GB_CS; i += 256) C[i] = 0.0f;
    __syncthreads();

    const int rl = tid >> 2, part = tid & 3;        // E-phase mapping: row, 64-unit slice
    const int rg = tid >> 5, cg = tid & 31;         // GEMM mapping: 8 rows x (4 + 4) cols

    for (int t = 0; t < L; ++t) {
        if (tid < GB_TM) {
            const int r = row0 + tid;
            snd[tid] = (tid < nrows && !done[((size_t)(r / W) * L + t) * W + (r % W)]) ? 1.0f : 0.0f;
        }
        __syncthreads();
        // ---------------- E-phase: element-wise gate backward ----------------
        float dx3 = 0.f, dx4 = 0.f;
        const size_t tok = (size_t)t * R + row0 + rl;
        if (rl < nrows) {
            float yh[8], dy[8], dl[8];
            { const float4* q = reinterpret_cast<const float4*>(y_hat + tok * 8); const float4 a = q[0], b = q[1];
              yh[0] = a.x; yh[1] = a.y; yh[2] = a.z; yh[3] = a.w; yh[4] = b.x; yh[5] = b.y; yh[6] = b.z; yh[7] = b.w; }
            { const float4* q = reinterpret_cast<const float4*>(d_y_hat + tok * 8); const float4 a = q[0], b = q[1];
              dy[0] = a.x; dy[1] = a.y; dy[2] = a.z; dy[3] = a.w; dy[4] = b.x; dy[5] = b.y; dy[6] = b.z; dy[7] = b.w; }
            float s = 0.f;
#pragma unroll
            for (int i = 0; i < 8; ++i) s = fmaf(yh[i], dy[i], s);
#pragma unroll
            for (int i = 0; i < 8; ++i) dl[i] = yh[i] * (dy[i] - s);          // softmax backward
            const float dpi = d_pi_hat[tok];
            if (part == 0) {                                                    // head-softmax logit cotangents
                float4* q = reinterpret_cast<float4*>(dl_out + tok * 8);
                q[0] = make_float4(dl[0], dl[1], dl[2], dl[3]);
                q[1] = make_float4(dl[4], dl[5], dl[6], dl[7]);
            }
            const bool has_next = (t + 1 < L) && snd[rl] != 0.0f;
            const size_t base = tok * LPG_H + part * 64;
            for (int j4 = 0; j4 < 64; j4 += 4) {
                const int j = part * 64 + j4;
                const float4 rr = *reinterpret_cast<const float4*>(gates + base + j4);
                const float4 zz = *reinterpret_cast<const float4*>(gates + gs + base + j4);
                const float4 nn = *reinterpret_cast<const float4*>(gates + 2 * gs + base + j4);
                const float4 hn = *reinterpret_cast<const float4*>(gates + 3 * gs + base + j4);
                const float4 ht = *reinterpret_cast<const float4*>(h + base + j4);
                float4 hp = make_float4(0.f, 0.f, 0.f, 0.f);
                if (has_next) hp = *reinterpret_cast<const float4*>(h + base + j4 + (size_t)R * LPG_H);
                const float4 cr = *reinterpret_cast<const float4*>(C + rl * GB_CS + j);
                float r_[4] = {rr.x, rr.y, rr.z, rr.w}, z_[4] = {zz.x, zz.y, zz.z, zz.w};
                float n_[4] = {nn.x, nn.y, nn.z, nn.w}, hn_[4] = {hn.x, hn.y, hn.z, hn.w};
                float ht_[4] = {ht.x, ht.y, ht.z, ht.w}, hp_[4] = {hp.x, hp.y, hp.z, hp.w};
                float c_[4] = {cr.x, cr.y, cr.z, cr.w};
                float dar[4], daz[4], dan[4], dhn[4], cz[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int u = j + e;
                    float dh = c_[e];
                    if (ht_[e] > 0.0f) {                                        // relu + heads (lpg.py:80-84)
                        float hd = dpi * swp[u];
#pragma unroll
                        for (int i = 0; i < 8; ++i) hd = fmaf(dl[i], sWy[u * 8 + i], hd);
                        dh += hd;
                    }
                    const float dn = dh * (1.0f - z_[e]);
                    const float dz = dh * (hp_[e] - n_[e]);
                    dan[e] = dn * (1.0f - n_[e] * n_[e]);
                    dhn[e] = dan[e] * r_[e];
                    dar[e] = dan[e] * hn_[e] * r_[e] * (1.0f - r_[e]);
                    daz[e] = dz * z_[e] * (1.0f - z_[e]);
                    cz[e] = dh * z_[e];
                    dx3 = fmaf(dar[e], sWi[u], fmaf(daz[e], sWi[LPG_H + u], fmaf(dan[e], sWi[2 * LPG_H + u], dx3)));
                    dx4 = fmaf(dar[e], sWi[LPG_G + u], fmaf(daz[e], sWi[LPG_G + LPG_H + u], fmaf(dan[e], sWi[LPG_G + 2 * LPG_H + u], dx4)));
                }
                *reinterpret_cast<float4*>(gates + base + j4) = make_float4(dar[0], dar[1], dar[2], dar[3]);
                *reinterpret_cast<float4*>(gates + gs + base + j4) = make_float4(daz[0], daz[1], daz[2], daz[3]);
                *reinterpret_cast<float4*>(gates + 2 * gs + base + j4) = make_float4(dan[0], dan[1], dan[2], dan[3]);
                *reinterpret_cast<float4*>(gates + 3 * gs + base + j4) = make_float4(dhn[0], dhn[1], dhn[2], dhn[3]);
                *reinterpret_cast<float4*>(C + rl * GB_CS + j) = make_float4(cz[0], cz[1], cz[2], cz[3]);
            }
        }
        dx3 += __shfl_xor_sync(0xffffffffu, dx3, 1); dx3 += __shfl_xor_sync(0xffffffffu, dx3, 2);
        dx4 += __shfl_xor_sync(0xffffffffu, dx4, 1); dx4 += __shfl_xor_sync(0xffffffffu, dx4, 2);
        if (part == 0 && rl < nrows) *reinterpret_cast<float2*>(dx + tok * 2) = make_float2(dx3, dx4);
        __syncthreads();
        if (t + 1 == L) break;
        // ---------------- GEMM: dh' = dGh[64][768] @ WhT[768][256] ----------------
        float acc[8][8];
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
        auto load_chunk = [&](int buf, int c0) {
            const int gate = c0 >> 8, u0 = c0 & 255;
            const size_t plane = (size_t)(gate == 2 ? 3 : gate) * gs;            // (dar, daz, dhn)
            {   // A: 64 rows x 16 floats -> one 16-byte copy per thread
                const int r = tid >> 2, q = tid & 3;
                const bool ok = r < nrows;
                const float* src = gates + plane + ((size_t)t * R + row0 + (ok ? r : 0)) * LPG_H + u0 + q * 4;
                cp_async16z(As + (buf * GB_TM + r) * GB_AS + q * 4, src, ok);
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {                                        // B: 16 x 256 floats
                const int f = tid + q * 256, kk = f >> 6, c4 = f & 63;
                cp_async16z(Bs + (buf * GB_KC + kk) * LPG_H + c4 * 4, WhT + (size_t)(c0 + kk) * LPG_H + c4 * 4, true);
            }
            cp_commit();
        };
        load_chunk(0, 0);
        for (int kc = 0; kc < LPG_G / GB_KC; ++kc) {
            if (kc + 1 < LPG_G / GB_KC) { load_chunk((kc + 1) & 1, (kc + 1) * GB_KC); cp_wait<1>(); }
            else cp_wait<0>();
            __syncthreads();
            const float* as = As + (kc & 1) * GB_TM * GB_AS;
            const float* bs = Bs + (kc & 1) * GB_KC * LPG_H;
#pragma unroll
            for (int k4 = 0; k4 < GB_KC; k4 += 4) {
                float4 a[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) a[i] = *reinterpret_cast<const float4*>(as + (rg * 8 + i) * GB_AS + k4);
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
                    const float4 b0 = *reinterpret_cast<const float4*>(bs + (k4 + kk) * LPG_H + cg * 4);
                    const float4 b1 = *reinterpret_cast<const float4*>(bs + (k4 + kk) * LPG_H + 128 + cg * 4);
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const float av = kk == 0 ? a[i].x : kk == 1 ? a[i].y : kk == 2 ? a[i].z : a[i].w;
                        acc[i][0] = fmaf(av, b0.x, acc[i][0]); acc[i][1] = fmaf(av, b0.y, acc[i][1]);
                        acc[i][2] = fmaf(av, b0.z, acc[i][2]); acc[i][3] = fmaf(av, b0.w, acc[i][3]);
                        acc[i][4] = fmaf(av, b1.x, acc[i][4]); acc[i][5] = fmaf(av, b1.y, acc[i][5]);
                        acc[i][6] = fmaf(av, b1.z, acc[i][6]); acc[i][7] = fmaf(av, b1.w, acc[i][7]);
                    }
                }
            }
            __syncthreads();
        }
        // carry for step t+1: (1 - done_t) * (dGh Wh^T + dh * z)
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int r = rg * 8 + i;
            const float nd = snd[r];
            float4* c0p = reinterpret_cast<float4*>(C + r * GB_CS + cg * 4);
            float4* c1p = reinterpret_cast<float4*>(C + r * GB_CS + 128 + cg * 4);
            const float4 c0 = *c0p, c1 = *c1p;
            *c0p = make_float4(nd * (acc[i][0] + c0.x), nd * (acc[i][1] + c0.y), nd * (acc[i][2] + c0.z), nd * (acc[i][3] + c0.w));
            *c1p = make_float4(nd * (acc[i][4] + c1.x), nd * (acc[i][5] + c1.y), nd * (acc[i][6] + c1.z), nd * (acc[i][7] + c1.w));
        }
        __syncthreads();
    }
}

static size_t gru_bwd_smem() {
    return sizeof(float) * (GB_TM * GB_CS + 2 * GB_TM * GB_AS + 2 * GB_KC * LPG_H + LPG_H + LPG_H * LPG_Y + 2 * LPG_G);
}

extern "C" int toued_gru_backward(const uint8_t* done, const float* lpg_params, const float* whT,
                                  const float* h, float* gates, const float* y_hat, const float* d_pi_hat,
                                  const float* d_y_hat, float* dl, float* dx, int n_agents, int n_workers,
                                  int rollout_len, int lifetime_conditioning, void* stream) {
    const int R = n_agents * n_workers;
    TOUED_CHECK(R > 0 && rollout_len > 0, "toued_gru_backward: empty problem");
    const size_t smem = gru_bwd_smem();
    TOUED_CUDA(cudaFuncSetAttribute(gru_backward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    gru_backward_kernel<<<(R + GB_TM - 1) / GB_TM, 256, smem, (cudaStream_t)stream>>>(
        done, lpg_params, lifetime_conditioning ? 7 : 5, whT, h, gates, y_hat, d_pi_hat, d_y_hat, dl, dx, R,
        rollout_len, n_workers);
    TOUED_LAUNCH_CHECK();
    return 0;
}

extern "C" int toued_transpose_wh(const float* lpg_params, float* whT, void* stream) {
    transpose_wh_kernel<<<dim3(LPG_G / 32, LPG_H / 32), dim3(32, 8), 0, (cudaStream_t)stream>>>(
        lpg_params + lpg_offsets(5).Wh, whT);
    TOUED_LAUNCH_CHECK();
    return 0;
}

// ------------------------------------------------------------------------------------------------
// dWh[j][c] = sum_tok h'[tok][j] * dGh[tok][c]      (tile 64 x 64, thread 4 x 4, token split S)
constexpr int WG_KC = 16;
__global__ void __launch_bounds__(256)
wgrad_wh_kernel(const uint8_t* __restrict__ done, const float* __restrict__ h, const float* __restrict__ gates,
                float* __restrict__ partial, int R, int L, int W, int chunks_per_split, int accumulate) {
    __shared__ __align__(16) float As[2][WG_KC][64];
    __shared__ __align__(16) float Bs[2][WG_KC][64];
    const int tid = threadIdx.x;
    const int c0 = blockIdx.x * 64, j0 = blockIdx.y * 64, split = blockIdx.z;
    const int gate = c0 >> 8, u0 = c0 & 255;
    const size_t gs = (size_t)L * R * LPG_H;
    const float* gp = gates + (size_t)(gate == 2 ? 3 : gate) * gs;
    const size_t ntok = (size_t)L * R;
    const size_t tok_begin = (size_t)split * chunks_per_split * WG_KC;
    const int tj = tid >> 4, tc = tid & 15;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    auto load_chunk = [&](int buf, int ch) {
        // 16 tokens x 64 floats for A and B = 256 16-byte copies each: one per thread
        const int kk = tid >> 4, q = tid & 15;
        const size_t tok = tok_begin + (size_t)ch * WG_KC + kk;
        const bool in = tok < ntok;
        const int t = in ? (int)(tok / R) : 0;
        const int row = in ? (int)(tok % R) : 0;
        const bool has_next = in && (t + 1 < L) && !done[((size_t)(row / W) * L + t) * W + (row % W)];
        const float* asrc = h + ((size_t)(has_next ? t + 1 : 0) * R + row) * LPG_H + j0 + q * 4;
        cp_async16z(&As[buf][kk][q * 4], asrc, has_next);
        const float* bsrc = gp + (in ? tok : 0) * LPG_H + u0 + q * 4;
        cp_async16z(&Bs[buf][kk][q * 4], bsrc, in);
        cp_commit();
    };
    load_chunk(0, 0);
    for (int ch = 0; ch < chunks_per_split; ++ch) {
        if (ch + 1 < chunks_per_split) { load_chunk((ch + 1) & 1, ch + 1); cp_wait<1>(); }
        else cp_wait<0>();
        __syncthreads();
        const int b = ch & 1;
#pragma unroll
        for (int kk = 0; kk < WG_KC; ++kk) {
            const float4 a = *reinterpret_cast<const float4*>(&As[b][kk][tj * 4]);
            const float4 v = *reinterpret_cast<const float4*>(&Bs[b][kk][tc * 4]);
            const float a_[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                acc[i][0] = fmaf(a_[i], v.x, acc[i][0]); acc[i][1] = fmaf(a_[i], v.y, acc[i][1]);
                acc[i][2] = fmaf(a_[i], v.z, acc[i][2]); acc[i][3] = fmaf(a_[i], v.w, acc[i][3]);
            }
        }
        __syncthreads();
    }
    float* out = partial + (size_t)split * LPG_H * LPG_G;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        float4* p = reinterpret_cast<float4*>(out + (size_t)(j0 + tj * 4 + i) * LPG_G + c0 + tc * 4);
        float4 v = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
        if (accumulate) { const float4 pv = *p; v.x += pv.x; v.y += pv.y; v.z += pv.z; v.w += pv.w; }
        *p = v;
    }
}

// streaming small gradients.  per split partial layout (floats):
//   [0, 8*768)            dWi rows 0..7 (row 7 = dbi because x[7] == 1)
//   [6144, +256)          dbhn
//   [6400, +256)          dw_pi
//   [6656, +256*8)        dW_y
//   [8704, +1)            db_pi ; [8705, +8) db_y
constexpr int SM_WI = 0, SM_BHN = 8 * LPG_G, SM_WPI = SM_BHN + LPG_H, SM_WY = SM_WPI + LPG_H,
              SM_BPI = SM_WY + LPG_H * LPG_Y, SM_BY = SM_BPI + 1, SM_TOTAL = SM_BY + LPG_Y;

__global__ void __launch_bounds__(256)
wgrad_small_kernel(const float* __restrict__ x, const float* __restrict__ h, const float* __restrict__ gates,
                   const float* __restrict__ d_pi_hat, const float* __restrict__ dl, float* __restrict__ partial,
                   int R, int L, int toks_per_split, int accumulate) {
    const int j = threadIdx.x, split = blockIdx.x;
    const size_t ntok = (size_t)L * R, gs = ntok * LPG_H;
    const size_t t0 = (size_t)split * toks_per_split;
    const size_t t1 = min(ntok, t0 + (size_t)toks_per_split);
    float wi[3][8], bhn = 0.f, head[9], hb = 0.f;
#pragma unroll
    for (int g = 0; g < 3; ++g)
#pragma unroll
        for (int q = 0; q < 8; ++q) wi[g][q] = 0.f;
#pragma unroll
    for (int i = 0; i < 9; ++i) head[i] = 0.f;
    for (size_t tok = t0; tok < t1; ++tok) {
        const float4 x0 = *reinterpret_cast<const float4*>(x + tok * 8), x1 = *reinterpret_cast<const float4*>(x + tok * 8 + 4);
        const float xv[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
        const float4 d0 = *reinterpret_cast<const float4*>(dl + tok * 8), d1 = *reinterpret_cast<const float4*>(dl + tok * 8 + 4);
        const float dv[9] = {d_pi_hat[tok], d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
        const float dar = gates[tok * LPG_H + j], daz = gates[gs + tok * LPG_H + j];
        const float dan = gates[2 * gs + tok * LPG_H + j], dhn = gates[3 * gs + tok * LPG_H + j];
        const float y = fmaxf(h[tok * LPG_H + j], 0.0f);
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            wi[0][q] = fmaf(xv[q], dar, wi[0][q]); wi[1][q] = fmaf(xv[q], daz, wi[1][q]); wi[2][q] = fmaf(xv[q], dan, wi[2][q]);
        }
        bhn += dhn;
#pragma unroll
        for (int i = 0; i < 9; ++i) head[i] = fmaf(y, dv[i], head[i]);
        if (j < 9) hb += dv[j];
    }
    float* out = partial + (size_t)split * SM_TOTAL;
    auto put = [&](int idx, float v) { out[idx] = accumulate ? out[idx] + v : v; };
#pragma unroll
    for (int g = 0; g < 3; ++g)
#pragma unroll
        for (int q = 0; q < 8; ++q) put(SM_WI + q * LPG_G + g * LPG_H + j, wi[g][q]);
    put(SM_BHN + j, bhn);
    put(SM_WPI + j, head[0]);
#pragma unroll
    for (int i = 0; i < 8; ++i) put(SM_WY + j * 8 + i, head[1 + i]);
    if (j < 9) put(SM_BPI + j, hb);
}

// embedding MLP backward: pyt = MLP(y_t), pyt1 = MLP(y_{t+1}) * (1 - d)   (lpg.py:66-69)
// per split partial layout = the parameter order e_w0[8][16] e_b0[16] e_w1[16] e_b1[1]  (161 floats)
constexpr int EM_TOTAL = LPG_Y * LPG_E + 2 * LPG_E + 1;
constexpr int EM_SREC = 44;            // y[8] | da[16] | relu(a) dp [16] | dp | pad 3: 176 B, float4 rows conflict-free
__global__ void __launch_bounds__(256, 2)
embed_backward_kernel(const int32_t* __restrict__ obs, const uint8_t* __restrict__ done,
                      const float* __restrict__ critic, const float* __restrict__ lpg, int emb_off,
                      const float* __restrict__ dx, float* __restrict__ partial, const uint32_t* __restrict__ cotmax,
                      int n_agents, int W, int L, int D, int accumulate) {
    // phase 1: each thread back-propagates its token through the two embedding-MLP applications (one pass over the
    //          weights for both) and leaves (y[8], da[16], relu(a)*dp [16], dp) per application in shared memory;
    // phase 2: the block's 2 x 256 samples are split over 4 pairs of warps; in a pair, 32 threads own a 1 x 4 block of
    //          e_w0 each (one scalar + one float4 load per sample and 4 FMAs), 4 threads a quad of e_b0, 4 a quad of
    //          e_w1 and one e_b1.  Sums stay in registers over the whole kernel; the 4 pair partials are combined in a
    //          fixed order at the end (deterministic).
    __shared__ float sp[EM_TOTAL];
    __shared__ float part[4][EM_TOTAL + 3];
    // dx of the tensor-core BPTT kernel is in units of the launch's cotangent scale S (tc.cuh)
    const float inv_s = cotmax ? 1.0f / cot_scale_from_max(*cotmax) : 1.0f;
    extern __shared__ __align__(16) float srec[];          // [2 * 256][44] = 88 KB (dynamic)
    const int tid = threadIdx.x;
    for (int i = tid; i < EM_TOTAL; i += 256) sp[i] = lpg[emb_off + i];
    __syncthreads();
    const size_t total = (size_t)n_agents * L * W;
    const size_t R = (size_t)n_agents * W;
    const size_t iters = (total + (size_t)gridDim.x * 256 - 1) / ((size_t)gridDim.x * 256);
    const int grp = tid >> 6, lt = tid & 63;               // pair of warps, thread within the pair
    // role of this thread in phase 2: src = float4 offset inside a record, ysrc = scalar multiplier offset (-1: 1.0)
    int src = -1, ysrc = -1, out0 = 0, nout = 0;
    if (lt < 32)      { ysrc = lt >> 2; src = 8 + 4 * (lt & 3); out0 = (lt >> 2) * LPG_E + 4 * (lt & 3); nout = 4; }
    else if (lt < 36) { src = 8 + 4 * (lt - 32); out0 = LPG_Y * LPG_E + 4 * (lt - 32); nout = 4; }
    else if (lt < 40) { src = 8 + LPG_E + 4 * (lt - 36); out0 = LPG_Y * LPG_E + LPG_E + 4 * (lt - 36); nout = 4; }
    else if (lt == 40) { src = 8 + 2 * LPG_E; out0 = LPG_Y * LPG_E + 2 * LPG_E; nout = 1; }
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (size_t it = 0; it < iters; ++it) {
        const size_t g = (it * gridDim.x + blockIdx.x) * 256 + tid;
        const bool ok = g < total;
        float y[2][8], dp[2] = {0.f, 0.f};
#pragma unroll
        for (int s = 0; s < 2; ++s)
#pragma unroll
            for (int i = 0; i < 8; ++i) y[s][i] = 0.f;
        if (ok) {
            const int w = (int)(g % W), t = (int)((g / W) % L), n = (int)(g / ((size_t)W * L));
            const float* ct = critic + (size_t)n * D * 8;
            float zy[8];
            tab_logits8<8>(ct, D, obs[((size_t)n * (L + 1) + t) * W + w], zy);
            softmax_c<8>(zy, y[0]);
            tab_logits8<8>(ct, D, obs[((size_t)n * (L + 1) + t + 1) * W + w], zy);
            softmax_c<8>(zy, y[1]);
            const float2 d = *reinterpret_cast<const float2*>(dx + ((size_t)t * R + (size_t)n * W + w) * 2);
            dp[0] = d.x * inv_s;
            dp[1] = done[g] ? 0.0f : d.y * inv_s;
        }
        float* r0 = srec + (size_t)tid * EM_SREC;
        float* r1 = srec + (size_t)(256 + tid) * EM_SREC;
        reinterpret_cast<float4*>(r0)[0] = make_float4(y[0][0], y[0][1], y[0][2], y[0][3]);
        reinterpret_cast<float4*>(r0)[1] = make_float4(y[0][4], y[0][5], y[0][6], y[0][7]);
        reinterpret_cast<float4*>(r1)[0] = make_float4(y[1][0], y[1][1], y[1][2], y[1][3]);
        reinterpret_cast<float4*>(r1)[1] = make_float4(y[1][4], y[1][5], y[1][6], y[1][7]);
#pragma unroll
        for (int eq = 0; eq < LPG_E / 4; ++eq) {
            float da[2][4], rd[2][4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int e = eq * 4 + k;
                float a0 = sp[LPG_Y * LPG_E + e], a1 = a0;
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float wgt = sp[i * LPG_E + e];
                    a0 = fmaf(y[0][i], wgt, a0);
                    a1 = fmaf(y[1][i], wgt, a1);
                }
                const float w1 = sp[LPG_Y * LPG_E + LPG_E + e];
                da[0][k] = a0 > 0.0f ? dp[0] * w1 : 0.0f;   rd[0][k] = fmaxf(a0, 0.0f) * dp[0];
                da[1][k] = a1 > 0.0f ? dp[1] * w1 : 0.0f;   rd[1][k] = fmaxf(a1, 0.0f) * dp[1];
            }
            reinterpret_cast<float4*>(r0 + 8)[eq] = make_float4(da[0][0], da[0][1], da[0][2], da[0][3]);
            reinterpret_cast<float4*>(r0 + 8 + LPG_E)[eq] = make_float4(rd[0][0], rd[0][1], rd[0][2], rd[0][3]);
            reinterpret_cast<float4*>(r1 + 8)[eq] = make_float4(da[1][0], da[1][1], da[1][2], da[1][3]);
            reinterpret_cast<float4*>(r1 + 8 + LPG_E)[eq] = make_float4(rd[1][0], rd[1][1], rd[1][2], rd[1][3]);
        }
        r0[8 + 2 * LPG_E] = dp[0];
        r1[8 + 2 * LPG_E] = dp[1];
        __syncthreads();
        if (nout == 4) {
            const float* base = srec + (size_t)grp * 128 * EM_SREC;
#pragma unroll 4
            for (int q = 0; q < 128; ++q) {
                const float* r = base + (size_t)q * EM_SREC;
                const float4 v = *reinterpret_cast<const float4*>(r + src);
                const float m = ysrc >= 0 ? r[ysrc] : 1.0f;
                acc[0] = fmaf(m, v.x, acc[0]); acc[1] = fmaf(m, v.y, acc[1]);
                acc[2] = fmaf(m, v.z, acc[2]); acc[3] = fmaf(m, v.w, acc[3]);
            }
        } else if (nout == 1) {
            const float* base = srec + (size_t)grp * 128 * EM_SREC + src;
            for (int q = 0; q < 128; ++q) acc[0] += base[(size_t)q * EM_SREC];
        }
        __syncthreads();
    }
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (k < nout) part[grp][out0 + k] = acc[k];
    __syncthreads();
    if (tid < EM_TOTAL) {
        const float v = (part[0][tid] + part[1][tid]) + (part[2][tid] + part[3][tid]);
        float* o = partial + (size_t)blockIdx.x * EM_TOTAL + tid;
        *o = accumulate ? *o + v : v;
    }
}

constexpr int WG_SPLITS = 37;        // capacity of the dWh partial area in token splits (SIMT kernel: 32, tensor-core kernel:
                                     // toued_wgrad_tc_splits() = 24; both checked against this capacity)
constexpr int WG_SPLITS_SIMT = 32;
constexpr int SM_SPLITS = 592;       // 4 per SM for the streaming kernels
constexpr int EM_SPLITS = 296;
constexpr int EM_SMEM = 2 * 256 * EM_SREC * (int)sizeof(float);

extern "C" int toued_lpg_wgrad_workspace_floats(void) {
    return WG_SPLITS * LPG_H * LPG_G + SM_SPLITS * SM_TOTAL + EM_SPLITS * EM_TOTAL;
}

extern "C" int toued_lpg_wgrad(const int32_t* obs, const uint8_t* done, const float* critic,
                               const float* lpg_params, const float* x, const float* h, const float* dgates,
                               const float* d_pi_hat, const float* dl, const float* dx, float* workspace,
                               int n_agents, int n_workers, int rollout_len, int obs_dim,
                               int lifetime_conditioning, int accumulate, void* stream) {
    const int R = n_agents * n_workers, L = rollout_len;
    TOUED_CHECK(R > 0 && L > 0, "toued_lpg_wgrad: empty problem");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t ntok = (size_t)L * R;
    float* p_wh = workspace;
    float* p_sm = p_wh + (size_t)WG_SPLITS * LPG_H * LPG_G;
    float* p_em = p_sm + (size_t)SM_SPLITS * SM_TOTAL;
    {
        const size_t chunks = (ntok + WG_KC - 1) / WG_KC;
        const int cps = (int)((chunks + WG_SPLITS_SIMT - 1) / WG_SPLITS_SIMT);
        wgrad_wh_kernel<<<dim3(LPG_G / 64, LPG_H / 64, WG_SPLITS_SIMT), 256, 0, st>>>(done, h, dgates, p_wh, R, L, n_workers, cps, accumulate);
        TOUED_LAUNCH_CHECK();
    }
    {
        const int tps = (int)((ntok + SM_SPLITS - 1) / SM_SPLITS);
        wgrad_small_kernel<<<SM_SPLITS, 256, 0, st>>>(x, h, dgates, d_pi_hat, dl, p_sm, R, L, tps, accumulate);
        TOUED_LAUNCH_CHECK();
    }
    TOUED_CUDA(cudaFuncSetAttribute(embed_backward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, EM_SMEM));
    embed_backward_kernel<<<EM_SPLITS, 256, EM_SMEM, st>>>(obs, done, critic, lpg_params, lpg_offsets(lifetime_conditioning ? 7 : 5).e_w0,
                                                      dx, p_em, nullptr, n_agents, n_workers, L, obs_dim, accumulate);
    TOUED_LAUNCH_CHECK();
    return 0;
}

// grad = sum over splits of the three partial groups, scattered to the flat parameter layout
__global__ void reduce_partials_kernel(const float* __restrict__ ws, float* __restrict__ grad, int X, int wh_splits, int sm_splits) {
    const LpgOffsets o = lpg_offsets(X);
    const float* p_wh = ws;
    const float* p_sm = p_wh + (size_t)WG_SPLITS * LPG_H * LPG_G;   // fixed offsets: the Wh area is sized for the largest split count
    const float* p_em = p_sm + (size_t)SM_SPLITS * SM_TOTAL;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < LPG_H * LPG_G) {
        float v = 0.f;
        for (int s = 0; s < wh_splits; ++s) v += p_wh[(size_t)s * LPG_H * LPG_G + i];
        grad[o.Wh + i] = v;
        return;
    }
    int k = i - LPG_H * LPG_G;
    if (k < SM_TOTAL) {
        float v = 0.f;
        for (int s = 0; s < sm_splits; ++s) v += p_sm[(size_t)s * SM_TOTAL + k];
        int dst;
        if (k < SM_BHN) { const int q = k / LPG_G, c = k % LPG_G; if (q == 7) dst = o.bi + c; else if (q < X) dst = o.Wi + q * LPG_G + c; else return; }
        else if (k < SM_WPI) dst = o.bhn + (k - SM_BHN);
        else if (k < SM_WY) dst = o.w_pi + (k - SM_WPI);
        else if (k < SM_BPI) dst = o.W_y + (k - SM_WY);
        else if (k < SM_BY) dst = o.b_pi;
        else dst = o.b_y + (k - SM_BY);
        grad[dst] = v;
        return;
    }
    k -= SM_TOTAL;
    if (k < EM_TOTAL) {
        float v = 0.f;
        for (int s = 0; s < EM_SPLITS; ++s) v += p_em[(size_t)s * EM_TOTAL + k];
        grad[o.e_w0 + k] = v;
    }
}

// split counts of the SIMT weight-gradient kernels: which = 0 -> dWh areas, 1 -> small-parameter areas
extern "C" int toued_lpg_wgrad_splits(int which) { return which == 0 ? WG_SPLITS_SIMT : SM_SPLITS; }

// offsets (in floats) of the three partial areas inside the workspace: {Wh, small, embed}
extern "C" int toued_lpg_wgrad_workspace_offset(int which) {
    if (which == 0) return 0;
    if (which == 1) return WG_SPLITS * LPG_H * LPG_G;
    return WG_SPLITS * LPG_H * LPG_G + SM_SPLITS * SM_TOTAL;
}

// embedding-MLP gradients only (shared by the fp32 and the tensor-core reverse pass)
extern "C" int toued_lpg_wgrad_embed(const int32_t* obs, const uint8_t* done, const float* critic, const float* lpg_params,
                                     const float* dx, float* workspace, const uint32_t* cotangent_max, int n_agents,
                                     int n_workers, int rollout_len, int obs_dim, int lifetime_conditioning, int accumulate,
                                     void* stream) {
    float* p_em = workspace + toued_lpg_wgrad_workspace_offset(2);
    TOUED_CUDA(cudaFuncSetAttribute(embed_backward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, EM_SMEM));
    embed_backward_kernel<<<EM_SPLITS, 256, EM_SMEM, (cudaStream_t)stream>>>(
        obs, done, critic, lpg_params, lpg_offsets(lifetime_conditioning ? 7 : 5).e_w0, dx, p_em, cotangent_max, n_agents,
        n_workers, rollout_len, obs_dim, accumulate);
    TOUED_LAUNCH_CHECK();
    return 0;
}

extern "C" int toued_reduce_partials(const float* workspace, float* grad, int lifetime_conditioning, int wh_splits,
                                     int sm_splits, void* stream) {
    const int n = LPG_H * LPG_G + SM_TOTAL + EM_TOTAL;
    // the producer says how many partial areas it filled (SIMT path: toued_lpg_wgrad_splits(); tensor-core path:
    // toued_wgrad_tc_splits() / toued_wgrad_tc_small_splits()); areas beyond that are never read
    TOUED_CHECK(wh_splits >= 1 && wh_splits <= WG_SPLITS, "toued_reduce_partials: wh_splits=%d out of range", wh_splits);
    TOUED_CHECK(sm_splits >= 1 && sm_splits <= SM_SPLITS, "toued_reduce_partials: sm_splits=%d out of range", sm_splits);
    reduce_partials_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(workspace, grad, lifetime_conditioning ? 7 : 5, wh_splits, sm_splits);
    TOUED_LAUNCH_CHECK();
    return 0;
}

// ------------------------------------------------------------------------------------------------
// optax.scale_by_adam(b1=.9, b2=.999, eps=1e-8, eps_root=0) -> scale(lr) -> scale(-1)
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, int n, float lr, float b1, float b2, float eps,
                            float c1, float c2) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float gi = g[i];
    const float mi = b1 * m[i] + (1.0f - b1) * gi;
    const float vi = b2 * v[i] + (1.0f - b2) * gi * gi;
    m[i] = mi; v[i] = vi;
    p[i] -= lr * (mi / c1) / (sqrtf(vi / c2) + eps);
}

extern "C" int toued_adam(float* params, const float* grad, float* mu, float* nu, int n, int count,
                          float lr, float b1, float b2, float eps, void* stream) {
    TOUED_CHECK(n > 0 && count >= 1, "toued_adam: bad arguments");
    const float c1 = 1.0f - powf(b1, (float)count), c2 = 1.0f - powf(b2, (float)count);
    adam_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(params, grad, mu, nu, n, lr, b1, b2, eps, c1, c2);
    TOUED_LAUNCH_CHECK();
    return 0;
}

// Same step with the 1-based update count kept on the device (count_dev holds the number of updates done so far and is
// incremented after the step): nothing of the call depends on host state, so it can sit inside a captured CUDA graph.
__global__ void adam_dev_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                float* __restrict__ v, const int* __restrict__ count_dev, int n, float lr, float b1,
                                float b2, float eps) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float cnt = (float)(*count_dev + 1);
    const float c1 = 1.0f - powf(b1, cnt), c2 = 1.0f - powf(b2, cnt);
    const float gi = g[i];
    const float mi = b1 * m[i] + (1.0f - b1) * gi;
    const float vi = b2 * v[i] + (1.0f - b2) * gi * gi;
    m[i] = mi; v[i] = vi;
    p[i] -= lr * (mi / c1) / (sqrtf(vi / c2) + eps);
}
__global__ void count_incr_kernel(int* count_dev) { *count_dev += 1; }

extern "C" int toued_adam_dev(float* params, const float* grad, float* mu, float* nu, int* count_dev, int n, float lr,
                              float b1, float b2, float eps, void* stream) {
    TOUED_CHECK(n > 0 && count_dev != nullptr, "toued_adam_dev: bad arguments");
    adam_dev_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(params, grad, mu, nu, count_dev, n, lr, b1, b2, eps);
    TOUED_LAUNCH_CHECK();
    count_incr_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(count_dev);
    TOUED_LAUNCH_CHECK();
    return 0;
}

// ------------------------------------------------------------------------------------------------
// --lpg_opt SGD (models/optim.py:6-11): optax.chain(clip_by_global_norm(max_norm), scale(lr), scale(-1)).
// One CTA reduces |g|^2 in a fixed order (deterministic), the update kernel reads it back: nothing depends on host state.
__global__ void __launch_bounds__(1024) sqnorm_kernel(const float* __restrict__ g, int n, float* __restrict__ out) {
    __shared__ float part[32];
    float s = 0.f;
    for (int i = threadIdx.x; i < n; i += 1024) s = fmaf(g[i], g[i], s);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x < 32) {
        s = part[threadIdx.x];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (threadIdx.x == 0) out[0] = s;
    }
}
__global__ void sgd_clip_kernel(float* __restrict__ p, const float* __restrict__ g, const float* __restrict__ sq, int n,
                                float lr, float max_norm) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float norm = sqrtf(sq[0]);
    // optax.clip_by_global_norm: where(norm < max_norm, g, g / norm * max_norm)
    const float gi = norm < max_norm ? g[i] : (g[i] / norm) * max_norm;
    p[i] -= lr * gi;
}
extern "C" int toued_sgd_clip(float* params, const float* grad, float* sqnorm_scratch, int n, float lr, float max_norm,
                              void* stream) {
    TOUED_CHECK(n > 0 && sqnorm_scratch != nullptr, "toued_sgd_clip: bad arguments");
    sqnorm_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(grad, n, sqnorm_scratch);
    TOUED_LAUNCH_CHECK();
    sgd_clip_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(params, grad, sqnorm_scratch, n, lr, max_norm);
    TOUED_LAUNCH_CHECK();
    return 0;
}

// ------------------------------------------------------------------------------------------------
// max |cotangent| of one reverse-pass launch (d pi_hat f32[n_tok], d y_hat f32[n_tok][8]) as the bit pattern of a
// non-negative float (integer order == float order, so atomicMax is exact and order-independent): the tensor-core
// reverse kernels derive their power-of-two operand scale from it (tc.cuh::cot_scale_from_max).  The maximum is taken
// over the bit patterns of |v|, in which NaN sorts above +inf: any non-finite cotangent gives +inf (S = 1) and sets
// TOUED_STATUS_NONFINITE_COT in out_bits[1] (fmaxf would skip a NaN and report the finite maximum).
__global__ void cot_max_kernel(const float* __restrict__ d_pi_hat, const float* __restrict__ d_y_hat, size_t n_tok,
                               uint32_t* __restrict__ out_bits) {
    uint32_t m = 0u;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_tok; i += stride)
        m = max(m, __float_as_uint(d_pi_hat[i]) & 0x7FFFFFFFu);
    const uint4* y4 = reinterpret_cast<const uint4*>(d_y_hat);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < 2 * n_tok; i += stride) {
        const uint4 v = y4[i];
        m = max(m, max(max(v.x & 0x7FFFFFFFu, v.y & 0x7FFFFFFFu), max(v.z & 0x7FFFFFFFu, v.w & 0x7FFFFFFFu)));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0 && m > 0u) {
        atomicMax(out_bits, min(m, 0x7F800000u));
        if (m >= 0x7F800000u) atomicOr(out_bits + 1, TOUED_STATUS_NONFINITE_COT);
    }
}

extern "C" int toued_cotangent_max(const float* d_pi_hat, const float* d_y_hat, int n_agents, int n_workers, int rollout_len,
                                   uint32_t* out_bits, void* stream) {
    const size_t n_tok = (size_t)n_agents * n_workers * rollout_len;
    TOUED_CHECK(n_tok > 0 && out_bits != nullptr, "toued_cotangent_max: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    TOUED_CUDA(cudaMemsetAsync(out_bits, 0, sizeof(uint32_t), st));     // word 0 only: the status word is sticky
    cot_max_kernel<<<296, 256, 0, st>>>(d_pi_hat, d_y_hat, n_tok, out_bits);
    TOUED_LAUNCH_CHECK();
    return 0;
}
