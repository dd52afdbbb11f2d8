// Tensor-core GRU backward (BPTT) for the LPG network — the reverse of gru_forward_tc.cu, i.e. the part
// of jax.grad(_train_agent) (meta/train.py:121-128) that flows through models/lpg.py:11-30,77-84.
//
// A CTA owns 128 sequences and walks t = 0 .. L-1 (the forward scan is reversed).  Per step
//     dh_t   = relu'(h_t) * (d pi_hat * w_pi + dl . W_y)  +  (1 - done_{t-1}) * carry
//     dG_g   = dh_t * f_g            (f_r, f_z, f_hn, f_an saved by the forward epilogue)
//     carry' = dGh @ Wh^T + z * dh_t
// The carry stays in fp32 in TMEM (two 256-column sets, ping-pong): dGh @ Wh^T is accumulated by
// tcgen05.mma from fp16 operands (dG written by the epilogue warps into SW128 smem chunks, Wh chunks
// streamed by a TMA-producer warp), and the element-wise z*dh_t term is injected into the same
// accumulator by a tiny identity MMA on an fp16 hi/lo pair, so the recurrent chain keeps ~22 mantissa
// bits without ever leaving tensor memory.
// Scaled arithmetic (tc.cuh, "scaled fp16 operands"): the kernel multiplies the incoming cotangents by the power of two
// S derived from `cotmax` and everything downstream -- carry, dG, dl, dx -- is in units of S; the consumers
// (toued_lpg_wgrad_tc, toued_lpg_wgrad_embed) take S back out.  A dG or z*dh value that leaves fp16's range (the
// conversion saturates it) or is not finite sets TOUED_STATUS_FP16_RANGE in cotmax[1]: the result is then unreliable.
// Round 1 used bf16 operands (8 significant bits; the rounding of Wh is systematic over all tokens) and left 0.6-1.6e-2
// of error on the GRU weight blocks of the meta-gradient.
// Outputs for the weight-gradient kernels: S * dG (dar, daz, dhn, dan) as an fp16 token-tile image,
// the head-logit cotangents S * dl and S * (d pyt, d pyt1).
#include "tc.cuh"
#include "lpg_common.cuh"
#include "../../include/toued.h"

constexpr int BT_M = 128;
// Epilogue warps 0..7: warp w owns TMEM lanes [32 (w & 3), +32) and the 32-unit half (w >> 2) of every 64-unit block,
// i.e. four 8-unit chunks per thread and unit block.  Eight warps keep the kernel at 168 registers; more epilogue warps
// lower the register cap until the chunk loop spills, and more than two warps per TMEM quadrant queue on the same
// tcgen05.ld port (DESIGN.md section 7.0).
constexpr int BT_THREADS = 11 * 32;              // 8 epilogue warps + TMA-load warp 8 + MMA warp 9 + TMA-store warp 10
constexpr int BT_ACHUNK = BT_M * 128;            // 16 KB: [128 rows][64 fp16], K-major SW128
constexpr int BT_SSTAGE = 4 * BT_ACHUNK;         // stored chunks dG_r, dG_z, dG_hn (also MMA operands), dG_an: DOUBLE-buffered over the unit blocks
constexpr int BT_CSTAGE = 2 * BT_ACHUNK;         // cz_hi, cz_lo (MMA operands only): single buffer, released K-step by K-step
constexpr int BT_BSLICE = LPG_H * 32;            // 8 KB: one K-step of Wh^T, [256 units][16 c] as a no-swizzle K = 16 block
constexpr int BT_NSB = 6;                        // two K-steps (x 3 gates) of Wh^T in flight
constexpr int BT_ICHUNK = 512;                   // 16 x 16 identity (no-swizzle K = 16 block)

// Wh[j][c] -> 48 fp16 K-step slices [s = c / 16][row j][k = c % 16], each an 8 KB K-major no-swizzle K = 16 block
__global__ void pack_wh_bwd_kernel(const float* __restrict__ Wh, __half* __restrict__ img) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= LPG_H * LPG_G) return;
    const int j = i / LPG_G, c = i % LPG_G;
    char* base = reinterpret_cast<char*>(img) + (size_t)(c >> 4) * BT_BSLICE;
    *reinterpret_cast<__half*>(base + k16_offset(j, c & 15)) = __float2half_rn(Wh[i]);
}

extern "C" int toued_pack_wh_backward(const float* lpg_params, void* whb_img, void* stream) {
    pack_wh_bwd_kernel<<<(LPG_H * LPG_G + 255) / 256, 256, 0, (cudaStream_t)stream>>>(
        lpg_params + lpg_offsets(5).Wh, (__half*)whb_img);
    TOUED_LAUNCH_CHECK();
    return 0;
}

// 16-byte read-only load that does not allocate in L1: with ~226 KB of the SM's 256 KB configured as shared memory the L1
// is a few KB, and the saved activations are read exactly once
__device__ __forceinline__ uint4 ldg_stream(const __half* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ void unpack8h(const uint4& r, float (&v)[8]) {
    const __half2* h = reinterpret_cast<const __half2*>(&r);
#pragma unroll
    for (int e = 0; e < 4; ++e) { const float2 f = __half22float2(h[e]); v[2 * e] = f.x; v[2 * e + 1] = f.y; }
}
__global__ void __launch_bounds__(BT_THREADS, 1)
gru_backward_tc_kernel(const uint8_t* __restrict__ done, const float* __restrict__ lpg, int X,
                       const unsigned char* __restrict__ whb_img, const __half* __restrict__ h16,
                       const __half* __restrict__ fac, const float* __restrict__ y_hat,
                       const float* __restrict__ d_pi_hat, const float* __restrict__ d_y_hat,
                       unsigned char* __restrict__ dgimg, float* __restrict__ dl_out, float* __restrict__ dx,
                       uint32_t* __restrict__ cotmax, int R, int L, int W) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    // (offset arithmetic on the __shared__ array, not an integer round trip: the compiler keeps the shared
    //  address space and emits LDS / STS instead of generic LD / ST)
    unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    unsigned char* sS = smem;                                   // 2 x 64 KB   stored chunks (dG_r, dG_z, dG_hn, dG_an), buffer = unit block & 1
    unsigned char* sC = sS + 2 * BT_SSTAGE;                     // 32 KB       cz_hi, cz_lo
    unsigned char* sB = sC + BT_CSTAGE;                         // BT_NSB x 8 KB Wh^T K-step slices
    unsigned char* sI = sB + BT_NSB * BT_BSLICE;                // 8 KB identity
    float* swp = reinterpret_cast<float*>(sI + BT_ICHUNK);      // [256]
    float* sWy = swp + LPG_H;                                   // [256][8]
    float* sWi = sWy + LPG_H * LPG_Y;                           // [256 units][4]: Wi row 3 x gates (r, z, n), Wi row 4 x gate r
    float* sWi2 = sWi + LPG_H * 4;                              // [256 units][2]: Wi row 4 x gates (z, n)
    float* sdx = sWi2 + LPG_H * 2;                              // [128][2]
    // k_full[ks]:  K-step ks of the current unit block is in shared memory (4 epilogue warps arrive)
    // k_empty[ks]: the MMAs of that K-step have read it (cz chunks may be overwritten; also orders the reuse of a stored buffer)
    //              AND the store warp has observed k_full[ks] of this unit block (two arrivals): no waiter on k_full can
    //              fall a whole phase behind the epilogue warps
    // s_empty[b]:  the bulk stores of stored buffer b have read it
    __shared__ __align__(8) uint64_t b_full[BT_NSB], b_empty[BT_NSB], k_full[4], k_empty[4], s_empty[2], q_full;
    __shared__ uint32_t tmem_base_s;

    const LpgOffsets o = lpg_offsets(X);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int row0 = blockIdx.x * BT_M;

    if (tid == 0) {
        for (int s = 0; s < BT_NSB; ++s) { mbar_init(&b_full[s], 1); mbar_init(&b_empty[s], 1); }
        for (int k = 0; k < 4; ++k) { mbar_init(&k_full[k], 4); mbar_init(&k_empty[k], 2); }
        mbar_init(&s_empty[0], 1); mbar_init(&s_empty[1], 1); mbar_init(&q_full, 1);
        mbar_fence_init();
    }
    if (warp == 9) tmem_alloc(&tmem_base_s, 512);
    for (int i = tid; i < LPG_H; i += BT_THREADS) swp[i] = lpg[o.w_pi + i];
    for (int i = tid; i < LPG_H * LPG_Y; i += BT_THREADS) sWy[i] = lpg[o.W_y + i];
    for (int i = tid; i < LPG_H * 6; i += BT_THREADS) {
        const int u = i / 6, q = i % 6;                // q = 3 * (input row - 3) + gate
        const float w = lpg[o.Wi + (3 + q / 3) * LPG_G + (q % 3) * LPG_H + u];
        if (q < 4) sWi[u * 4 + q] = w; else sWi2[u * 2 + q - 4] = w;
    }
    for (int i = tid; i < 16 * 16; i += BT_THREADS) {
        const int n = i >> 4, k = i & 15;
        *reinterpret_cast<__half*>(sI + k16_offset(n, k)) = __float2half_rn(n == k ? 1.0f : 0.0f);
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;
    const size_t R32 = ((size_t)R + 31) >> 5;                   // 32-row blocks of the RB32 layout
    const size_t tstride = R32 * 32 * LPG_H;                    // RB32 elements per timestep

    if (warp == 8) {
        // ===================== TMA producer: Wh^T K-step slices in (unit block, K-step, gate) order ====
        if (lane == 0) {
            uint32_t it = 0;
            for (int t = 0; t < L; ++t) {
                if (t + 1 == L) break;                                   // the last step issues no MMAs
                for (int ub = 0; ub < 4; ++ub)
                    for (int kk = 0; kk < 4; ++kk) {
                        const int ks = ((kk & 1) << 1) | (kk >> 1);
                        for (int g = 0; g < 3; ++g, ++it) {
                            const int s = it % BT_NSB;
                            mbar_wait(&b_empty[s], ((it / BT_NSB) & 1) ^ 1);
                            mbar_expect_tx(&b_full[s], BT_BSLICE);
                            bulk_g2s(sB + s * BT_BSLICE, whb_img + (size_t)(g * 16 + ub * 4 + ks) * BT_BSLICE, BT_BSLICE, &b_full[s]);
                        }
                    }
            }
        }
    } else if (warp == 9) {
        // ===================== MMA issuer =============================================================
        // The whole warp walks the loop (all lanes wait on the barriers); one elected lane issues (tc.cuh::elect_one).
        {
            constexpr uint32_t idesc256 = tc_idesc(BT_M, 256, 0), idesc16 = tc_idesc(BT_M, 16, 0);     // fp16 operands
            const uint32_t s_addr = smem_u32(sS), c_addr = smem_u32(sC), i_addr = smem_u32(sI);
            const uint64_t cd0 = tc_smem_desc(c_addr), idd = tc_smem_desc_k16(i_addr);
            uint32_t it = 0;
            uint32_t ait = 0;
            for (int t = 0; t < L; ++t) {
                const uint32_t q_addr = tmem_base + (t & 1) * 256;
                const bool mma = t + 1 < L;                          // the last step only stores its dG tiles
                for (int ub = 0; ub < 4; ++ub, ++ait) {
                    // The stage is consumed K-step by K-step (16 units = what four epilogue warps finish every two
                    // chunks): the MMAs of a unit block are spread over the time the epilogue warps need to produce it.
                    const uint64_t ad0 = tc_smem_desc(s_addr + (ait & 1) * BT_SSTAGE);
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk) {
                        // K-steps in the order the epilogue completes them: 0, 2, 1, 3 (the two unit halves progress together)
                        const int ks = ((kk & 1) << 1) | (kk >> 1);
                        uint32_t sg[3];
                        if (mma) {
#pragma unroll
                            for (int g = 0; g < 3; ++g, ++it) {
                                sg[g] = it % BT_NSB;
                                mbar_wait(&b_full[sg[g]], (it / BT_NSB) & 1);
                            }
                        }
                        mbar_wait(&k_full[ks], ait & 1);
                        tc_fence_after();
                        if (elect_one()) {
                            if (mma) {
#pragma unroll
                                for (int g = 0; g < 3; ++g)
                                    tc_mma(q_addr, ad0 + (uint64_t)((g * BT_ACHUNK) >> 4) + 2 * ks,
                                           tc_smem_desc_k16(smem_u32(sB + sg[g] * BT_BSLICE)), idesc256, (ub | kk | g) != 0);
                                // z * dh_t (fp16 hi + lo) through a 16 x 16 identity: accumulates onto the 16 columns of this K-step
                                tc_mma(q_addr + ub * 64 + ks * 16, cd0 + 2 * ks, idd, idesc16, 1u);
                                tc_mma(q_addr + ub * 64 + ks * 16, cd0 + (uint64_t)(BT_ACHUNK >> 4) + 2 * ks, idd, idesc16, 1u);
#pragma unroll
                                for (int g = 0; g < 3; ++g) tc_commit(&b_empty[sg[g]]);
                            }
                            tc_commit(&k_empty[ks]);                 // (no MMAs outstanding on the last step: arrives at once)
                            if (mma && ub == 3 && kk == 3) tc_commit(&q_full);
                        }
                        __syncwarp();
                    }
                }
            }
        }
    } else if (warp == 10) {
        // ===================== TMA store warp: dG tiles of every unit block -> token-tile image ==========
        // The SW128 chunks in smem ARE the image's 8 KB sub-tiles of the weight-gradient GEMM, so they leave as
        // full-line bulk stores.  The stored chunks are double-buffered: the stores of unit block n drain while the
        // epilogue warps fill the other buffer with unit block n + 1 (round 1 had ONE stage, and ncu showed the epilogue
        // warps waiting 15 % of their time for the stores to release it: profiles/r02 stall table in DESIGN.md section 7).
        if (lane == 0) {
            const uint32_t s_addr = smem_u32(sS);
            const size_t Rp = ((size_t)R + 63) & ~(size_t)63;
            const int nsub = ((size_t)row0 + 64 < Rp) ? 2 : 1;      // 64-token sub-tiles of this CTA inside the image
            uint32_t ait = 0;
            for (int t = 0; t < L; ++t) {
                for (int ub = 0; ub < 4; ++ub, ++ait) {
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk) {                 // in completion order
                        const int ks = ((kk & 1) << 1) | (kk >> 1);
                        mbar_wait(&k_full[ks], ait & 1);
                        mbar_arrive(&k_empty[ks]);
                    }
                    const size_t itok0 = (size_t)t * Rp + row0;
                    const uint32_t src0 = s_addr + (ait & 1) * BT_SSTAGE;
#pragma unroll
                    for (int g = 0; g < 4; ++g)
                        for (int sub = 0; sub < nsub; ++sub)
                            bulk_s2g(dgimg + tile_img_offset(itok0 + sub * 64, 16, (g * 4 + ub) * 64), src0 + g * BT_ACHUNK + sub * 8192, 8192);
                    bulk_commit();
                    if (ait > 0) {
                        bulk_wait_read_1();                          // the group of the previous unit block has been read
                        mbar_arrive(&s_empty[(ait - 1) & 1]);
                    }
                }
            }
            bulk_wait_read();
            mbar_arrive(&s_empty[(ait - 1) & 1]);
            bulk_wait_all();
        }
    } else {
        // ===================== epilogue / producer-of-A warps 0 .. 7 ====================================
        const int q = warp & 3, hf = warp >> 2;
        const int rl = q * 32 + lane;
        const int row = row0 + rl;
        const bool rv = row < R;
        const int rsafe = rv ? row : 0;
        const int n_ag = rsafe / W, w_ag = rsafe % W;
        uint32_t ait = 0;
        // Some fp16 operand of this thread left fp16's range (the conversion saturated it) or was not finite: reported in
        // cotmax[1].  Two checks per element cover all five operands: |cz| <= |dh|, |gan|, |ghn| <= |dh| and
        // |gz| <= |dh| / 2 (z, r, n, h' in their ranges), so |dh| bounds all but gr; a NaN anywhere in the chain (dh, or
        // a saved gate) reaches gr through gan and ghn.  A NaN stays in the running maximum.  Checking dh rather than
        // z * dh also reports a carry grown past 65504 / S where z happens to be small.
        float range_max = 0.0f;                  // NaN-propagating running max of |dh|, |gr|
        const uint32_t sS_u32 = smem_u32(sS), sC_u32 = smem_u32(sC);
        const float S = cotmax ? cot_scale_from_max(*cotmax) : 1.0f;      // power of two: scaling is exact
        // ---- software pipeline: the factor loads of the next 8-unit chunk and the head cotangents of the
        //      next timestep are issued one iteration ahead (across unit-block / timestep boundaries) ----
        struct FacLoads { uint4 r, z, n, hn, hx; };              // gates of step t, h of step t+1 (the carry h')
        // per-thread element index of (t = 0, this row, this thread's first unit); chunk (ub, c8) adds (ub * 8 + c8) * 256
        const size_t fbase = rb32_index(0, R32, rsafe, hf * 32);
        const __half* p_r = fac + fac_index(0, R32, rsafe, hf * 32, 0);
        const __half* p_z = fac + fac_index(0, R32, rsafe, hf * 32, 1);
        const __half* p_n = fac + fac_index(0, R32, rsafe, hf * 32, 2);
        const __half* p_hn = fac + fac_index(0, R32, rsafe, hf * 32, 3);
        const __half* p_hx = h16 + fbase;                        // + (t + 1) * tstride at use
        const int tlast = L - 1;
        auto issue_fac = [&](int t_, int ub_, int c8_) {
            FacLoads l;
            const size_t off = (size_t)t_ * tstride + (size_t)((ub_ * 8 + c8_) << 8);
            const size_t foff = 4 * (size_t)t_ * tstride + (size_t)((ub_ * 8 + c8_) << 8);     // gate planes: interleaved per 32-row block
            l.r = ldg_stream(p_r + foff);
            l.z = ldg_stream(p_z + foff);
            l.n = ldg_stream(p_n + foff);
            l.hn = ldg_stream(p_hn + foff);
            // h of step t+1; at the last step the (unused: masked by nd_hp = 0) load stays inside the tensor
            l.hx = ldg_stream(p_hx + off + (t_ < tlast ? tstride : 0));
            return l;
        };
        struct RowLoads { float4 y0, y1, d0, d1; float dpi; uint8_t dn, dn_hp; };
        auto issue_row = [&](int t_) {
            RowLoads r;
            const size_t tok_ = (size_t)t_ * R + rsafe;
            const float4* q0 = reinterpret_cast<const float4*>(y_hat + tok_ * 8);
            const float4* q1 = reinterpret_cast<const float4*>(d_y_hat + tok_ * 8);
            r.y0 = q0[0]; r.y1 = q0[1]; r.d0 = q1[0]; r.d1 = q1[1];
            r.dpi = d_pi_hat[tok_];
            r.dn = t_ > 0 ? done[((size_t)n_ag * L + (t_ - 1)) * W + w_ag] : (uint8_t)1;
            r.dn_hp = t_ + 1 < L ? done[((size_t)n_ag * L + t_) * W + w_ag] : (uint8_t)1;   // the cell at t consumed (1 - done_t) h_{t+1}
            return r;
        };
        FacLoads nxt = issue_fac(0, 0, 0);
        RowLoads rnx = issue_row(0);
        for (int t = 0; t < L; ++t) {
            const size_t tok = (size_t)t * R + rsafe;
            // head cotangents of this row (softmax backward of y_hat), lpg.py:83-84
            float dl[8], dpi;
            const RowLoads rc = rnx;
            if (t + 1 < L) rnx = issue_row(t + 1);
            {
                const float yh[8] = {rc.y0.x, rc.y0.y, rc.y0.z, rc.y0.w, rc.y1.x, rc.y1.y, rc.y1.z, rc.y1.w};
                const float dy[8] = {rc.d0.x, rc.d0.y, rc.d0.z, rc.d0.w, rc.d1.x, rc.d1.y, rc.d1.z, rc.d1.w};
                float s = 0.f;
#pragma unroll
                for (int i = 0; i < 8; ++i) s = fmaf(yh[i], dy[i], s);
#pragma unroll
                for (int i = 0; i < 8; ++i) dl[i] = rv ? S * (yh[i] * (dy[i] - s)) : 0.0f;
                dpi = rv ? S * rc.dpi : 0.0f;
                if (hf == 0 && rv) {
                    float4* qo = reinterpret_cast<float4*>(dl_out + tok * 8);
                    qo[0] = make_float4(dl[0], dl[1], dl[2], dl[3]);
                    qo[1] = make_float4(dl[4], dl[5], dl[6], dl[7]);
                }
            }
            // carry mask: the cell at step t-1 consumed (1 - done_{t-1}) * h_t
            const float nd = (t > 0 && rv && !rc.dn) ? 1.0f : 0.0f;
            const float nd_hp = rc.dn_hp ? 0.0f : 1.0f;
            if (t > 0) { mbar_wait(&q_full, (t - 1) & 1); tc_fence_after(); }
            const uint32_t p_addr = tmem_base + ((t - 1) & 1) * 256 + ((uint32_t)(q * 32) << 16);
            float dx3 = 0.f, dx4 = 0.f;
            for (int ub = 0; ub < 4; ++ub) {
                const int ubase = ub * 64 + hf * 32;                 // first of this thread's 32 units
                const uint32_t sSb = sS_u32 + (ait & 1) * BT_SSTAGE;
#pragma unroll
                for (int c8 = 0; c8 < 4; ++c8) {
                    const int u0 = ubase + c8 * 8;
                    float carry[8];
                    if (t > 0) tmem_ld8(p_addr + u0, carry);
                    const FacLoads cur = nxt;
                    {   // prefetch the next chunk (next c8, else next unit block, else next timestep; past the end: a harmless reload)
                        int t2 = t, ub2 = ub, c2 = c8 + 1;
                        if (c2 == 4) { c2 = 0; ++ub2; if (ub2 == 4) { ub2 = 0; t2 = min(t + 1, tlast); } }
                        nxt = issue_fac(t2, ub2, c2);
                    }
                    if (t > 0) tmem_ld_wait();
                    else {
#pragma unroll
                        for (int e = 0; e < 8; ++e) carry[e] = 0.f;
                    }
                    float gr_[8], zz[8], gn_[8], hn_[8], hx[8];
                    // the saved z plane carries relu'(h_t) in its sign bits (z itself is in [0, 1]): set = h_t <= 0
                    const uint32_t zw[4] = {cur.z.x, cur.z.y, cur.z.z, cur.z.w};
                    unpack8h(cur.r, gr_); unpack8h(make_uint4(zw[0] & 0x7FFF7FFFu, zw[1] & 0x7FFF7FFFu, zw[2] & 0x7FFF7FFFu, zw[3] & 0x7FFF7FFFu), zz);
                    unpack8h(cur.n, gn_); unpack8h(cur.hn, hn_); unpack8h(cur.hx, hx);
                    float gr[8], gz[8], ghn[8], gan[8], cz[8];
#pragma unroll
                    for (int e = 0; e < 8; ++e) {
                        const int u = u0 + e;
                        float dh = nd * carry[e];
                        {
                            const float4 w0 = *reinterpret_cast<const float4*>(sWy + u * 8), w1 = *reinterpret_cast<const float4*>(sWy + u * 8 + 4);
                            float hd = dpi * swp[u];
                            hd = fmaf(dl[0], w0.x, hd); hd = fmaf(dl[1], w0.y, hd); hd = fmaf(dl[2], w0.z, hd); hd = fmaf(dl[3], w0.w, hd);
                            hd = fmaf(dl[4], w1.x, hd); hd = fmaf(dl[5], w1.y, hd); hd = fmaf(dl[6], w1.z, hd); hd = fmaf(dl[7], w1.w, hd);
                            dh += ((zw[e >> 1] >> (15 + 16 * (e & 1))) & 1u) ? 0.0f : hd;
                        }
                        if (!rv) dh = 0.0f;
                        // GRUCell backward factors from the saved gates (models/lpg.py:11-30):
                        //   d a_n = dh (1-z)(1-n^2);  d(Whn h + bhn) = d a_n * r;  d a_r = d a_n * hn * r(1-r);
                        //   d a_z = dh (h' - n) z(1-z)
                        const float omz = 1.0f - zz[e];
                        gan[e] = dh * omz * (1.0f - gn_[e] * gn_[e]);
                        ghn[e] = gan[e] * gr_[e];
                        gr[e] = ghn[e] * hn_[e] * (1.0f - gr_[e]);
                        gz[e] = dh * (nd_hp * hx[e] - gn_[e]) * zz[e] * omz;
                        cz[e] = dh * zz[e];
                        range_max = fmax3_nan(range_max, fabsf(dh), fabsf(gr[e]));
                        {
                            const float4 w0 = *reinterpret_cast<const float4*>(sWi + u * 4);
                            const float2 w1 = *reinterpret_cast<const float2*>(sWi2 + u * 2);
                            dx3 = fmaf(gr[e], w0.x, fmaf(gz[e], w0.y, fmaf(gan[e], w0.z, dx3)));
                            dx4 = fmaf(gr[e], w0.w, fmaf(gz[e], w1.x, fmaf(gan[e], w1.y, dx4)));
                        }
                    }
                    // z * dh as an fp16 hi / lo pair (saturating conversions; the residual of a saturated value saturates too)
                    uint4 czh4, czl4;
                    {
                        uint32_t hi[4], lo[4];
#pragma unroll
                        for (int e2 = 0; e2 < 4; ++e2) {
                            hi[e2] = pack_h2_sat(cz[2 * e2], cz[2 * e2 + 1]);
                            const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&hi[e2]));
                            lo[e2] = pack_h2_sat(cz[2 * e2] - f.x, cz[2 * e2 + 1] - f.y);
                        }
                        czh4 = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                        czl4 = make_uint4(lo[0], lo[1], lo[2], lo[3]);
                    }
                    // Reuse of the shared-memory stage (both waits have long been satisfied in steady state: the wait is one
                    // unit block / half a unit block behind the consumer):
                    //   first chunk of a unit block: the bulk stores of unit block ait - 2 have read this stored buffer;
                    //   first chunk of each K-step: the MMAs of the previous unit block have read that K-step (cz chunks; the
                    //   MMAs that read this stored buffer two unit blocks ago completed before those).
                    if (c8 == 0 && ait >= 2) mbar_wait(&s_empty[ait & 1], ((ait >> 1) & 1) ^ 1);
                    if ((c8 & 1) == 0 && ait > 0) mbar_wait(&k_empty[hf * 2 + (c8 >> 1)], (ait & 1) ^ 1);
                    const uint32_t so = sw128_offset(BT_M, rl, hf * 32 + c8 * 8);
                    st_shared_v4(sSb + so + 0 * BT_ACHUNK, pack8h_sat(gr));
                    st_shared_v4(sSb + so + 1 * BT_ACHUNK, pack8h_sat(gz));
                    st_shared_v4(sSb + so + 2 * BT_ACHUNK, pack8h_sat(ghn));
                    st_shared_v4(sSb + so + 3 * BT_ACHUNK, pack8h_sat(gan));
                    st_shared_v4(sC_u32 + so, czh4);
                    st_shared_v4(sC_u32 + so + BT_ACHUNK, czl4);
                    if (c8 & 1) {                                  // K-step 2 hf + (c8 >> 1) of this unit block is complete
                        fence_proxy_async_smem();
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&k_full[hf * 2 + (c8 >> 1)]);
                    }
                }
                ++ait;
            }
            // d pyt / d pyt1: combine the two unit halves of the row (fixed order)
            if (hf > 0) { sdx[((hf - 1) * BT_M + rl) * 2] = dx3; sdx[((hf - 1) * BT_M + rl) * 2 + 1] = dx4; }
            asm volatile("bar.sync 1, 256;" ::: "memory");
            if (hf == 0 && rv) {
                dx3 += sdx[rl * 2]; dx4 += sdx[rl * 2 + 1];
                *reinterpret_cast<float2*>(dx + ((size_t)t * R + row) * 2) = make_float2(dx3, dx4);
            }
            asm volatile("bar.sync 1, 256;" ::: "memory");
        }
        if (__any_sync(0xffffffffu, !(range_max <= 65504.0f)) && lane == 0 && cotmax) atomicOr(cotmax + 1, TOUED_STATUS_FP16_RANGE);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 9) tmem_dealloc(tmem_base, 512);
}

static size_t gru_bwd_tc_smem() {
    return 2 * BT_SSTAGE + BT_CSTAGE + BT_NSB * BT_BSLICE + BT_ICHUNK + sizeof(float) * (LPG_H + LPG_H * LPG_Y + LPG_H * 6 + BT_M * 2) + 1024;
}

extern "C" int toued_gru_backward_tc(const uint8_t* done, const float* lpg_params, const void* whb_img,
                                     const void* h16, const void* fac, const float* y_hat, const float* d_pi_hat,
                                     const float* d_y_hat, void* dgimg, float* dl, float* dx, uint32_t* cotangent_max,
                                     int n_agents, int n_workers, int rollout_len, int lifetime_conditioning, void* stream) {
    const int R = n_agents * n_workers;
    TOUED_CHECK(R > 0 && rollout_len > 0, "toued_gru_backward_tc: empty problem");
    const size_t smem = gru_bwd_tc_smem();
    TOUED_CUDA(cudaFuncSetAttribute(gru_backward_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    gru_backward_tc_kernel<<<(R + BT_M - 1) / BT_M, BT_THREADS, smem, (cudaStream_t)stream>>>(
        done, lpg_params, lifetime_conditioning ? 7 : 5, (const unsigned char*)whb_img, (const __half*)h16,
        (const __half*)fac, y_hat, d_pi_hat, d_y_hat, (unsigned char*)dgimg, dl, dx, cotangent_max, R, rollout_len, n_workers);
    TOUED_LAUNCH_CHECK();
    return 0;
}
