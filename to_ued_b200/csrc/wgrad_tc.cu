// Tensor-core weight gradient of the recurrent matrix:  dWh[j][c] = sum_tok h'[tok][j] * dGh[tok][c]
// (the parameter-gradient sum of jax.grad through models/lpg.py:29, flax GRUCell hr/hz/hn kernels).
//
// Both operands are contracted over tokens, i.e. they are MN-major for tcgen05: the 64-token x 64-column
// sub-tiles of the fp16 token tile images written by the forward (h') and backward (S * dG, tc.cuh) kernels are
// bulk-copied (cp.async.bulk) into shared memory and used as-is.  A CTA owns one 128 (j) x 384 (c)
// output tile (fp32 accumulators in 384 TMEM columns) and a contiguous range of token blocks; the four
// tile types of one token range are adjacent CTAs so they share their operand stream through L2.
// Output: per-split partial sums (deterministic; reduced by toued_reduce_partials).
#include "tc.cuh"
#include "lpg_common.cuh"
#include "../../include/toued.h"

// small-gradient partial layout (identical to wgrad_small_kernel in lpg_backward.cu)
constexpr int SMT_WI = 0, SMT_BHN = 8 * LPG_G, SMT_WPI = SMT_BHN + LPG_H, SMT_WY = SMT_WPI + LPG_H,
              SMT_BPI = SMT_WY + LPG_H * LPG_Y, SMT_BY = SMT_BPI + 1, SMT_TOTAL = SMT_BY + LPG_Y;
constexpr int WT_THREADS = 192;            // 4 epilogue warps + producer warp + MMA warp
constexpr int WT_NS = 3;
constexpr int WT_STAGE = 9 * 8192;         // dWh tiles: 2 A + 6 B sub-tiles of 8 KB; x tiles: 1 A + 8 B

__global__ void __launch_bounds__(WT_THREADS, 1)
wgrad_wh_tc_kernel(const unsigned char* __restrict__ hpimg, const unsigned char* __restrict__ dgimg,
                   const unsigned char* __restrict__ ximg, float* __restrict__ partial, float* __restrict__ small_partial,
                   const uint32_t* __restrict__ cotmax, int n_tok_blocks, int blocks_per_split, int accumulate) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    // (offset arithmetic on the __shared__ array, not an integer round trip: the compiler keeps the shared
    //  address space and emits LDS / STS instead of generic LD / ST)
    unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    __shared__ __align__(8) uint64_t full[WT_NS], empty[WT_NS], done_bar;
    __shared__ uint32_t tmem_base_s;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // tile types 0-3: dWh tile (jt, ct) = h'^T [128 j] x dG [384 c];
    // tile types 4-5: input-side gradients  x^T [8 (of 64) inputs] x dG column groups 8*(type-4) .. +8
    const int type = blockIdx.x % 6, split = blockIdx.x / 6;
    const bool xt = type >= 4;
    const int jt = (type >> 1) & 1, ct = type & 1;
    const int tb0 = split * blocks_per_split;
    const int tb1 = min(n_tok_blocks, tb0 + blocks_per_split);
    const int nblk = max(0, tb1 - tb0);

    if (tid == 0) {
        for (int s = 0; s < WT_NS; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(&done_bar, 1);
        mbar_fence_init();
    }
    if (warp == 5) tmem_alloc(&tmem_base_s, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;

    if (warp == 4) {
        if (lane == 0) {
            for (int i = 0; i < nblk; ++i) {
                const int s = i % WT_NS;
                mbar_wait(&empty[s], ((i / WT_NS) & 1) ^ 1);
                mbar_expect_tx(&full[s], xt ? 9 * 8192 : 8 * 8192);
                unsigned char* st = smem + s * WT_STAGE;
                const size_t tb = (size_t)(tb0 + i);
                if (!xt) {
                    bulk_g2s(st, hpimg + ((tb * 4 + 2 * jt) << 13), 2 * 8192, &full[s]);            // j groups 2jt, 2jt+1
                    bulk_g2s(st + 2 * 8192, dgimg + ((tb * 16 + 6 * ct) << 13), 6 * 8192, &full[s]);  // c groups 6ct .. 6ct+5
                } else {
                    bulk_g2s(st, ximg + (tb << 13), 8192, &full[s]);                                  // the x group
                    bulk_g2s(st + 8192, dgimg + ((tb * 16 + 8 * ct) << 13), 7 * 8192, &full[s]);      // c groups 8ct .. 8ct+6
                    bulk_g2s(st + 8 * 8192, dgimg + ((tb * 16 + 8 * ct + 7) << 13), 8192, &full[s]);  // c group 8ct+7
                }
            }
        }
    } else if (warp == 5) {
        {   // all lanes wait, one elected lane issues (tc.cuh::elect_one)
            constexpr uint32_t idesc = tc_idesc_mn(128, 192, 0), idesc_x = tc_idesc_mn(64, 256, 0);   // fp16; x tiles: M = 64 (one group, 8 rows used)
            for (int i = 0; i < nblk; ++i) {
                const int s = i % WT_NS;
                mbar_wait(&full[s], (i / WT_NS) & 1);
                tc_fence_after();
                const uint32_t a0 = smem_u32(smem + s * WT_STAGE);
                if (elect_one()) {
                if (!xt) {
                    const uint32_t b0 = a0 + 2 * 8192;
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks) {
                        const uint64_t ad = tc_smem_desc_mn(a0 + ks * 2048, 8192);
                        tc_mma(tmem_base, ad, tc_smem_desc_mn(b0 + ks * 2048, 8192), idesc, (i | ks) != 0);
                        tc_mma(tmem_base + 192, ad, tc_smem_desc_mn(b0 + 3 * 8192 + ks * 2048, 8192), idesc, (i | ks) != 0);
                    }
                } else {
                    const uint32_t b0 = a0 + 8192;
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks) {
                        // M = 64: the single x group (halves the A fetch of these operand-fetch-bound MMAs)
                        const uint64_t ad = tc_smem_desc_mn(a0 + ks * 2048, 0);
                        tc_mma(tmem_base, ad, tc_smem_desc_mn(b0 + ks * 2048, 8192), idesc_x, (i | ks) != 0);
                        tc_mma(tmem_base + 256, ad, tc_smem_desc_mn(b0 + 4 * 8192 + ks * 2048, 8192), idesc_x, (i | ks) != 0);
                    }
                }
                tc_commit(&empty[s]);
                }
                __syncwarp();
            }
            if (elect_one()) tc_commit(&done_bar);
            __syncwarp();
        }
    } else {
        // epilogue: TMEM lane = j within the tile
        mbar_wait(&done_bar, 0);
        tc_fence_after();
        // the dG image is in units of the launch's cotangent scale S (tc.cuh): take it back out of the fp32 sums
        const float inv_s = cotmax ? 1.0f / cot_scale_from_max(*cotmax) : 1.0f;
        if (xt) {
            // rows 0..7 of the x tile: dWi (rows q < X), dbi (row 7) and dbhn (row 7 of the dhn columns).
            // Always accumulates: the head-gradient kernel has initialised this split's small-partial area.
            if (warp == 0) {
                float* out = small_partial + (size_t)split * SMT_TOTAL;
                auto dst_of = [&](int cc) {
                    if (ct == 0) return SMT_WI + lane * LPG_G + cc;                            // dar, daz columns
                    if (cc >= 256) return SMT_WI + lane * LPG_G + 512 + (cc - 256);           // dan columns
                    return lane == 7 ? SMT_BHN + cc : -1;                                     // sum of dhn
                };
                for (int c = 0; c < 512; c += 32) {          // 32 columns per round: loads first, then the stores
                    float v[4][8], o[4][8];
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        if (nblk > 0) tmem_ld8(tmem_base + c + 8 * i, v[i]);
                        else {
#pragma unroll
                            for (int e = 0; e < 8; ++e) v[i][e] = 0.f;
                        }
                    }
                    if (nblk > 0) tmem_ld_wait();
                    if (lane < 8) {
#pragma unroll
                        for (int i = 0; i < 4; ++i)
#pragma unroll
                            for (int e = 0; e < 8; ++e) { const int d = dst_of(c + 8 * i + e); o[i][e] = d >= 0 ? out[d] : 0.0f; }
#pragma unroll
                        for (int i = 0; i < 4; ++i)
#pragma unroll
                            for (int e = 0; e < 8; ++e) { const int d = dst_of(c + 8 * i + e); if (d >= 0) out[d] = fmaf(v[i][e], inv_s, o[i][e]); }
                    }
                }
            }
        } else {
        const int j = jt * 128 + warp * 32 + lane;
        float* out = partial + (size_t)split * LPG_H * LPG_G + (size_t)j * LPG_G + ct * 384;
        // 64 columns per round: the previous partials are fetched with 16 independent loads in flight
        // (one dependent load -> add -> store round trip per 8 columns would serialise 48 DRAM latencies)
        for (int c = 0; c < 384; c += 64) {
            float4 pre[16];
            float4* p = reinterpret_cast<float4*>(out + c);
            if (accumulate) {
#pragma unroll
                for (int i = 0; i < 16; ++i) pre[i] = p[i];
            } else {
#pragma unroll
                for (int i = 0; i < 16; ++i) pre[i] = make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                float v[8];
                if (nblk > 0) {
                    tmem_ld8(tmem_base + ((uint32_t)(warp * 32) << 16) + c + 8 * i, v);
                    tmem_ld_wait();
                } else {
#pragma unroll
                    for (int e = 0; e < 8; ++e) v[e] = 0.f;
                }
                p[2 * i] = make_float4(fmaf(v[0], inv_s, pre[2 * i].x), fmaf(v[1], inv_s, pre[2 * i].y), fmaf(v[2], inv_s, pre[2 * i].z), fmaf(v[3], inv_s, pre[2 * i].w));
                p[2 * i + 1] = make_float4(fmaf(v[4], inv_s, pre[2 * i + 1].x), fmaf(v[5], inv_s, pre[2 * i + 1].y), fmaf(v[6], inv_s, pre[2 * i + 1].z), fmaf(v[7], inv_s, pre[2 * i + 1].w));
            }
        }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 5) tmem_dealloc(tmem_base, 512);
}

// head gradients (dw_pi, dW_y, db_pi, db_y) + initialisation of the split's input-side area (TC path).
// A warp owns one 8-unit chunk of the RB32 layout: lane = row of a 32-row block, so every h16 access is a
// coalesced 512-byte line; each lane keeps 8 x 9 accumulators over all the row blocks of its split and the
// 32 rows are combined once at the end by a fixed shuffle tree (deterministic).
constexpr int HT_SPLITS = 148;
// Every lane only ever needs its own row's data, so each lane runs a private
// HT_DEPTH-deep cp.async ring (no barriers, no producer warp): 16 B of h16, 32 B of dl and 4 B of d_pi_hat
// per row block in flight HT_DEPTH blocks ahead.
constexpr int HT_DEPTH = 6;
constexpr int HT_SLOT = 64;                  // bytes per lane per stage: h16 [0,16) | dl [16,48) | d_pi_hat [48,52)
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async4(uint32_t dst, const void* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory");
}
__global__ void __launch_bounds__(256)
wgrad_heads_stream_kernel(const __half* __restrict__ h16, const float* __restrict__ d_pi_hat, const float* __restrict__ dl,
                          float* __restrict__ partial, const uint32_t* __restrict__ cotmax, int R, int L, int blocks_per_split,
                          int accumulate) {
    const float inv_s = cotmax ? 1.0f / cot_scale_from_max(*cotmax) : 1.0f;      // dl arrives in units of S, d_pi_hat does not
    extern __shared__ __align__(128) unsigned char hsm[];     // [HT_DEPTH][256 threads][HT_SLOT]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int chunk = blockIdx.x * 8 + warp;            // 0..31
    const int split = blockIdx.y;
    const int R32 = (R + 31) >> 5;
    const int nrb = L * R32;
    const int b0 = split * blocks_per_split, b1 = min(nrb, b0 + blocks_per_split);
    const uint32_t slot0 = smem_u32(hsm) + threadIdx.x * HT_SLOT;
    // producer-side cursor (block ib = (it, irb), ring stage istage); all counters advance incrementally:
    // divisions in this loop cost more than its 72 FMAs
    int ib = b0, it = b0 / R32, irb = b0 % R32, istage = 0;
    auto issue = [&]() {
        if (ib < b1) {
            const int row = irb * 32 + lane;
            if (row < R) {
                const size_t tok = (size_t)it * R + row;
                const uint32_t d = slot0 + istage * (256 * HT_SLOT);
                cp_async16(d, h16 + (((size_t)ib * 32 + chunk) << 8) + (lane << 3));
                cp_async16(d + 16, dl + tok * 8);
                cp_async16(d + 32, dl + tok * 8 + 4);
                cp_async4(d + 48, d_pi_hat + tok);
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        ++ib;
        if (++irb == R32) { irb = 0; ++it; }
        if (++istage == HT_DEPTH) istage = 0;
    };
    float acc[8][9], hb[9];
#pragma unroll
    for (int e = 0; e < 8; ++e)
#pragma unroll
        for (int i = 0; i < 9; ++i) acc[e][i] = 0.f;
#pragma unroll
    for (int i = 0; i < 9; ++i) hb[i] = 0.f;
#pragma unroll
    for (int i = 0; i < HT_DEPTH - 1; ++i) issue();
    int crb = b0 % R32, cstage = 0;
    for (int b = b0; b < b1; ++b) {
        issue();
        asm volatile("cp.async.wait_group %0;" ::"n"(HT_DEPTH - 1) : "memory");
        const int row = crb * 32 + lane;
        const unsigned char* st = hsm + cstage * (256 * HT_SLOT) + threadIdx.x * HT_SLOT;
        if (++crb == R32) crb = 0;
        if (++cstage == HT_DEPTH) cstage = 0;
        if (row >= R) continue;
        const uint4 raw = *reinterpret_cast<const uint4*>(st);
        const float4 d0 = *reinterpret_cast<const float4*>(st + 16), d1 = *reinterpret_cast<const float4*>(st + 32);
        const float dv[9] = {*reinterpret_cast<const float*>(st + 48), d0.x * inv_s, d0.y * inv_s, d0.z * inv_s, d0.w * inv_s,
                             d1.x * inv_s, d1.y * inv_s, d1.z * inv_s, d1.w * inv_s};
        const __half2* hh = reinterpret_cast<const __half2*>(&raw);
#pragma unroll
        for (int e2 = 0; e2 < 4; ++e2) {
            const float2 f = __half22float2(hh[e2]);
            const float y0 = fmax_nan(f.x, 0.0f), y1 = fmax_nan(f.y, 0.0f);       // relu that keeps NaN
#pragma unroll
            for (int i = 0; i < 9; ++i) { acc[2 * e2][i] = fmaf(y0, dv[i], acc[2 * e2][i]); acc[2 * e2 + 1][i] = fmaf(y1, dv[i], acc[2 * e2 + 1][i]); }
        }
        if (chunk == 0) {
#pragma unroll
            for (int i = 0; i < 9; ++i) hb[i] += dv[i];
        }
    }
    float* out = partial + (size_t)split * SMT_TOTAL;
    auto put = [&](int idx, float v) { out[idx] = accumulate ? out[idx] + v : v; };
    // butterfly sums leave the total in every lane; lane (j mod 32) owns value j, so the read-modify-writes
    // of a warp go out in parallel instead of 72 dependent round trips from lane 0
#pragma unroll
    for (int e = 0; e < 8; ++e)
#pragma unroll
        for (int i = 0; i < 9; ++i) {
            float v = acc[e][i];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (lane == ((e * 9 + i) & 31)) { if (i == 0) put(SMT_WPI + chunk * 8 + e, v); else put(SMT_WY + (chunk * 8 + e) * 8 + (i - 1), v); }
        }
    if (chunk == 0) {
#pragma unroll
        for (int i = 0; i < 9; ++i) {
            float v = hb[i];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (lane == 16 + i) put(SMT_BPI + i, v);
        }
    }
    if (!accumulate) {                    // the x-tile CTAs of the GEMM kernel add into the input-side area
        for (int i = blockIdx.x * 256 + threadIdx.x; i < SMT_WPI; i += 4 * 256) out[i] = 0.0f;
    }
}

// ---- head gradients on the tensor cores (R % 32 == 0) ---------------------------------------------------
// dw_pi / dW_y = relu(h)^T [256 units x tokens] . [d pi_hat | dl] [tokens x 9]: a GEMM contracted over tokens.
// A 32-row block of the RB32 activation layout (16 KB contiguous) is, as it lies in memory, an MN-major
// no-swizzle tcgen05 operand (k = rows).  Per block: TMA bulk copy -> four warps apply relu in place (fp16) and
// build the B operand from the fp32 cotangents, scaled by the launch's S (tc.cuh), as an fp16 hi + lo pair (N = 32:
// columns 0..15 hi, 16..31 lo, so the cotangents keep ~22 mantissa bits) -> 4 MMAs (M128 N32 K16).
constexpr int HM_NS = 4;
constexpr int HM_A = 16384, HM_RAW = 1024 + 128, HM_B = 2048;
constexpr int HM_STAGE = HM_A + HM_RAW + HM_B;            // 19584 B (multiple of 128)
constexpr int HM_THREADS = 192;
__global__ void __launch_bounds__(HM_THREADS, 1)
wgrad_heads_mma_kernel(const __half* __restrict__ h16, const float* __restrict__ d_pi_hat, const float* __restrict__ dl,
                       float* __restrict__ partial, uint32_t* __restrict__ cotmax, int R, int L, int blocks_per_split,
                       int accumulate) {
    extern __shared__ __align__(1024) unsigned char hm_raw[];
    unsigned char* smem = hm_raw + ((128u - (smem_u32(hm_raw) & 127u)) & 127u);
    __shared__ __align__(8) uint64_t full[HM_NS], ready[HM_NS], empty[HM_NS], done_bar;
    __shared__ uint32_t tmem_base_s;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int split = blockIdx.x;
    const int R32 = R >> 5;
    const int nrb = L * R32;
    const int b0 = split * blocks_per_split, b1 = min(nrb, b0 + blocks_per_split);
    const int nblk = max(0, b1 - b0);
    if (tid == 0) {
        for (int s = 0; s < HM_NS; ++s) { mbar_init(&full[s], 1); mbar_init(&ready[s], 4); mbar_init(&empty[s], 1); }
        mbar_init(&done_bar, 1);
        mbar_fence_init();
    }
    if (warp == 5) tmem_alloc(&tmem_base_s, 64);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;

    if (warp == 4) {
        if (lane == 0) {
            int t = b0 / R32, rb = b0 % R32;
            for (int i = 0; i < nblk; ++i) {
                const int s = i % HM_NS;
                mbar_wait(&empty[s], ((i / HM_NS) & 1) ^ 1);
                unsigned char* st = smem + s * HM_STAGE;
                const size_t tok0 = (size_t)t * R + (size_t)rb * 32;
                mbar_expect_tx(&full[s], HM_A + HM_RAW);
                bulk_g2s(st, h16 + ((size_t)(b0 + i) << 13), HM_A, &full[s]);
                bulk_g2s(st + HM_A, dl + tok0 * 8, 1024, &full[s]);
                bulk_g2s(st + HM_A + 1024, d_pi_hat + tok0, 128, &full[s]);
                if (++rb == R32) { rb = 0; ++t; }
            }
        }
    } else if (warp == 5) {
        {
            // (kind::f16 needs A and B in the same 16-bit format on this part: fp16 x bf16 traps; both are fp16 here)
            constexpr uint32_t idesc = tc_idesc_mn(128, 32, 0);
            for (int i = 0; i < nblk; ++i) {
                const int s = i % HM_NS;
                mbar_wait(&ready[s], (i / HM_NS) & 1);
                tc_fence_after();
                const uint32_t a0 = smem_u32(smem + s * HM_STAGE), bb = a0 + HM_A + HM_RAW;
                if (elect_one()) {
#pragma unroll
                for (int ks = 0; ks < 2; ++ks) {
                    const uint64_t bd = tc_smem_desc_mn_plain(bb + ks * 256, 128, 512);
#pragma unroll
                    for (int mh = 0; mh < 2; ++mh)
                        tc_mma(tmem_base + mh * 32, tc_smem_desc_mn_plain(a0 + mh * 8192 + ks * 256, 128, 512), bd, idesc,
                               (i | ks) != 0);
                }
                tc_commit(&empty[s]);
                }
                __syncwarp();
            }
            if (elect_one()) tc_commit(&done_bar);
            __syncwarp();
        }
    } else {
        // ---- transform warps (0..3), later the epilogue ----
        float hb[9];
#pragma unroll
        for (int i = 0; i < 9; ++i) hb[i] = 0.f;
        const float S = cotmax ? cot_scale_from_max(*cotmax) : 1.0f, inv_s = 1.0f / S;
        bool range_bad = false;                   // an operand was clamped to fp16's range or is not finite (cotmax[1])
        for (int i = 0; i < nblk; ++i) {
            const int s = i % HM_NS;
            mbar_wait(&full[s], (i / HM_NS) & 1);
            unsigned char* st = smem + s * HM_STAGE;
            // relu in place (fp16): 1024 16-byte groups, 8 per thread (consecutive threads, consecutive groups)
            const __half2 z2 = __float2half2_rn(0.0f);
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                uint4* pp = reinterpret_cast<uint4*>(st) + q * 128 + tid;
                uint4 raw = *pp;
                __half2* hh = reinterpret_cast<__half2*>(&raw);
#pragma unroll
                for (int e = 0; e < 4; ++e) hh[e] = __hmax2_nan(hh[e], z2);
                *pp = raw;
            }
            if (warp == 0) {
                // B operand for row `lane`: [n-group g][k = row][8] bf16; groups 0,1 = hi of (d pi_hat, dl[0..7], 0..),
                // groups 2,3 = lo
                const float4 d0 = *reinterpret_cast<const float4*>(st + HM_A + lane * 32), d1 = *reinterpret_cast<const float4*>(st + HM_A + lane * 32 + 16);
                // in units of S: d_pi_hat is scaled here, dl was written scaled by the BPTT kernel
                const float dv[9] = {S * *reinterpret_cast<const float*>(st + HM_A + 1024 + lane * 4), d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
                float hi[9], lo[9];
#pragma unroll
                for (int j = 0; j < 9; ++j) {
                    // (a NaN passes the clamp instead of becoming -65504)
                    range_bad |= !(fabsf(dv[j]) <= 65504.0f);
                    hi[j] = __half2float(__float2half_rn(fmin_nan(fmax_nan(dv[j], -65504.0f), 65504.0f)));
                    lo[j] = dv[j] - hi[j];
                    hb[j] += dv[j];
                }
                auto pk = [](float a, float b) { return pack_h2_sat(a, b); };
                unsigned char* bp = st + HM_A + HM_RAW + lane * 16;
                *reinterpret_cast<uint4*>(bp) = make_uint4(pk(hi[0], hi[1]), pk(hi[2], hi[3]), pk(hi[4], hi[5]), pk(hi[6], hi[7]));
                *reinterpret_cast<uint4*>(bp + 512) = make_uint4(pk(hi[8], 0.f), 0u, 0u, 0u);
                *reinterpret_cast<uint4*>(bp + 1024) = make_uint4(pk(lo[0], lo[1]), pk(lo[2], lo[3]), pk(lo[4], lo[5]), pk(lo[6], lo[7]));
                *reinterpret_cast<uint4*>(bp + 1536) = make_uint4(pk(lo[8], 0.f), 0u, 0u, 0u);
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(&ready[s]);
        }
        if (warp == 0 && __any_sync(0xffffffffu, range_bad) && lane == 0 && cotmax) atomicOr(cotmax + 1, TOUED_STATUS_FP16_RANGE);
        // ---- epilogue: TMEM lane = unit within the 128-unit half ----
        mbar_wait(&done_bar, 0);
        tc_fence_after();
        float* out = partial + (size_t)split * SMT_TOTAL;
#pragma unroll
        for (int mh = 0; mh < 2; ++mh) {
            const int u = mh * 128 + warp * 32 + lane;
            float v[4][8];
            if (nblk > 0) {
#pragma unroll
                for (int q = 0; q < 4; ++q) tmem_ld8(tmem_base + ((uint32_t)(warp * 32) << 16) + mh * 32 + 8 * q, v[q]);
                tmem_ld_wait();
            } else {
#pragma unroll
                for (int q = 0; q < 4; ++q)
#pragma unroll
                    for (int e = 0; e < 8; ++e) v[q][e] = 0.f;
            }
            float g[9];
#pragma unroll
            for (int j = 0; j < 8; ++j) g[j] = v[0][j] + v[2][j];
            g[8] = v[1][0] + v[3][0];
            // (SMT_TOTAL is odd: no vector accesses into a split's area)
            float* wy = out + SMT_WY + u * 8;
            float prev[9];
#pragma unroll
            for (int j = 0; j < 9; ++j) prev[j] = 0.f;
            if (accumulate) {
                prev[0] = out[SMT_WPI + u];
#pragma unroll
                for (int j = 0; j < 8; ++j) prev[1 + j] = wy[j];
            }
            out[SMT_WPI + u] = fmaf(g[0], inv_s, prev[0]);
#pragma unroll
            for (int j = 0; j < 8; ++j) wy[j] = fmaf(g[1 + j], inv_s, prev[1 + j]);
        }
        if (warp == 0) {
#pragma unroll
            for (int i = 0; i < 9; ++i) {
                float v = hb[i];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
                v *= inv_s;
                if (lane == i) out[SMT_BPI + i] = accumulate ? out[SMT_BPI + i] + v : v;
            }
        }
        if (!accumulate) {                // the x-tile CTAs of the GEMM kernel add into the input-side area
            for (int i = tid; i < SMT_WPI; i += 128) out[i] = 0.0f;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 5) tmem_dealloc(tmem_base, 64);
}

constexpr int WT_SPLITS = 24;              // 6 tile types x 24 = 144 CTAs
static_assert(WT_SPLITS <= 37 && HT_SPLITS <= 592, "partial areas of toued_lpg_wgrad_workspace_floats (lpg_backward.cu) are sized for 37 / 592 splits");
extern "C" int toued_wgrad_tc_splits(void) { return WT_SPLITS; }
extern "C" int toued_wgrad_tc_small_splits(void) { return HT_SPLITS; }

extern "C" int toued_lpg_wgrad_tc(const void* hpimg, const void* dgimg, const void* ximg, const void* h16,
                                  const float* d_pi_hat, const float* dl, float* wh_partials, float* small_partials,
                                  uint32_t* cotangent_max, int n_agents, int n_workers, int rollout_len, int accumulate,
                                  void* stream) {
    const int R = n_agents * n_workers, L = rollout_len;
    TOUED_CHECK(R > 0 && L > 0, "toued_lpg_wgrad_tc: empty problem");
    cudaStream_t st = (cudaStream_t)stream;
    const int Rp = (R + 63) / 64 * 64;
    const int n_tb = L * Rp / 64;
    const int bps = (n_tb + WT_SPLITS - 1) / WT_SPLITS;
    // head gradients first: also zero-initialises the input-side area the GEMM's x tiles accumulate into
    const int nrb = L * ((R + 31) / 32);
    const int rbps = (nrb + HT_SPLITS - 1) / HT_SPLITS;
    if (R % 32 == 0) {
        constexpr int msmem = HM_NS * HM_STAGE + 128;
        TOUED_CUDA(cudaFuncSetAttribute(wgrad_heads_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, msmem));
        wgrad_heads_mma_kernel<<<HT_SPLITS, HM_THREADS, msmem, st>>>((const __half*)h16, d_pi_hat, dl, small_partials,
                                                                    cotangent_max, R, L, rbps, accumulate);
    } else {
        constexpr int hsmem = HT_DEPTH * 256 * HT_SLOT;
        TOUED_CUDA(cudaFuncSetAttribute(wgrad_heads_stream_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, hsmem));
        wgrad_heads_stream_kernel<<<dim3(4, HT_SPLITS), 256, hsmem, st>>>((const __half*)h16, d_pi_hat, dl, small_partials,
                                                                         cotangent_max, R, L, rbps, accumulate);
    }
    TOUED_LAUNCH_CHECK();
    const size_t smem = WT_NS * WT_STAGE + 1024;
    TOUED_CUDA(cudaFuncSetAttribute(wgrad_wh_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    wgrad_wh_tc_kernel<<<6 * WT_SPLITS, WT_THREADS, smem, st>>>((const unsigned char*)hpimg, (const unsigned char*)dgimg,
                                                                (const unsigned char*)ximg, wh_partials, small_partials,
                                                                cotangent_max, n_tb, bps, accumulate);
    TOUED_LAUNCH_CHECK();
    return 0;
}
