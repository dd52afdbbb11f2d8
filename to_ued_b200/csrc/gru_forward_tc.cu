// Tensor-core GRU forward (tcgen05 / TMEM / TMA), the production path for models/lpg.py:11-30,77-84.
//
// A CTA owns 128 sequences (UMMA_M = 128, cta_group::1) for all L reverse-scan steps; 19 warps, warp-specialised.
//   * Hidden state: lives in TENSOR MEMORY as fp16 pairs (2 x 128 columns, ping-pong over the steps) and is the
//     TMEM-resident A operand of the recurrent MMAs (tcgen05.mma with [a_tmem]).  It never touches shared memory: a
//     64 KB smem A tile re-read by each of the 16 passes of a step was the bound of the first version (the tensor core
//     fetches shared-memory operands at ~64 B/clk).
//   * Recurrent matrix: pre-packed once per meta-step into 16 fp16 "pass" images of 26 KB (pass p = hidden units
//     [16p, 16p+16) x gates (r, z, n): [48 rows][256 k] as four SW128 K-blocks, plus a 2 KB no-swizzle K = 16 block
//     holding W_i and b_i of those units as an fp16 hi / lo pair).  A TMA-producer warp streams the 16 images per step
//     from L2 with cp.async.bulk into a ring of FT_NS = 6 stages (mbarrier full / empty pairs).  (The images are NOT
//     resident: one CTA owns all 768 gate columns = 416 KB per step; VERDICT r01 "weak" #4 / DESIGN.md section 7.)
//   * MMA warp (all lanes wait on the barriers, one lane elected with elect.sync issues): per pass the input projection
//     x_t W_i + b_i first (A = the x tile [128 x 16] in smem, N = 64, initialises the accumulator columns
//     r | z | 0 | i_n -- i_n keeps its own columns because r gates only the hidden part of the candidate), then 16
//     recurrent MMAs M128 N48 K16 accumulating onto r | z | h_n; two accumulators (even / odd passes).
//   * Epilogue: two sets of 8 warps (set 0 = even passes / accumulator 0, set 1 = odd passes / accumulator 1; in a set
//     warp q + 4 hf owns TMEM lanes [32q, 32q + 32) and units [8 hf, 8 hf + 8) of the pass).  tcgen05.ld the
//     pre-activations and h', flax GRUCell gate math (ex2.approx / rcp.approx), tcgen05.st h_t into the other hidden
//     buffer, and save h16, the four gate planes (fp16, RB32 layout; the sign bits of the z plane carry relu'(h_t)) and the
//     fp16 token-tile image of the masked carry.
//   * Heads on the tensor cores: relu(h_t) of each pass goes to 8 TMEM columns (ring of 4 tiles) and is the A operand of
//     a K = 16 MMA against [w_pi | W_y] (fp16 hi / lo, N = 32); the per-step epilogue adds biases and does the softmax.
//   * The x tile of step s + 2 overwrites the tile step s used: it is written by SET 1 (whose last pass, 15, is the last
//     MMA reader of the tile), never by set 0 -- the round-1 write-after-read race (DESIGN.md section 6).
// fp16 operands / fp32 accumulate: the hidden state is quantised to fp16 once per step (|h| < 1).
// Parity is checked against the exact-fp32 SIMT kernel and the fp64 oracle with a stated tolerance.
#include "tc.cuh"
#include "lpg_common.cuh"
#include "../../include/toued.h"

constexpr int FT_M = 128;                 // rows per CTA
constexpr int FT_PU = 16;                 // hidden units per pass
constexpr int FT_PN = 3 * FT_PU;          // 48 accumulator columns per pass
constexpr int FT_NPASS = LPG_H / FT_PU;   // 16
constexpr int FT_KB = LPG_H / 64;         // 4 K-blocks
constexpr int FT_BH = FT_KB * FT_PN * 128;         // 24576 B: recurrent part of a pass image (SW128 K-blocks)
constexpr int FT_XN = 64;                          // x-part rows: Wi_r, Wi_z, 0, Wi_n (16 each) -> accumulator cols 0..63
constexpr int FT_BX = (FT_XN / 8) * 256;           // 2048 B: input part (no-swizzle K=16 block: x[0..7] incl. the bias 1)
constexpr int FT_BSTAGE = FT_BH + FT_BX;           // 26624 B per pass image (multiple of 1024)
constexpr int FT_AX = (FT_M / 8) * 256;            // 4096 B: x tile of the A operand
constexpr int FT_NS = 6;                  // B stages (7 measured: see DESIGN.md section 7.0)
constexpr int FT_THEADS = 128, FT_TTILE = 192, FT_THOLD = 256;   // tensor-memory columns: 2 x 64 gate accumulators at 0, 2 x 32 head
                                                                 // accumulators, 4 x 8 relu(h) tiles, 2 x 128 columns of hidden state
// The heads MMAs (one K = 16 MMA per pass on the relu(h) tile) are issued by a warp of their own, not by the gate-MMA warp:
// the gate-MMA warp is a serial resource (16 passes x ~200 uniform-datapath instructions and three barrier waits per step)
// and the epilogue warps spend 20 % of their time waiting for its MMAs.
constexpr int FT_THREADS = 608;           // 2 sets of 8 epilogue warps (even / odd passes) + producer warp + MMA warp + heads-MMA warp

// Wh[k][c] (fp32, c = g*256 + unit) -> fp16 pass images: image[p][kb][row = g*16 + u][128 B swizzled]
__global__ void pack_wh_fwd_kernel(const float* __restrict__ Wh, __half* __restrict__ img, size_t lpg_stride) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= LPG_H * LPG_G) return;
    Wh += (size_t)blockIdx.y * lpg_stride;                       // one parameter set per blockIdx.y
    img += (size_t)blockIdx.y * (FT_NPASS * FT_BSTAGE / 2);
    const int k = i / LPG_G, c = i % LPG_G;
    const int g = c / LPG_H, unit = c % LPG_H, p = unit / FT_PU, u = unit % FT_PU;
    char* base = reinterpret_cast<char*>(img) + (size_t)p * FT_BSTAGE;
    *reinterpret_cast<__half*>(base + sw128_offset(FT_PN, g * FT_PU + u, k)) = __float2half_rn(Wh[i]);
}

// input part of the pass images: rows [0,16) Wi_r, [16,32) Wi_z, [32,48) zero, [48,64) Wi_n of the pass's
// 16 units; k = input index (k < X: Wi[k], k == 7: bias b_i, else 0)
__global__ void pack_wi_fwd_kernel(const float* __restrict__ lpg, int X, __half* __restrict__ img, size_t lpg_stride) {
    const LpgOffsets o = lpg_offsets(X);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= FT_NPASS * FT_XN * 16) return;
    lpg += (size_t)blockIdx.y * lpg_stride;
    img += (size_t)blockIdx.y * (FT_NPASS * FT_BSTAGE / 2);
    const int k = i & 15, row = (i >> 4) % FT_XN, p = i / (16 * FT_XN);
    const int blk = row >> 4, u = p * FT_PU + (row & 15);
    // k in [8,16) holds the fp16 residual of slot k-8 (the x tile repeats x there): raw step / lifetime
    // inputs reach a few hundred, so W_i is carried to ~22 bits
    float v = 0.0f;
    if (blk != 2) {
        const int g = blk == 3 ? 2 : blk, kk = k & 7;
        if (kk < X) v = lpg[o.Wi + kk * LPG_G + g * LPG_H + u];
        else if (kk == 7) v = lpg[o.bi + g * LPG_H + u];
        if (k >= 8) v -= __half2float(__float2half_rn(v));
    }
    char* base = reinterpret_cast<char*>(img) + (size_t)p * FT_BSTAGE + FT_BH;
    *reinterpret_cast<__half*>(base + k16_offset(row, k)) = __float2half_rn(v);
}

static int pack_wh_forward(const float* lpg_params, void* wh_img, int lifetime_conditioning, int n_sets, size_t lpg_stride,
                           void* stream) {
    const int X = lifetime_conditioning ? 7 : 5;
    pack_wh_fwd_kernel<<<dim3((LPG_H * LPG_G + 255) / 256, n_sets), 256, 0, (cudaStream_t)stream>>>(
        lpg_params + lpg_offsets(X).Wh, (__half*)wh_img, lpg_stride);
    TOUED_LAUNCH_CHECK();
    pack_wi_fwd_kernel<<<dim3((FT_NPASS * FT_XN * 16 + 255) / 256, n_sets), 256, 0, (cudaStream_t)stream>>>(
        lpg_params, X, (__half*)wh_img, lpg_stride);
    TOUED_LAUNCH_CHECK();
    return 0;
}

extern "C" int toued_pack_wh_forward(const float* lpg_params, void* wh_img, int lifetime_conditioning, void* stream) {
    return pack_wh_forward(lpg_params, wh_img, lifetime_conditioning, 1, 0, stream);
}

extern "C" int toued_pack_wh_forward_multi(const float* lpg_params, void* wh_img, int lifetime_conditioning, int n_sets,
                                           int lpg_stride, void* stream) {
    TOUED_CHECK(n_sets > 0 && lpg_stride > 0, "toued_pack_wh_forward_multi: bad arguments");
    return pack_wh_forward(lpg_params, wh_img, lifetime_conditioning, n_sets, (size_t)lpg_stride, stream);
}

template <int X>
__global__ void __launch_bounds__(FT_THREADS, 1)
gru_forward_tc_kernel(const float* __restrict__ x, const uint8_t* __restrict__ done,
                      const float* __restrict__ lpg, const __half* __restrict__ wh_img,
                      __half* __restrict__ h16, __half* __restrict__ fac, unsigned char* __restrict__ hpimg,
                      float* __restrict__ pi_hat, float* __restrict__ y_hat, int R, int L, int W,
                      int rows_per_cta, size_t lpg_stride) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    // (offset arithmetic on the __shared__ array, not an integer round trip: the compiler keeps the shared
    //  address space and emits LDS / STS instead of generic LD / ST)
    unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    unsigned char* sAx = smem;                                  // 2 x 4 KB    x tile (no-swizzle K = 16 block)
    unsigned char* sB = sAx + 2 * FT_AX;                        // FT_NS x 26 KB
    unsigned char* sHB = sB + FT_NS * FT_BSTAGE;                // 16 x 1 KB   head weights [w_pi | W_y] as fp16 hi / lo, per pass
    float* sbhn = reinterpret_cast<float*>(sHB + FT_NPASS * 1024);    // [256]
    __shared__ __align__(8) uint64_t b_full[FT_NS], b_empty[FT_NS], acc_full[2], acc_empty[2], a_ready;
    __shared__ __align__(8) uint64_t stage_full[4], stage_empty[4], heads_full[2], h0_ready;
    __shared__ uint32_t tmem_base_s;

    const LpgOffsets o = lpg_offsets(X);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // rows_per_cta = 128: shared parameters, dense 128-row tiles.  rows_per_cta = W (<= 128) with lpg_stride != 0: one
    // agent and one parameter set (own pass images) per CTA -- the per-candidate forward of the ES path.
    const int row0 = blockIdx.x * rows_per_cta;
    lpg += (size_t)blockIdx.x * lpg_stride;
    if (lpg_stride) wh_img += (size_t)blockIdx.x * (FT_NPASS * FT_BSTAGE / 2);

    if (tid == 0) {
        for (int s = 0; s < FT_NS; ++s) { mbar_init(&b_full[s], 1); mbar_init(&b_empty[s], 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(&acc_full[a], 1); mbar_init(&acc_empty[a], 8); }
        mbar_init(&a_ready, 16);
        for (int a = 0; a < 4; ++a) { mbar_init(&stage_full[a], 8); mbar_init(&stage_empty[a], 1); }
        for (int a = 0; a < 2; ++a) mbar_init(&heads_full[a], 1);
        mbar_init(&h0_ready, 1);
        mbar_fence_init();
    }
    if (warp == 17) tmem_alloc(&tmem_base_s, 512);     // column map: FT_THEADS / FT_TTILE / FT_THOLD above

    for (int i = tid; i < LPG_H; i += FT_THREADS) sbhn[i] = lpg[o.bhn + i];
    // head weights as the B operand of the heads MMA: per pass a [32 n][16 k] no-swizzle block; n < 16: fp16 of
    // (w_pi, W_y[.,0..7], 0..), n >= 16: the fp16 residual, so the heads keep ~22 weight bits
    for (int i = tid; i < FT_NPASS * 32 * 16; i += FT_THREADS) {
        const int p = i >> 9, n = (i >> 4) & 31, k = i & 15, u = p * FT_PU + k, nn = n & 15;
        const float w = nn == 0 ? lpg[o.w_pi + u] : (nn < 1 + LPG_Y ? lpg[o.W_y + u * LPG_Y + nn - 1] : 0.0f);
        const float hi = __half2float(__float2half_rn(w));
        *reinterpret_cast<__half*>(sHB + p * 1024 + k16_offset(n, k)) = __float2half_rn(n < 16 ? hi : w - hi);
    }
    // initial carry = 0 (both A buffers); x tiles zero, then x_{L-1} into tile 0 (twice: W_i hi / lo parts)
    for (int i = tid; i < (2 * FT_AX) / 16; i += FT_THREADS) reinterpret_cast<uint4*>(sAx)[i] = make_uint4(0u, 0u, 0u, 0u);
    __syncthreads();
    if (tid < FT_M) {
        const int r_ = row0 + tid;
        if (tid < rows_per_cta && r_ < R) {
            const float4* xp = reinterpret_cast<const float4*>(x + ((size_t)(L - 1) * R + r_) * LPG_XP);
            const float4 x0 = xp[0], x1 = xp[1];
            __half2 h0 = __floats2half2_rn(x0.x, x0.y), h1 = __floats2half2_rn(x0.z, x0.w);
            __half2 h2 = __floats2half2_rn(x1.x, x1.y), h3 = __floats2half2_rn(x1.z, x1.w);
            uint4 pk;
            pk.x = *reinterpret_cast<uint32_t*>(&h0); pk.y = *reinterpret_cast<uint32_t*>(&h1);
            pk.z = *reinterpret_cast<uint32_t*>(&h2); pk.w = *reinterpret_cast<uint32_t*>(&h3);
            *reinterpret_cast<uint4*>(sAx + k16_offset(tid, 0)) = pk;
            *reinterpret_cast<uint4*>(sAx + k16_offset(tid, 8)) = pk;
        }
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;

    if (warp == 16) {
        // ===================== TMA producer: stream the 16 pass images per step =====================
        if (lane == 0) {
            uint32_t it = 0;
            for (int t = L - 1; t >= 0; --t) {
                for (int p = 0; p < FT_NPASS; ++p, ++it) {
                    const int s = it % FT_NS;
                    mbar_wait(&b_empty[s], ((it / FT_NS) & 1) ^ 1);
                    mbar_expect_tx(&b_full[s], FT_BSTAGE);
                    bulk_g2s(sB + s * FT_BSTAGE, reinterpret_cast<const char*>(wh_img) + (size_t)p * FT_BSTAGE,
                             FT_BSTAGE, &b_full[s]);
                }
            }
        }
    } else if (warp == 17) {
        // ===================== MMA issuer ==========================================================
        // The whole warp walks the loop (all lanes wait on the barriers); one elected lane issues.
        {
            constexpr uint32_t idesc = tc_idesc(FT_M, FT_PN, 0), idesc_x = tc_idesc(FT_M, FT_XN, 0);
            uint32_t it = 0;
            int cur = 0;
            for (int t = L - 1, step = 0; t >= 0; --t, ++step) {
                if (step > 0) { mbar_wait(&a_ready, (step - 1) & 1); } else { mbar_wait(&h0_ready, 0); }
                tc_fence_after();
                const uint64_t axd = tc_smem_desc_k16(smem_u32(sAx + cur * FT_AX));
                for (int p = 0; p < FT_NPASS; ++p, ++it) {
                    const int s = it % FT_NS, a = it & 1;
                    mbar_wait(&acc_empty[a], ((it >> 1) & 1) ^ 1);
                    mbar_wait(&b_full[s], (it / FT_NS) & 1);
                    tc_fence_after();
                    if (elect_one()) {
                        const uint32_t b_addr = smem_u32(sB + s * FT_BSTAGE);
                        const uint32_t d_addr = tmem_base + a * 64;
                        // input projection + bias first: initialises all 64 accumulator columns
                        // (r | z | 0 | i_n); the recurrent part then accumulates onto columns 0..47 (r | z | h_n)
                        tc_mma(d_addr, axd, tc_smem_desc_k16(b_addr + FT_BH), idesc_x, 0u);
                        const uint64_t bd0 = tc_smem_desc(b_addr);
                        const uint32_t ha = tmem_base + FT_THOLD + cur * 128;     // h' of this step: 8 columns per K = 16 step
#pragma unroll
                        for (int kb = 0; kb < FT_KB; ++kb) {
#pragma unroll
                            for (int ks = 0; ks < 4; ++ks)      // descriptor address field is in 16-byte units
                                tc_mma_ts(d_addr, ha + (kb * 4 + ks) * 8,
                                          bd0 + (uint64_t)((kb * FT_PN * 128 + ks * 32) >> 4), idesc, 1u);
                        }
                        tc_commit(&b_empty[s]);
                        tc_commit(&acc_full[a]);
                    }
                    __syncwarp();
                }
                cur ^= 1;
            }
        }
    } else if (warp == 18) {
        // ===================== heads-MMA issuer: follows the relu(h) tiles as the epilogue warps publish them.  Ordering with
        // the readout of the head accumulators two steps earlier is transitive: readout(s) precedes that warp's passes of step
        // s + 1, hence a_ready(s + 1), hence the gate MMAs and relu tiles of step s + 2 this warp waits for.
        // Per pass q: (pi_hat, y logits) += relu(h_t)[:, 16 units of pass q] . W_heads[16 units][32]; the A tile is read from
        // tensor memory (written by the epilogue warps with tcgen05.st: no shared-memory staging, no proxy fence).
        constexpr uint32_t idesc_h = tc_idesc(FT_M, 32, 0);
        const uint32_t hb_addr = smem_u32(sHB);
        const uint32_t nq = (uint32_t)L * FT_NPASS;
        for (uint32_t q = 0; q < nq; ++q) {
            const uint32_t sb = q & 3, p = q & 15, stp = q >> 4;
            mbar_wait(&stage_full[sb], (q >> 2) & 1);
            tc_fence_after();
            if (elect_one()) {
                tc_mma_ts(tmem_base + FT_THEADS + (stp & 1) * 32, tmem_base + FT_TTILE + sb * 8, tc_smem_desc_k16(hb_addr + p * 1024),
                          idesc_h, p != 0);
                tc_commit(&stage_empty[sb]);
                if (p == 15) tc_commit(&heads_full[stp & 1]);
            }
            __syncwarp();
        }
    } else {
        // ===================== epilogue warps: set 0 (warps 0..7) takes the even passes / accumulator 0,
        // set 1 (warps 8..15) the odd passes / accumulator 1.  A pass is one long dependent chain per warp
        // (LDTM -> gates -> pack -> stores); two sets in flight give every scheduler four warps to interleave.
        const int set = warp >> 3, q = warp & 3, hf = (warp >> 2) & 1;
        const int rl = q * 32 + lane;                 // row within the tile == TMEM lane
        const int row = row0 + rl;
        const bool rv = rl < rows_per_cta && row < R;
        const int rsafe = rv ? row : 0;
        const int n_ag = rsafe / W, w_ag = rsafe % W;
        const size_t R32 = ((size_t)R + 31) >> 5;             // 32-row blocks of the RB32 layout
        const size_t Rp = ((size_t)R + 63) & ~(size_t)63;     // rows padded to the 64-token image blocks
        int cur = 0;
        // initial carry = 0: hidden-state buffer 0 (this thread's columns)
#pragma unroll
        for (int pp = 0; pp < FT_NPASS / 2; ++pp)
            tmem_st4(tmem_base + ((uint32_t)(q * 32) << 16) + FT_THOLD + (2 * pp + set) * 8 + hf * 4, make_uint4(0u, 0u, 0u, 0u));
        tmem_st_wait();
        tc_fence_before();
        asm volatile("bar.sync 1, 512;" ::: "memory");
        if (warp == 0 && lane == 0) mbar_arrive(&h0_ready);
        float b_heads[1 + LPG_Y];
        b_heads[0] = lpg[o.b_pi];
#pragma unroll
        for (int c = 0; c < LPG_Y; ++c) b_heads[1 + c] = lpg[o.b_y + c];
        for (int t = L - 1, step = 0; t >= 0; --t, ++step) {
            // x_{t-1} (the next processed step) goes into the other x tile as fp16 (one thread per row).  That tile was
            // the A operand of the input-projection MMAs of the PREVIOUS step, the last of which (pass 15) belongs to
            // set 1: only a set-1 warp has observed acc_full of that pass, i.e. knows that every MMA reading the tile
            // has completed.  (Round 1 wrote it from set 0, whose last pass is 14: when set 1 lagged by one pass the
            // MMA of pass 15 read x of the wrong time step for 16 units -- the source of the run-to-run differences
            // of the BASELINE-size step.)
            if (set == 1 && hf == 0 && t > 0) {
                uint4 pk = make_uint4(0u, 0u, 0u, 0u);
                if (rv) {
                    const float4* xp = reinterpret_cast<const float4*>(x + ((size_t)(t - 1) * R + row) * LPG_XP);
                    const float4 x0 = xp[0], x1 = xp[1];
                    __half2 h0 = __floats2half2_rn(x0.x, x0.y), h1 = __floats2half2_rn(x0.z, x0.w);
                    __half2 h2 = __floats2half2_rn(x1.x, x1.y), h3 = __floats2half2_rn(x1.z, x1.w);
                    pk.x = *reinterpret_cast<uint32_t*>(&h0); pk.y = *reinterpret_cast<uint32_t*>(&h1);
                    pk.z = *reinterpret_cast<uint32_t*>(&h2); pk.w = *reinterpret_cast<uint32_t*>(&h3);
                }
                *reinterpret_cast<uint4*>(sAx + (cur ^ 1) * FT_AX + k16_offset(rl, 0)) = pk;
                *reinterpret_cast<uint4*>(sAx + (cur ^ 1) * FT_AX + k16_offset(rl, 8)) = pk;
            }
            // mask for the NEXT processed step (t-1): its carry is zero where done[t-1]
            const bool zero_next = (t > 0) && done[((size_t)n_ag * L + (t - 1)) * W + w_ag];
            // per-step output pointers (64-bit address arithmetic once per step; the passes add 32-bit offsets)
            __half* const h16_t = h16 + rb32_index((size_t)t, R32, rsafe, 0);
            __half* const fac_t = fac ? fac + fac_index((size_t)t, R32, rsafe, 0, 0) : nullptr;
            const size_t hp_tok = (size_t)(t > 0 ? t - 1 : 0) * Rp + row;              // token of the masked carry h' consumed at step t-1
            unsigned char* const hp_t = hpimg ? hpimg + (((hp_tok >> 6) * 4) << 13) + (hp_tok & 63) * 128 : nullptr;
            const uint32_t hp_r7 = (uint32_t)(hp_tok & 7);
            for (int p = set; p < FT_NPASS; p += 2) {
                const uint32_t it = (uint32_t)step * FT_NPASS + p;
                const int a = set;
                mbar_wait(&acc_full[a], (it >> 1) & 1);
                tc_fence_after();
                float ar[8], az[8], an[8], ai[8];
                const uint32_t ta = tmem_base + ((uint32_t)(q * 32) << 16) + a * 64 + hf * 8;
                tmem_ld8(ta, ar);
                tmem_ld8(ta + FT_PU, az);
                tmem_ld8(ta + 2 * FT_PU, an);
                tmem_ld8(ta + 3 * FT_PU, ai);
                const uint4 hp_tm = tmem_ld4(tmem_base + ((uint32_t)(q * 32) << 16) + FT_THOLD + cur * 128 + p * 8 + hf * 4);   // h' of these units
                tmem_ld_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&acc_empty[a]);
                const int u0 = p * FT_PU + hf * 8;              // first of this thread's 8 units
                const uint4 hp_raw = hp_tm;
                const __half2* hp2 = reinterpret_cast<const __half2*>(&hp_raw);
                float hp[8];
#pragma unroll
                for (int e = 0; e < 4; ++e) { const float2 f = __half22float2(hp2[e]); hp[2 * e] = f.x; hp[2 * e + 1] = f.y; }
                float hv[8], rr[8], zz[8], nn[8], hn[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    const int u = u0 + e;
                    // The epilogue is bound by the MUFU pipe (16 results / clk / SM; 6 MUFU operations per unit with three
                    // ex2 + rcp activations).  The two sigmoids share ONE reciprocal: inv = 1/(a b), r = b inv, z = a inv
                    // (exponents clamped at 60 so that the product stays finite; sigmoid is 0 to fp32 there anyway; the clamp
                    // keeps a NaN pre-activation NaN).
                    const float ea = ex2_approx(fmin_nan(-1.4426950408889634f * ar[e], 60.0f));
                    const float eb = ex2_approx(fmin_nan(-1.4426950408889634f * az[e], 60.0f));
                    const float da = 1.0f + ea, db = 1.0f + eb;
                    const float inv = rcp_approx(da * db);
                    rr[e] = inv * db;                                     // input projection + bias already inside
                    zz[e] = inv * da;
                    hn[e] = an[e] + sbhn[u];
                    nn[e] = tanh_fast(ai[e] + rr[e] * hn[e]);
                    hv[e] = (1.0f - zz[e]) * nn[e] + zz[e] * hp[e];
                }
                auto pack8 = [](const float (&v)[8]) {
                    uint4 r;
                    __half2 h0 = __floats2half2_rn(v[0], v[1]), h1 = __floats2half2_rn(v[2], v[3]);
                    __half2 h2 = __floats2half2_rn(v[4], v[5]), h3 = __floats2half2_rn(v[6], v[7]);
                    r.x = *reinterpret_cast<uint32_t*>(&h0); r.y = *reinterpret_cast<uint32_t*>(&h1);
                    r.z = *reinterpret_cast<uint32_t*>(&h2); r.w = *reinterpret_cast<uint32_t*>(&h3);
                    return r;
                };
                const uint4 hpk = pack8(hv);
                {   // relu(h_t) of this pass -> K = 16 tile (8 TMEM columns) for the heads MMA
                    const uint32_t sb = it & 3;
                    mbar_wait(&stage_empty[sb], ((it >> 2) & 1) ^ 1);
                    // the (masked) next carry goes into the other hidden-state buffer of tensor memory
                    tmem_st4(tmem_base + ((uint32_t)(q * 32) << 16) + FT_THOLD + (cur ^ 1) * 128 + p * 8 + hf * 4, zero_next ? make_uint4(0u, 0u, 0u, 0u) : hpk);
                    uint4 rl4;
                    const __half2 z2 = __float2half2_rn(0.0f);
                    const __half2* hs = reinterpret_cast<const __half2*>(&hpk);
                    __half2 r0 = __hmax2_nan(hs[0], z2), r1 = __hmax2_nan(hs[1], z2), r2 = __hmax2_nan(hs[2], z2), r3 = __hmax2_nan(hs[3], z2);
                    rl4.x = *reinterpret_cast<uint32_t*>(&r0); rl4.y = *reinterpret_cast<uint32_t*>(&r1);
                    rl4.z = *reinterpret_cast<uint32_t*>(&r2); rl4.w = *reinterpret_cast<uint32_t*>(&r3);
                    tmem_st4(tmem_base + ((uint32_t)(q * 32) << 16) + FT_TTILE + sb * 8 + hf * 4, rl4);
                    tmem_st_wait();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&stage_full[sb]);
                }
                if (rv) {
                    const uint32_t so = (uint32_t)(u0 >> 3) << 8;                   // RB32: chunk stride 256 elements
                    if (h16) *reinterpret_cast<uint4*>(h16_t + so) = hpk;
                    if (fac) {
                        // the reverse pass rebuilds its factors from the gates (and h' from h16 of step t+1)
                        __half* const fo = fac_t + so;                              // planes 8192 elements apart (tc.cuh::fac_index)
                        *reinterpret_cast<uint4*>(fo) = pack8(rr);
                        // z is in [0, 1]: its sign bits carry relu'(h_t) for the reverse pass (set = the fp16 h_t is <= 0)
                        uint4 zp = pack8(zz);
                        {
                            const __half2 zero2 = __float2half2_rn(0.0f);
                            const __half2* hs2 = reinterpret_cast<const __half2*>(&hpk);
                            zp.x |= __hle2_mask(hs2[0], zero2) & 0x80008000u; zp.y |= __hle2_mask(hs2[1], zero2) & 0x80008000u;
                            zp.z |= __hle2_mask(hs2[2], zero2) & 0x80008000u; zp.w |= __hle2_mask(hs2[3], zero2) & 0x80008000u;
                        }
                        *reinterpret_cast<uint4*>(fo + 8192) = zp;
                        *reinterpret_cast<uint4*>(fo + 2 * 8192) = pack8(nn);
                        *reinterpret_cast<uint4*>(fo + 3 * 8192) = pack8(hn);
                    }
                    if (hpimg) {
                        // h' consumed at step t-1 (= masked h_t): fp16 token-tile image for the weight-gradient GEMM (the very fp16
                        // values the recurrence used: no second rounding)
                        if (t > 0)       // tile_img_offset(hp_tok, 4, u0) with the per-step part hoisted
                            *reinterpret_cast<uint4*>(hp_t + ((uint32_t)(u0 >> 6) << 13) + ((((uint32_t)(u0 & 63) >> 3) ^ hp_r7) << 4)) =
                                zero_next ? make_uint4(0u, 0u, 0u, 0u) : hpk;
                        if (t == L - 1)
                            *reinterpret_cast<uint4*>(hpimg + tile_img_offset((size_t)t * Rp + row, 4, u0)) = make_uint4(0u, 0u, 0u, 0u);
                    }
                }
            }
            // this warp's part of h_t is in tensor memory: signal the MMA warp.  The x tile of the next step was written
            // with generic-proxy stores and is read by the tensor core (async proxy): proxy fence before the arrival.
            fence_proxy_async_smem();
            tmem_st_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&a_ready);
            // heads: the 16 heads MMAs of this step are complete -> bias, softmax, outputs (one thread per row)
            if (set == 1 && hf == 0) {
                mbar_wait(&heads_full[step & 1], (step >> 1) & 1);
                tc_fence_after();
                float v[4][8];
                const uint32_t th = tmem_base + ((uint32_t)(q * 32) << 16) + FT_THEADS + (step & 1) * 32;
#pragma unroll
                for (int j = 0; j < 4; ++j) tmem_ld8(th + 8 * j, v[j]);
                tmem_ld_wait();
                tc_fence_before();
                if (rv) {
                    float zl[LPG_Y], pr[LPG_Y];
#pragma unroll
                    for (int c = 0; c < 7; ++c) zl[c] = v[0][1 + c] + v[2][1 + c] + b_heads[1 + c];
                    zl[7] = v[1][0] + v[3][0] + b_heads[8];
                    softmax_c<LPG_Y>(zl, pr);
                    const size_t tok = (size_t)t * R + row;
                    pi_hat[tok] = v[0][0] + v[2][0] + b_heads[0];
                    float4* yo = reinterpret_cast<float4*>(y_hat + tok * LPG_Y);
                    yo[0] = make_float4(pr[0], pr[1], pr[2], pr[3]);
                    yo[1] = make_float4(pr[4], pr[5], pr[6], pr[7]);
                }
            }
            cur ^= 1;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 17) tmem_dealloc(tmem_base, 512);
}

static size_t gru_fwd_tc_smem(int X) {
    (void)X;
    return 2 * FT_AX + FT_NS * FT_BSTAGE + FT_NPASS * 1024 + sizeof(float) * LPG_H + 1024;
}

static int gru_forward_tc_launch(const float* x, const uint8_t* done, const float* lpg_params, const void* wh_img,
                                 void* h16, void* fac, void* hpimg, float* pi_hat, float* y_hat, int n_agents,
                                 int n_workers, int rollout_len, int lifetime_conditioning, size_t lpg_stride, void* stream) {
    const int R = n_agents * n_workers;
    const int rows = lpg_stride ? n_workers : FT_M;
    const int blocks = lpg_stride ? n_agents : (R + FT_M - 1) / FT_M;
    cudaStream_t st = (cudaStream_t)stream;
    if (lifetime_conditioning) {
        const size_t smem = gru_fwd_tc_smem(7);
        TOUED_CUDA(cudaFuncSetAttribute(gru_forward_tc_kernel<7>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        gru_forward_tc_kernel<7><<<blocks, FT_THREADS, smem, st>>>(x, done, lpg_params, (const __half*)wh_img, (__half*)h16,
                                                                    (__half*)fac, (unsigned char*)hpimg, pi_hat, y_hat, R, rollout_len, n_workers,
                                                                    rows, lpg_stride);
    } else {
        const size_t smem = gru_fwd_tc_smem(5);
        TOUED_CUDA(cudaFuncSetAttribute(gru_forward_tc_kernel<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        gru_forward_tc_kernel<5><<<blocks, FT_THREADS, smem, st>>>(x, done, lpg_params, (const __half*)wh_img, (__half*)h16,
                                                                    (__half*)fac, (unsigned char*)hpimg, pi_hat, y_hat, R, rollout_len, n_workers,
                                                                    rows, lpg_stride);
    }
    TOUED_LAUNCH_CHECK();
    return 0;
}

extern "C" int toued_gru_forward_tc(const float* x, const uint8_t* done, const float* lpg_params, const void* wh_img,
                                    void* h16, void* fac, void* hpimg, float* pi_hat, float* y_hat, int n_agents,
                                    int n_workers, int rollout_len, int lifetime_conditioning, void* stream) {
    TOUED_CHECK(n_agents * n_workers > 0 && rollout_len > 0, "toued_gru_forward_tc: empty problem");
    // h16 is read only by the reverse pass, which also needs fac / hpimg: inference may pass NULL for all three
    TOUED_CHECK(h16 != nullptr || (fac == nullptr && hpimg == nullptr), "toued_gru_forward_tc: h16 is required with fac / hpimg");
    return gru_forward_tc_launch(x, done, lpg_params, wh_img, h16, fac, hpimg, pi_hat, y_hat, n_agents, n_workers, rollout_len,
                                 lifetime_conditioning, 0, stream);
}

extern "C" int toued_gru_forward_tc_multi(const float* x, const uint8_t* done, const float* lpg_params, const void* wh_img,
                                          float* pi_hat, float* y_hat, int n_agents, int n_workers, int rollout_len,
                                          int lifetime_conditioning, int lpg_stride, void* stream) {
    TOUED_CHECK(n_agents > 0 && n_workers > 0 && rollout_len > 0, "toued_gru_forward_tc_multi: empty problem");
    TOUED_CHECK(n_workers <= FT_M && lpg_stride > 0, "toued_gru_forward_tc_multi: n_workers=%d must be <= 128 and lpg_stride > 0", n_workers);
    return gru_forward_tc_launch(x, done, lpg_params, wh_img, nullptr, nullptr, nullptr, pi_hat, y_hat, n_agents, n_workers,
                                 rollout_len, lifetime_conditioning, (size_t)lpg_stride, stream);
}
