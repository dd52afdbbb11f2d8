// Unit kernel for the tcgen05 building blocks: D[128][N] = A[128][K] * B[N][K]^T with fp16 operands
// (fp32 in global, converted on the fly), K = 256, N = 48 — the tile shape the GRU kernels use.
// Exercises: SW128 K-major operand tiles, smem/instruction descriptors, cp.async.bulk of a pre-swizzled
// B image, tcgen05.mma accumulation in TMEM, tcgen05.commit -> mbarrier, tcgen05.ld.
#include "tc.cuh"
#include "../../include/toued.h"

// B[N][K] fp32 (row-major) -> fp16 SW128 image: K-block kb at byte kb*N*128
__global__ void pack_b_sw128_kernel(const float* __restrict__ B, __half* __restrict__ img, int N, int K) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N * K) return;
    const int n = i / K, k = i % K;
    *reinterpret_cast<__half*>(reinterpret_cast<char*>(img) + sw128_offset(N, n, k)) = __float2half_rn(B[i]);
}

template <int N, int K>
__global__ void __launch_bounds__(128, 1)
tc_gemm_test_kernel(const float* __restrict__ A, const __half* __restrict__ Bimg, float* __restrict__ D) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    // (offset arithmetic on the __shared__ array, not an integer round trip: the compiler keeps the shared
    //  address space and emits LDS / STS instead of generic LD / ST)
    unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    unsigned char* sA = smem;                              // K/64 K-blocks x 128 rows x 128 B
    unsigned char* sB = smem + (K / 64) * 128 * 128;       // K/64 K-blocks x N rows x 128 B
    __shared__ __align__(8) uint64_t bar_b, bar_mma;
    __shared__ uint32_t tmem_base;
    const int tid = threadIdx.x, warp = tid >> 5;
    if (warp == 0) tmem_alloc(&tmem_base, 64);
    if (tid == 0) { mbar_init(&bar_b, 1); mbar_init(&bar_mma, 1); mbar_fence_init(); }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tb = tmem_base;
    if (tid == 0) {
        mbar_expect_tx(&bar_b, (K / 64) * N * 128);
        bulk_g2s(sB, Bimg, (K / 64) * N * 128, &bar_b);
    }
    // A: row = tid, convert fp32 -> fp16 into the swizzled tile
    for (int k = 0; k < K; k += 8) {
        __half2 h[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) h[e] = __floats2half2_rn(A[tid * K + k + 2 * e], A[tid * K + k + 2 * e + 1]);
        *reinterpret_cast<uint4*>(sA + sw128_offset(128, tid, k)) = *reinterpret_cast<uint4*>(h);
    }
    fence_proxy_async_smem();
    __syncthreads();
    if (tid == 0) {
        mbar_wait(&bar_b, 0);
        tc_fence_after();
        constexpr uint32_t idesc = tc_idesc(128, N, 0);
#pragma unroll
        for (int kb = 0; kb < K / 64; ++kb) {
            const uint64_t ad = tc_smem_desc(smem_u32(sA + kb * 128 * 128));
            const uint64_t bd = tc_smem_desc(smem_u32(sB + kb * N * 128));
#pragma unroll
            for (int s = 0; s < 4; ++s) tc_mma(tb, ad + 2 * s, bd + 2 * s, idesc, (kb | s) != 0);
        }
        tc_commit(&bar_mma);
    }
    mbar_wait(&bar_mma, 0);
    tc_fence_after();
    for (int c = 0; c < N; c += 8) {
        float v[8];
        tmem_ld8(tb + ((uint32_t)(warp * 32) << 16) + c, v);
        tmem_ld_wait();
#pragma unroll
        for (int e = 0; e < 8; ++e) D[tid * N + c + e] = v[e];
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tb, 64);
}

extern "C" int toued_tc_gemm_test(const float* A, const float* B, void* scratch_img, float* D, void* stream) {
    constexpr int N = 48, K = 256;
    cudaStream_t st = (cudaStream_t)stream;
    pack_b_sw128_kernel<<<(N * K + 255) / 256, 256, 0, st>>>(B, (__half*)scratch_img, N, K);
    TOUED_LAUNCH_CHECK();
    const size_t smem = (K / 64) * 128 * 128 + (K / 64) * N * 128 + 1024;
    TOUED_CUDA(cudaFuncSetAttribute(tc_gemm_test_kernel<N, K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    tc_gemm_test_kernel<N, K><<<1, 128, smem, st>>>(A, (const __half*)scratch_img, D);
    TOUED_LAUNCH_CHECK();
    return 0;
}

// ------------------------------------------------------------------------------------------------
// MN-major check: D[128][128] = sum_k A[k][m] * B[k][n], K = 128 "tokens", bf16 token tile images.
__global__ void pack_tile_img_kernel(const float* __restrict__ X, __nv_bfloat16* __restrict__ img, int K, int C) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= K * C) return;
    const int k = i / C, c = i % C;
    *reinterpret_cast<__nv_bfloat16*>(reinterpret_cast<char*>(img) + tile_img_offset(k, C / 64, c)) = __float2bfloat16_rn(X[i]);
}

__global__ void __launch_bounds__(128, 1)
tc_gemm_mn_test_kernel(const unsigned char* __restrict__ Aimg, const unsigned char* __restrict__ Bimg, float* __restrict__ D,
                       uint32_t lbo, uint32_t sbo, uint32_t kadv) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    // (offset arithmetic on the __shared__ array, not an integer round trip: the compiler keeps the shared
    //  address space and emits LDS / STS instead of generic LD / ST)
    unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    unsigned char* sA = smem;               // 2 token blocks x [2 col groups][8 KB]
    unsigned char* sB = smem + 32768;
    __shared__ __align__(8) uint64_t bar_ld, bar_mma;
    __shared__ uint32_t tmem_base;
    const int tid = threadIdx.x, warp = tid >> 5;
    if (warp == 0) tmem_alloc(&tmem_base, 128);
    if (tid == 0) { mbar_init(&bar_ld, 1); mbar_init(&bar_mma, 1); mbar_fence_init(); }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tb = tmem_base;
    if (tid == 0) {
        mbar_expect_tx(&bar_ld, 65536);
        bulk_g2s(sA, Aimg, 32768, &bar_ld);
        bulk_g2s(sB, Bimg, 32768, &bar_ld);
        mbar_wait(&bar_ld, 0);
        tc_fence_after();
        constexpr uint32_t idesc = tc_idesc_mn(128, 128, 1);
        for (int blk = 0; blk < 2; ++blk)
            for (int ks = 0; ks < 4; ++ks) {
                auto mk = [&](uint32_t addr) {
                    return (uint64_t)((addr >> 4) & 0x3FFFu) | ((uint64_t)((lbo >> 4) & 0x3FFFu) << 16) |
                           ((uint64_t)((sbo >> 4) & 0x3FFFu) << 32) | (1ull << 46) | (2ull << 61);
                };
                const uint64_t ad = mk(smem_u32(sA + blk * 16384 + ks * kadv));
                const uint64_t bd = mk(smem_u32(sB + blk * 16384 + ks * kadv));
                tc_mma(tb, ad, bd, idesc, (blk | ks) != 0);
            }
        tc_commit(&bar_mma);
    }
    mbar_wait(&bar_mma, 0);
    tc_fence_after();
    for (int c = 0; c < 128; c += 8) {
        float v[8];
        tmem_ld8(tb + ((uint32_t)(warp * 32) << 16) + c, v);
        tmem_ld_wait();
#pragma unroll
        for (int e = 0; e < 8; ++e) D[tid * 128 + c + e] = v[e];
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tb, 128);
}

extern "C" int toued_tc_gemm_mn_test(const float* A, const float* B, void* scratch_img, float* D, int lbo, int sbo,
                                     int kadv, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    unsigned char* ia = (unsigned char*)scratch_img;
    unsigned char* ib = ia + 32768;
    pack_tile_img_kernel<<<(128 * 128 + 255) / 256, 256, 0, st>>>(A, (__nv_bfloat16*)ia, 128, 128);
    pack_tile_img_kernel<<<(128 * 128 + 255) / 256, 256, 0, st>>>(B, (__nv_bfloat16*)ib, 128, 128);
    TOUED_LAUNCH_CHECK();
    const size_t smem = 65536 + 1024;
    TOUED_CUDA(cudaFuncSetAttribute(tc_gemm_mn_test_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    tc_gemm_mn_test_kernel<<<1, 128, smem, st>>>(ia, ib, D, (uint32_t)lbo, (uint32_t)sbo, (uint32_t)kadv);
    TOUED_LAUNCH_CHECK();
    return 0;
}

// ------------------------------------------------------------------------------------------------
// CTA pair (cta_group::2), both operands MN-major: D[256 m][256 n] = sum_k A[k][m] B[k][n], K = 128 tokens.
// CTA r of the 2-cluster holds column groups {2r, 2r+1} of the A image (its 128 rows of M) and {2r, 2r+1} of the B image
// (its half of N); the leader issues M256 N256 K16 MMAs; every CTA reads back its own 128 rows x 256 columns.
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(128, 1)
tc_gemm_mn2_test_kernel(const unsigned char* __restrict__ Aimg, const unsigned char* __restrict__ Bimg, float* __restrict__ D) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    unsigned char* sA = smem;               // 2 token blocks x [2 col groups][8 KB]
    unsigned char* sB = smem + 32768;
    __shared__ __align__(8) uint64_t bar_ld, bar_peer, bar_mma;
    __shared__ uint32_t tmem_base;
    const int tid = threadIdx.x, warp = tid >> 5;
    const uint32_t rank = cluster_ctarank();
    if (tid == 0) { mbar_init(&bar_ld, 1); mbar_init(&bar_peer, 1); mbar_init(&bar_mma, 1); mbar_fence_init(); }
    if (warp == 0) tmem_alloc2(&tmem_base, 256);
    tc_fence_before();
    __syncthreads();
    cluster_sync();                          // barriers of both CTAs are initialised before anyone arrives remotely
    tc_fence_after();
    const uint32_t tb = tmem_base;
    if (tid == 0) {
        mbar_expect_tx(&bar_ld, 65536);
        for (int blk = 0; blk < 2; ++blk) {  // image: [token block][4 col groups][8 KB]
            bulk_g2s(sA + blk * 16384, Aimg + ((size_t)(blk * 4 + 2 * rank) << 13), 16384, &bar_ld);
            bulk_g2s(sB + blk * 16384, Bimg + ((size_t)(blk * 4 + 2 * rank) << 13), 16384, &bar_ld);
        }
        mbar_wait(&bar_ld, 0);
        if (rank != 0) {
            mbar_arrive_remote(&bar_peer, 0);            // my operands have landed: tell the leader
        } else {
            mbar_wait_cluster(&bar_peer, 0);
            tc_fence_after();
            constexpr uint32_t idesc = tc_idesc_mn(256, 256, 1);
            for (int blk = 0; blk < 2; ++blk)
                for (int ks = 0; ks < 4; ++ks)
                    tc_mma2(tb, tc_smem_desc_mn(smem_u32(sA + blk * 16384 + ks * 2048), 8192),
                            tc_smem_desc_mn(smem_u32(sB + blk * 16384 + ks * 2048), 8192), idesc, (blk | ks) != 0);
            tc_commit2(&bar_mma, 3);
        }
    }
    mbar_wait_cluster(&bar_mma, 0);
    tc_fence_after();
    for (int c = 0; c < 256; c += 8) {
        float v[8];
        tmem_ld8(tb + ((uint32_t)(warp * 32) << 16) + c, v);
        tmem_ld_wait();
#pragma unroll
        for (int e = 0; e < 8; ++e) D[(size_t)(rank * 128 + tid) * 256 + c + e] = v[e];
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync();                          // both CTAs are done with tensor memory before it is released
    if (warp == 0) tmem_dealloc2(tb, 256);
}

extern "C" int toued_tc_gemm_mn2_test(const float* A, const float* B, void* scratch_img, float* D, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    unsigned char* ia = (unsigned char*)scratch_img;
    unsigned char* ib = ia + 65536;
    pack_tile_img_kernel<<<(128 * 256 + 255) / 256, 256, 0, st>>>(A, (__nv_bfloat16*)ia, 128, 256);
    pack_tile_img_kernel<<<(128 * 256 + 255) / 256, 256, 0, st>>>(B, (__nv_bfloat16*)ib, 128, 256);
    TOUED_LAUNCH_CHECK();
    const size_t smem = 65536 + 1024;
    TOUED_CUDA(cudaFuncSetAttribute(tc_gemm_mn2_test_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    tc_gemm_mn2_test_kernel<<<2, 128, smem, st>>>(ia, ib, D);
    TOUED_LAUNCH_CHECK();
    return 0;
}

// ------------------------------------------------------------------------------------------------
// K = 256 (SW128 blocks) + 16 (no-swizzle block): D[128][48] = A[128][272] * B[48][272]^T, fp16.
__global__ void pack_b_mixed_kernel(const float* __restrict__ B, __half* __restrict__ img, int N, int K) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N * K) return;
    const int n = i / K, k = i % K;
    char* base = reinterpret_cast<char*>(img);
    if (k < 256) *reinterpret_cast<__half*>(base + sw128_offset(N, n, k)) = __float2half_rn(B[i]);
    else *reinterpret_cast<__half*>(base + 4 * N * 128 + k16_offset(n, k - 256)) = __float2half_rn(B[i]);
}

__global__ void __launch_bounds__(128, 1)
tc_gemm_mixed_test_kernel(const float* __restrict__ A, const __half* __restrict__ Bimg, float* __restrict__ D) {
    constexpr int N = 48, K = 272;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    // (offset arithmetic on the __shared__ array, not an integer round trip: the compiler keeps the shared
    //  address space and emits LDS / STS instead of generic LD / ST)
    unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    unsigned char* sA = smem;                               // 4 x 16 KB SW128 + 4 KB k16 tile
    unsigned char* sAx = sA + 4 * 128 * 128;
    unsigned char* sB = sAx + 4096;                         // 4 x 6 KB SW128 + 1.5 KB k16 tile (1024-aligned)
    __shared__ __align__(8) uint64_t bar_b, bar_mma;
    __shared__ uint32_t tmem_base;
    const int tid = threadIdx.x, warp = tid >> 5;
    if (warp == 0) tmem_alloc(&tmem_base, 64);
    if (tid == 0) { mbar_init(&bar_b, 1); mbar_init(&bar_mma, 1); mbar_fence_init(); }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tb = tmem_base;
    constexpr uint32_t BBYTES = 4 * N * 128 + (N / 8) * 256;
    if (tid == 0) { mbar_expect_tx(&bar_b, BBYTES); bulk_g2s(sB, Bimg, BBYTES, &bar_b); }
    for (int k = 0; k < K; ++k) {
        const __half h = __float2half_rn(A[tid * K + k]);
        if (k < 256) *reinterpret_cast<__half*>(sA + sw128_offset(128, tid, k)) = h;
        else *reinterpret_cast<__half*>(sAx + k16_offset(tid, k - 256)) = h;
    }
    fence_proxy_async_smem();
    __syncthreads();
    if (tid == 0) {
        mbar_wait(&bar_b, 0);
        tc_fence_after();
        constexpr uint32_t idesc = tc_idesc(128, N, 0);
        for (int kb = 0; kb < 4; ++kb) {
            const uint64_t ad = tc_smem_desc(smem_u32(sA + kb * 128 * 128));
            const uint64_t bd = tc_smem_desc(smem_u32(sB + kb * N * 128));
            for (int s = 0; s < 4; ++s) tc_mma(tb, ad + 2 * s, bd + 2 * s, idesc, (kb | s) != 0);
        }
        tc_mma(tb, tc_smem_desc_k16(smem_u32(sAx)), tc_smem_desc_k16(smem_u32(sB + 4 * N * 128)), idesc, 1u);
        tc_commit(&bar_mma);
    }
    mbar_wait(&bar_mma, 0);
    tc_fence_after();
    for (int c = 0; c < N; c += 8) {
        float v[8];
        tmem_ld8(tb + ((uint32_t)(warp * 32) << 16) + c, v);
        tmem_ld_wait();
#pragma unroll
        for (int e = 0; e < 8; ++e) D[tid * N + c + e] = v[e];
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tb, 64);
}

extern "C" int toued_tc_gemm_mixed_test(const float* A, const float* B, void* scratch_img, float* D, void* stream) {
    constexpr int N = 48, K = 272;
    cudaStream_t st = (cudaStream_t)stream;
    pack_b_mixed_kernel<<<(N * K + 255) / 256, 256, 0, st>>>(B, (__half*)scratch_img, N, K);
    TOUED_LAUNCH_CHECK();
    const size_t smem = 4 * 128 * 128 + 4096 + 4 * N * 128 + 2048 + 1024;
    TOUED_CUDA(cudaFuncSetAttribute(tc_gemm_mixed_test_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    tc_gemm_mixed_test_kernel<<<1, 128, smem, st>>>(A, (const __half*)scratch_img, D);
    TOUED_LAUNCH_CHECK();
    return 0;
}

// ------------------------------------------------------------------------------------------------
// The weight-gradient GEMM's operand roles (wgrad_tc.cu), fp16, K = 128 tokens: one MN-major A of 128 columns
// (two 64-column groups) against (a) B = 256 columns (four groups, N = 256) and (b) B = the first 16 columns of a
// single 64-column group (N = 16: an MN-major SW128 operand narrower than its 64-element swizzle atom, as the x image
// is used).  D[128][256 + 16] = A^T [B | X[:, 0:16]].
__global__ void pack_tile_img_f16_kernel(const float* __restrict__ X, __half* __restrict__ img, int K, int C) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= K * C) return;
    const int k = i / C, c = i % C;
    *reinterpret_cast<__half*>(reinterpret_cast<char*>(img) + tile_img_offset(k, C / 64, c)) = __float2half_rn(X[i]);
}

__global__ void __launch_bounds__(128, 1)
tc_gemm_mn_x16_test_kernel(const unsigned char* __restrict__ Aimg, const unsigned char* __restrict__ Bimg,
                           const unsigned char* __restrict__ Ximg, float* __restrict__ D) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    unsigned char* sA = smem;               // 2 token blocks x [2 col groups][8 KB]
    unsigned char* sB = smem + 32768;       // 2 token blocks x [4 col groups][8 KB]
    unsigned char* sX = smem + 98304;       // 2 token blocks x [1 col group][8 KB]
    __shared__ __align__(8) uint64_t bar_ld, bar_mma;
    __shared__ uint32_t tmem_base;
    const int tid = threadIdx.x, warp = tid >> 5;
    if (warp == 0) tmem_alloc(&tmem_base, 512);
    if (tid == 0) { mbar_init(&bar_ld, 1); mbar_init(&bar_mma, 1); mbar_fence_init(); }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tb = tmem_base;
    if (tid == 0) {
        mbar_expect_tx(&bar_ld, 32768 + 65536 + 16384);
        bulk_g2s(sA, Aimg, 32768, &bar_ld);
        bulk_g2s(sB, Bimg, 65536, &bar_ld);
        bulk_g2s(sX, Ximg, 16384, &bar_ld);
        mbar_wait(&bar_ld, 0);
        tc_fence_after();
        constexpr uint32_t idesc = tc_idesc_mn(128, 256, 0), idesc_x = tc_idesc_mn(128, 16, 0);
        for (int blk = 0; blk < 2; ++blk)
            for (int ks = 0; ks < 4; ++ks) {
                const uint64_t ad = tc_smem_desc_mn(smem_u32(sA + blk * 16384 + ks * 2048), 8192);
                tc_mma(tb, ad, tc_smem_desc_mn(smem_u32(sB + blk * 32768 + ks * 2048), 8192), idesc, (blk | ks) != 0);
                tc_mma(tb + 256, ad, tc_smem_desc_mn(smem_u32(sX + blk * 8192 + ks * 2048), 8192), idesc_x, (blk | ks) != 0);
            }
        tc_commit(&bar_mma);
    }
    mbar_wait(&bar_mma, 0);
    tc_fence_after();
    for (int c = 0; c < 272; c += 8) {
        float v[8];
        tmem_ld8(tb + ((uint32_t)(warp * 32) << 16) + c, v);
        tmem_ld_wait();
#pragma unroll
        for (int e = 0; e < 8; ++e) D[tid * 272 + c + e] = v[e];
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tb, 512);
}

extern "C" int toued_tc_gemm_mn_x16_test(const float* A, const float* B, const float* X, void* scratch_img, float* D,
                                         void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    unsigned char* ia = (unsigned char*)scratch_img;
    unsigned char* ib = ia + 32768;
    unsigned char* ix = ib + 65536;
    pack_tile_img_f16_kernel<<<(128 * 128 + 255) / 256, 256, 0, st>>>(A, (__half*)ia, 128, 128);
    pack_tile_img_f16_kernel<<<(128 * 256 + 255) / 256, 256, 0, st>>>(B, (__half*)ib, 128, 256);
    pack_tile_img_f16_kernel<<<(128 * 64 + 255) / 256, 256, 0, st>>>(X, (__half*)ix, 128, 64);
    TOUED_LAUNCH_CHECK();
    const size_t smem = 32768 + 65536 + 16384 + 1024;
    TOUED_CUDA(cudaFuncSetAttribute(tc_gemm_mn_x16_test_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    tc_gemm_mn_x16_test_kernel<<<1, 128, smem, st>>>(ia, ib, ix, D);
    TOUED_LAUNCH_CHECK();
    return 0;
}
