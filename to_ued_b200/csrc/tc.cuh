// tcgen05 / TMEM / mbarrier helpers (sm_100a inline PTX).
//
// Operand convention used by every tensor-core kernel here: both operands K-major fp16/bf16 in shared
// memory as "SW128 K-block tiles": a K-block is 64 elements (128 B) wide; row r of a K-block occupies
// bytes [r*128, r*128+128) and its 16-byte chunk c is stored at chunk position c ^ (r & 7)
// (the 128-byte swizzle, Swizzle<3,4,3>).  Tiles are 1024-byte aligned; groups of 8 rows are 1024 B
// apart (SBO).  Matches cute::UMMA K-major SWIZZLE_128B canonical layout
// ((8,n),2):((8,SBO),1) in 16-byte units (descriptor fields: version=1, LBO=1, SBO=64, layout=2).
#pragma once
#include "common.cuh"
#include <cuda_fp16.h>
#include <cuda_bf16.h>

constexpr int TC_KB_ELEMS = 64;        // elements per K-block (128 B of fp16/bf16)
constexpr int TC_UMMA_K = 16;          // K per tcgen05.mma for 16-bit inputs

// byte offset of element (row, k) inside a K-major SW128 tile set whose K-blocks are `rows*128` B apart
__host__ __device__ __forceinline__ uint32_t sw128_offset(int rows, int row, int k) {
    const int kb = k >> 6, kin = k & 63;
    const int chunk = kin >> 3;
    return (uint32_t)kb * (uint32_t)rows * 128u + (uint32_t)row * 128u + (uint32_t)((chunk ^ (row & 7)) << 4) +
           (uint32_t)((kin & 7) << 1);
}

// "Token tile image": a [tokens][C] 16-bit matrix stored as 64-token x 64-column sub-tiles of 8 KB,
// each already in the SW128 pattern (row = token, 128 B per row, chunk ^= row & 7), sub-tiles ordered
// [token block][column group].  A sub-tile is at once (a) a K-major SW128 K-block with K = columns and
// (b) an MN-major SW128 atom column with K = tokens, so it can be bulk-copied into shared memory and
// fed to tcgen05.mma for both the recurrence GEMMs and the weight-gradient GEMMs.
__host__ __device__ __forceinline__ size_t tile_img_offset(size_t tok, int n_col_groups, int col) {
    const size_t tb = tok >> 6; const int r = (int)(tok & 63), cg = col >> 6, cin = col & 63;
    return ((tb * n_col_groups + cg) << 13) + (size_t)r * 128 + (size_t)(((cin >> 3) ^ (r & 7)) << 4) + (size_t)((cin & 7) << 1);
}

// "RB32" layout of per-(token, unit) 16-bit tensors saved between the tensor-core forward and reverse
// kernels: [t][row block of 32][chunk of 8 units][32 rows][8 units].  A warp of the epilogue (32 rows, one
// 16-byte chunk each) reads / writes 512 contiguous bytes.  Returns an element (2-byte) index.
__host__ __device__ __forceinline__ size_t rb32_index(size_t t, size_t n_row_blocks, int row, int u) {
    return (((t * n_row_blocks + (size_t)(row >> 5)) * 32 + (size_t)(u >> 3)) << 8) + (size_t)((row & 31) << 3) + (size_t)(u & 7);
}

// The four saved gate planes (r, z, n, hn) of the tensor-core forward: RB32 blocks with the planes INTERLEAVED per
// (t, 32-row block): [t][row block][plane][chunk][32 rows][8 units].  (Four separate [L][R]-sized planes put the four
// loads a reverse-pass thread issues together exactly 160 MiB apart at the BASELINE shape.)
__host__ __device__ __forceinline__ size_t fac_index(size_t t, size_t n_row_blocks, int row, int u, int plane) {
    return ((((t * n_row_blocks + (size_t)(row >> 5)) * 4 + (size_t)plane) * 32 + (size_t)(u >> 3)) << 8) + (size_t)((row & 31) << 3) + (size_t)(u & 7);
}

__device__ __forceinline__ uint64_t tc_smem_desc(uint32_t smem_addr) {
    return (uint64_t)((smem_addr >> 4) & 0x3FFFu) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// K-major, NO swizzle ("interleave") operand for a narrow K = 16 block: 8-row x 16-byte core matrices
// (128 B contiguous); the second 8-element K chunk is `lbo` bytes further, the next 8-row group `sbo`
// bytes further.  byte offset of element (row, k), k < 16, with lbo = 128, sbo = 256:
__host__ __device__ __forceinline__ uint32_t k16_offset(int row, int k) {
    return (uint32_t)(row >> 3) * 256u + (uint32_t)(k >> 3) * 128u + (uint32_t)(row & 7) * 16u + (uint32_t)(k & 7) * 2u;
}
__device__ __forceinline__ uint64_t tc_smem_desc_k16(uint32_t smem_addr) {
    return (uint64_t)((smem_addr >> 4) & 0x3FFFu) | ((uint64_t)(128u >> 4) << 16) | ((uint64_t)(256u >> 4) << 32) |
           (1ull << 46);                                   // layout type 0 = no swizzle
}
// MN-major SW128 operand (contraction index = rows of the tile image): 64 MN-elements (128 B) per k-row,
// 8 k-rows per 1024-byte swizzle atom (SBO), next group of 64 MN-elements `lbo_bytes` away (LBO).
__device__ __forceinline__ uint64_t tc_smem_desc_mn(uint32_t smem_addr, uint32_t lbo_bytes) {
    return (uint64_t)((smem_addr >> 4) & 0x3FFFu) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) | (64ull << 32) |
           (1ull << 46) | (2ull << 61);
}
// MN-major operand WITHOUT swizzle: 8 (k) x 16-byte (8 MN-elements) core matrices of 128 contiguous bytes;
// in this mode (unlike the swizzled MN-major modes) `lbo_bytes` = distance to the next 8 k-rows and
// `sbo_bytes` = distance to the next 8 MN-elements.  The RB32 activation layout [chunk][32 rows][8 units]
// is exactly this with lbo = 128, sbo = 512 (k = rows).
__device__ __forceinline__ uint64_t tc_smem_desc_mn_plain(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((smem_addr >> 4) & 0x3FFFu) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}
// instruction descriptor with both operands MN-major (weight-gradient GEMMs)
__host__ __device__ constexpr uint32_t tc_idesc_mn(int M, int N, int fmt) {
    return (1u << 4) | ((uint32_t)fmt << 7) | ((uint32_t)fmt << 10) | (1u << 15) | (1u << 16) |
           ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// instruction descriptor, kind::f16, fp32 accumulate, both operands K-major. fmt: 0 = f16, 1 = bf16
__host__ __device__ constexpr uint32_t tc_idesc(int M, int N, int fmt) {
    return (1u << 4) | ((uint32_t)fmt << 7) | ((uint32_t)fmt << 10) | ((uint32_t)(N >> 3) << 17) |
           ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void tc_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
                 ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// same with the A operand read from tensor memory (M rows = lanes, two 16-bit K elements per 32-bit column)
__device__ __forceinline__ void tc_mma_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n"
                 ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// One lane of a converged warp (elect.sync).  Issuing tcgen05.mma / commit under `if (elect_one())` instead of
// `if (lane == 0)` lets the compiler prove the branch is taken by exactly one thread and emit the uniform-datapath
// instructions directly; under a plain lane test it wraps EVERY UTCHMMA in an ELECT / BRA.U.ANY loop (~10 extra
// instructions per MMA on the single issuing thread -- the bottleneck of a stream of small MMAs).
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
// arrive on an mbarrier when all previously issued MMAs of this thread have completed
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// TMEM allocation: executed by ONE full warp; column count a power of two >= 32
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// 32 lanes x 8 consecutive columns: thread i of the warp gets row (lane quadrant base + i)
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8]) {
    uint32_t r[8];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
// 32 lanes x 4 consecutive columns: thread i of the warp writes row (lane quadrant base + i)
__device__ __forceinline__ void tmem_st4(uint32_t taddr, const uint4& v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ uint4 tmem_ld4(uint32_t taddr) {
    uint4 r;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(taddr));
    return r;
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// smem -> global 1-D bulk copy (TMA store) tracked by the issuing thread's bulk group
__device__ __forceinline__ void bulk_s2g(void* dst_gmem, uint32_t src_smem, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(src_smem), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read_1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void st_shared_v4(uint32_t addr, const uint4& v) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// ---- CTA pairs (cta_group::2): two CTAs of a 2-cluster share one MMA of M = 256 -------------------------------------
// Each CTA holds its own 128 rows of A and HALF of the N columns of B at the same shared-memory offsets; the leader (rank
// 0) issues the MMA, both CTAs' tensor memory receives its 128 rows x N columns.  Per CTA and K-step the tensor core then
// fetches 128 x 16 of A and N/2 x 16 of B instead of N x 16: what an operand-fetch-bound 1-CTA MMA stream needs.
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_alloc2(uint32_t* smem_dst, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_mma2(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
                 ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// arrive on the mbarrier at this shared-memory offset in every CTA of `cta_mask` once all MMAs issued so far completed
__device__ __forceinline__ void tc_commit2(uint64_t* bar, uint16_t cta_mask) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"(cta_mask) : "memory");
}
// arrive (release at cluster scope) on the mbarrier at the same shared-memory offset in CTA `cta` of the cluster
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t cta) {
    asm volatile("{\n\t.reg .b32 ra;\n\tmapa.shared::cluster.u32 ra, %0, %1;\n\t"
                 "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n\t}" ::"r"(smem_u32(bar)), "r"(cta) : "memory");
}
// wait with acquire at cluster scope (the arrivals come from the peer CTA)
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tWAITC_%=:\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONEC_%=;\n\tbra WAITC_%=;\n\tDONEC_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}

// ---- scaled fp16 operands of the tensor-core reverse pass -----------------------------------------------------------
// The reverse pass is linear in the cotangents (d pi_hat, d y_hat), which are tiny (pre-scaled by 1 / N_global): far
// below fp16's range but fine for bf16 -- at 8 instead of 11 significant bits.  The tensor-core reverse kernels therefore
// run on cotangents multiplied by a power of two S chosen per launch from max |cotangent| (toued_cotangent_max), use fp16
// operands everywhere (dG, z * dh, Wh, h', x: 8x finer than bf16; h' is even exact, it IS fp16), convert with saturation,
// and multiply their fp32 results by 1 / S when they leave the kernel.  S puts the largest cotangent at [2^3, 2^4): a
// factor 2^12 of headroom for growth along the 20-step chain before saturation, ~2^-27 of the maximum before underflow.
// A saturated or non-finite operand is not corrected but reported in the launch's status word (include/toued.h).
__device__ __forceinline__ float cot_scale_from_max(uint32_t max_bits) {
    if (max_bits == 0u || max_bits >= 0x7F800000u) return 1.0f;           // no signal, or inf / nan: leave unscaled
    const int e = (int)(max_bits >> 23) - 127;                            // floor(log2(max))
    const int s = min(max(3 - e, -100), 100);
    return __uint_as_float((uint32_t)(s + 127) << 23);                     // 2^s
}
// two fp32 -> packed fp16x2 with saturation to +-65504 (lo in the low half)
__device__ __forceinline__ uint32_t pack_h2_sat(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
__device__ __forceinline__ uint4 pack8h_sat(const float (&v)[8]) {
    return make_uint4(pack_h2_sat(v[0], v[1]), pack_h2_sat(v[2], v[3]), pack_h2_sat(v[4], v[5]), pack_h2_sat(v[6], v[7]));
}
