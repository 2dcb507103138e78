// prefill_gemm.cuh -- the batched-prefill building block: C[M,N] (fp32) = A[M,K] (fp16) * B[N,K]^T (fp16)
// on the 5th-generation tensor cores (sm_100a): TMA (cp.async.bulk.tensor, SWIZZLE_128B) -> shared
// memory ring -> tcgen05.mma (kind::f16, cta_group::1, 128 x BN x 16 per instruction, accumulator in
// TMEM) -> tcgen05.ld epilogue.  Replaces the reference's mma.sync m16n8k16 GEMMs gemmMMA / gemmMMAQKV /
// gemmMMAGateUp (TransformerBatchPrefillKernels.java:792-915, 971, 1132), which stage BK=16 through a
// single shared-memory buffer.  A = activations rounded to FP16 (batchedRmsApplyFP16, :61), B = the FP16
// weight matrix exactly as stored in GGUF ([N][K], K contiguous = "K-major" for both operands).
//
// Warp roles (256 threads): warp 0 lane 0 = TMA producer, warp 1 lane 0 = MMA issuer, warp 2 = TMEM
// allocator, warps 4-7 = epilogue (warp w owns TMEM lanes 32*(w%4) .. +31, i.e. 32 rows of the tile).
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace pg {

constexpr int BM = 128, BK = 64, BN = 128;
// Epilogue modes: F32 store (QKV), F32 read-add-store (x += A*W^T: Wo and W2), and the gate/up pair:
// the B tile is 64 rows of W1 and 64 rows of W3 for the same 64 hidden units, so accumulator columns
// [0,64) = gate, [64,128) = up, and the epilogue emits f16(silu(gate)*up) (InferenceCore.java:150-158).
enum { GEMM_F32 = 0, GEMM_RESID = 1, GEMM_GATEUP = 2 };

__device__ __forceinline__ uint32_t s32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t cnt) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(cnt)); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "PG_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra PG_DONE;\n"
        "bra PG_WAIT;\n"
        "PG_DONE:\n"
        "}\n" ::"r"(bar), "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap *map, int c0, int c1, uint32_t bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
                 "l"(map), "r"(c0), "r"(c1), "r"(bar)
                 : "memory");
}
// UMMA shared-memory matrix descriptor, K-major operand, 128-byte swizzle (cute/arch/mma_sm100_desc.hpp
// SmemDescriptor): start address >> 4 | LBO (unused for swizzled K-major, 1) << 16 | SBO = 8 rows * 128 B >> 4
// << 32 | version 1 << 46 | layout SWIZZLE_128B (2) << 61.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
    return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// Instruction descriptor for kind::f16: D = f32 (bit 4), A = B = f16 (0), both K-major, N >> 3 at bit 17, M >> 4 at bit 24.
__host__ __device__ constexpr uint32_t umma_idesc_f16(int m, int n) { return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24); }

__device__ __forceinline__ void umma_f16(uint32_t tmem_c, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_c),
        "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// 32 lanes x 32 consecutive fp32 accumulator columns: thread `lane` of the warp gets row (lane quarter base + lane)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
          "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
          "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}

template <int STAGES> constexpr size_t smem_bytes() { return (size_t)STAGES * (BM * BK * 2 + BN * BK * 2) + (2 * STAGES + 1) * 8 + 16 + 1024; }

// grid = (M tiles, N tiles): the CTAs that share a weight (B) tile are adjacent in launch order, so the
// tile comes from HBM once and from L2 for the others; A (activations, a few MB) lives in L2.
// C: row stride ldc (elements); rows >= m_valid are not stored.  GEMM_GATEUP: N tiles index 64 hidden units.
template <int MODE, int STAGES>
__global__ void __launch_bounds__(256) k_gemm_f16_tcgen05(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b,
                                                         const __grid_constant__ CUtensorMap tma_b2, const __grid_constant__ CUtensorMap tma_c,
                                                         void *__restrict__ Cv, int ldc, int m_valid, int K) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023); // SWIZZLE_128B tiles need 1024-byte alignment
    constexpr int A_BYTES = BM * BK * 2, B_BYTES = BN * BK * 2;
    static_assert(STAGES * (A_BYTES + B_BYTES) >= BM * BN * 4, "the C tile is staged in the operand ring");
    uint8_t *sA = smem, *sB = smem + STAGES * A_BYTES;
    uint64_t *bars = reinterpret_cast<uint64_t *>(sB + STAGES * B_BYTES);
    const uint32_t full0 = s32(bars), empty0 = s32(bars + STAGES), tmem_full = s32(bars + 2 * STAGES);
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * STAGES + 1);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; s++) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, 1); }
        mbar_init(tmem_full, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) { // TMEM: BN fp32 accumulator columns x 128 lanes
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(s32(tmem_slot)), "r"((uint32_t)BN) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;
    const int nk = (K + BK - 1) / BK, m0 = blockIdx.x * BM;
    const int n0 = blockIdx.y * (MODE == GEMM_GATEUP ? BN / 2 : BN);

    if (warp == 0 && lane == 0) {
        // ===== TMA producer =====
        for (int kb = 0; kb < nk; kb++) {
            const int st = kb % STAGES;
            mbar_wait(empty0 + 8 * st, ((kb / STAGES) & 1) ^ 1);
            mbar_expect_tx(full0 + 8 * st, A_BYTES + B_BYTES);
            tma_load_2d(s32(sA + st * A_BYTES), &tma_a, kb * BK, m0, full0 + 8 * st);
            if (MODE == GEMM_GATEUP) {
                tma_load_2d(s32(sB + st * B_BYTES), &tma_b, kb * BK, n0, full0 + 8 * st);
                tma_load_2d(s32(sB + st * B_BYTES + B_BYTES / 2), &tma_b2, kb * BK, n0, full0 + 8 * st);
            } else {
                tma_load_2d(s32(sB + st * B_BYTES), &tma_b, kb * BK, n0, full0 + 8 * st);
            }
        }
    } else if (warp == 1 && lane == 0) {
        // ===== MMA issuer: one thread issues tcgen05.mma for the whole CTA =====
        constexpr uint32_t idesc = umma_idesc_f16(BM, BN);
        for (int kb = 0; kb < nk; kb++) {
            const int st = kb % STAGES;
            mbar_wait(full0 + 8 * st, (kb / STAGES) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint64_t da = umma_desc_sw128(s32(sA + st * A_BYTES)), db = umma_desc_sw128(s32(sB + st * B_BYTES));
#pragma unroll
            for (int k = 0; k < BK / 16; k++) // UMMA_K = 16 fp16 = 32 bytes = +2 in the (addr >> 4) field
                umma_f16(tmem_base, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
            umma_commit(empty0 + 8 * st); // smem slot free once these MMAs have read it
        }
        umma_commit(tmem_full); // accumulator complete
    } else if (warp >= 4) {
        // ===== epilogue: TMEM -> registers -> global (fp32) =====
        mbar_wait(tmem_full, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const int q = warp & 3; // TMEM lane quarter this warp may touch
        const int row = m0 + q * 32 + lane;
        const uint32_t tlane = tmem_base + ((uint32_t)(q * 32) << 16);
        if (MODE == GEMM_GATEUP) {
            __half *C = reinterpret_cast<__half *>(Cv);
#pragma unroll 1
            for (int c0 = 0; c0 < BN / 2; c0 += 32) {
                uint32_t g[32], u[32];
                tmem_ld32(tlane + (uint32_t)c0, g);
                tmem_ld32(tlane + (uint32_t)(BN / 2 + c0), u);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (row < m_valid) {
                    uint4 *dst = reinterpret_cast<uint4 *>(C + (size_t)row * ldc + n0 + c0);
#pragma unroll
                    for (int v = 0; v < 4; v++) {
                        uint32_t w[4];
#pragma unroll
                        for (int e = 0; e < 4; e++) {
                            const float g0 = __uint_as_float(g[8 * v + 2 * e]), g1 = __uint_as_float(g[8 * v + 2 * e + 1]);
                            const float h0 = (g0 / (1.0f + expf(-g0))) * __uint_as_float(u[8 * v + 2 * e]);
                            const float h1 = (g1 / (1.0f + expf(-g1))) * __uint_as_float(u[8 * v + 2 * e + 1]);
                            const __half2 hh = __floats2half2_rn(h0, h1);
                            w[e] = *reinterpret_cast<const uint32_t *>(&hh);
                        }
                        dst[v] = make_uint4(w[0], w[1], w[2], w[3]);
                    }
                }
            }
        } else {
            // FP32 tile -> shared memory (the ring is idle now: every TMA load has landed and every MMA has
            // read it) in the SWIZZLE_128B layout of the C tensor map, then ONE thread hands the four
            // 128 x 32 boxes to TMA: a plain tensor store (QKV) or an f32 reduce-add performed by the memory
            // system (x += A W^T for Wo / W2 -- no read-modify-write through the SM).  Rows past m_valid add 0.
            const int rloc = q * 32 + lane;
#pragma unroll 1
            for (int c = 0; c < BN / 32; c++) {
                uint32_t r[32];
                tmem_ld32(tlane + (uint32_t)(c * 32), r);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                uint8_t *buf = smem + c * (BM * 32 * 4) + rloc * 128;
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    uint4 o = make_uint4(r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
                    if (row >= m_valid) o = make_uint4(0u, 0u, 0u, 0u);
                    *reinterpret_cast<uint4 *>(buf + ((j ^ (rloc & 7)) << 4)) = o;
                }
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            asm volatile("bar.sync 1, 128;" ::: "memory"); // the four epilogue warps
            if (warp == 4 && lane == 0) {
#pragma unroll
                for (int c = 0; c < BN / 32; c++) {
                    const uint32_t src = s32(smem + c * (BM * 32 * 4));
                    if (MODE == GEMM_RESID)
                        asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.bulk_group [%0, {%2, %3}], [%1];" ::"l"(&tma_c), "r"(src),
                                     "r"(n0 + c * 32), "r"(m0)
                                     : "memory");
                    else
                        asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(&tma_c), "r"(src), "r"(n0 + c * 32),
                                     "r"(m0)
                                     : "memory");
                }
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 2) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)BN) : "memory");
}

// =====================================================================================================
// CTA-pair version: two CTAs of a cluster (the two SMs of a TPC) compute one 256 x BN tile with
// tcgen05.mma.cta_group::2.  Each CTA loads ITS 128 rows of A and ITS half of the B tile (BN/2 weight rows),
// so an SM ingests 16 KB + BN/2 * 128 B per 128 x BN x 64 MACs -- twice the arithmetic intensity of the
// single-CTA kernel at BN = 256 (the 128 x 128 tile is bound by the ~64 B/clk an SM can pull from L2).
// Protocol (CUTLASS PipelineTmaUmmaAsync, cutlass/pipeline/sm100_pipeline.hpp): both producers issue
// cta_group::2 TMA loads whose complete_tx lands on the LEADER's full barrier (peer bit cleared); only the
// leader arms it (expect_tx for both CTAs' bytes), waits on it and issues the MMAs; tcgen05.commit with a
// multicast mask frees the stage in both CTAs and finally publishes the accumulator (rows 0-127 in the
// leader's TMEM, 128-255 in the peer's) to both epilogues, which are identical to the single-CTA ones.
// GEMM_GATEUP (persistent kernel below): the leader's half of B is BN/2 rows of W1, the peer's half BN/2 rows of W3.
// =====================================================================================================
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() { // every thread of both CTAs
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tma_load_2d_2sm(uint32_t dst, const CUtensorMap *map, int c0, int c1, uint32_t bar) {
    asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst), "l"(map),
                 "r"(bar & 0xFEFFFFFFu), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void umma_f16_2cta(uint32_t tmem_c, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    const uint32_t z = 0u;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n"
        "}\n" ::"r"(tmem_c),
        "l"(da), "l"(db), "r"(idesc), "r"(accumulate), "r"(z)
        : "memory");
}
__device__ __forceinline__ void umma_commit_2cta(uint32_t bar) { // arrives on the barrier at this offset in BOTH CTAs
    const uint16_t mask = 3;
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"(mask) : "memory");
}

template <int BN, int STAGES> constexpr size_t smem_bytes_2cta() {
    return (size_t)STAGES * (BM * BK * 2 + (BN / 2) * BK * 2) + (2 * STAGES + 1) * 8 + 16 + 1024;
}

// x += A W^T for Wo and W2 (GEMM_RESID), split K over blockIdx.z: every split reduce-adds its partial product into x.
template <int BN, int STAGES>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(256, 1)
    k_gemm_f16_2cta(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b, const __grid_constant__ CUtensorMap tma_c,
                    int m_valid, int K, int kb_per_split) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    constexpr int A_BYTES = BM * BK * 2, B_BYTES = (BN / 2) * BK * 2; // per CTA and stage
    static_assert(BN == 128 || BN == 256 || BN == 512, "TMEM allocations are powers of two");
    static_assert(STAGES * (A_BYTES + B_BYTES) >= BM * BN * 4, "the C tile is staged in the operand ring");
    uint8_t *sA = smem, *sB = smem + STAGES * A_BYTES;
    uint64_t *bars = reinterpret_cast<uint64_t *>(sB + STAGES * B_BYTES);
    const uint32_t full0 = s32(bars), empty0 = s32(bars + STAGES), tmem_full = s32(bars + 2 * STAGES);
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * STAGES + 1);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; s++) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, 1); }
        mbar_init(tmem_full, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) { // the same warp of both CTAs allocates the pair's accumulator columns
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(s32(tmem_slot)), "r"((uint32_t)BN) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    cluster_sync_all(); // barriers of both CTAs initialised before any remote complete_tx / commit can land
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;
    // split-K: blockIdx.z owns k-blocks [kb0, kb0 + nk)
    const int nk_all = (K + BK - 1) / BK, kb0 = blockIdx.z * kb_per_split;
    const int nk = nk_all - kb0 < kb_per_split ? nk_all - kb0 : kb_per_split;
    // rows of this CTA: m0 .. m0 + 127 of the pair tile
    const int m0 = (int)(blockIdx.x >> 1) * (2 * BM) + (int)rank * BM;
    const int n0 = blockIdx.y * BN;

    if (warp == 0 && lane == 0) {
        // ===== TMA producer (both CTAs): own A rows, own half of the B tile =====
        const int brow = n0 + (int)rank * (BN / 2);
        for (int kb = 0; kb < nk; kb++) {
            const int st = kb % STAGES;
            mbar_wait(empty0 + 8 * st, ((kb / STAGES) & 1) ^ 1);
            if (rank == 0) mbar_expect_tx(full0 + 8 * st, 2 * (A_BYTES + B_BYTES));
            tma_load_2d_2sm(s32(sA + st * A_BYTES), &tma_a, (kb0 + kb) * BK, m0, full0 + 8 * st);
            tma_load_2d_2sm(s32(sB + st * B_BYTES), &tma_b, (kb0 + kb) * BK, brow, full0 + 8 * st);
        }
    } else if (warp == 1 && lane == 0 && rank == 0) {
        // ===== MMA issuer: one thread of the leader CTA drives both SMs' tensor cores =====
        constexpr uint32_t idesc = umma_idesc_f16(2 * BM, BN);
        for (int kb = 0; kb < nk; kb++) {
            const int st = kb % STAGES;
            mbar_wait(full0 + 8 * st, (kb / STAGES) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint64_t da = umma_desc_sw128(s32(sA + st * A_BYTES)), db = umma_desc_sw128(s32(sB + st * B_BYTES));
#pragma unroll
            for (int k = 0; k < BK / 16; k++) umma_f16_2cta(tmem_base, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
            umma_commit_2cta(empty0 + 8 * st);
        }
        umma_commit_2cta(tmem_full);
    }
    __syncwarp(); // the elected producer / MMA lanes rejoin their warps
    {
        // ===== epilogue (both CTAs, own 128 rows): all 8 warps -- warp w reads TMEM lanes 32*(w%4).., warps 0-3 take the first
        // half of the columns and warps 4-7 the second =====
        mbar_wait(tmem_full, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const int q = warp & 3, half = warp >> 2;
        const int row = m0 + q * 32 + lane;
        const uint32_t tlane = tmem_base + ((uint32_t)(q * 32) << 16);
        if (m0 < m_valid) { // CTA-uniform: nothing of this tile is stored otherwise
            const int rloc = q * 32 + lane;
#pragma unroll 1
            for (int c = half * (BN / 64); c < (half + 1) * (BN / 64); c++) {
                uint32_t r[32];
                tmem_ld32(tlane + (uint32_t)(c * 32), r);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                uint8_t *buf = smem + c * (BM * 32 * 4) + rloc * 128;
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    uint4 o = make_uint4(r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
                    if (row >= m_valid) o = make_uint4(0u, 0u, 0u, 0u);
                    *reinterpret_cast<uint4 *>(buf + ((j ^ (rloc & 7)) << 4)) = o;
                }
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncthreads();
            if (threadIdx.x == 0) {
#pragma unroll
                for (int c = 0; c < BN / 32; c++) {
                    const uint32_t src = s32(smem + c * (BM * 32 * 4));
                    asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.bulk_group [%0, {%2, %3}], [%1];" ::"l"(&tma_c), "r"(src),
                                 "r"(n0 + c * 32), "r"(m0)
                                 : "memory");
                }
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    cluster_sync_all(); // neither CTA may exit (or free TMEM) while the pair can still touch its shared memory / TMEM
    if (warp == 2) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)BN) : "memory");
}

// =====================================================================================================
// The CTA-pair GEMM as a PERSISTENT kernel (the QKV and gate/up GEMMs).  One cluster per TPC walks tiles t = cluster + i * clusters (M pair tiles fastest, so neighbouring
// clusters share a weight tile in L2); the accumulator is double buffered in TMEM (2 x BN columns), so while the four
// epilogue warps drain tile i the MMA thread already accumulates tile i+1 and the producers are loading tile i+2 --
// prologue, pipeline fill and epilogue no longer sit on the critical path of every tile (they are ~25 % of a K = 4096 tile
// in k_gemm_f16_2cta).  New synchronisation relative to the non-persistent kernel: tmem_full[2] (leader MMA -> both
// epilogues, multicast commit) and tmem_empty[2] on the LEADER (count 8 = 4 epilogue warps x 2 CTAs, remote
// mbarrier.arrive through the cluster window), plus two 16 KB C staging buffers of their own (the operand ring is busy).
// =====================================================================================================
__device__ __forceinline__ void mbar_arrive_leader(uint32_t bar) { // arrive on the barrier at this offset in the pair's even CTA
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(bar & 0xFEFFFFFFu) : "memory");
}

template <int BN, int STAGES> constexpr size_t smem_bytes_2cta_persist() {
    return (size_t)STAGES * (BM * BK * 2 + (BN / 2) * BK * 2) + 2 * (BM * 32 * 4) + (2 * STAGES + 4) * 8 + 16 + 1024;
}

template <int MODE, int BN, int STAGES>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(256, 1)
    k_gemm_f16_2cta_persist(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b, const __grid_constant__ CUtensorMap tma_b2,
                            const __grid_constant__ CUtensorMap tma_c, void *__restrict__ Cv, int ldc, int m_valid, int K, int m_pairs, int n_tiles) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    constexpr int A_BYTES = BM * BK * 2, B_BYTES = (BN / 2) * BK * 2, CST_BYTES = BM * 32 * 4;
    static_assert(2 * BN <= 512, "two accumulators must fit the 512 TMEM columns");
    uint8_t *sA = smem, *sB = smem + STAGES * A_BYTES, *sC = sB + STAGES * B_BYTES; // sC: two staging buffers, 1024-byte aligned
    uint64_t *bars = reinterpret_cast<uint64_t *>(sC + 2 * CST_BYTES);
    const uint32_t full0 = s32(bars), empty0 = s32(bars + STAGES), tfull0 = s32(bars + 2 * STAGES), tempty0 = s32(bars + 2 * STAGES + 2);
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * STAGES + 4);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; s++) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, 1); }
        for (int b = 0; b < 2; b++) { mbar_init(tfull0 + 8 * b, 1); mbar_init(tempty0 + 8 * b, 8); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(s32(tmem_slot)), "r"((uint32_t)(2 * BN)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    cluster_sync_all();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;
    const int nk = (K + BK - 1) / BK;
    const int n_clusters = (int)(gridDim.x >> 1), cid = (int)(blockIdx.x >> 1), total = m_pairs * n_tiles;

    if (warp == 0 && lane == 0) {
        // ===== TMA producer (both CTAs) =====
        const CUtensorMap *bmap = (MODE == GEMM_GATEUP && rank == 1) ? &tma_b2 : &tma_b;
        int it = 0; // running k-block counter across tiles: the ring never drains between tiles
        for (int t = cid; t < total; t += n_clusters) {
            const int mp = t % m_pairs, nt = t / m_pairs;
            const int m0 = mp * 2 * BM + (int)rank * BM;
            const int n0 = nt * (MODE == GEMM_GATEUP ? BN / 2 : BN);
            const int brow = MODE == GEMM_GATEUP ? n0 : n0 + (int)rank * (BN / 2);
            for (int kb = 0; kb < nk; kb++, it++) {
                const int st = it % STAGES;
                mbar_wait(empty0 + 8 * st, ((it / STAGES) & 1) ^ 1);
                if (rank == 0) mbar_expect_tx(full0 + 8 * st, 2 * (A_BYTES + B_BYTES));
                tma_load_2d_2sm(s32(sA + st * A_BYTES), &tma_a, kb * BK, m0, full0 + 8 * st);
                tma_load_2d_2sm(s32(sB + st * B_BYTES), bmap, kb * BK, brow, full0 + 8 * st);
            }
        }
    } else if (warp == 1 && lane == 0 && rank == 0) {
        // ===== MMA issuer (leader): accumulator buffer i & 1 =====
        constexpr uint32_t idesc = umma_idesc_f16(2 * BM, BN);
        int it = 0, i = 0;
        for (int t = cid; t < total; t += n_clusters, i++) {
            const int buf = i & 1;
            mbar_wait(tempty0 + 8 * buf, ((i >> 1) & 1) ^ 1); // both CTAs' epilogues have drained this buffer (first two uses pass at once)
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            for (int kb = 0; kb < nk; kb++, it++) {
                const int st = it % STAGES;
                mbar_wait(full0 + 8 * st, (it / STAGES) & 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint64_t da = umma_desc_sw128(s32(sA + st * A_BYTES)), db = umma_desc_sw128(s32(sB + st * B_BYTES));
#pragma unroll
                for (int k = 0; k < BK / 16; k++) umma_f16_2cta(tmem_base + (uint32_t)(buf * BN), da + 2 * k, db + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
                umma_commit_2cta(empty0 + 8 * st);
            }
            umma_commit_2cta(tfull0 + 8 * buf);
        }
    } else if (warp >= 4) {
        // ===== epilogue (both CTAs): four warps, warp w owns TMEM lanes 32 * (w - 4) =====
        const int q = warp & 3, et = threadIdx.x - 128; // et: 0..127 within the epilogue group
        int i = 0, chunk = 0;                         // chunk: running count of staged 32-column chunks (staging buffer = chunk & 1)
        for (int t = cid; t < total; t += n_clusters, i++) {
            const int buf = i & 1;
            const int mp = t % m_pairs, nt = t / m_pairs;
            const int m0 = mp * 2 * BM + (int)rank * BM;
            const int n0 = nt * (MODE == GEMM_GATEUP ? BN / 2 : BN);
            const int row = m0 + q * 32 + lane;
            mbar_wait(tfull0 + 8 * buf, (i >> 1) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t tlane = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * BN);
            if (MODE == GEMM_GATEUP) {
                __half *C = reinterpret_cast<__half *>(Cv);
#pragma unroll 1
                for (int c0 = 0; c0 < BN / 2; c0 += 32) {
                    uint32_t g[32], u[32];
                    tmem_ld32(tlane + (uint32_t)c0, g);
                    tmem_ld32(tlane + (uint32_t)(BN / 2 + c0), u);
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                    if (c0 + 32 >= BN / 2) { // last TMEM read of this tile: hand the accumulator back before the (slow) stores
                        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                        __syncwarp();
                        if (lane == 0) mbar_arrive_leader(tempty0 + 8 * buf);
                    }
                    if (row < m_valid) {
                        uint4 *dst = reinterpret_cast<uint4 *>(C + (size_t)row * ldc + n0 + c0);
#pragma unroll
                        for (int v = 0; v < 4; v++) {
                            uint32_t w[4];
#pragma unroll
                            for (int e = 0; e < 4; e++) {
                                const float g0 = __uint_as_float(g[8 * v + 2 * e]), g1 = __uint_as_float(g[8 * v + 2 * e + 1]);
                                const float h0 = (g0 / (1.0f + expf(-g0))) * __uint_as_float(u[8 * v + 2 * e]);
                                const float h1 = (g1 / (1.0f + expf(-g1))) * __uint_as_float(u[8 * v + 2 * e + 1]);
                                const __half2 hh = __floats2half2_rn(h0, h1);
                                w[e] = *reinterpret_cast<const uint32_t *>(&hh);
                            }
                            dst[v] = make_uint4(w[0], w[1], w[2], w[3]);
                        }
                    }
                }
            } else {
                const int rloc = q * 32 + lane;
#pragma unroll 1
                for (int c = 0; c < BN / 32; c++, chunk++) {
                    uint32_t r[32];
                    tmem_ld32(tlane + (uint32_t)(c * 32), r);
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                    if (c == BN / 32 - 1) {
                        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                        __syncwarp();
                        if (lane == 0) mbar_arrive_leader(tempty0 + 8 * buf);
                    }
                    uint8_t *cst = sC + (chunk & 1) * CST_BYTES;
                    if (et == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); // the store that used this buffer two chunks ago has read it
                    asm volatile("bar.sync 2, 128;" ::: "memory");
                    uint8_t *dstp = cst + rloc * 128;
#pragma unroll
                    for (int j = 0; j < 8; j++) {
                        uint4 o = make_uint4(r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
                        if (row >= m_valid) o = make_uint4(0u, 0u, 0u, 0u);
                        *reinterpret_cast<uint4 *>(dstp + ((j ^ (rloc & 7)) << 4)) = o;
                    }
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    asm volatile("bar.sync 2, 128;" ::: "memory");
                    if (et == 0) {
                        asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(&tma_c), "r"(s32(cst)),
                                     "r"(n0 + c * 32), "r"(m0)
                                     : "memory");
                        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    }
                }
            }
        }
        if (et == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    }
    __syncwarp(); // the elected producer / MMA / store lanes rejoin their warps before the aligned cluster barrier
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    cluster_sync_all();
    if (warp == 2) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)(2 * BN)) : "memory");
}

// ---- host side ----
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                                  const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr) == cudaSuccess && qr == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

// [rows][K] fp16 row-major, box = {BK (inner, 128 bytes), box_rows}, 128-byte swizzle
inline int make_map(CUtensorMap *map, const void *base, uint64_t rows, uint64_t K, uint32_t box_rows) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) return -1;
    cuuint64_t dims[2] = {K, rows};
    cuuint64_t strides[1] = {K * 2};
    cuuint32_t box[2] = {(cuuint32_t)BK, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void *>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : -2;
}

// C / x as [rows][cols] fp32 row-major, box = 32 columns (128 bytes) x 128 rows, 128-byte swizzle (matches the epilogue's staging)
inline int make_map_c(CUtensorMap *map, const void *base, uint64_t rows, uint64_t cols) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) return -1;
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {cols * 4};
    cuuint32_t box[2] = {32, (cuuint32_t)BM};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void *>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : -2;
}

template <int MODE, int STAGES>
inline int gemm_launch(const CUtensorMap &a, const CUtensorMap &b, const CUtensorMap &b2, const CUtensorMap &c, void *C, int ldc, int m_valid, int m_tiles,
                       int n_tiles, int K, cudaStream_t stream) {
    static bool attr = false; // one flag per instantiation
    if (!attr) {
        if (cudaFuncSetAttribute(k_gemm_f16_tcgen05<MODE, STAGES>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes<STAGES>()) != cudaSuccess) return -4;
        attr = true;
    }
    k_gemm_f16_tcgen05<MODE, STAGES><<<dim3(m_tiles, n_tiles), 256, smem_bytes<STAGES>(), stream>>>(a, b, b2, c, C, ldc, m_valid, K);
    return cudaGetLastError() == cudaSuccess ? 0 : -5;
}

// x += A W^T through the CTA-pair kernel, K split `splits` ways.  m_tiles = 128-row tiles of M, even (M padded to 256).
// B maps must have box rows = BN / 2.
template <int BN, int STAGES>
inline int gemm2_launch(const CUtensorMap &a, const CUtensorMap &b, const CUtensorMap &c, int m_valid, int m_tiles, int n_tiles, int K, cudaStream_t stream,
                        int splits = 1) {
    static bool attr = false;
    if (!attr) {
        if (cudaFuncSetAttribute(k_gemm_f16_2cta<BN, STAGES>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes_2cta<BN, STAGES>()) != cudaSuccess)
            return -4;
        attr = true;
    }
    if (m_tiles % 2 || splits < 1) return -6;
    const int nk = (K + BK - 1) / BK, per = (nk + splits - 1) / splits;
    if ((splits - 1) * per >= nk) return -6; // an empty split would publish an unwritten accumulator
    k_gemm_f16_2cta<BN, STAGES><<<dim3(m_tiles, n_tiles, splits), 256, smem_bytes_2cta<BN, STAGES>(), stream>>>(a, b, c, m_valid, K, per);
    return cudaGetLastError() == cudaSuccess ? 0 : -5;
}
constexpr int GEMM2_STAGES_256 = 6; // 192 KB of operand ring per CTA

// Persistent variant (GEMM_F32, GEMM_GATEUP).  n_sms: SMs of the device; the grid is the largest even number of CTAs <= n_sms.
template <int MODE, int BN, int STAGES>
inline int gemm2_persist_launch(const CUtensorMap &a, const CUtensorMap &b, const CUtensorMap &b2, const CUtensorMap &c, void *C, int ldc, int m_valid, int m_tiles,
                                int n_tiles, int K, int n_sms, cudaStream_t stream) {
    static_assert(MODE != GEMM_RESID, "the residual GEMMs run on k_gemm_f16_2cta");
    static bool attr = false;
    if (!attr) {
        if (cudaFuncSetAttribute(k_gemm_f16_2cta_persist<MODE, BN, STAGES>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes_2cta_persist<BN, STAGES>()) !=
            cudaSuccess)
            return -4;
        attr = true;
    }
    if (m_tiles & 1) return -6;
    const int m_pairs = m_tiles / 2, total = m_pairs * n_tiles;
    int clusters = n_sms / 2;
    if (clusters > total) clusters = total;
    if (clusters < 1) return -6;
    k_gemm_f16_2cta_persist<MODE, BN, STAGES><<<dim3(2 * clusters), 256, smem_bytes_2cta_persist<BN, STAGES>(), stream>>>(a, b, b2, c, C, ldc, m_valid, K, m_pairs, n_tiles);
    return cudaGetLastError() == cudaSuccess ? 0 : -5;
}
constexpr int GEMM2_PERSIST_STAGES_256 = 5; // 5 x 32 KB of operands + 2 x 16 KB of C staging

// 3 stages of 32 KB: two CTAs fit one SM (2 x 99 KB shared memory, 2 x 128 TMEM columns), so one CTA's
// epilogue overlaps the other's main loop.
constexpr int GEMM_STAGES = 3, GEMM_STAGES_DEEP = 6;

// Test/measurement entry: C[M,N] (+)= A[M,K] * B[N,K]^T ; M, N multiples of 128, K multiple of 64.  Device pointers.
// The kernels of the prefill: two_cta = 0: single-CTA F32 (resid = 0) or residual GEMM at `stages` = 3 or 6 (0 = 3);
// two_cta = 256: the CTA-pair residual GEMM split `resid` ways over K; two_cta = 1256: the persistent CTA-pair F32 GEMM.
inline int gemm_f16(const __half *A, const __half *B, float *C, int M, int N, int K, int stages, int resid, int two_cta, cudaStream_t stream) {
    if (M % BM || N % BN || K % BK) return -3;
    CUtensorMap ma, mb, mc;
    int rc;
    if (two_cta) { // 256-wide pair tiles
        if (M % 256 || N % 256) return -3;
        if ((rc = make_map(&ma, A, (uint64_t)M, (uint64_t)K, BM))) return rc;
        if ((rc = make_map(&mb, B, (uint64_t)N, (uint64_t)K, 128))) return rc;
        if ((rc = make_map_c(&mc, C, (uint64_t)M, (uint64_t)N))) return rc;
        if (resid) return gemm2_launch<256, GEMM2_STAGES_256>(ma, mb, mc, M, M / BM, N / 256, K, stream, resid);
        int dev = 0, sms = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        return gemm2_persist_launch<GEMM_F32, 256, GEMM2_PERSIST_STAGES_256>(ma, mb, mb, mc, C, N, M, M / BM, N / 256, K, sms, stream);
    }
    if ((rc = make_map(&ma, A, (uint64_t)M, (uint64_t)K, BM))) return rc;
    if ((rc = make_map(&mb, B, (uint64_t)N, (uint64_t)K, BN))) return rc;
    if ((rc = make_map_c(&mc, C, (uint64_t)M, (uint64_t)N))) return rc;
    if (resid && stages == 6) return gemm_launch<GEMM_RESID, 6>(ma, mb, mb, mc, C, N, M, M / BM, N / BN, K, stream);
    if (resid) return gemm_launch<GEMM_RESID, GEMM_STAGES>(ma, mb, mb, mc, C, N, M, M / BM, N / BN, K, stream);
    if (stages == 6) return gemm_launch<GEMM_F32, 6>(ma, mb, mb, mc, C, N, M, M / BM, N / BN, K, stream);
    return gemm_launch<GEMM_F32, GEMM_STAGES>(ma, mb, mb, mc, C, N, M, M / BM, N / BN, K, stream);
}

} // namespace pg
