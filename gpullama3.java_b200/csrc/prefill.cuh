// prefill.cuh -- batched prefill (--batch-prefill-size N) on the tensor cores.
//
// One chunk of n <= B prompt tokens at positions start .. start+n-1 goes through every layer as GEMMs
// (prefill_gemm.cuh: TMA + tcgen05.mma, FP32 accumulation in TMEM) instead of n matvec passes:
//
//   X[n][dim] <- embedding rows                                      k_pf_embed
//   per layer:  A16 <- f16(rmsnorm(X) * w)                            k_pf_rmsnorm_f16   (batchedRmsReduce + batchedRmsApplyFP16)
//               QKV <- A16 * [Wq;Wk;Wv]^T                             GEMM_F32           (gemmMMAQKV)
//               q,k <- (Qwen3: per-head RMSNorm) RoPE; k,v -> cache   k_pf_rope_kv       (batchedRopeWithKVCachePacked)
//               ATT16 <- causal softmax(q k^T / sqrt(hs)) v           k_pf_attention_mma (batchedFlashAttentionFP16Out)
//               X += ATT16 * Wo^T                                     GEMM_RESID         (gemmMMA + residual)
//               A16 <- f16(rmsnorm(X) * w)
//               H16 <- f16(silu(A16 W1^T) * (A16 W3^T))               GEMM_GATEUP        (gemmMMAGateUp + batchedFFNSwiGLUFP16Packed)
//               X += H16 * W2^T                                       GEMM_RESID         (gemmMMA + batchedResidualAddFP32)
//   no logits (InferenceCoreBatchPrefillDecode.java:166-167): the product of prefill is the KV cache.
//
// Task list mirrored from LlamaFP16LayersBatchPrefillMMA.java:84-219 / TransformerBatchPrefillKernels.java.
// Numerics: activations are rounded to FP16 before each GEMM (as the reference's tensor-core path does),
// so the KV cache agrees with the exact CPU path to FP16 tolerance, not bit for bit; the exact
// token-by-token path stays available (b200_set_prefill_mode).
#pragma once
#include "../../include/b200llama.h"
#include "decode_kernels.cuh"
#include "prefill_gemm.cuh"
#include <vector>

struct PrefillLayerMaps {
    CUtensorMap qkv, wo, w1, w3, w2; // weight boxes of 128 rows; w1 / w3: 128 on CTA pairs, 64 on single CTAs (gate/up tile 64 + 64)
};

struct PrefillCtx {
    int batch = 0, bpad = 0;
    bool ready = false; // tensor-core path usable for this plan
    int mode = 0;       // 0 = exact token-by-token graph, 1 = tensor-core GEMMs
    bool pair = true;      // CTA-pair (cta_group::2) GEMMs; single-CTA ones for shapes the 256-wide pair tiles do not divide
    float *X = nullptr, *QKV = nullptr;
    __half *A16 = nullptr, *ATT16 = nullptr, *H16 = nullptr;
    int *tok = nullptr;
    __half *KH = nullptr, *VH = nullptr; // f16 K / V rows [0, start+n) of the layer in flight
    CUtensorMap mA, mATT, mH; // GEMM A operands (f16 activations)
    CUtensorMap mX, mQKV;     // GEMM outputs written by TMA (f32)
    std::vector<PrefillLayerMaps> maps;
    const char *why = "the plan was created without a prefill batch size (prefill_batch_size <= 1)";
};

// ---- elementwise kernels ------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_pf_embed(const int *__restrict__ tok, DevMat emb, float *__restrict__ X, int dim) {
    const int b = blockIdx.x, token = tok[b];
    for (int i = threadIdx.x; i < dim; i += 256) X[(size_t)b * dim + i] = emb_get(emb, token, i);
}

__device__ __forceinline__ float pf_block_sum(float v, float *red) { // blockDim.x multiple of 32, <= 256
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) red[warp] = v;
    __syncthreads();
    float t = 0.0f;
    for (int w = 0; w < nw; w++) t += red[w];
    __syncthreads();
    return t;
}

// out16[b][i] = f16(w[i] * (rsqrt(mean(x^2) + eps) * x[b][i]))
__global__ void __launch_bounds__(256) k_pf_rmsnorm_f16(const float *__restrict__ X, const float *__restrict__ w, float eps, int dim, __half *__restrict__ out) {
    __shared__ float red[8];
    const float *x = X + (size_t)blockIdx.x * dim;
    float ss = 0.0f;
    for (int i = threadIdx.x * 4; i < dim; i += 1024) {
        const float4 v = *reinterpret_cast<const float4 *>(x + i);
        ss += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
    }
    ss = pf_block_sum(ss, red);
    const float sc = (float)(1.0 / sqrt((double)(ss / (float)dim + eps)));
    __half *o = out + (size_t)blockIdx.x * dim;
    for (int i = threadIdx.x * 4; i < dim; i += 1024) {
        const float4 v = *reinterpret_cast<const float4 *>(x + i);
        const float4 g = *reinterpret_cast<const float4 *>(w + i);
        const __half2 a = __floats2half2_rn(g.x * (sc * v.x), g.y * (sc * v.y)), c = __floats2half2_rn(g.z * (sc * v.z), g.w * (sc * v.w));
        uint2 pk;
        pk.x = *reinterpret_cast<const uint32_t *>(&a);
        pk.y = *reinterpret_cast<const uint32_t *>(&c);
        *reinterpret_cast<uint2 *>(o + i) = pk;
    }
}

// One CTA per token, one warp per head at a time.  Llama rotates interleaved pairs (InferenceCore.java:75-87);
// Qwen3 normalises the head, then rotates NeoX pairs (:594-619).  q is rotated in place; k and v go to the
// FP32 KV cache (what decode reads) and, as f16, to the per-layer scratch the attention kernel streams.
template <int HS>
__global__ void __launch_bounds__(256) k_pf_rope_kv(float *__restrict__ qkv, int ldq, float *__restrict__ kc, float *__restrict__ vc, __half *__restrict__ kh,
                                                   __half *__restrict__ vh, int kvd, int n_heads, int n_kv_heads, int arch, const float *__restrict__ qnw,
                                                   const float *__restrict__ knw, float eps, const float *__restrict__ cr, const float *__restrict__ ci,
                                                   int start_pos) {
    constexpr int HALF = HS / 2, PPL = HALF / 32; // pairs per lane
    const int b = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5, pos = start_pos + b;
    const int qd = n_heads * HS;
    for (int hh = warp; hh < n_heads + n_kv_heads; hh += 8) {
        const bool is_q = hh < n_heads;
        const int kvh = hh - n_heads;
        float *src = qkv + (size_t)b * ldq + (is_q ? hh * HS : qd + kvh * HS);
        float v0[PPL], v1[PPL];
        int i0[PPL], i1[PPL];
        float ss = 0.0f;
#pragma unroll
        for (int u = 0; u < PPL; u++) {
            const int p = lane + 32 * u;
            if (arch & KF_NEOX) { i0[u] = p; i1[u] = p + HALF; } else { i0[u] = 2 * p; i1[u] = 2 * p + 1; }
            v0[u] = src[i0[u]];
            v1[u] = src[i1[u]];
            ss += v0[u] * v0[u] + v1[u] * v1[u];
        }
        if (arch & KF_QKNORM) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
            const float sc = (float)(1.0 / sqrt((double)(ss / (float)HS + eps)));
            const float *nw = is_q ? qnw : knw;
#pragma unroll
            for (int u = 0; u < PPL; u++) { v0[u] = nw[i0[u]] * (sc * v0[u]); v1[u] = nw[i1[u]] * (sc * v1[u]); }
        }
#pragma unroll
        for (int u = 0; u < PPL; u++) {
            const int p = lane + 32 * u;
            const float fcr = cr[(size_t)pos * HALF + p], fci = ci[(size_t)pos * HALF + p];
            const float r0 = v0[u] * fcr - v1[u] * fci, r1 = v0[u] * fci + v1[u] * fcr;
            if (is_q) {
                src[i0[u]] = r0;
                src[i1[u]] = r1;
            } else {
                const size_t o = (size_t)pos * kvd + kvh * HS;
                const float *vsrc = qkv + (size_t)b * ldq + qd + kvd + kvh * HS;
                const float w0 = vsrc[i0[u]], w1 = vsrc[i1[u]];
                kc[o + i0[u]] = r0; kc[o + i1[u]] = r1;
                vc[o + i0[u]] = w0; vc[o + i1[u]] = w1;
                kh[o + i0[u]] = __float2half_rn(r0); kh[o + i1[u]] = __float2half_rn(r1);
                vh[o + i0[u]] = __float2half_rn(w0); vh[o + i1[u]] = __float2half_rn(w1);
            }
        }
    }
}

// f16 copies of cache rows written before this chunk (start_pos > 0): rows [0, rows) of one layer
__global__ void __launch_bounds__(256) k_pf_kv_to_f16(const float *__restrict__ kc, const float *__restrict__ vc, __half *__restrict__ kh, __half *__restrict__ vh,
                                                     size_t n4) {
    for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < n4; i += (size_t)gridDim.x * 256) {
        const float4 a = reinterpret_cast<const float4 *>(kc)[i], c = reinterpret_cast<const float4 *>(vc)[i];
        const __half2 a0 = __floats2half2_rn(a.x, a.y), a1 = __floats2half2_rn(a.z, a.w), c0 = __floats2half2_rn(c.x, c.y), c1 = __floats2half2_rn(c.z, c.w);
        uint2 pk;
        pk.x = *reinterpret_cast<const uint32_t *>(&a0); pk.y = *reinterpret_cast<const uint32_t *>(&a1);
        reinterpret_cast<uint2 *>(kh)[i] = pk;
        pk.x = *reinterpret_cast<const uint32_t *>(&c0); pk.y = *reinterpret_cast<const uint32_t *>(&c1);
        reinterpret_cast<uint2 *>(vh)[i] = pk;
    }
}

// ---- causal attention over the chunk + everything already in the cache, on the warp-level tensor cores ----
// FlashAttention-2 layout with mma.sync.m16n8k16 (f16 operands, f32 accumulation): CTA = one KV head x 64
// query rows (4 warps x 16 rows), key tiles of 64.  Q (pre-scaled), K and V are converted to f16 on their
// way into shared memory; S = Q K^T stays in registers, its accumulator layout is re-used directly as the
// A operand of P V, and V's B fragments come from ldmatrix.trans.  This op is 1 % of the prefill FLOPs
// (0.07 of 7.2 TFLOP at pp512); the GEMMs that carry the rest run on tcgen05.
constexpr int PM_THREADS = 128, PM_ROWS = 64, PM_KT = 64;
template <int HS> constexpr size_t pm_smem_bytes() { return (size_t)5 * PM_ROWS * (HS + 8) * 2; } // Q + 2 x (K, V)

__device__ __forceinline__ void mma_f16_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ float ex2_approx(float x) { // 2^x on the SFU (ex2(-inf) = 0)
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ uint32_t pack_h2(float lo, float hi) {
    const __half2 h = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<const uint32_t *>(&h);
}

template <int HS>
__global__ void __launch_bounds__(PM_THREADS) k_pf_attention_mma(const float *__restrict__ qkv, int ldq, const __half *__restrict__ kh, const __half *__restrict__ vh,
                                                                int kvd, int kv_mul, int n, int start_pos, float inv_sqrt_hs, __half *__restrict__ out, int ldo) {
    extern __shared__ __align__(16) unsigned char pm_sm[];
    constexpr int RP = HS + 8, H4 = HS / 4, KS = HS / 16, NB = HS / 8; // row pitch (halves): 16 B of padding keeps fragment loads conflict-free
    __half *sQ = reinterpret_cast<__half *>(pm_sm), *sKV = sQ + PM_ROWS * RP; // stage s: K at sKV + s*2*64*RP, V right after it
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
    const int QT = PM_ROWS / kv_mul, q0 = ((int)gridDim.x - 1 - (int)blockIdx.x) * QT, grp = blockIdx.y; // longest (latest) query tiles first
    const int q_end = (q0 + QT < n ? q0 + QT : n), nkeys = start_pos + q_end, ntiles = (nkeys + PM_KT - 1) / PM_KT;
    const uint32_t sKV_addr = (uint32_t)__cvta_generic_to_shared(sKV);
    // K/V tile -> shared memory with cp.async (16 bytes per request, rows past nkeys zero-filled), double buffered
    constexpr int C8 = HS / 8, JSTEP = PM_THREADS / C8; // 16-byte chunks per row; rows covered by one pass of the CTA
    const int lc8 = tid % C8, lj0 = tid / C8;
    const size_t gcol = (size_t)grp * HS + lc8 * 8;
    const uint32_t ldst0 = sKV_addr + (uint32_t)((lj0 * RP + lc8 * 8) * 2);
    auto load_tile = [&](int it) {
        uint32_t d = ldst0 + (uint32_t)((it & 1) * 2 * PM_KT * RP * 2);
        int tk = it * PM_KT + lj0;
#pragma unroll
        for (int i = 0; i < PM_KT / JSTEP; i++, tk += JSTEP, d += (uint32_t)(JSTEP * RP * 2)) {
            const int ok = tk < nkeys ? 16 : 0;
            const size_t goff = (size_t)(ok ? tk : 0) * kvd + gcol;
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(kh + goff), "r"(ok) : "memory");
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d + (uint32_t)(PM_KT * RP * 2)), "l"(vh + goff), "r"(ok) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    if (ntiles > 0) load_tile(0);

    const float qscale = inv_sqrt_hs * 1.4426950408889634f;
    for (int idx = tid; idx < PM_ROWS * H4; idx += PM_THREADS) {
        const int r = idx / H4, d4 = idx % H4, b = q0 + r / kv_mul, h = grp * kv_mul + r % kv_mul;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (b < n) v = *reinterpret_cast<const float4 *>(qkv + (size_t)b * ldq + h * HS + d4 * 4);
        uint2 pk;
        pk.x = pack_h2(v.x * qscale, v.y * qscale); // scores come out in units of log2: softmax below uses ex2
        pk.y = pack_h2(v.z * qscale, v.w * qscale);
        *reinterpret_cast<uint2 *>(sQ + r * RP + d4 * 4) = pk;
    }
    __syncthreads();
    uint32_t qf[KS][4];
    {
        const __half *base = sQ + (warp * 16 + g) * RP + 2 * t;
#pragma unroll
        for (int kk = 0; kk < KS; kk++) {
            qf[kk][0] = *reinterpret_cast<const uint32_t *>(base + kk * 16);
            qf[kk][1] = *reinterpret_cast<const uint32_t *>(base + 8 * RP + kk * 16);
            qf[kk][2] = *reinterpret_cast<const uint32_t *>(base + kk * 16 + 8);
            qf[kk][3] = *reinterpret_cast<const uint32_t *>(base + 8 * RP + kk * 16 + 8);
        }
    }
    float o[NB][4];
#pragma unroll
    for (int nb = 0; nb < NB; nb++) o[nb][0] = o[nb][1] = o[nb][2] = o[nb][3] = 0.0f;
    float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.0f, l1 = 0.0f;
    const int row0 = warp * 16 + g, row1 = row0 + 8;
    const int tb0 = q0 + row0 / kv_mul, tb1 = q0 + row1 / kv_mul;
    const int qpos0 = tb0 < n ? start_pos + tb0 : -1, qpos1 = tb1 < n ? start_pos + tb1 : -1; // -1: every key masked
    // smallest position among this warp's 16 rows (-1 when the warp holds padding rows): tiles entirely at or before it need no mask
    const int wlast_tok = q0 + (warp * 16 + 15) / kv_mul;
    const int wmin_pos = wlast_tok < n ? start_pos + q0 + (warp * 16) / kv_mul : -1;

#pragma unroll 1
    for (int it = 0; it < ntiles; it++) {
        const int k0 = it * PM_KT;
        if (it + 1 < ntiles) {
            load_tile(it + 1); // the buffer it overwrites was released by the barrier that ended iteration it-1
            asm volatile("cp.async.wait_group 1;" ::: "memory");
        } else {
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        __syncthreads();
        const uint32_t sK_addr = sKV_addr + (uint32_t)((it & 1) * 2 * PM_KT * RP * 2);
        const uint32_t sV_addr = sKV_addr + (uint32_t)(((it & 1) * 2 + 1) * PM_KT * RP * 2);
        float s[8][4];
#pragma unroll
        for (int nb = 0; nb < 8; nb++) s[nb][0] = s[nb][1] = s[nb][2] = s[nb][3] = 0.0f;
        {
            // four 8x8 blocks of K per ldmatrix: (keys nb*8.., d kk*16..), (same keys, d+8), (keys (nb+1)*8.., d), (.., d+8)
            const uint32_t kaddr0 = sK_addr + (uint32_t)((((lane & 7) + ((lane >> 4) << 3)) * RP + (((lane >> 3) & 1) << 3)) * 2);
#pragma unroll
            for (int kk = 0; kk < KS; kk++)
#pragma unroll
                for (int nb = 0; nb < 8; nb += 2) {
                    uint32_t b0, b1, b2, b3;
                    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                                 : "=r"(b0), "=r"(b1), "=r"(b2), "=r"(b3)
                                 : "r"(kaddr0 + (uint32_t)((nb * 8 * RP + kk * 16) * 2)));
                    mma_f16_16816(s[nb], qf[kk], b0, b1);
                    mma_f16_16816(s[nb + 1], qf[kk], b2, b3);
                }
        }
        float mx0 = -INFINITY, mx1 = -INFINITY;
        if (k0 + PM_KT - 1 > wmin_pos) { // warp-uniform: some key of this tile is ahead of some row of this warp (or a row is padding)
#pragma unroll
            for (int nb = 0; nb < 8; nb++) {
                const int key = k0 + nb * 8 + 2 * t;
                if (key > qpos0) s[nb][0] = -INFINITY;
                if (key + 1 > qpos0) s[nb][1] = -INFINITY;
                if (key > qpos1) s[nb][2] = -INFINITY;
                if (key + 1 > qpos1) s[nb][3] = -INFINITY;
            }
        }
#pragma unroll
        for (int nb = 0; nb < 8; nb++) {
            mx0 = fmaxf(mx0, fmaxf(s[nb][0], s[nb][1]));
            mx1 = fmaxf(mx1, fmaxf(s[nb][2], s[nb][3]));
        }
        mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
        mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
        const float mn0 = fmaxf(m0, mx0), mn1 = fmaxf(m1, mx1);
        // a row with nothing visible yet keeps m = -inf: use 0 as the reference so that ex2(-inf - 0) = 0 and alpha = ex2(-inf) = 0 on l = 0
        const float r0 = mn0 == -INFINITY ? 0.0f : mn0, r1 = mn1 == -INFINITY ? 0.0f : mn1;
        const float al0 = ex2_approx(m0 - r0), al1 = ex2_approx(m1 - r1);
        float sum0 = 0.0f, sum1 = 0.0f;
#pragma unroll
        for (int nb = 0; nb < 8; nb++) {
            s[nb][0] = ex2_approx(s[nb][0] - r0);
            s[nb][1] = ex2_approx(s[nb][1] - r0);
            s[nb][2] = ex2_approx(s[nb][2] - r1);
            s[nb][3] = ex2_approx(s[nb][3] - r1);
            sum0 += s[nb][0] + s[nb][1];
            sum1 += s[nb][2] + s[nb][3];
        }
        sum0 += __shfl_xor_sync(0xffffffffu, sum0, 1); sum0 += __shfl_xor_sync(0xffffffffu, sum0, 2);
        sum1 += __shfl_xor_sync(0xffffffffu, sum1, 1); sum1 += __shfl_xor_sync(0xffffffffu, sum1, 2);
        l0 = l0 * al0 + sum0; l1 = l1 * al1 + sum1;
        m0 = mn0; m1 = mn1;
#pragma unroll
        for (int nb = 0; nb < NB; nb++) { o[nb][0] *= al0; o[nb][1] *= al0; o[nb][2] *= al1; o[nb][3] *= al1; }
#pragma unroll
        for (int ks = 0; ks < PM_KT / 16; ks++) {
            uint32_t pa[4];
            pa[0] = pack_h2(s[2 * ks][0], s[2 * ks][1]);
            pa[1] = pack_h2(s[2 * ks][2], s[2 * ks][3]);
            pa[2] = pack_h2(s[2 * ks + 1][0], s[2 * ks + 1][1]);
            pa[3] = pack_h2(s[2 * ks + 1][2], s[2 * ks + 1][3]);
#pragma unroll
            for (int nb = 0; nb < NB; nb += 2) {
                // four 8x8 blocks of V (keys ks*16 .. +15, columns nb*8 .. +15), transposed on the way into registers
                const uint32_t addr = sV_addr + (uint32_t)(((ks * 16 + (lane & 15)) * RP + nb * 8 + ((lane >> 4) << 3)) * 2);
                uint32_t b0, b1, b2, b3;
                asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(b0), "=r"(b1), "=r"(b2), "=r"(b3) : "r"(addr));
                mma_f16_16816(o[nb], pa, b0, b1);
                mma_f16_16816(o[nb + 1], pa, b2, b3);
            }
        }
        __syncthreads(); // every warp is done with this stage before the next iteration's prefetch overwrites it
    }
    const float inv0 = l0 > 0.0f ? 1.0f / l0 : 0.0f, inv1 = l1 > 0.0f ? 1.0f / l1 : 0.0f;
    if (tb0 < n) {
        __half *op = out + (size_t)tb0 * ldo + (grp * kv_mul + row0 % kv_mul) * HS + 2 * t;
#pragma unroll
        for (int nb = 0; nb < NB; nb++) *reinterpret_cast<uint32_t *>(op + nb * 8) = pack_h2(o[nb][0] * inv0, o[nb][1] * inv0);
    }
    if (tb1 < n) {
        __half *op = out + (size_t)tb1 * ldo + (grp * kv_mul + row1 % kv_mul) * HS + 2 * t;
#pragma unroll
        for (int nb = 0; nb < NB; nb++) *reinterpret_cast<uint32_t *>(op + nb * 8) = pack_h2(o[nb][2] * inv1, o[nb][3] * inv1);
    }
}

inline void prefill_free(PrefillCtx &) {} // device buffers are owned by the plan's allocation list
