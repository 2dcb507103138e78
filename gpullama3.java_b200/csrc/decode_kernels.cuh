// decode_kernels.cuh -- single-token decode kernels (Q8_0 and FP16 weights), bit-exact with the
// reference's CPU path.  One CUDA graph strings them together per token (plan.cu).
//
// Replaces (reference kernel inventory, SURVEY.md 2.K):
//   k_rmsnorm_quant  <- reductionOneBlockWithLayer + reductionOneBlock2WithLayer / mapContextWithQuantize
//                       (TransformerComputeKernelsLayered.java:387-454) + convertQ8_0toFP32 embedding
//   k_matvec_q8      <- fusedQKVMatmulQ8 / matrixVectorGenericWithResidualQ8_0Byte / matrixVectorGenericQ8Byte
//                       (TransformerComputeKernelsLayered.java:3038-3223, 2888-2906, 2773-2787)
//   k_gateup_q8      <- fullyFusedRmsNormFFNGateUpQ8 (:3386-3549)
//   k_rope_kv        <- ropeRotationWithCacheCopy (:495-542), Qwen3 fusedQKRmsNorm + NeoX rope (Qwen3Kernels.java:302-361,973-1064)
//   k_attention      <- processHeadsFlashAttention (:784-906)
//   k_argmax_advance <- argmaxLogits (TransformerComputeKernels.java:25-56), with CPU tie-break semantics
// but the arithmetic they implement is the CPU path's (InferenceCore.java:50-172, 565-697).
#pragma once
#include "common.cuh"
#include "seqsum2.cuh"

enum { MODE_STORE = 0, MODE_RESID = 1 };

// ------------------------------------------------------------------------------------------
// Embedding row lookup: FloatTensor.copyTo -> getFloat per element (InferenceCore.java:61).
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float emb_get(const DevMat &e, int token, int i) {
    size_t idx = (size_t)token * e.cols + i;
    if (e.type == 8) { // Q8_0FloatTensor.getFloat: quant * scale (Q8_0FloatTensor.java:55-63)
        float q = (float)((const int8_t *)e.qs)[idx];
        return __fmul_rn(q, __half2float(e.sc[idx >> 5]));
    } else if (e.type == 1) { // FP16FloatTensor.getFloat: Float.float16ToFloat (IEEE, subnormals kept)
        return __half2float(((const __half *)e.qs)[idx]);
    }
    return ((const float *)e.qs)[idx];
}

// ------------------------------------------------------------------------------------------
// RMSNorm (+ optional embedding gather, + Q8_0 activation quantisation).
// InferenceCore.rmsnorm (InferenceCore.java:39-48): ss = sequential float sum of x*x;
// ss = ss/size + eps; ss = (float)(1.0/Math.sqrt(ss)); out = w * (ss * x).
// The sum is order-sensitive, so one thread walks it (squares precomputed in parallel).
// One CTA.  Outputs: xq/xs (Q8_0 activation for the following matvec) and/or xb (float).
// ------------------------------------------------------------------------------------------
#define NORM_THREADS SEQSUM2_THREADS
__host__ __device__ inline int norm_padded(int dim) { return (dim + SEQSUM2_THREADS - 1) / SEQSUM2_THREADS * SEQSUM2_THREADS; }
// squares (padded to whole thread chunks) | the accumulator's scratch (seqsum2.cuh)
__host__ __device__ inline size_t norm_smem_bytes(int dim) { return (size_t)norm_padded(dim) * 4 + 16 + seqsum2_scratch_bytes(); }

template <bool EMBED>
__global__ void __launch_bounds__(NORM_THREADS, 1) k_rmsnorm_quant(float *__restrict__ x, const StepState *__restrict__ st,
                                                               DevMat emb, const float *__restrict__ w, float eps, int dim,
                                                               int8_t *__restrict__ xq, float *__restrict__ xs,
                                                               float *__restrict__ xb, TraceBuf tr, TpCtx tp, int tp_wait_op) {
    // One CTA of 1024 threads.  Under PDL this CTA only has to fit next to ONE streaming-matvec CTA
    // (the following matvec's CTA for this SM simply starts a little later).
    extern __shared__ __align__(16) float sm[];
    float *sq = sm;
    __shared__ float s_ss;
    const int tid = threadIdx.x;
    trace_entry(tr);
    pdl_launch_dependents();
    pdl_wait();
    trace_mark(tr, 2);
    if (tp.n > 1 && tp_wait_op >= 0) { // x is gathered from all ranks: wait for their slices
        if (tid == 0) tp_wait(tp, TP_SLOT_X, tp_seq(tp, (unsigned)tp_wait_op));
        __syncthreads();
    }
    int token = 0;
    if (EMBED) token = st->token;
    for (int i = tid; i < dim; i += NORM_THREADS) {
        float v;
        if (EMBED) { v = emb_get(emb, token, i); x[i] = v; }
        else v = ldcg_f32c(x + i);
        sq[i] = __fmul_rn(v, v);
    }
    for (int i = dim + tid; i < norm_padded(dim); i += NORM_THREADS) sq[i] = 0.0f;
    __syncthreads();
    // ss = sequential float sum of the squares (exact, parallel)
    SeqSum2Scratch scratch = seqsum2_carve(reinterpret_cast<unsigned char *>(sm + norm_padded(dim)));
    float ss = block_seqsum_exact_v2(sq, dim, scratch);
    if (EMBED) __threadfence_block(); // x[] written above by other threads of this block
    if (tid == 0) {
        ss = __fdiv_rn(ss, (float)dim);
        ss = __fadd_rn(ss, eps);
        s_ss = (float)(1.0 / sqrt((double)ss));
    }
    __syncthreads();
    ss = s_ss;
    const int lane = tid & 31, warp = tid >> 5;
    constexpr int NWN = NORM_THREADS / 32;
    const int nb = dim / 32;
#pragma unroll 1
    for (int b0 = warp; b0 < nb; b0 += 4 * NWN) { // 8 loads in flight per lane
        float xv[4], wv[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int b = b0 + u * NWN;
            xv[u] = 0.0f; wv[u] = 0.0f;
            if (b < nb) { xv[u] = ldcg_f32c(x + b * 32 + lane); wv[u] = w[b * 32 + lane]; } // x: L2 hit (or this block's own store)
        }
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int b = b0 + u * NWN;
            if (b < nb) {
                const int i = b * 32 + lane;
                const float v = __fmul_rn(wv[u], __fmul_rn(ss, xv[u]));
                if (xb) xb[i] = v;
                if (xq) {
                    float as;
                    int q = quant_block_lane(v, as);
                    xq[i] = (int8_t)q;
                    if (lane == 0) xs[b] = as;
                }
            }
        }
    }
    trace_mark(tr, 3);
}

// Test hook: the sequential-sum emulation on arbitrary non-negative terms (padded with zeros: adding +0 never
// changes a sum of non-negative floats), seqsum2.cuh with T threads (1024: the norm kernel's form; 256: the persistent decode kernel's form)
template <int T>
__global__ void __launch_bounds__(T, 1) k_test_seqsum2(const float *__restrict__ terms, int n, float *__restrict__ out, int *__restrict__ info) {
    extern __shared__ __align__(16) float sm[];
    float *sq = sm;
    const int E = (n + T - 1) / T, np = T * E;
    SeqSum2Scratch scratch = seqsum2_carve(reinterpret_cast<unsigned char *>(sm + np), T);
    for (int i = threadIdx.x; i < np; i += T) sq[i] = i < n ? terms[i] : 0.0f;
    if (threadIdx.x == 0) { scratch.info[0] = -1; scratch.info[1] = -2; }
    __syncthreads();
    const float s = block_seqsum_exact_v2_t<T>(sq, n, scratch, (int)threadIdx.x, SeqSum2BlockSync());
    if (threadIdx.x == 0) { out[0] = s; info[0] = scratch.info[0]; info[1] = scratch.info[1]; }
}

// ------------------------------------------------------------------------------------------
// Q8_0 dequant-matvec, bit-exact with Q8_0FloatTensor.dotQ8Activation (Q8_0FloatTensor.java:90-123):
//   per 32-block b:  isum_b = sum aq*wq (int32, exact);  term_b = (float)isum_b * (wScale_b * aScale_b)
//   result = ((term_0 + term_1) + term_2) + ...      strictly in block order.
// The activation quantisation is row-independent, so it arrives pre-quantised (xq, xs).
// Mapping: a warp owns R rows; lane l owns blocks l, l+32, ... of each row (one LDG.256 per block,
// the warp reads 1 KB contiguous per instruction); block terms go to shared memory and lanes
// 0..R-1 then walk their row's terms in order.
// ------------------------------------------------------------------------------------------
template <int R>
__device__ __forceinline__ void q8_row_terms(const int8_t *__restrict__ qs, const __half *__restrict__ sc, size_t row0,
                                             int cols, int nb, const int4 *__restrict__ sxq, const float *__restrict__ sxs,
                                             float *__restrict__ terms, int nbp, int lane) {
    constexpr int JB = R >= 4 ? 2 : 4; // 64 registers of weights in flight per lane
    for (int b0 = 0; b0 < nb; b0 += 32 * JB) {
        int wv[R][JB][8];
        __half sv[R][JB];
#pragma unroll
        for (int r = 0; r < R; r++)
#pragma unroll
            for (int j = 0; j < JB; j++) {
                int b = b0 + j * 32 + lane;
                if (b < nb) {
                    ldg256_stream(qs + (row0 + r) * (size_t)cols + (size_t)b * 32, wv[r][j]);
                    sv[r][j] = sc[(row0 + r) * (size_t)nb + b];
                }
            }
#pragma unroll
        for (int j = 0; j < JB; j++) {
            int b = b0 + j * 32 + lane;
            if (b < nb) {
                int4 a0 = sxq[b], a1 = sxq[nb + b];
                float as = sxs[b];
#pragma unroll
                for (int r = 0; r < R; r++) {
                    int isum = __dp4a(wv[r][j][0], a0.x, 0);
                    isum = __dp4a(wv[r][j][1], a0.y, isum);
                    isum = __dp4a(wv[r][j][2], a0.z, isum);
                    isum = __dp4a(wv[r][j][3], a0.w, isum);
                    isum = __dp4a(wv[r][j][4], a1.x, isum);
                    isum = __dp4a(wv[r][j][5], a1.y, isum);
                    isum = __dp4a(wv[r][j][6], a1.z, isum);
                    isum = __dp4a(wv[r][j][7], a1.w, isum);
                    terms[r * nbp + b] = __fmul_rn((float)isum, __fmul_rn(__half2float(sv[r][j]), as));
                }
            }
        }
    }
}

// Stage the quantised activation in shared memory as two planes of 16-byte half-blocks
// (plane p holds bytes [16p,16p+16) of every block) so that lanes reading consecutive
// blocks hit consecutive 16-byte slots: conflict-free LDS.128.
__device__ __forceinline__ void stage_activation(const int8_t *__restrict__ xq, const float *__restrict__ xs, int cols,
                                                 int4 *sxq, float *sxs) {
    const int nb = cols >> 5;
    const int4 *src = reinterpret_cast<const int4 *>(xq);
    for (int c = threadIdx.x; c < cols / 16; c += blockDim.x) sxq[(c & 1) * nb + (c >> 1)] = src[c];
    for (int b = threadIdx.x; b < nb; b += blockDim.x) sxs[b] = xs[b];
}

__host__ __device__ inline size_t q8_smem_bytes(int cols, int rows_per_warp, int warps) {
    int nb = cols / 32, nbp = nb | 1;
    return (size_t)cols + (size_t)nb * 4 + (size_t)warps * rows_per_warp * nbp * 4 + 64;
}

template <int R, int MODE>
__global__ void __launch_bounds__(256) k_matvec_q8(const int8_t *__restrict__ qs, const __half *__restrict__ sc,
                                                   const int8_t *__restrict__ xq, const float *__restrict__ xs, int rows,
                                                   int cols, float *__restrict__ out) {
    extern __shared__ __align__(16) unsigned char smraw[];
    const int nb = cols >> 5, nbp = nb | 1;
    int4 *sxq = reinterpret_cast<int4 *>(smraw);
    float *sxs = reinterpret_cast<float *>(smraw + cols);
    float *terms_all = sxs + nb;
    stage_activation(xq, xs, cols, sxq, sxs);
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float *terms = terms_all + (size_t)warp * R * nbp;
    const int nwarps_total = gridDim.x * (blockDim.x >> 5);
    for (size_t row0 = (size_t)(blockIdx.x * (blockDim.x >> 5) + warp) * R; row0 < (size_t)rows; row0 += (size_t)nwarps_total * R) {
        q8_row_terms<R>(qs, sc, row0, cols, nb, sxq, sxs, terms, nbp, lane);
        __syncwarp();
        if (lane < R) {
            const float *t = terms + lane * nbp;
            float acc = 0.0f;
            for (int b = 0; b < nb; b++) acc = __fadd_rn(acc, t[b]);
            size_t row = row0 + lane;
            if (MODE == MODE_RESID) out[row] = __fadd_rn(out[row], acc); // x[i] = x[i] + xb2[i]  (InferenceCore.java:143,164)
            else out[row] = acc;
        }
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------
// Fused gate/up projection + SwiGLU + Q8_0 quantisation of the result (the activation of the
// down projection).  InferenceCore.java:150-158: hb = hb / (float)(1.0 + Math.exp(-hb)); hb *= hb2.
// One CTA (8 warps) = one 32-element block of hb, so the CTA can quantise it in its epilogue.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float swiglu(float g, float u) {
    float s = __fdiv_rn(g, (float)(1.0 + exp((double)(-g))));
    return __fmul_rn(s, u);
}

__global__ void __launch_bounds__(256) k_gateup_q8(const int8_t *__restrict__ qs1, const __half *__restrict__ sc1,
                                                   const int8_t *__restrict__ qs3, const __half *__restrict__ sc3,
                                                   const int8_t *__restrict__ xq, const float *__restrict__ xs, int hidden,
                                                   int cols, int8_t *__restrict__ hq, float *__restrict__ hs,
                                                   float *__restrict__ hb_dbg) {
    extern __shared__ __align__(16) unsigned char smraw[];
    __shared__ float hvals[32];
    const int nb = cols >> 5, nbp = nb | 1;
    int4 *sxq = reinterpret_cast<int4 *>(smraw);
    float *sxs = reinterpret_cast<float *>(smraw + cols);
    float *terms_all = sxs + nb;
    stage_activation(xq, xs, cols, sxq, sxs);
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float *terms = terms_all + (size_t)warp * 4 * nbp; // 2 hidden units x {gate, up}
    for (int blk = blockIdx.x; blk < hidden / 32; blk += gridDim.x) {
#pragma unroll 1
        for (int half = 0; half < 2; half++) {
            int u0 = blk * 32 + warp * 4 + half * 2; // this warp: hidden units u0, u0+1
            q8_row_terms<2>(qs1, sc1, (size_t)u0, cols, nb, sxq, sxs, terms, nbp, lane);
            q8_row_terms<2>(qs3, sc3, (size_t)u0, cols, nb, sxq, sxs, terms + 2 * nbp, nbp, lane);
            __syncwarp();
            float acc = 0.0f;
            if (lane < 4) {
                const float *t = terms + lane * nbp;
                for (int b = 0; b < nb; b++) acc = __fadd_rn(acc, t[b]);
            }
            float up = __shfl_down_sync(0xffffffffu, acc, 2); // lanes 0,1 = gate(u0,u0+1); lanes 2,3 = up
            if (lane < 2) hvals[warp * 4 + half * 2 + lane] = swiglu(acc, up);
            __syncwarp();
        }
        __syncthreads();
        if (warp == 0) {
            float v = hvals[lane];
            if (hb_dbg) hb_dbg[blk * 32 + lane] = v;
            float as;
            int q = quant_block_lane(v, as);
            hq[blk * 32 + lane] = (int8_t)q;
            if (lane == 0) hs[blk] = as;
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------
// FP16 dequant-matvec, bit-exact with FP16FloatTensor.vectorDot (FP16FloatTensor.java:62-110)
// for an L-lane species: L independent strided FMA chains (fused, as FloatVector.fma), then
// reduceLanes(ADD) in ascending lane order, then the IEEE scalar tail.
// A warp owns 32/L rows at a time... see k_matvec_f16 below: thread (r, c) owns chain c of row r;
// the warp stages 16-byte coalesced loads through shared memory so every thread reads its
// stride-L elements from there.
// ------------------------------------------------------------------------------------------
template <int MODE>
__global__ void __launch_bounds__(256) k_matvec_f16(const __half *__restrict__ w, const float *__restrict__ x, int rows,
                                                    int cols, int lanes, float *__restrict__ out) {
    // Each warp processes RW = 32/lanes rows at once; thread t of the warp: row r = t / lanes, chain c = t % lanes.
    // Shared: activation x (cols floats) + per-warp weight tile RW x TC halves.
    extern __shared__ __align__(16) unsigned char smraw[];
    float *sx = reinterpret_cast<float *>(smraw);
    constexpr int TC = 256; // columns per staged tile
    __half *tiles = reinterpret_cast<__half *>(smraw + (size_t)cols * 4);
    for (int i = threadIdx.x; i < cols; i += blockDim.x) sx[i] = x[i];
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int L = lanes > 0 ? lanes : 1;
    const int RW = 32 / L;
    __half *tile = tiles + (size_t)warp * RW * TC;
    const int r = lane / L, c = lane % L;
    const int nwarps_total = gridDim.x * (blockDim.x >> 5);
    const int upper = lanes > 0 ? cols - (cols % L) : 0;
    for (size_t row0 = (size_t)(blockIdx.x * (blockDim.x >> 5) + warp) * RW; row0 < (size_t)rows; row0 += (size_t)nwarps_total * RW) {
        float acc = 0.0f;
        for (int c0 = 0; c0 < cols; c0 += TC) {
            int tc = min(TC, cols - c0);
            // coalesced stage: RW rows x tc halves, 8 halves (16 B) per lane per load
            int chunks_per_row = tc >> 3;
            for (int q = lane; q < RW * chunks_per_row; q += 32) {
                int rr = q / chunks_per_row, cc = q % chunks_per_row;
                size_t row = row0 + rr;
                int4 v = make_int4(0, 0, 0, 0);
                if (row < (size_t)rows) v = ldg128_stream(w + row * (size_t)cols + c0 + cc * 8);
                *reinterpret_cast<int4 *>(tile + rr * TC + cc * 8) = v;
            }
            __syncwarp();
            if (lanes > 0) {
                int lim = min(tc, upper - c0);
                for (int i = c; i < lim; i += L) {
                    float wf = f16_bits_to_f32_daz(__half_as_ushort(tile[r * TC + i]));
                    acc = fmaf(wf, sx[c0 + i], acc);
                }
            } else {
                // llama.VectorBitSize=0: FloatTensor.scalarDot, sequential, IEEE conversion, unfused
                for (int i = 0; i < tc; i++) acc = __fadd_rn(acc, __fmul_rn(__half2float(tile[r * TC + i]), sx[c0 + i]));
            }
            __syncwarp();
        }
        // reduceLanes(ADD), ascending lane order starting from the identity, then scalar tail
        float result = acc;
        if (lanes > 0) {
            result = 0.0f;
            for (int k = 0; k < L; k++) {
                float a = __shfl_sync(0xffffffffu, acc, r * L + k);
                result = __fadd_rn(result, a);
            }
            size_t row = row0 + r;
            if (row < (size_t)rows)
                for (int j = upper; j < cols; j++)
                    result = __fadd_rn(result, __fmul_rn(__half2float(w[row * (size_t)cols + j]), sx[j]));
        }
        size_t row = row0 + r;
        if (c == 0 && row < (size_t)rows) {
            if (MODE == MODE_RESID) out[row] = __fadd_rn(out[row], result);
            else out[row] = result;
        }
    }
}

// SwiGLU over separately computed gate/up vectors (FP16 path): hb = silu(hb) * hb2.
__global__ void k_swiglu(float *__restrict__ hb, const float *__restrict__ hb2, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) hb[i] = swiglu(hb[i], hb2[i]);
}

// ------------------------------------------------------------------------------------------
// Fused RoPE + KV-cache write + attention, one query head per CTA, exact CPU-path order.
//   prologue : (Qwen3: per-head RMSNorm of q and k, InferenceCore.java:594-600) then RoPE of this
//              head's q and of its KV head's k (InferenceCore.java:75-87 interleaved pairs / :604-619 NeoX);
//              every query head of a KV group rotates the same k redundantly (cheaper than a
//              kernel boundary); the group's first head writes k,v into the cache (:92-93)
//   scores   : score_t = scalarDot(q, k_t) / sqrt(head)   (sequential unfused mul/add, FloatTensor.java:86-92)
//   softmax  : max, (float)Math.exp(f - max), sequential sum, divide        (FloatTensor.java:211-219)
//   output   : xb = sum_t a_t * v_t, sequentially over t per element (saxpyInPlace, FloatTensor.java:221-227)
// The current position's k/v come from shared memory / the packed qkv vector, older ones from the
// FP32 cache.  Output as floats (xb) and/or quantised to Q8_0 (activation of the Wo matvec).
// ------------------------------------------------------------------------------------------
#define ATT_THREADS 512 // four threads per key (scores) and per output element (weighted sum): head size <= ATT_THREADS / 4

template <int HS>
__global__ void __launch_bounds__(ATT_THREADS) k_attention(float *__restrict__ qkv, float *__restrict__ kc, float *__restrict__ vc,
                                                          const StepState *__restrict__ st, const float *__restrict__ cr,
                                                          const float *__restrict__ ci, int n_heads, int n_kv_heads, int arch /* KF_* flags */,
                                                          const float *__restrict__ qnorm_w, const float *__restrict__ knorm_w,
                                                          float eps, float sqrt_hs, int8_t *__restrict__ xq,
                                                          float *__restrict__ xs, float *__restrict__ xb, TraceBuf tr, TpCtx tp,
                                                          unsigned tp_out_op, int head_base, float *att_scratch, int ctx) {
    extern __shared__ __align__(16) float sm[]; // q[HS] | k[HS] | out[HS] | att[ctx] (att in global scratch for long contexts)
    __shared__ float red[ATT_THREADS / 32];
    __shared__ float s_val[2];
    float *sq = sm, *sk = sm + HS, *so = sm + 2 * HS;
    float *att = att_scratch ? att_scratch + (size_t)blockIdx.x * ctx : sm + 3 * HS;
    const int h = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int HALF = HS / 2;
    trace_entry(tr);
    pdl_launch_dependents();
    const int kv_mul = n_heads / n_kv_heads, kvh = h / kv_mul;
    const int qd = n_heads * HS, kvd = n_kv_heads * HS;
    pdl_wait();
    trace_mark(tr, 2);
    const int pos = st->pos, nt = pos + 1;
    { // K/V rows of the earlier positions -> L2, one 128-byte line per request, so the score loads below hit L2 (the weight stream carries an
      // evict_first policy; without the prefetch these rows come from HBM every layer)
        constexpr int LINES = HS / 32;
        for (int i = tid; i < pos * LINES; i += ATT_THREADS) {
            const size_t off = (size_t)(i / LINES) * kvd + kvh * HS + (i % LINES) * 32;
            asm volatile("prefetch.global.L2 [%0];" ::"l"(kc + off));
            asm volatile("prefetch.global.L2 [%0];" ::"l"(vc + off));
        }
    }
    const float *qsrc = qkv + h * HS, *ksrc = qkv + qd + kvh * HS, *vsrc = qkv + qd + kvd + kvh * HS;
    // ---- prologue: threads [0,HALF) rotate q pairs, threads [HALF,HS) rotate k pairs
    if (tid < HS) {
        const bool is_q = tid < HALF;
        const int p = is_q ? tid : tid - HALF;
        const float *src = is_q ? qsrc : ksrc;
        int i0, i1;
        if (arch & KF_NEOX) { i0 = p; i1 = p + HALF; } else { i0 = 2 * p; i1 = 2 * p + 1; }
        float v0 = src[i0], v1 = src[i1];
        if (arch & KF_QKNORM) { // Qwen3 per-head RMSNorm: literal sequential sum over the head
            float *sqr = is_q ? so : sk; // scratch: HS squares each
            sqr[i0] = __fmul_rn(v0, v0);
            sqr[i1] = __fmul_rn(v1, v1);
        }
        if (arch & KF_QKNORM) {
            asm volatile("bar.sync 3, %0;" ::"n"(HS) : "memory");
            if (p == 0) {
                const float *sqr = is_q ? so : sk;
                float ss = 0.0f;
                for (int i = 0; i < HS; i++) ss = __fadd_rn(ss, sqr[i]);
                ss = __fdiv_rn(ss, (float)HS);
                ss = __fadd_rn(ss, eps);
                s_val[is_q ? 0 : 1] = (float)(1.0 / sqrt((double)ss));
            }
            asm volatile("bar.sync 3, %0;" ::"n"(HS) : "memory");
            const float ss = s_val[is_q ? 0 : 1];
            const float *nw = is_q ? qnorm_w : knorm_w;
            v0 = __fmul_rn(nw[i0], __fmul_rn(ss, v0));
            v1 = __fmul_rn(nw[i1], __fmul_rn(ss, v1));
            asm volatile("bar.sync 3, %0;" ::"n"(HS) : "memory"); // scratch reads done before sk/so are overwritten
        }
        const float fcr = cr[(size_t)pos * HALF + p], fci = ci[(size_t)pos * HALF + p];
        const float r0 = __fsub_rn(__fmul_rn(v0, fcr), __fmul_rn(v1, fci));
        const float r1 = __fadd_rn(__fmul_rn(v0, fci), __fmul_rn(v1, fcr));
        float *dst = is_q ? sq : sk;
        dst[i0] = r0;
        dst[i1] = r1;
        if (h % kv_mul == 0) { // first query head of the KV group owns the cache / debug write-back
            if (!is_q) {
                const size_t o = (size_t)pos * kvd + kvh * HS;
                kc[o + i0] = r0;
                kc[o + i1] = r1;
                vc[o + i0] = vsrc[i0];
                vc[o + i1] = vsrc[i1];
                // (the rotated k is NOT written back into qkv: the other query heads of this group read the
                //  unrotated k from there concurrently)
            }
        }
        if (is_q) { qkv[h * HS + i0] = r0; qkv[h * HS + i1] = r1; }
    }
    __syncthreads();
    // ---- scores (scalarDot, FloatTensor.java:86-92: one sequential unfused mul/add chain per key).  Four threads share a key: each loads
    // ITS quarter of the K row at once (one round trip per pass of ATT_THREADS/4 keys), then the chain runs through the quad in element
    // order, handed on by shuffle.  The V rows of the first round of the weighted sum are requested here too (they do not depend on the scores).
    constexpr int QE = HS / 4, QV = HS / 16, VB = 32;
    const int quad = tid & 3, qbase = lane & ~3, vd = tid >> 2;
    const bool vlive = vd < HS;
    float vv[VB];
    {
        const float *vcol = vc + kvh * HS + vd;
#pragma unroll
        for (int u = 0; u < VB; u++) vv[u] = (vlive && quad * VB + u < pos) ? __ldg(vcol + (size_t)(quad * VB + u) * kvd) : 0.0f;
    }
    float lmax = -INFINITY;
#pragma unroll 1
    for (int t0 = 0; t0 < nt; t0 += ATT_THREADS / 4) {
        const int t = t0 + (tid >> 2);
        float4 kk[QV];
        if (t < pos) {
            const float4 *k = reinterpret_cast<const float4 *>(kc + (size_t)t * kvd + kvh * HS + quad * QE);
#pragma unroll
            for (int u = 0; u < QV; u++) kk[u] = __ldg(k + u);
        } else {
#pragma unroll
            for (int u = 0; u < QV; u++) kk[u] = t == pos ? *reinterpret_cast<const float4 *>(sk + quad * QE + 4 * u) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        float acc = 0.0f;
#pragma unroll 1
        for (int qd4 = 0; qd4 < 4; qd4++) {
            if (quad == qd4) {
                const float *qq = sq + qd4 * QE;
#pragma unroll
                for (int u = 0; u < QV; u++) {
                    acc = __fadd_rn(acc, __fmul_rn(qq[4 * u + 0], kk[u].x));
                    acc = __fadd_rn(acc, __fmul_rn(qq[4 * u + 1], kk[u].y));
                    acc = __fadd_rn(acc, __fmul_rn(qq[4 * u + 2], kk[u].z));
                    acc = __fadd_rn(acc, __fmul_rn(qq[4 * u + 3], kk[u].w));
                }
            }
            acc = __shfl_sync(0xffffffffu, acc, qbase + qd4);
        }
        if (quad == 0 && t < nt) {
            const float s = __fdiv_rn(acc, sqrt_hs);
            att[t] = s;
            lmax = fmaxf(lmax, s);
        }
    }
    lmax = warp_max_f(lmax);
    if (lane == 0) red[warp] = lmax;
    __syncthreads();
    float mx = red[0];
#pragma unroll
    for (int w = 1; w < ATT_THREADS / 32; w++) mx = fmaxf(mx, red[w]);
    for (int t = tid; t < nt; t += ATT_THREADS) att[t] = (float)exp((double)__fsub_rn(att[t], mx));
    __syncthreads();
    if (tid == 0) {
        float sum = 0.0f;
        int t = 0;
        for (; t + 4 <= nt; t += 4) {
            const float a0 = att[t], a1 = att[t + 1], a2 = att[t + 2], a3 = att[t + 3];
            sum = __fadd_rn(sum, a0); sum = __fadd_rn(sum, a1); sum = __fadd_rn(sum, a2); sum = __fadd_rn(sum, a3);
        }
        for (; t < nt; t++) sum = __fadd_rn(sum, att[t]);
        s_val[0] = sum;
    }
    __syncthreads();
    const float sum = s_val[0];
    for (int t = tid; t < nt; t += ATT_THREADS) att[t] = __fdiv_rn(att[t], sum);
    __syncthreads();
    // ---- output: xb = sum_t a_t * v_t sequentially over t per element (saxpyInPlace, FloatTensor.java:221-227); four threads per element, thread
    // `quad` holds rows [128 r + 32 quad, +32) of round r, the chain runs through the quad in row order
#pragma unroll 1
    for (int vd0 = 0; vd0 < HS; vd0 += ATT_THREADS / 4) { // one pass for head sizes up to 128
        const int d = vd0 + vd;
        const bool live = d < HS;
        const float *vcol = vc + kvh * HS + d;
        const float vcur = live ? vsrc[d] : 0.0f; // current position: straight from the packed qkv vector
        float acc = 0.0f;
#pragma unroll 1
        for (int r0 = 0; r0 < pos; r0 += 4 * VB) {
            if (r0 > 0 || vd0 > 0) { // (round 0 of the first pass was requested before the scores)
                const int vt0 = r0 + quad * VB;
#pragma unroll
                for (int u = 0; u < VB; u++) vv[u] = (live && vt0 + u < pos) ? __ldg(vcol + (size_t)(vt0 + u) * kvd) : 0.0f;
            }
#pragma unroll 1
            for (int qd4 = 0; qd4 < 4; qd4++) {
                if (quad == qd4) {
                    const int vt0 = r0 + qd4 * VB;
#pragma unroll
                    for (int u = 0; u < VB; u++)
                        if (vt0 + u < pos) acc = __fadd_rn(__fmul_rn(att[vt0 + u], vv[u]), acc);
                }
                acc = __shfl_sync(0xffffffffu, acc, qbase + qd4);
            }
        }
        if (live && quad == 0) {
            acc = __fadd_rn(__fmul_rn(att[pos], vcur), acc);
            so[d] = acc;
            if (xb) xb[h * HS + d] = acc;
        }
    }
    __syncthreads();
    if (xq) {
        for (int b = warp; b < HS / 32; b += ATT_THREADS / 32) {
            float as;
            int q = quant_block_lane(so[b * 32 + lane], as);
            if (tp.n > 1) { // all-gather: this head's quantised output goes straight into every rank's buffer
                const int gh = head_base + h;
                for (int k = 0; k < tp.n; k++) {
                    tp_ptr<int8_t>(tp, k, tp.off_attq)[gh * HS + b * 32 + lane] = (int8_t)q;
                    if (lane == 0) tp_ptr<float>(tp, k, tp.off_atts)[(gh * HS) / 32 + b] = as;
                }
            } else {
                xq[h * HS + b * 32 + lane] = (int8_t)q;
                if (lane == 0) xs[(h * HS) / 32 + b] = as;
            }
        }
    }
    if (tp.n > 1) {
        __syncthreads();
        if (tid == 0) tp_cta_done(tp, TP_SLOT_ATT, tp_seq(tp, tp_out_op), gridDim.x);
    }
    trace_mark(tr, 3);
}

// ------------------------------------------------------------------------------------------
// Greedy sampler + step advance.  FloatTensor.argmax (FloatTensor.java:138-151): first strict
// maximum.  One CTA; each thread keeps (max, lowest index) over a strided slice, then a tree
// merge that prefers the lower index on ties -- equal to the sequential scan for NaN-free input.
// Also advances the device-resident StepState so graph replays chain without the host.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void argmax_merge(float &v, int &i, float ov, int oi) {
    if (ov > v || (ov == v && oi < i)) { v = ov; i = oi; }
}

__global__ void __launch_bounds__(1024) k_argmax_advance(const float *__restrict__ logits, int vocab, StepState *st,
                                                        const int *__restrict__ seq_tokens, int *__restrict__ out_ids,
                                                        int do_argmax, const float *__restrict__ part_val,
                                                        const int *__restrict__ part_idx, int n_part, TraceBuf tr, TpCtx tp, int tp_wait_x_op) {
    __shared__ float sv[32];
    __shared__ int si[32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    trace_entry(tr);
    pdl_launch_dependents();
    pdl_wait();
    trace_mark(tr, 2);
    int best_i = 0;
    if (do_argmax) {
        float best = -INFINITY;
        best_i = 0x7fffffff;
        if (part_val) { // per-CTA (max, first index) pairs produced by the lm_head kernel
            for (int i = tid; i < n_part; i += blockDim.x) {
                float v = part_val[i];
                int ix = part_idx[i];
                argmax_merge(best, best_i, v, ix);
            }
        } else {
            for (int i = tid; i < vocab; i += blockDim.x) {
                float v = logits[i];
                if (v > best) { best = v; best_i = i; }
            }
        }
        // a thread that saw nothing > -inf keeps INT_MAX; index 0 wins below if all are -inf
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            float ov = __shfl_xor_sync(0xffffffffu, best, o);
            int oi = __shfl_xor_sync(0xffffffffu, best_i, o);
            argmax_merge(best, best_i, ov, oi);
        }
        if (lane == 0) { sv[warp] = best; si[warp] = best_i; }
        __syncthreads();
        if (warp == 0) {
            int nw = blockDim.x >> 5;
            best = lane < nw ? sv[lane] : -INFINITY;
            best_i = lane < nw ? si[lane] : 0x7fffffff;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                float ov = __shfl_xor_sync(0xffffffffu, best, o);
                int oi = __shfl_xor_sync(0xffffffffu, best_i, o);
                argmax_merge(best, best_i, ov, oi);
            }
            if (tp.n > 1) { // exchange every rank's (max, lowest global index) and merge identically everywhere
                const unsigned seq = tp_seq(tp, tp.ops_per_fwd - 1u);
                if (lane == 0) {
                    for (int k = 0; k < tp.n; k++) {
                        tp_ptr<float>(tp, k, tp.off_pv)[tp.rank] = best;
                        tp_ptr<int>(tp, k, tp.off_pi)[tp.rank] = best_i;
                    }
                    tp_signal(tp, TP_SLOT_ARG, seq);
                    tp_wait(tp, TP_SLOT_ARG, seq);
                }
                __syncwarp();
                best = lane < tp.n ? ldcg_f32c(tp_ptr<float>(tp, tp.rank, tp.off_pv) + lane) : -INFINITY;
                best_i = lane < tp.n ? (int)__float_as_int(ldcg_f32c(reinterpret_cast<const float *>(tp_ptr<int>(tp, tp.rank, tp.off_pi)) + lane)) : 0x7fffffff;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    float ov = __shfl_xor_sync(0xffffffffu, best, o);
                    int oi = __shfl_xor_sync(0xffffffffu, best_i, o);
                    argmax_merge(best, best_i, ov, oi);
                }
            }
            if (best_i == 0x7fffffff) best_i = 0;
        }
    } else if (tp.n > 1 && tp_wait_x_op >= 0) {
        // prefill graph: no argmax exchange, but the next forward's embedding write must not race the peers'
        // last residual-stream pushes of this forward
        if (tid == 0) tp_wait(tp, TP_SLOT_X, tp_seq(tp, (unsigned)tp_wait_x_op));
        __syncthreads();
    }
    if (tid == 0) {
        int step = st->step;
        if (do_argmax && out_ids) out_ids[step] = best_i;
        int next = step + 1;
        if (st->feedback && do_argmax) st->token = best_i;
        else if (next < st->n_seq) st->token = seq_tokens[next];
        st->step = next;
        st->pos = st->pos + 1;
        if (tp.n > 1) *reinterpret_cast<volatile unsigned *>(tp.peer[tp.rank] + tp.off_tick) += 1u; // next forward's flag epoch
    }
    trace_mark(tr, 3);
}
