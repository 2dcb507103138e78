// decode_persistent.cuh -- ONE persistent kernel per decoded token (sm_100a), replacing the 227 dependent launches of
// the round-1 decode graph (and, in the reference, TornadoVMMasterPlanSingleToken.tornadoVMForwardDecode's N+2 TaskGraph
// executions, TornadoVMMasterPlanSingleToken.java:68-95).  The arithmetic of every phase is the bit-exact CPU order of
// decode_kernels.cuh / stream_matvec.cuh (InferenceCore.java:50-172, 565-697); what this file adds is the orchestration:
//
//   * grid = one CTA per SM (cooperative launch: co-residency is checked by the driver), 8 consumer warps + 1 producer
//     warp, resident for the whole token;
//   * the producer thread walks the tile-major weight stream of EVERY matrix of the token in consumption order (QKV, Wo,
//     gate/up, W2 per layer, then lm_head) through one shared-memory ring of 1-D bulk copies: weight addresses never
//     depend on activations, so HBM keeps streaming across what used to be kernel boundaries; the copies carry an L2
//     evict_first policy, so 8 GB of single-use weights per token do not push the KV rows, x and the norm weights out of L2;
//   * phases are separated by epoch counters instead of kernel boundaries, five per layer:
//         QKV rows -> attention | attention heads -> Wo | x -> ffn norm | hidden activation -> W2 | x -> next layer.
//     Counters are monotone and never reset: target = (tick * layers + layer + 1) * arrivers, where tick counts launches.
//     Under tensor parallelism the last local arriver of an exchanging phase raises epoch flags on every rank (NVLink
//     peer stores, system-scope fences) and waiters poll the flags of all ranks: the all-gathers of common.cuh, now
//     inside one kernel;
//   * RMSNorm is computed REDUNDANTLY by every CTA straight into its own shared-memory activation buffer (exact
//     accumulator: seqsum2.cuh on the 256 consumer threads), which removes two of the seven dependencies of a layer
//     and the xq/xs round trip;
//   * attention heads run on the first n_heads CTAs with the consumer warps; the score row lives in shared memory, or
//     in a global scratch row when the context is too long for it;
//   * the embedding row is consumed in place: layer 0's norm squares the embedding row and layer 0's Wo epilogue
//     writes x = emb + Wo*att, so there is no "x = embedding" pass and no grid sync before the first layer;
//   * every spin has a deadline (%globaltimer): a lost peer or a desynchronised call sequence sets an error word the
//     host checks after the launch instead of hanging the GPU.
#pragma once
#include "decode_kernels.cuh"
#include "seqsum2.cuh"
#include "stream_matvec.cuh"

#define PD_WARPS 16                     // consumer warps: 4 per SM sub-partition -- every phase of this kernel is a chain of dependent instructions,
                                        // and the ncu samples (profiles/r2_pd_full_v2.summary.txt) show warps waiting on their own previous result
#define PD_CT (PD_WARPS * 32)           // consumer threads
#define PD_THREADS (PD_CT + 32)         // + the producer warp
#define PD_MAX_STAGES 32
#define PD_TIMEOUT_NS 4000000000ull    // 4 s: far beyond any legitimate wait, well under gpurun's limits
#define PD_STAMPS 20                    // trace stamps per layer and CTA (0-9 phases, 10-15 inside the attn norm / the attention)

enum { PD_S_QKV = 0, PD_S_ATT = 1, PD_S_WO = 2, PD_S_GU = 3, PD_S_W2 = 4, PD_S_LM = 5, PD_S_ARG = 6, PD_S_SLOTS = 8,
       PD_S_TICK = 8, PD_S_LMTICK = 9, PD_S_ERR = 10, PD_S_WORDS = 16 };
// PD_S_TICK counts launches (epoch of the per-layer counters); PD_S_LMTICK counts launches that ran the lm_head (the prefill
// graph does not), which is the epoch of PD_S_LM / PD_S_ARG.  PD_S_ERR != 0: a wait timed out (value = 1 + slot).

struct PdLayer {
    TileMat qkv, wo, gu, w2;
    const float *attn_norm, *ffn_norm, *q_norm, *k_norm;
    float *kc, *vc; // this layer's FP32 KV cache (this rank's KV heads)
};

struct PdArgs {
    const PdLayer *layers; // device array [n_layers]
    int n_layers;
    TileMat lm_head;
    const float *out_norm;
    DevMat emb;
    int dim, hidden, qd;     // full widths (qd = columns of Wo)
    int n_heads, n_kv_heads; // of THIS rank
    int head_size, arch /* KF_* flags */, ctx;
    float eps, sqrt_hs;
    const float *rope_cr, *rope_ci;
    StepState *st;
    const int *seq_tokens;
    int *out_ids;
    float *x, *qkv, *hb, *logits;
    int8_t *attq;
    float *atts;
    int8_t *hq;
    float *hs;
    unsigned *blk_cnt;
    float *part_val;
    int *part_idx;
    unsigned *sync;            // [PD_S_WORDS] local epoch counters, ticks, error word
    unsigned *host_err;        // mapped pinned host word: receives the error code so the host sees it without a copy
    float *att_scratch;        // [n_heads][ctx] score rows in global memory, or NULL: rows live in shared memory
    unsigned long long *trace; // [gridDim.x][n_layers + 1][PD_STAMPS] %globaltimer stamps, or NULL
    int with_logits;
    // tensor parallelism (tp.n == 1: everything below unused)
    TpCtx tp;
    unsigned pd_flags_off;     // offset of the persistent kernel's epoch flags [PD_S_SLOTS][TP_MAX] in every rank's comm buffer
    int head_base, dim_base, hid_base, voc_base; // global index of this rank's first head / residual row / hidden unit / vocab row
};

struct PdSmem {
    size_t off_bar, off_xq, off_xs, off_nbuf, off_wbuf, off_rope, off_seq, off_terms, off_hvals, off_misc, off_ring, total;
    int stages, stage_bytes, tstride, nbuf_floats;
};

// max_seg = widest column segment of any matrix of the plan; att_floats = 3*head_size + ctx when the score row lives in
// shared memory, 3*head_size otherwise.
__host__ __device__ inline PdSmem pd_layout(int dim, int qd, int hidden, int head_size, int att_floats, int max_seg, size_t budget) {
    PdSmem L;
    const int unit = smv_unit_bytes(max_seg);
    L.stage_bytes = (4 * unit + 127) & ~127;
    L.tstride = ((max_seg / 32 + 3) & ~3) + 4; // per-row stride of the term buffer: 16-byte aligned rows, the four walker lanes on distinct banks
    int maxc = dim > qd ? dim : qd;
    if (hidden > maxc) maxc = hidden;
    const int E = (dim + PD_CT - 1) / PD_CT;
    const int sq_floats = PD_CT * seqsum2_stride(E); // squares of the norm in the accumulator's bank-conflict-free chunk layout
    L.nbuf_floats = sq_floats > att_floats ? sq_floats : att_floats;
    size_t o = 0;
    L.off_bar = o; o += 2 * PD_MAX_STAGES * 8 + PD_MAX_STAGES * 4;
    o = (o + 15) & ~(size_t)15;
    L.off_xq = o; o += (size_t)maxc;
    L.off_xs = o; o += (size_t)(maxc / 32) * 4;
    o = (o + 15) & ~(size_t)15;
    L.off_nbuf = o; o += (size_t)L.nbuf_floats * 4; // squares of the norm | q,k,out,att of the attention (time-disjoint)
    o = (o + 15) & ~(size_t)15;
    L.off_wbuf = o; o += (size_t)dim * 4; // weights of the NEXT norm (attn, ffn or final), fetched one phase ahead (cp.async) as soon as
                                          // the previous norm has read its own out of this buffer
    L.off_rope = o; o += (size_t)head_size * 4; // this position's rope row: cos | sin
    o = (o + 15) & ~(size_t)15;
    L.off_seq = o; o += seqsum2_scratch_bytes(PD_CT);
    o = (o + 15) & ~(size_t)15;
    L.off_terms = o; o += (size_t)PD_WARPS * 4 * L.tstride * 4;
    L.off_hvals = o; o += SMV_HVALS * 4;
    L.off_misc = o; o += 96 * 4; // red[16], s_val[2] @16, scale @20, argmax merge scratch @32 (16 floats) / @48 (16 ints)
    o = (o + 127) & ~(size_t)127;
    L.off_ring = o;
    long room = (long)budget - (long)o;
    int s = room > 0 ? (int)(room / L.stage_bytes) : 0;
    if (s > PD_MAX_STAGES) s = PD_MAX_STAGES;
    L.stages = s;
    L.total = o + (size_t)s * L.stage_bytes;
    return L;
}

// ---- bounded waits ----------------------------------------------------------------------------------------------------------
// Polls are RELAXED loads; ONE acquire load of the same word follows the successful one.  (ld.acquire in the loop compiles to a
// load plus CCTL.IVALL: every poll of thread 0 threw away the whole L1 of its SM; a trailing fence.acq_rel.sys instead costs a
// MEMBAR.SYS per wait, which made tensor-parallel steps ~20 % slower -- profiles/r2_tp2_fences.log.)
__device__ __forceinline__ unsigned pd_ld_relaxed_gpu(const unsigned *p) {
    unsigned v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned pd_ld_relaxed_sys(const unsigned *p) {
    unsigned v;
    asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// one thread: spin until *p >= target (wrap-safe); gives up after PD_TIMEOUT_NS or as soon as another waiter gave up
template <bool SYS> __device__ __noinline__ void pd_spin(const unsigned *p, unsigned target, unsigned *err, unsigned *host_err, unsigned code) {
    unsigned it = 0;
    unsigned long long t0 = 0;
    for (;;) {
        const unsigned v = SYS ? pd_ld_relaxed_sys(p) : pd_ld_relaxed_gpu(p);
        if ((int)(v - target) >= 0) { // counters and flags are monotone: the acquire re-read observes a value >= the relaxed one
            unsigned w;
            if (SYS) asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(w) : "l"(p) : "memory");
            else asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(w) : "l"(p) : "memory");
            return;
        }
        if ((++it & 255u) == 0u) {
            if (*reinterpret_cast<volatile unsigned *>(err)) return;
            const unsigned long long now = gtime();
            if (!t0) t0 = now;
            else if (now - t0 > PD_TIMEOUT_NS) {
                atomicCAS(err, 0u, code);
                *reinterpret_cast<volatile unsigned *>(host_err) = code;
                return;
            }
        }
    }
}

__device__ __forceinline__ void pd_bar_sync() { asm volatile("bar.sync 1, %0;" ::"n"(PD_CT) : "memory"); }

struct PdConsumerSync {
    __device__ __forceinline__ void operator()() const { pd_bar_sync(); }
};

// Every consumer thread calls these.  `cross`: the phase's outputs are consumed by other ranks too (tensor parallelism):
// the CTA's peer stores (made before the barrier) are published by thread 0's system-scope fence, and the LAST local
// arriver raises this rank's epoch flag on every rank.
__device__ __noinline__ void pd_arrive(const PdArgs &a, int slot, unsigned target, unsigned epoch, bool cross, int tid) {
    pd_bar_sync();
    if (tid == 0) {
        const bool x = cross && a.tp.n > 1;
        // gpu-scope fence per CTA, ONE system-scope fence by the last arriver below: the CTAs' peer stores reach system scope through the
        // cumulativity of the fence chain (CTA store -> fence.gpu -> atomic -> last arriver's atomic -> fence.sys -> flag).  A per-CTA
        // __threadfence_system() here cost ~7 us per exchange at tp2 (148 MEMBAR.SYS waiting on NVLink round trips).
        __threadfence();
        const unsigned old = atomicAdd(a.sync + slot, 1u);
        if (x && old + 1u == target) {
            __threadfence_system();
            for (int k = 0; k < a.tp.n; k++) {
                unsigned *f = reinterpret_cast<unsigned *>(a.tp.peer[k] + a.pd_flags_off) + slot * TP_MAX + a.tp.rank;
                asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(f), "r"(epoch) : "memory");
            }
        }
    }
}
__device__ __noinline__ void pd_wait(const PdArgs &a, int slot, unsigned target, unsigned epoch, bool cross, int tid) {
    if (tid == 0) {
        if (cross && a.tp.n > 1) {
            const unsigned *f = reinterpret_cast<const unsigned *>(a.tp.peer[a.tp.rank] + a.pd_flags_off) + slot * TP_MAX;
            for (int k = 0; k < a.tp.n; k++) pd_spin<true>(f + k, epoch, a.sync + PD_S_ERR, a.host_err, 1u + (unsigned)slot);
        } else pd_spin<false>(a.sync + slot, target, a.sync + PD_S_ERR, a.host_err, 1u + (unsigned)slot);
    }
    pd_bar_sync();
}

__device__ __forceinline__ void pd_stamp(const PdArgs &a, int layer, int k, int tid) {
    if (a.trace && tid == 0) a.trace[((size_t)blockIdx.x * (a.n_layers + 1) + layer) * PD_STAMPS + k] = gtime();
}

// ---- producer: the whole token's weight stream, in consumption order ----------------------------------------------------
// Cursor over this CTA's tiles of matrix 0..n_mats-1 (4 per layer, then the lm_head): the same walk the consumers make.
struct PdWalk {
    const PdArgs *a;
    int n_mats, mi;
    TileMat W;
    int g1, gb, nw, s, w;
    unsigned tile_bytes;
    __device__ __forceinline__ void open() { // position on the first tile of matrix mi (skipping matrices this CTA has no rows of)
        for (; mi < n_mats; mi++) {
            const int l = mi >> 2;
            if (l < a->n_layers) {
                const PdLayer &Ly = a->layers[l];
                const int k = mi & 3;
                W = k == 0 ? Ly.qkv : k == 1 ? Ly.wo : k == 2 ? Ly.gu : Ly.w2;
            } else W = a->lm_head;
            const int ngroups = W.rows >> 2;
            gb = (int)(((long long)blockIdx.x * ngroups) / gridDim.x);
            g1 = (int)(((long long)(blockIdx.x + 1) * ngroups) / gridDim.x);
            if (gb < g1) {
                nw = min(PD_WARPS, g1 - gb);
                s = 0; w = 0;
                tile_bytes = 4u * (unsigned)W.unit_bytes;
                return;
            }
        }
    }
    __device__ __forceinline__ void init(const PdArgs *args) {
        a = args;
        n_mats = 4 * a->n_layers + (a->with_logits ? 1 : 0);
        mi = 0;
        open();
    }
    __device__ __forceinline__ bool valid() const { return mi < n_mats; }
    __device__ __forceinline__ const unsigned char *addr() const { return W.base + ((size_t)(gb + w) * W.nseg + s) * tile_bytes; }
    __device__ __forceinline__ void next() {
        if (++w < nw) return;
        w = 0;
        if (++s < W.nseg) return;
        s = 0;
        gb += PD_WARPS;
        if (gb < g1) { nw = min(PD_WARPS, g1 - gb); return; }
        mi++;
        open();
    }
};

__device__ __forceinline__ void pd_produce(const PdArgs &a, unsigned char *smem, const PdSmem &L, unsigned bar0) {
    const int S = L.stages;
    const unsigned long long pol = l2_policy_evict_first();
    PdWalk cur;
    cur.init(&a);
    for (unsigned seq = 0; cur.valid(); cur.next(), seq++) {
        const int st = seq % S;
        const unsigned ph = (seq / S) & 1u;
        mbar_wait(bar0 + 8 * (PD_MAX_STAGES + st), ph ^ 1u); // slot free (first pass returns at once)
        const unsigned full = bar0 + 8 * st;
        mbar_expect_tx(full, cur.tile_bytes);
        bulk_g2s_evict_first(smem_u32(smem + L.off_ring + (size_t)st * L.stage_bytes), cur.addr(), cur.tile_bytes, full, pol);
    }
}

// Fat scalar helpers kept OUT OF LINE: the kernel's phases execute on a cold instruction cache every layer (the loop body of a
// layer is several times the cache), so static code size and taken branches cost more than call overhead.
__device__ __noinline__ float pd_walk_rolled(float acc, const float *t, int nbs) { // strictly in block order (Q8_0FloatTensor.java:117-121)
    int b = 0;
    if (nbs >= 4) {
        float4 c = *reinterpret_cast<const float4 *>(t);
#pragma unroll 1
        for (; b + 4 <= nbs; b += 4) {
            float4 n = c;
            if (b + 8 <= nbs) n = *reinterpret_cast<const float4 *>(t + b + 4); // next four terms in flight during the adds
            acc = __fadd_rn(acc, c.x); acc = __fadd_rn(acc, c.y); acc = __fadd_rn(acc, c.z); acc = __fadd_rn(acc, c.w);
            c = n;
        }
    }
#pragma unroll 1
    for (; b < nbs; b++) acc = __fadd_rn(acc, t[b]);
    return acc;
}
__device__ __noinline__ float pd_swiglu(float g, float u) { return swiglu_exact(g, u); }
__device__ __noinline__ int pd_quant_block(float v, float *ascale) {
    float as;
    const int q = quant_block_lane(v, as);
    *ascale = as;
    return q;
}
__device__ __noinline__ float pd_emb_get(const DevMat &e, int token, int i) { return emb_get(e, token, i); }
__device__ __noinline__ float pd_exp_narrow(float x) { return (float)exp((double)x); } // (float) Math.exp(double)

// ---- consumers: one matrix (the loop of k_stream_matvec_q8, activation already in shared memory) --------------------------
// l0_emb: layer 0's Wo writes x = embedding + acc (the embedding row is never copied into x beforehand).
// row_base: global index of this rank's first output row (RESID, STORE/argmax) or hidden unit (GATEUP).
template <int MODE>
__device__ __noinline__ void pd_consume_matrix(const TileMat &W, const PdArgs &a, unsigned char *smem, const PdSmem &L, unsigned bar0, volatile unsigned *rel,
                                                  unsigned &seq_base, float *out, bool argmax, bool l0_emb, int token, int row_base, int tid) {
    // every descriptor field into a register once: the waits below are asm with a memory clobber, after which the compiler would
    // otherwise re-read W.* (global memory) and L.* on every use inside the tile loop
    const int lane = tid & 31, warp = tid >> 5, S = L.stages, tstride = L.tstride, stage_bytes = L.stage_bytes;
    const int w_unit = W.unit_bytes, w_seg = W.seg;
    const int ngroups = W.rows >> 2;
    const int g0 = (int)(((long long)blockIdx.x * ngroups) / gridDim.x), g1 = (int)(((long long)(blockIdx.x + 1) * ngroups) / gridDim.x);
    const int nseg = W.nseg, nbs = w_seg >> 5;
    const unsigned char *ring = smem + L.off_ring;
    const int tp_n = a.tp.n;
    float *terms = reinterpret_cast<float *>(smem + L.off_terms) + (size_t)warp * 4 * tstride;
    const unsigned char *sact = smem + L.off_xq;
    const float *sxs = reinterpret_cast<const float *>(smem + L.off_xs);
    float *hvals = reinterpret_cast<float *>(smem + L.off_hvals);
    const int hsel = (lane >> 2) & 1;
    float best = -INFINITY;
    int best_i = 0x7fffffff;
#pragma unroll 1
    for (int gb = g0; gb < g1; gb += PD_WARPS) {
        const int nw = min(PD_WARPS, g1 - gb);
        if (warp < nw) {
            const int G = gb + warp;
            float acc = 0.0f;
#pragma unroll 1
            for (int s = 0; s < nseg; s++) {
                const unsigned seq = seq_base + (unsigned)(s * nw + warp);
                const int st = seq % S;
                const unsigned lap = seq / S;
                if (lane == 0)
                    while (rel[st] != lap) {}
                __syncwarp();
                mbar_wait(bar0 + 8 * st, lap & 1u);
                const unsigned char *tile = ring + (size_t)st * stage_bytes;
#pragma unroll 1
                for (int b = lane; b < nbs; b += 32) {
                    const unsigned char *ab = sact + ((size_t)(s * nbs + b) << 5);
                    const int4 a0 = *reinterpret_cast<const int4 *>(ab + 16 * hsel);
                    const int4 a1 = *reinterpret_cast<const int4 *>(ab + 16 * (hsel ^ 1));
                    const float as = sxs[s * nbs + b];
#pragma unroll
                    for (int r = 0; r < 4; r++) {
                        const unsigned char *wb = tile + (size_t)r * w_unit + ((size_t)b << 5);
                        const int4 w0 = *reinterpret_cast<const int4 *>(wb + 16 * hsel);
                        const int4 w1 = *reinterpret_cast<const int4 *>(wb + 16 * (hsel ^ 1));
                        const __half sc = *reinterpret_cast<const __half *>(tile + (size_t)r * w_unit + w_seg + 2 * b);
                        int isum = __dp4a(w0.x, a0.x, 0);
                        isum = __dp4a(w0.y, a0.y, isum);
                        isum = __dp4a(w0.z, a0.z, isum);
                        isum = __dp4a(w0.w, a0.w, isum);
                        isum = __dp4a(w1.x, a1.x, isum);
                        isum = __dp4a(w1.y, a1.y, isum);
                        isum = __dp4a(w1.z, a1.z, isum);
                        isum = __dp4a(w1.w, a1.w, isum);
                        terms[r * tstride + b] = __fmul_rn((float)isum, __fmul_rn(__half2float(sc), as));
                    }
                }
                __syncwarp();
                if (lane == 0) {
                    rel[st] = lap + 1u;
                    mbar_arrive(bar0 + 8 * (PD_MAX_STAGES + st));
                }
                if (lane < 4) acc = pd_walk_rolled(acc, terms + lane * tstride, nbs);
                __syncwarp();
            }
            if (MODE == SMV_GATEUP) {
                const float up = __shfl_down_sync(0xffffffffu, acc, 2);
                if (lane < 2) {
                    const int unit = 2 * G + lane;
                    const float hval = pd_swiglu(acc, up);
                    out[unit] = hval;
                    hvals[unit - 2 * g0] = hval;
                }
            } else if (lane < 4) {
                const size_t row = (size_t)4 * G + lane;
                if (MODE == SMV_RESID) {
                    const size_t grow = (size_t)row_base + row;
                    const float base = l0_emb ? pd_emb_get(a.emb, token, (int)grow) : out[grow];
                    const float v = __fadd_rn(base, acc); // x[i] = x[i] + xb2[i]
                    if (tp_n > 1) { // all-gather of the residual stream: this rank's rows go to every rank
                        for (int k = 0; k < tp_n; k++) tp_ptr<float>(a.tp, k, a.tp.off_x)[grow] = v;
                    } else out[grow] = v;
                } else {
                    out[row] = acc;
                    const int grow = row_base + (int)row;
                    if (acc > best) { best = acc; best_i = grow; } // rows ascend per lane: first maximum kept
                }
            }
        }
        seq_base += (unsigned)(nseg * nw);
    }
    if (MODE == SMV_GATEUP) { // Q8_0 quantisation of the hidden activation: k_stream_matvec_q8's epilogue
        pd_bar_sync();
        const int u0 = 2 * g0, u1 = 2 * g1;
        if (u1 > u0) {
            for (int blk = (u0 >> 5) + warp; blk <= ((u1 - 1) >> 5); blk += PD_WARPS) {
                const int lo = max(blk << 5, u0), hi = min((blk << 5) + 32, u1);
                float v = 0.0f;
                bool mine = true;
                if (hi - lo == 32) v = hvals[(blk << 5) + lane - u0];
                else {
                    unsigned old = 0;
                    if (lane == 0) {
                        __threadfence(); // cumulative: publishes the hb stores of the whole CTA (ordered by the barrier above)
                        old = atomicAdd(&a.blk_cnt[blk], (unsigned)(hi - lo));
                    }
                    old = __shfl_sync(0xffffffffu, old, 0);
                    mine = (old + (unsigned)(hi - lo) == 32u);
                    if (mine) {
                        __threadfence();
                        v = ldcg_f32(out + (blk << 5) + lane);
                        if (lane == 0) a.blk_cnt[blk] = 0u;
                    }
                }
                if (mine) {
                    float as;
                    const int q = pd_quant_block(v, &as);
                    const int gblk = (row_base >> 5) + blk;
                    if (a.tp.n > 1) {
                        for (int k = 0; k < a.tp.n; k++) {
                            tp_ptr<int8_t>(a.tp, k, a.tp.off_hq)[(gblk << 5) + lane] = (int8_t)q;
                            if (lane == 0) tp_ptr<float>(a.tp, k, a.tp.off_hs)[gblk] = as;
                        }
                    } else {
                        a.hq[(gblk << 5) + lane] = (int8_t)q;
                        if (lane == 0) a.hs[gblk] = as;
                    }
                }
            }
        }
    } else if (MODE == SMV_STORE && argmax) {
        int *cand_i = reinterpret_cast<int *>(hvals + 64);
        pd_bar_sync(); // hvals may still be read by a previous phase
        if (lane < 4) { hvals[warp * 4 + lane] = best; cand_i[warp * 4 + lane] = best_i; }
        pd_bar_sync();
        if (tid == 0) {
            float bv = -INFINITY;
            int bi = 0x7fffffff;
            for (int k = 0; k < PD_WARPS * 4; k++) {
                const float v = hvals[k];
                const int ix = cand_i[k];
                if (v > bv || (v == bv && ix < bi)) { bv = v; bi = ix; }
            }
            a.part_val[blockIdx.x] = bv;
            a.part_idx[blockIdx.x] = bi;
        }
    }
}

// ---- RMSNorm of the residual stream into THIS CTA's activation buffer (arithmetic of k_rmsnorm_quant) ----------------------
__device__ __forceinline__ float4 pd_ldcg128(const float *p) {
    float4 v;
    asm volatile("ld.global.cg.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}

// One out-of-line copy of the exact accumulator for every caller (attn norm, ffn norm, final norm, long softmax rows): the
// kernel's code must stay inside the instruction cache, every cold fetch queues behind the weight stream.
__device__ __noinline__ float pd_seqsum(const float *sq, int n, int S, unsigned char *smem, const PdSmem &L, int tid) {
    SeqSum2Scratch scratch = seqsum2_carve(smem + L.off_seq, PD_CT);
    return block_seqsum_exact_v2_t<PD_CT>(sq, n, scratch, tid, PdConsumerSync(), S);
}

// Norm weights are fetched with cp.async one phase ahead into their shared-memory buffer (slot i4 by the thread that will
// read slot i4: no barrier needed, only that thread's own wait_group).
__device__ __forceinline__ void pd_prefetch_w(const float *w, float *sbuf, int dim, int tid) {
    const int n4 = dim >> 2;
    for (int i4 = tid; i4 < n4; i4 += PD_CT)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(sbuf + 4 * i4)), "l"(w + 4 * i4) : "memory");
    asm volatile("cp.async.commit_group;" ::: "memory");
}

// Thread t owns the 16-byte slots i4 = u * PD_CT + t (u < U) of the vector: x and the norm weights stay in REGISTERS between
// the two passes; a 32-element quantisation block is eight consecutive slots = eight consecutive lanes, so its amax is three
// shuffles.  Only the squares go through shared memory (the exact accumulator's chunk layout).  wbuf: this norm's weights,
// already on their way into shared memory (pd_prefetch_w).
template <int U>
__device__ __noinline__ void pd_norm_u(const PdArgs &a, const float *wbuf, bool from_emb, int token, unsigned char *smem, const PdSmem &L, int tid, int stamp_layer) {
    const int dim = a.dim, n4 = dim >> 2;
    float *sq = reinterpret_cast<float *>(smem + L.off_nbuf);
    float *misc = reinterpret_cast<float *>(smem + L.off_misc);
    const int E = (dim + PD_CT - 1) / PD_CT, S = seqsum2_stride(E);
    float4 xv[U];
#pragma unroll
    for (int u = 0; u < U; u++) { // every load of this thread in flight at once: one L2 round trip
        const int i4 = u * PD_CT + tid;
        xv[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i4 < n4) {
            if (from_emb) { // first layer: the embedding row (quantised table: element-wise, FloatTensor.copyTo)
                xv[u] = make_float4(pd_emb_get(a.emb, token, 4 * i4), pd_emb_get(a.emb, token, 4 * i4 + 1), pd_emb_get(a.emb, token, 4 * i4 + 2), pd_emb_get(a.emb, token, 4 * i4 + 3));
            } else xv[u] = pd_ldcg128(a.x + 4 * i4);
        }
    }
    // squares -> chunk layout: element i belongs to accumulator thread i / E at offset i % E of its S-float chunk
    for (int i = dim + tid; i < PD_CT * E; i += PD_CT) sq[(i / E) * S + (i % E)] = 0.0f; // zero padding of the last chunks
#pragma unroll
    for (int u = 0; u < U; u++) {
        const int i4 = u * PD_CT + tid;
        if (i4 < n4) {
            const int i = 4 * i4;
            const float4 q = make_float4(__fmul_rn(xv[u].x, xv[u].x), __fmul_rn(xv[u].y, xv[u].y), __fmul_rn(xv[u].z, xv[u].z), __fmul_rn(xv[u].w, xv[u].w));
            if ((E & 3) == 0) *reinterpret_cast<float4 *>(sq + (i / E) * S + (i % E)) = q; // the four elements share a chunk
            else {
                sq[(i / E) * S + (i % E)] = q.x; sq[((i + 1) / E) * S + ((i + 1) % E)] = q.y;
                sq[((i + 2) / E) * S + ((i + 2) % E)] = q.z; sq[((i + 3) / E) * S + ((i + 3) % E)] = q.w;
            }
        }
    }
    pd_bar_sync();
    if (stamp_layer >= 0) pd_stamp(a, stamp_layer, 10, tid);
    float ss = pd_seqsum(sq, dim, S, smem, L, tid);
    if (stamp_layer >= 0) pd_stamp(a, stamp_layer, 11, tid);
    if (tid == 0) {
        ss = __fdiv_rn(ss, (float)dim);
        ss = __fadd_rn(ss, a.eps);
        misc[20] = (float)(1.0 / sqrt((double)ss));
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory"); // this thread's slots of the norm weights have landed
    pd_bar_sync();
    ss = misc[20];
    unsigned *sxq = reinterpret_cast<unsigned *>(smem + L.off_xq);
    float *sxs = reinterpret_cast<float *>(smem + L.off_xs);
#pragma unroll
    for (int u = 0; u < U; u++) { // out = w * (ss * x) (InferenceCore.java:45-47), then Q8_0FloatTensor.java:100-117 per 32-block
        const int i4 = u * PD_CT + tid;
        if (u * PD_CT < n4) { // warp-uniform (n4 is a multiple of 8 and whole 8-lane groups are in or out)
            float v0 = 0.f, v1 = 0.f, v2 = 0.f, v3 = 0.f;
            if (i4 < n4) {
                const float4 wv = *reinterpret_cast<const float4 *>(wbuf + 4 * i4);
                v0 = __fmul_rn(wv.x, __fmul_rn(ss, xv[u].x)); v1 = __fmul_rn(wv.y, __fmul_rn(ss, xv[u].y));
                v2 = __fmul_rn(wv.z, __fmul_rn(ss, xv[u].z)); v3 = __fmul_rn(wv.w, __fmul_rn(ss, xv[u].w));
            }
            float amax = fmaxf(fmaxf(fabsf(v0), fabsf(v1)), fmaxf(fabsf(v2), fabsf(v3)));
            amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, 1));
            amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, 2));
            amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, 4));
            const float qs = __fdiv_rn(amax, 127.0f);
            const float ascale = __half2float(__float2half_rn(qs));
            const float ainv = qs != 0.0f ? __fdiv_rn(1.0f, qs) : 0.0f;
            const float s0 = __fmul_rn(v0, ainv), s1 = __fmul_rn(v1, ainv), s2 = __fmul_rn(v2, ainv), s3 = __fmul_rn(v3, ainv);
            const int q0 = __float2int_rz(__fadd_rn(s0, copysignf(0.5f, s0))), q1 = __float2int_rz(__fadd_rn(s1, copysignf(0.5f, s1)));
            const int q2 = __float2int_rz(__fadd_rn(s2, copysignf(0.5f, s2))), q3 = __float2int_rz(__fadd_rn(s3, copysignf(0.5f, s3)));
            if (i4 < n4) {
                sxq[i4] = (unsigned)(q0 & 0xff) | ((unsigned)(q1 & 0xff) << 8) | ((unsigned)(q2 & 0xff) << 16) | ((unsigned)(q3 & 0xff) << 24);
                if ((tid & 7) == 0) sxs[i4 >> 3] = ascale;
            }
        }
    }
    pd_bar_sync();
}

// U = 16-byte slots per consumer thread = ceil(dim / (4 * PD_CT)): only the instantiation the model needs ever executes
__device__ __forceinline__ void pd_norm_to_smem(const PdArgs &a, const float *wbuf, bool from_emb, int token, unsigned char *smem, const PdSmem &L, int tid, int stamp_layer = -1) {
    const int U = ((a.dim >> 2) + PD_CT - 1) / PD_CT;
    if (U <= 1) pd_norm_u<1>(a, wbuf, from_emb, token, smem, L, tid, stamp_layer);
    else if (U == 2) pd_norm_u<2>(a, wbuf, from_emb, token, smem, L, tid, stamp_layer);
    else pd_norm_u<4>(a, wbuf, from_emb, token, smem, L, tid, stamp_layer); // dim <= 4 * PD_CT * 4 = 8192 (checked at plan creation)
}

// a quantised activation vector produced by other CTAs / ranks (attention output, hidden activation) -> shared memory
__device__ __noinline__ void pd_load_act(const int8_t *q, const float *s, int cols, unsigned char *smem, const PdSmem &L, int tid) {
    int4 *sxq = reinterpret_cast<int4 *>(smem + L.off_xq);
    float *sxs = reinterpret_cast<float *>(smem + L.off_xs);
    const int4 *src = reinterpret_cast<const int4 *>(q);
    const int n16 = cols >> 4, nb = cols >> 5;
    for (int c0 = 0; c0 < n16; c0 += 4 * PD_CT) { // four 16-byte loads + one scale load in flight per thread: one L2 round trip for 16 K columns
        int4 v[4];
        float sc[2];
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int c = c0 + u * PD_CT + tid;
            v[u] = c < n16 ? __ldcg(src + c) : make_int4(0, 0, 0, 0);
        }
#pragma unroll
        for (int u = 0; u < 2; u++) {
            const int b = (c0 >> 1) + u * PD_CT + tid;
            sc[u] = b < nb ? __ldcg(s + b) : 0.0f;
        }
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int c = c0 + u * PD_CT + tid;
            if (c < n16) sxq[c] = v[u];
        }
#pragma unroll
        for (int u = 0; u < 2; u++) {
            const int b = (c0 >> 1) + u * PD_CT + tid;
            if (b < nb) sxs[b] = sc[u];
        }
    }
    pd_bar_sync();
}

// ---- one attention head with the consumer warps: k_attention's body (exact CPU order, InferenceCore.java:98-137) -------------
// h = local head index on this rank.
template <int HS>
__device__ __noinline__ void pd_attention_head(const PdArgs &a, const PdLayer &Ly, int h, int pos, unsigned char *smem, const PdSmem &L, int tid, int layer) {
    float *sm = reinterpret_cast<float *>(smem + L.off_nbuf);
    float *misc = reinterpret_cast<float *>(smem + L.off_misc);
    float *red = misc, *s_val = misc + 16;
    float *sq = sm, *sk = sm + HS, *so = sm + 2 * HS;
    const int ctx_pad = (a.ctx + PD_CT - 1) / PD_CT * PD_CT; // score rows are padded to whole accumulator chunks
    float *att = a.att_scratch ? a.att_scratch + (size_t)h * ctx_pad : sm + 3 * HS;
    const int lane = tid & 31, warp = tid >> 5;
    constexpr int HALF = HS / 2;
    const int nt = pos + 1;
    const int kv_mul = a.n_heads / a.n_kv_heads, kvh = h / kv_mul;
    const int qd = a.n_heads * HS, kvd = a.n_kv_heads * HS;
    float *qkv = a.qkv, *kc = Ly.kc, *vc = Ly.vc;
    const float *qsrc = qkv + h * HS, *ksrc = qkv + qd + kvh * HS, *vsrc = qkv + qd + kvd + kvh * HS;
    if (tid < HS) {
        const bool is_q = tid < HALF;
        const int p = is_q ? tid : tid - HALF;
        const float *src = is_q ? qsrc : ksrc;
        int i0, i1;
        if (a.arch & KF_NEOX) { i0 = p; i1 = p + HALF; } else { i0 = 2 * p; i1 = 2 * p + 1; }
        float v0 = ldcg_f32c(src + i0), v1 = ldcg_f32c(src + i1); // written by other CTAs in this kernel: bypass L1
        const float *srope = reinterpret_cast<const float *>(smem + L.off_rope); // this position's rope row, staged at kernel start
        const float fcr = srope[p], fci = srope[HALF + p];
        float cv0 = 0.f, cv1 = 0.f;
        const bool owner = (h % kv_mul == 0) && !is_q; // first query head of the KV group owns the cache write (InferenceCore.java:92-93)
        if (owner) { cv0 = ldcg_f32c(vsrc + i0); cv1 = ldcg_f32c(vsrc + i1); }
        if (a.arch & KF_QKNORM) { // Qwen3 per-head RMSNorm: literal sequential sum over the head (InferenceCore.java:594-600)
            float *sqr = is_q ? so : sk;
            sqr[i0] = __fmul_rn(v0, v0);
            sqr[i1] = __fmul_rn(v1, v1);
            asm volatile("bar.sync 3, %0;" ::"n"(HS) : "memory");
            if (p == 0) {
                float ss = 0.0f;
                for (int i = 0; i < HS; i++) ss = __fadd_rn(ss, sqr[i]);
                ss = __fdiv_rn(ss, (float)HS);
                ss = __fadd_rn(ss, a.eps);
                s_val[is_q ? 0 : 1] = (float)(1.0 / sqrt((double)ss));
            }
            asm volatile("bar.sync 3, %0;" ::"n"(HS) : "memory");
            const float ss = s_val[is_q ? 0 : 1];
            const float *nw = is_q ? Ly.q_norm : Ly.k_norm;
            v0 = __fmul_rn(nw[i0], __fmul_rn(ss, v0));
            v1 = __fmul_rn(nw[i1], __fmul_rn(ss, v1));
            asm volatile("bar.sync 3, %0;" ::"n"(HS) : "memory");
        }
        const float r0 = __fsub_rn(__fmul_rn(v0, fcr), __fmul_rn(v1, fci));
        const float r1 = __fadd_rn(__fmul_rn(v0, fci), __fmul_rn(v1, fcr));
        float *dst = is_q ? sq : sk;
        dst[i0] = r0;
        dst[i1] = r1;
        if (owner) {
            const size_t o = (size_t)pos * kvd + kvh * HS;
            kc[o + i0] = r0;
            kc[o + i1] = r1;
            vc[o + i0] = cv0;
            vc[o + i1] = cv1;
        }
    }
    pd_bar_sync();
    // ---- scores (scalarDot, FloatTensor.java:86-92: one sequential unfused mul/add chain per key).  Four threads share a key: each
    // loads ITS quarter of the K row at once (one L2 round trip per pass of PD_CT/4 keys instead of two dependent ones per key), then
    // the chain runs through the quad in element order, handed on by shuffle.  The V rows this thread will need are requested
    // here as well: they do not depend on the scores, so their round trip overlaps with everything up to the weighted sum.
    constexpr int QE = HS / 4, QV = HS / 16; // elements / 16-byte loads per quarter row
    const int quad = tid & 3, qbase = lane & ~3;
    constexpr int VB = 32;                   // V rows per thread and round of the weighted sum (4 threads per output element -> 128 keys per round)
    const int vd = tid >> 2;                 // output element of the weighted sum owned by this quad (HS <= PD_CT / 4)
    const bool vlive = vd < HS;
    float vv[VB];
    {
        const float *vcol = vc + kvh * HS + vd;
        const int vt0 = quad * VB;           // rows [vt0, vt0 + VB) of round 0
#pragma unroll
        for (int u = 0; u < VB; u++) vv[u] = (vlive && vt0 + u < pos) ? __ldcg(vcol + (size_t)(vt0 + u) * kvd) : 0.0f;
    }
    float lmax = -INFINITY;
#pragma unroll 1
    for (int t0 = 0; t0 < nt; t0 += PD_CT / 4) {
        const int t = t0 + (tid >> 2);
        float4 kk[QV];
        if (t < pos) { // rows of earlier tokens: written by earlier launches
            const float4 *k = reinterpret_cast<const float4 *>(kc + (size_t)t * kvd + kvh * HS + quad * QE);
#pragma unroll
            for (int u = 0; u < QV; u++) kk[u] = __ldcg(k + u);
        } else { // t == pos: this step's rotated k (shared memory); t > pos: idle slot
#pragma unroll
            for (int u = 0; u < QV; u++) kk[u] = t == pos ? *reinterpret_cast<const float4 *>(sk + quad * QE + 4 * u) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        float acc = 0.0f;
#pragma unroll 1
        for (int qd = 0; qd < 4; qd++) {
            if (quad == qd) {
                const float *qq = sq + qd * QE;
#pragma unroll
                for (int u = 0; u < QV; u++) {
                    acc = __fadd_rn(acc, __fmul_rn(qq[4 * u + 0], kk[u].x));
                    acc = __fadd_rn(acc, __fmul_rn(qq[4 * u + 1], kk[u].y));
                    acc = __fadd_rn(acc, __fmul_rn(qq[4 * u + 2], kk[u].z));
                    acc = __fadd_rn(acc, __fmul_rn(qq[4 * u + 3], kk[u].w));
                }
            }
            acc = __shfl_sync(0xffffffffu, acc, qbase + qd); // the chain so far, to the whole quad
        }
        if (quad == 0 && t < nt) {
            const float sc = __fdiv_rn(acc, a.sqrt_hs);
            att[t] = sc;
            lmax = fmaxf(lmax, sc);
        }
    }
    lmax = warp_max_f(lmax);
    if (lane == 0) red[warp] = lmax;
    pd_bar_sync();
    pd_stamp(a, layer, 13, tid);
    float mx = red[0];
#pragma unroll
    for (int w = 1; w < PD_WARPS; w++) mx = fmaxf(mx, red[w]);
    for (int t = tid; t < nt; t += PD_CT) att[t] = pd_exp_narrow(__fsub_rn(att[t], mx));
    pd_bar_sync();
    // sequential float sum (FloatTensor.softmaxInPlace, FloatTensor.java:211-219): short rows by one thread (16-byte loads ahead of
    // the add chain), long rows with the exact parallel accumulator (the terms are non-negative)
    float sum;
    if (nt >= 512) {
        const int E = (nt + PD_CT - 1) / PD_CT;
        for (int t = nt + tid; t < PD_CT * E; t += PD_CT) att[t] = 0.0f;
        pd_bar_sync();
        sum = pd_seqsum(att, nt, 0, smem, L, tid);
    } else {
        if (tid == 0) s_val[0] = seq2_literal(0.0f, att, nt, (reinterpret_cast<uintptr_t>(att) & 15) == 0);
        pd_bar_sync();
        sum = s_val[0];
    }
    for (int t = tid; t < nt; t += PD_CT) att[t] = __fdiv_rn(att[t], sum);
    pd_bar_sync();
    pd_stamp(a, layer, 14, tid);
    { // xb = sum_t a_t * v_t, sequentially over t per element (saxpyInPlace, FloatTensor.java:221-227).  Four threads per element: thread
      // `quad` holds rows [128 r + 32 quad, +32) of round r, all requested before the chain starts; the chain itself (4 cycles per key, the
      // floor of this phase) runs through the quad in row order.
        const float *vcol = vc + kvh * HS + vd;
        const float vcur = vlive ? ldcg_f32c(vsrc + vd) : 0.0f; // the current position's v, straight from the packed q|k|v vector
        float acc = 0.0f;
#pragma unroll 1
        for (int r0 = 0; r0 < pos; r0 += 4 * VB) {
            if (r0 > 0) { // round 0 was requested before the scores
                const int vt0 = r0 + quad * VB;
#pragma unroll
                for (int u = 0; u < VB; u++) vv[u] = (vlive && vt0 + u < pos) ? __ldcg(vcol + (size_t)(vt0 + u) * kvd) : 0.0f;
            }
#pragma unroll 1
            for (int qd = 0; qd < 4; qd++) {
                if (quad == qd) {
                    const int vt0 = r0 + qd * VB;
#pragma unroll
                    for (int u = 0; u < VB; u++)
                        if (vt0 + u < pos) acc = __fadd_rn(__fmul_rn(att[vt0 + u], vv[u]), acc);
                }
                acc = __shfl_sync(0xffffffffu, acc, qbase + qd);
            }
        }
        if (vlive && quad == 0) so[vd] = __fadd_rn(__fmul_rn(att[pos], vcur), acc);
    }
    pd_bar_sync();
    const int gh = a.head_base + h;
    for (int b = warp; b < HS / 32; b += PD_WARPS) {
        float as;
        const int q = pd_quant_block(so[b * 32 + lane], &as);
        if (a.tp.n > 1) { // all-gather: this head's quantised output goes straight into every rank's buffer
            for (int k = 0; k < a.tp.n; k++) {
                tp_ptr<int8_t>(a.tp, k, a.tp.off_attq)[gh * HS + b * 32 + lane] = (int8_t)q;
                if (lane == 0) tp_ptr<float>(a.tp, k, a.tp.off_atts)[(gh * HS) / 32 + b] = as;
            }
        } else {
            a.attq[gh * HS + b * 32 + lane] = (int8_t)q;
            if (lane == 0) a.atts[(gh * HS) / 32 + b] = as;
        }
    }
    pd_stamp(a, layer, 15, tid);
}

// ---- the kernel -----------------------------------------------------------------------------------------------------------
template <int HS>
__global__ void __launch_bounds__(PD_THREADS, 1) k_decode_persistent(const __grid_constant__ PdArgs a, const __grid_constant__ PdSmem L) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int S = L.stages;
    const unsigned bar0 = smem_u32(smem + L.off_bar);
    volatile unsigned *rel = reinterpret_cast<volatile unsigned *>(smem + L.off_bar + 2 * PD_MAX_STAGES * 8);
    if (tid == 0) {
        for (int s = 0; s < S; s++) {
            mbar_init(bar0 + 8 * s, 1);
            mbar_init(bar0 + 8 * (PD_MAX_STAGES + s), 1);
            rel[s] = 0u;
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (warp == PD_WARPS) { // ===== producer =====
        if (lane == 0) pd_produce(a, smem, L, bar0);
        return;
    }

    // ===== consumers =====
    const int token = a.st->token, pos = a.st->pos;
    const unsigned tick = *reinterpret_cast<volatile unsigned *>(a.sync + PD_S_TICK);
    const unsigned lmtick = *reinterpret_cast<volatile unsigned *>(a.sync + PD_S_LMTICK);
    const unsigned nC = gridDim.x, nL = (unsigned)a.n_layers, nH = (unsigned)a.n_heads;
    float *wbufA = reinterpret_cast<float *>(smem + L.off_wbuf), *wbufF = wbufA; // one buffer: every thread re-fills exactly the slots it has just read
    pd_prefetch_w(a.n_layers ? a.layers[0].attn_norm : a.out_norm, wbufA, a.dim, tid);
    if (tid < a.head_size) { // this position's rope row (RoPE.precomputeFreqsCis table), the same for every layer
        const int half = a.head_size >> 1;
        float *srope = reinterpret_cast<float *>(smem + L.off_rope);
        srope[tid] = tid < half ? __ldg(a.rope_cr + (size_t)pos * half + tid) : __ldg(a.rope_ci + (size_t)pos * half + (tid - half));
    }
    unsigned seq_base = 0;
#pragma unroll 1
    for (int l = 0; l < a.n_layers; l++) {
        const PdLayer &Ly = a.layers[l];
        const unsigned e = tick * nL + (unsigned)l + 1u; // this layer's epoch
        pd_stamp(a, l, 0, tid);
        pd_norm_to_smem(a, wbufA, l == 0, token, smem, L, tid, l);
        if (a.trace && l == 1) { // diagnostic (traced launch only): the same exact sum again, instruction cache warm -- stamps 16 -> 17 vs 10 -> 11
            const int E = (a.dim + PD_CT - 1) / PD_CT;
            pd_stamp(a, l, 16, tid);
            const float again = pd_seqsum(reinterpret_cast<const float *>(smem + L.off_nbuf), a.dim, seqsum2_stride(E), smem, L, tid);
            if (tid == 0) reinterpret_cast<float *>(smem + L.off_misc)[30] = again;
            pd_stamp(a, l, 17, tid);
        }
        pd_prefetch_w(Ly.ffn_norm, wbufF, a.dim, tid); // needed after the attention block
        pd_stamp(a, l, 1, tid);
        pd_consume_matrix<SMV_STORE>(Ly.qkv, a, smem, L, bar0, rel, seq_base, a.qkv, false, false, token, 0, tid);
        pd_stamp(a, l, 2, tid);
        if (blockIdx.x < nH) { // head CTAs: pull this layer's K/V rows of their KV head into L2 NOW -- a line survives only ~20 us in L2 under
            // the weight stream (126 MB at 5.6 TB/s), so the prefetch must sit just ahead of the scores, not at the top of the layer
            const int kvh = (int)blockIdx.x / (a.n_heads / a.n_kv_heads), kvd = a.n_kv_heads * a.head_size;
            const int lines = a.head_size >> 5; // 128-byte lines per row of one KV head
            for (int i = tid; i < pos * lines; i += PD_CT) { // plain L2 prefetches through the LSU: the TMA queue is busy refilling the ring right now
                const size_t off = (size_t)(i / lines) * kvd + kvh * a.head_size + (i % lines) * 32;
                asm volatile("prefetch.global.L2 [%0];" ::"l"(Ly.kc + off));
                asm volatile("prefetch.global.L2 [%0];" ::"l"(Ly.vc + off));
            }
        }
        pd_arrive(a, PD_S_QKV, e * nC, e, false, tid); // q/k/v of this rank's heads stay on this rank
        if (blockIdx.x < nH) { // attention: the first n_heads CTAs, one head each
            pd_wait(a, PD_S_QKV, e * nC, e, false, tid);
            pd_stamp(a, l, 12, tid);
            pd_attention_head<HS>(a, Ly, blockIdx.x, pos, smem, L, tid, l);
            pd_arrive(a, PD_S_ATT, e * nH, e, true, tid);
        }
        pd_wait(a, PD_S_ATT, e * nH, e, true, tid);
        pd_stamp(a, l, 3, tid);
        pd_load_act(a.attq, a.atts, a.qd, smem, L, tid);
        pd_consume_matrix<SMV_RESID>(Ly.wo, a, smem, L, bar0, rel, seq_base, a.x, false, l == 0, token, a.dim_base, tid);
        pd_stamp(a, l, 4, tid);
        pd_arrive(a, PD_S_WO, e * nC, e, true, tid);
        pd_wait(a, PD_S_WO, e * nC, e, true, tid);
        pd_stamp(a, l, 5, tid);
        pd_norm_to_smem(a, wbufF, false, token, smem, L, tid);
        pd_prefetch_w(l + 1 < a.n_layers ? a.layers[l + 1].attn_norm : a.out_norm, wbufA, a.dim, tid); // the next attn norm (or the final norm)
        pd_stamp(a, l, 6, tid);
        pd_consume_matrix<SMV_GATEUP>(Ly.gu, a, smem, L, bar0, rel, seq_base, a.hb, false, false, token, a.hid_base, tid);
        pd_stamp(a, l, 7, tid);
        pd_arrive(a, PD_S_GU, e * nC, e, true, tid);
        pd_wait(a, PD_S_GU, e * nC, e, true, tid);
        pd_load_act(a.hq, a.hs, a.hidden, smem, L, tid);
        pd_stamp(a, l, 8, tid);
        pd_consume_matrix<SMV_RESID>(Ly.w2, a, smem, L, bar0, rel, seq_base, a.x, false, false, token, a.dim_base, tid);
        pd_stamp(a, l, 9, tid);
        pd_arrive(a, PD_S_W2, e * nC, e, true, tid);
        pd_wait(a, PD_S_W2, e * nC, e, true, tid);
    }
    int best_i = 0;
    if (a.with_logits) {
        const unsigned le = lmtick + 1u;
        pd_stamp(a, a.n_layers, 0, tid);
        pd_norm_to_smem(a, wbufA, false, token, smem, L, tid);
        pd_stamp(a, a.n_layers, 1, tid);
        pd_consume_matrix<SMV_STORE>(a.lm_head, a, smem, L, bar0, rel, seq_base, a.logits, true, false, token, a.voc_base, tid);
        pd_stamp(a, a.n_layers, 2, tid);
        pd_arrive(a, PD_S_LM, le * nC, le, false, tid);
        if (blockIdx.x != 0) return;
        pd_wait(a, PD_S_LM, le * nC, le, false, tid);
        // FloatTensor.argmax over the per-CTA (max, first index) pairs: k_argmax_advance
        float best = -INFINITY;
        best_i = 0x7fffffff;
        for (int i = tid; i < (int)nC; i += PD_CT) argmax_merge(best, best_i, ldcg_f32c(a.part_val + i), __ldcg(a.part_idx + i));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, best, o);
            const int oi = __shfl_xor_sync(0xffffffffu, best_i, o);
            argmax_merge(best, best_i, ov, oi);
        }
        float *sv = reinterpret_cast<float *>(smem + L.off_misc) + 32;
        int *si = reinterpret_cast<int *>(sv + 16);
        if (lane == 0) { sv[warp] = best; si[warp] = best_i; }
        pd_bar_sync();
        if (tid == 0) {
            best = sv[0]; best_i = si[0];
            for (int w = 1; w < PD_WARPS; w++) argmax_merge(best, best_i, sv[w], si[w]);
            if (a.tp.n > 1) { // exchange every rank's (max, lowest global index) and merge identically everywhere
                for (int k = 0; k < a.tp.n; k++) {
                    tp_ptr<float>(a.tp, k, a.tp.off_pv)[a.tp.rank] = best;
                    tp_ptr<int>(a.tp, k, a.tp.off_pi)[a.tp.rank] = best_i;
                }
                __threadfence_system();
                for (int k = 0; k < a.tp.n; k++) {
                    unsigned *f = reinterpret_cast<unsigned *>(a.tp.peer[k] + a.pd_flags_off) + PD_S_ARG * TP_MAX + a.tp.rank;
                    asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(f), "r"(le) : "memory");
                }
                const unsigned *f = reinterpret_cast<const unsigned *>(a.tp.peer[a.tp.rank] + a.pd_flags_off) + PD_S_ARG * TP_MAX;
                for (int k = 0; k < a.tp.n; k++) pd_spin<true>(f + k, le, a.sync + PD_S_ERR, a.host_err, 1u + PD_S_ARG);
                best = -INFINITY; best_i = 0x7fffffff;
                for (int k = 0; k < a.tp.n; k++)
                    argmax_merge(best, best_i, ldcg_f32c(tp_ptr<float>(a.tp, a.tp.rank, a.tp.off_pv) + k),
                                 __float_as_int(ldcg_f32c(reinterpret_cast<const float *>(tp_ptr<int>(a.tp, a.tp.rank, a.tp.off_pi)) + k)));
            }
            if (best_i == 0x7fffffff) best_i = 0;
        }
    } else if (blockIdx.x != 0) {
        return;
    }
    if (tid == 0) { // step advance (k_argmax_advance's tail) + the next launch's epoch
        StepState *st = a.st;
        const int step = st->step;
        if (a.with_logits && a.out_ids) a.out_ids[step] = best_i;
        const int next = step + 1;
        if (st->feedback && a.with_logits) st->token = best_i;
        else if (next < st->n_seq) st->token = a.seq_tokens[next];
        st->step = next;
        st->pos = st->pos + 1;
        *reinterpret_cast<volatile unsigned *>(a.sync + PD_S_TICK) = tick + 1u;
        if (a.with_logits) *reinterpret_cast<volatile unsigned *>(a.sync + PD_S_LMTICK) = lmtick + 1u;
        pd_stamp(a, a.n_layers, 3, tid);
    }
}
