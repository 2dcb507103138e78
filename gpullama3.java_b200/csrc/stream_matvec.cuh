// stream_matvec.cuh -- the decode hot kernel: Q8_0 dequant-matvec as a persistent, TMA-fed
// weight stream (sm_100a).
//
// One CTA per SM.  A single producer thread walks this CTA's static slice of the weight matrix
// and keeps a ring of shared-memory stages full with 1-D bulk async copies
// (cp.async.bulk ... mbarrier::complete_tx, SASS UBLKCP); eight consumer warps pop tiles, do the
// int8 x int8 dot products with dp4a and reduce each row's per-block terms in the exact order of
// Q8_0FloatTensor.dotQ8Activation (Q8_0FloatTensor.java:90-123).  The producer never waits for
// anything but ring space: under programmatic dependent launch the NEXT matvec kernel is already
// resident and fills its ring with (immutable) weights while the current kernel, the RMSNorm or
// the attention kernel are still running, so HBM keeps streaming across kernel boundaries.
//
// Device weight layout ("tile-major", built once at upload; same 1.0625 B/element as GGUF):
//   rows are taken in groups of 4; a row is cut into nseg segments of SEG columns;
//   unit(r, s)  = SEG int8 quants followed by SEG/32 f16 block scales, padded to 16 bytes;
//   tile(G, s)  = units (4G..4G+3, s) back to back   -> ONE bulk copy;
//   tiles are stored in (G, s) order, so a CTA's slice [G0, G1) is one contiguous byte range.
//   For the fused gate/up projection group G holds rows {gate 2G, gate 2G+1, up 2G, up 2G+1}.
#pragma once
#include "common.cuh"

#define SMV_CONSUMER_WARPS 8
#define SMV_THREADS ((SMV_CONSUMER_WARPS + 1) * 32)
#define SMV_MAX_STAGES 16
#define SMV_HVALS 512 // capacity (hidden units per CTA) of the gate/up epilogue buffer

enum { SMV_STORE = 0, SMV_RESID = 1, SMV_GATEUP = 2 };

struct TileMat { // device weight matrix in tile-major layout
    const unsigned char *base;
    int rows, cols;  // rows = 4 * groups (for gate/up: 2 * hidden)
    int seg, nseg;   // columns per segment, segments per row
    int unit_bytes;  // seg + seg/16 rounded up to 16
};

__host__ __device__ inline int smv_pick_nseg(int cols) {
    for (int n = 1; n <= 64; n++)
        if (cols % n == 0 && (cols / n) % 32 == 0 && cols / n <= 2560) return n;
    return 0;
}
__host__ __device__ inline int smv_unit_bytes(int seg) { return (seg + seg / 16 + 15) & ~15; }

struct SmvSmem {
    size_t off_bar, off_xq, off_xs, off_terms, off_hvals, off_ring, total;
    int stages, stage_bytes, nbs_pad;
};

__host__ __device__ inline SmvSmem smv_layout(int cols, int seg, size_t budget) {
    SmvSmem L;
    int unit = smv_unit_bytes(seg);
    L.stage_bytes = (4 * unit + 127) & ~127;
    L.nbs_pad = ((seg / 32 + 3) & ~3) + 4; // row stride of the term buffer: 16-byte aligned rows, the four walker lanes on distinct banks
    size_t o = 0;
    L.off_bar = o; o += 2 * SMV_MAX_STAGES * 8 + SMV_MAX_STAGES * 4; // full[], empty[] mbarriers + release counters
    L.off_xq = o; o += (size_t)cols;
    L.off_xs = o; o += (size_t)(cols / 32) * 4;
    o = (o + 15) & ~(size_t)15;
    L.off_terms = o; o += (size_t)SMV_CONSUMER_WARPS * 4 * L.nbs_pad * 4;
    L.off_hvals = o; o += SMV_HVALS * 4; // GATEUP: this CTA's swiglu outputs; STORE+argmax: per-warp candidates
    o = (o + 127) & ~(size_t)127;
    L.off_ring = o;
    long room = (long)budget - (long)o;
    int s = room > 0 ? (int)(room / L.stage_bytes) : 0;
    if (s > SMV_MAX_STAGES) s = SMV_MAX_STAGES;
    L.stages = s;
    L.total = o + (size_t)s * L.stage_bytes;
    return L;
}

// ---- mbarrier / bulk-copy / PDL primitives (inline PTX) ---------------------------------------
__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(unsigned bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(bar), "r"(parity)
        : "memory");
}
// Global -> shared bulk copy with an L2 evict_first policy: single-use weight tiles must not push the KV rows, activations and norm weights out of L2
// (measured on the persistent kernel: +6 % tokens/s, profiles/r2_run6_evict_first_qwen3.log).
__device__ __forceinline__ unsigned long long l2_policy_evict_first() {
    unsigned long long pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void bulk_g2s_evict_first(unsigned dst, const void *src, unsigned bytes, unsigned bar, unsigned long long pol) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(dst), "l"(src),
                 "r"(bytes), "r"(bar), "l"(pol)
                 : "memory");
}
__device__ __forceinline__ void consumer_bar_sync() { asm volatile("bar.sync 1, %0;" ::"n"(SMV_CONSUMER_WARPS * 32) : "memory"); }

__device__ __forceinline__ float ldcg_f32(const float *p) {
    float v;
    asm volatile("ld.global.cg.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}

__device__ __forceinline__ float swiglu_exact(float g, float u) { // InferenceCore.java:150-158
    float s = __fdiv_rn(g, (float)(1.0 + exp((double)(-g))));
    return __fmul_rn(s, u);
}

// The ordered sum of one row's block terms (Q8_0FloatTensor.java:117-121: result += ..., block after block).  The add chain is
// inherently serial (4 cycles per term); what can be taken off it is the shared-memory latency: 16 terms are fetched with four
// 16-byte loads while the previous 16 are being added.
__device__ __forceinline__ float pd_walk_terms(float acc, const float *t, int nbs) {
    int b = 0;
    if (nbs >= 16) {
        float4 c0 = *reinterpret_cast<const float4 *>(t), c1 = *reinterpret_cast<const float4 *>(t + 4);
        float4 c2 = *reinterpret_cast<const float4 *>(t + 8), c3 = *reinterpret_cast<const float4 *>(t + 12);
        for (; b + 16 <= nbs; b += 16) {
            float4 n0 = c0, n1 = c1, n2 = c2, n3 = c3;
            if (b + 32 <= nbs) {
                n0 = *reinterpret_cast<const float4 *>(t + b + 16); n1 = *reinterpret_cast<const float4 *>(t + b + 20);
                n2 = *reinterpret_cast<const float4 *>(t + b + 24); n3 = *reinterpret_cast<const float4 *>(t + b + 28);
            }
            acc = __fadd_rn(acc, c0.x); acc = __fadd_rn(acc, c0.y); acc = __fadd_rn(acc, c0.z); acc = __fadd_rn(acc, c0.w);
            acc = __fadd_rn(acc, c1.x); acc = __fadd_rn(acc, c1.y); acc = __fadd_rn(acc, c1.z); acc = __fadd_rn(acc, c1.w);
            acc = __fadd_rn(acc, c2.x); acc = __fadd_rn(acc, c2.y); acc = __fadd_rn(acc, c2.z); acc = __fadd_rn(acc, c2.w);
            acc = __fadd_rn(acc, c3.x); acc = __fadd_rn(acc, c3.y); acc = __fadd_rn(acc, c3.z); acc = __fadd_rn(acc, c3.w);
            c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        }
    }
    for (; b + 4 <= nbs; b += 4) {
        const float4 v = *reinterpret_cast<const float4 *>(t + b);
        acc = __fadd_rn(acc, v.x); acc = __fadd_rn(acc, v.y); acc = __fadd_rn(acc, v.z); acc = __fadd_rn(acc, v.w);
    }
    for (; b < nbs; b++) acc = __fadd_rn(acc, t[b]);
    return acc;
}

struct SmvArgs {
    TileMat W;
    const int8_t *xq;   // pre-quantised activation [cols]
    const float *xs;    // its block scales [cols/32]
    float *out;         // STORE: out[row] = r; RESID: out[row] += r; GATEUP: hb[unit] (float, also read back)
    int8_t *hq;         // GATEUP: quantised hb
    float *hs;          // GATEUP: hb block scales
    unsigned *blk_cnt;  // GATEUP: per-32-block arrival counters (self-resetting)
    float *part_val;    // STORE (lm_head): per-CTA running maximum of the rows it produced ...
    int *part_idx;      // ... and the lowest row index attaining it (FloatTensor.argmax tie-break), or NULL
    TraceBuf tr;
    // tensor parallelism (tp.n == 1: unused)
    TpCtx tp;
    int wait_slot;      // slot whose flags gate the activation (-1: none)
    unsigned wait_op;
    int out_slot;       // slot to raise after this kernel's peer stores (-1: outputs stay local)
    unsigned out_op;
    int row_base;       // global index of this rank's first output row (RESID/STORE) or hidden unit (GATEUP)
};

template <int MODE>
__global__ void __launch_bounds__(SMV_THREADS, 1) k_stream_matvec_q8(SmvArgs a, SmvSmem L) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const TileMat W = a.W;
    const int S = L.stages;
    const unsigned bar0 = smem_u32(smem + L.off_bar); // full[s] at bar0 + 8s, empty[s] at bar0 + 8(S_MAX + s)
    const int ngroups = W.rows >> 2;
    const int g0 = (int)(((long long)blockIdx.x * ngroups) / gridDim.x);
    const int g1 = (int)(((long long)(blockIdx.x + 1) * ngroups) / gridDim.x);
    const int nseg = W.nseg;
    const unsigned tile_bytes = 4u * (unsigned)W.unit_bytes;

    // rel[st] = number of tiles consumed from stage st so far.  The consumer warps advance
    // independently, so a warp can reach the tile of lap k+2 of a stage while lap k+1 is still in
    // flight; a parity wait cannot tell those apart, the counter can.
    volatile unsigned *rel = reinterpret_cast<volatile unsigned *>(smem + L.off_bar + 2 * SMV_MAX_STAGES * 8);
    if (tid == 0) {
        for (int s = 0; s < S; s++) {
            mbar_init(bar0 + 8 * s, 1);
            mbar_init(bar0 + 8 * (SMV_MAX_STAGES + s), 1);
            rel[s] = 0u;
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    trace_entry(a.tr);
    pdl_launch_dependents(); // let the next kernel become resident and start prefetching its weights

    if (warp == SMV_CONSUMER_WARPS) {
        // ===== producer: weights are immutable, so it does not wait for the previous kernel =====
        if (lane == 0) {
            unsigned seq = 0;
            const unsigned long long pol = l2_policy_evict_first();
            for (int gb = g0; gb < g1; gb += SMV_CONSUMER_WARPS) {
                int nw = min(SMV_CONSUMER_WARPS, g1 - gb);
                for (int s = 0; s < nseg; s++)
#pragma unroll 1 // one copy per iteration: the producer is a single thread, its code size is what matters
                    for (int w = 0; w < nw; w++, seq++) {
                        int st = seq % S;
                        unsigned ph = (seq / S) & 1u;
                        mbar_wait(bar0 + 8 * (SMV_MAX_STAGES + st), ph ^ 1u); // slot free (first pass returns at once)
                        unsigned full = bar0 + 8 * st;
                        mbar_expect_tx(full, tile_bytes);
                        const unsigned char *src = W.base + ((size_t)(gb + w) * nseg + s) * tile_bytes;
                        bulk_g2s_evict_first(smem_u32(smem + L.off_ring + (size_t)st * L.stage_bytes), src, tile_bytes, full, pol);
                    }
            }
        }
        return;
    }

    // ===== consumers =====
    pdl_wait(); // activations come from the previous kernel
    trace_mark(a.tr, 2);
    if (a.tp.n > 1 && a.wait_slot >= 0) { // ... and, under TP, from every rank
        if (tid == 0) tp_wait(a.tp, a.wait_slot, tp_seq(a.tp, a.wait_op));
        consumer_bar_sync();
    }
    {
        const int nb = W.cols >> 5;
        int4 *sxq = reinterpret_cast<int4 *>(smem + L.off_xq);
        float *sxs = reinterpret_cast<float *>(smem + L.off_xs);
        const int4 *src = reinterpret_cast<const int4 *>(a.xq);
        for (int c = tid; c < W.cols / 16; c += SMV_CONSUMER_WARPS * 32) sxq[c] = __ldcg(src + c);
        for (int b = tid; b < nb; b += SMV_CONSUMER_WARPS * 32) sxs[b] = __ldcg(a.xs + b);
    }
    consumer_bar_sync();

    const int nbs = W.seg >> 5; // blocks per segment
    float *terms = reinterpret_cast<float *>(smem + L.off_terms) + (size_t)warp * 4 * L.nbs_pad;
    const unsigned char *sact = smem + L.off_xq;
    const float *sxs = reinterpret_cast<const float *>(smem + L.off_xs);
    const int hsel = (lane >> 2) & 1; // half-swap: conflict-free LDS.128 over 32-byte strides

    float *hvals = reinterpret_cast<float *>(smem + L.off_hvals);
    float best = -INFINITY;
    int best_i = 0x7fffffff;

    unsigned seq_base = 0;
    for (int gb = g0; gb < g1; gb += SMV_CONSUMER_WARPS) {
        const int nw = min(SMV_CONSUMER_WARPS, g1 - gb);
        if (warp < nw) {
            const int G = gb + warp;
            float acc = 0.0f; // lanes 0..3: running row sums
            for (int s = 0; s < nseg; s++) {
                const unsigned seq = seq_base + (unsigned)(s * nw + warp);
                const int st = seq % S;
                const unsigned lap = seq / S;
                if (lane == 0)
                    while (rel[st] != lap) {} // every earlier occupant of this stage has been consumed
                __syncwarp();
                mbar_wait(bar0 + 8 * st, lap & 1u);
                const unsigned char *tile = smem + L.off_ring + (size_t)st * L.stage_bytes;
                for (int b = lane; b < nbs; b += 32) {
                    const unsigned char *ab = sact + ((size_t)(s * nbs + b) << 5);
                    const int4 a0 = *reinterpret_cast<const int4 *>(ab + 16 * hsel);
                    const int4 a1 = *reinterpret_cast<const int4 *>(ab + 16 * (hsel ^ 1));
                    const float as = sxs[s * nbs + b];
#pragma unroll
                    for (int r = 0; r < 4; r++) {
                        const unsigned char *wb = tile + (size_t)r * W.unit_bytes + ((size_t)b << 5);
                        const int4 w0 = *reinterpret_cast<const int4 *>(wb + 16 * hsel);
                        const int4 w1 = *reinterpret_cast<const int4 *>(wb + 16 * (hsel ^ 1));
                        const __half sc = *reinterpret_cast<const __half *>(tile + (size_t)r * W.unit_bytes + W.seg + 2 * b);
                        int isum = __dp4a(w0.x, a0.x, 0);
                        isum = __dp4a(w0.y, a0.y, isum);
                        isum = __dp4a(w0.z, a0.z, isum);
                        isum = __dp4a(w0.w, a0.w, isum);
                        isum = __dp4a(w1.x, a1.x, isum);
                        isum = __dp4a(w1.y, a1.y, isum);
                        isum = __dp4a(w1.z, a1.z, isum);
                        isum = __dp4a(w1.w, a1.w, isum);
                        terms[r * L.nbs_pad + b] = __fmul_rn((float)isum, __fmul_rn(__half2float(sc), as));
                    }
                }
                __syncwarp();
                if (lane == 0) { // weights consumed: slot back to the producer
                    rel[st] = lap + 1u;
                    mbar_arrive(bar0 + 8 * (SMV_MAX_STAGES + st));
                }
                if (lane < 4) acc = pd_walk_terms(acc, terms + lane * L.nbs_pad, nbs); // strictly in block order
                __syncwarp();
            }
            // rows 4G..4G+3 are complete in lanes 0..3
            if (MODE == SMV_GATEUP) {
                const float up = __shfl_down_sync(0xffffffffu, acc, 2);
                if (lane < 2) {
                    const int unit = 2 * G + lane;
                    const float hval = swiglu_exact(acc, up);
                    a.out[unit] = hval;
                    hvals[unit - 2 * g0] = hval;
                }
            } else if (lane < 4) {
                const size_t row = (size_t)4 * G + lane;
                if (MODE == SMV_RESID) {
                    if (a.tp.n > 1) { // all-gather of the residual stream: this rank's rows go to every rank
                        const size_t grow = (size_t)a.row_base + row;
                        const float v = __fadd_rn(ldcg_f32c(a.out + grow), acc);
                        for (int k = 0; k < a.tp.n; k++) tp_ptr<float>(a.tp, k, a.tp.off_x)[grow] = v;
                    } else a.out[row] = __fadd_rn(a.out[row], acc); // x[i] = x[i] + xb2[i]
                } else {
                    a.out[row] = acc;
                    const int grow = a.row_base + (int)row;
                    if (acc > best) { best = acc; best_i = grow; } // rows ascend per lane: first maximum kept
                }
            }
        }
        seq_base += (unsigned)(nseg * nw);
    }

    if (MODE == SMV_GATEUP) {
        // Quantise hb = silu(gate)*up to Q8_0 (the activation of the down projection,
        // Q8_0FloatTensor.java:100-117).  Blocks of 32 units that lie wholly inside this CTA's range are
        // quantised from shared memory; the (at most two) blocks shared with a neighbouring CTA are finished
        // by whichever CTA arrives last (fence + counter), so no warp ever fences inside the streaming loop.
        consumer_bar_sync();
        const int u0 = 2 * g0, u1 = 2 * g1;
        if (u1 > u0) {
            for (int blk = (u0 >> 5) + warp; blk <= ((u1 - 1) >> 5); blk += SMV_CONSUMER_WARPS) {
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
                        v = ldcg_f32(a.out + (blk << 5) + lane);
                        if (lane == 0) a.blk_cnt[blk] = 0u;
                    }
                }
                if (mine) {
                    float as;
                    int q = quant_block_lane(v, as);
                    if (a.tp.n > 1) {
                        const int gblk = (a.row_base >> 5) + blk;
                        for (int k = 0; k < a.tp.n; k++) {
                            tp_ptr<int8_t>(a.tp, k, a.tp.off_hq)[(gblk << 5) + lane] = (int8_t)q;
                            if (lane == 0) tp_ptr<float>(a.tp, k, a.tp.off_hs)[gblk] = as;
                        }
                    } else {
                        a.hq[(blk << 5) + lane] = (int8_t)q;
                        if (lane == 0) a.hs[blk] = as;
                    }
                }
            }
        }
    } else if (MODE == SMV_STORE) {
        if (a.part_val) { // on-device greedy sampler, stage 1: this CTA's (max, first index)
            int *cand_i = reinterpret_cast<int *>(hvals + 64);
            if (lane < 4) { hvals[warp * 4 + lane] = best; cand_i[warp * 4 + lane] = best_i; }
            consumer_bar_sync();
            if (tid == 0) {
                float bv = -INFINITY;
                int bi = 0x7fffffff;
                for (int k = 0; k < SMV_CONSUMER_WARPS * 4; k++) {
                    float v = hvals[k];
                    int ix = cand_i[k];
                    if (v > bv || (v == bv && ix < bi)) { bv = v; bi = ix; }
                }
                a.part_val[blockIdx.x] = bv;
                a.part_idx[blockIdx.x] = bi;
            }
        }
    }
    if (a.tp.n > 1 && a.out_slot >= 0) { // publish: all peer stores of this CTA, then (last CTA) the flag
        consumer_bar_sync(); // the CTA's stores are ordered before thread 0's device-scope fence + counter (tp_cta_done);
        if (tid == 0) tp_cta_done(a.tp, a.out_slot, tp_seq(a.tp, a.out_op), gridDim.x); // only the LAST CTA pays the system-scope fence
    }
    trace_mark(a.tr, 3);
}

// ---- upload-time repack: GGUF Q8_0 blocks (34 B: f16 scale + 32 int8) -> tile-major -----------
// One thread per 16-bit word of the destination tile payload.  src_row(g, r) gives the source row
// of group g, slot r: identity for plain matrices, the gate/up interleave for the fused FFN matrix.
struct RepackSrc {
    const unsigned char *raw[3]; // up to three source tensors stacked by rows (q|k|v), or gate/up
    int rows[3];
    int row0[3];                 // first source row of each part (tensor-parallel slices)
    int gateup;                  // 1: raw[0] = gate, raw[1] = up, group G = {g 2G, g 2G+1, u 2G, u 2G+1}
};

__global__ void k_repack_tiles(RepackSrc src, unsigned char *dst, int rows, int cols, int seg, int nseg, int unit_bytes) {
    // grid.x over (group, segment, slot) units; threads over 16-bit words of one unit
    const long long unit_id = blockIdx.x;
    const int r = (int)(unit_id % 4);
    const int s = (int)((unit_id / 4) % nseg);
    const long long G = unit_id / (4LL * nseg);
    long long row;
    const unsigned char *raw;
    if (src.gateup) {
        raw = src.raw[r >> 1];
        row = src.row0[r >> 1] + 2 * G + (r & 1);
    } else {
        row = 4 * G + r;
        int k = 0;
        while (k < 2 && row >= src.rows[k]) { row -= src.rows[k]; k++; }
        raw = src.raw[k];
        row += src.row0[k];
    }
    const int nbs = seg / 32;
    const unsigned char *blocks = raw + ((size_t)row * (cols / 32) + (size_t)s * nbs) * 34; // first source block of this unit
    unsigned char *u = dst + (size_t)unit_id * unit_bytes;
    const int words = unit_bytes / 2;
    for (int w = threadIdx.x; w < words; w += blockDim.x) {
        unsigned short v = 0;
        if (w < seg / 2) { // quant payload: word w -> block w/16, word-in-block w%16
            int b = w >> 4, k = w & 15;
            v = *reinterpret_cast<const unsigned short *>(blocks + (size_t)b * 34 + 2 + 2 * k);
        } else if (w < seg / 2 + nbs) {
            int b = w - seg / 2;
            v = *reinterpret_cast<const unsigned short *>(blocks + (size_t)b * 34);
        }
        reinterpret_cast<unsigned short *>(u)[w] = v;
    }
}

// ---- inverse of the repack: tile-major Q8_0 stream -> row-major f16 matrix (value = f16(q * scale)) ----------------
// One CTA per unit (group G, segment s, slot r).  Plain matrices: row 4G + r of out0.  Gate/up stream: slots 0,1 are
// gate rows 2G, 2G+1 (out0), slots 2,3 the up rows (out1).
__global__ void k_tiles_to_f16(TileMat W, int gateup, __half *__restrict__ out0, __half *__restrict__ out1) {
    const long long unit_id = blockIdx.x;
    const int r = (int)(unit_id % 4);
    const int s = (int)((unit_id / 4) % W.nseg);
    const long long G = unit_id / (4LL * W.nseg);
    __half *out = gateup && (r >> 1) ? out1 : out0;
    const long long row = gateup ? 2 * G + (r & 1) : 4 * G + r;
    const unsigned char *u = W.base + (size_t)unit_id * W.unit_bytes;
    const __half *sc = reinterpret_cast<const __half *>(u + W.seg);
    __half2 *dst = reinterpret_cast<__half2 *>(out + (size_t)row * W.cols + (size_t)s * W.seg);
    for (int i = threadIdx.x; i < W.seg / 2; i += blockDim.x) {
        const unsigned short w = reinterpret_cast<const unsigned short *>(u)[i];
        const float f = __half2float(sc[i >> 4]);
        dst[i] = __floats2half2_rn((float)(signed char)(w & 0xFF) * f, (float)(signed char)(w >> 8) * f);
    }
}
