// seqsum2.cuh -- the exact sequential-sum accumulator of the decode path's RMSNorms (round 2; the algorithm is validated on
// the CPU by tools/seqsum2/proto.c, on the GPU by tools/seqsum2/harness.cu and tests/test_gpu_parity.py).
//
// The bit-exact value of  s = 0; for (i) s = s + t[i]  for non-negative float terms (InferenceCore.rmsnorm's accumulator,
// InferenceCore.java:39-48), evaluated by one CTA.  Float addition is not associative, so a tree reduction gives different
// bits, and a literal chain costs ~8-10 cycles per term on one thread.  While the running sum s stays inside one binade
// [2^e, 2^(e+1)) its mantissa M is an integer in units of u = 2^(e-23), and adding a term t rounds to  M + k + [f > 1/2]
// with t/u = k + f (on an exact tie, f == 1/2, round-half-even makes the increment depend on the parity of M).  So inside a
// binade a step is the integer map  M -> M + a[M & 1], and such maps compose associatively.  The sum is three block-wide
// scans and a ~25-item serial walk:
//   1. float prefix P over per-thread sums (E consecutive terms per thread)            -> predicted binade per thread
//   2. a thread whose P range lies well inside one binade composes its E steps  M -> M + a[M & 1]  (SeqPair)
//      into one pair ("clean"); any other thread is "literal"
//   3. segmented scan of the pairs over runs of clean threads with equal binade          (pairs compose associatively)
//   4. item list (ballot/popc compaction): one item per literal thread and one per run
//   5. one thread walks the items: literal = E real float adds; run = verify (exponent on entry, mantissa < 2^24 on
//      exit) and add the integer; a failed check replays the run literally.  Predictions decide speed, never the result.
// CPU model (20000 adversarial cases, n = 2048/4096/8192): 0 mismatches, ~3 head threads + ~24 items per sum.
#pragma once
#include "common.cuh"

#define SEQSUM2_THREADS 1024
#define SEQSUM2_LITERAL INT_MIN

struct SeqPair { // the step  M -> M + a[M & 1]
    unsigned a0, a1;
};
__device__ __forceinline__ SeqPair seq_compose(SeqPair L, SeqPair R) { // apply L, then R
    SeqPair o;
    o.a0 = L.a0 + ((L.a0 & 1u) ? R.a1 : R.a0);
    o.a1 = L.a1 + (((1u + L.a1) & 1u) ? R.a1 : R.a0);
    o.a0 = min(o.a0, 1u << 26); // saturate: anything >= 2^24 fails verification anyway
    o.a1 = min(o.a1, 1u << 26);
    return o;
}

__device__ __forceinline__ int f32_exponent(float f) { return (int)((__float_as_uint(f) >> 23) & 0xffu) - 127; }

// Parity pair of adding t to a running sum in binade e (ulp 2^(e-23)).  Returns false when t >= 2^(e+1)
// (not a within-binade step).
__device__ __forceinline__ bool seq_pair(float t, int e, SeqPair &pr) {
    const unsigned tb = __float_as_uint(t);
    const int et = (int)(tb >> 23);
    pr.a0 = pr.a1 = 0u;
    if (et == 0) return true; // zero / denormal term: far below half an ulp (e >= -90)
    const unsigned m = (tb & 0x7fffffu) | 0x800000u;
    int shift = (e + 127) - et; // t / ulp = m * 2^-shift
    if (shift < 0) return false;
    if (shift > 25) shift = 25;
    const unsigned k = m >> shift;
    const unsigned rem = m & ((1u << shift) - 1u);
    const unsigned half = shift ? (1u << (shift - 1)) : 0u;
    if (shift && rem == half) { // exact tie: the result mantissa M + k + r must be even
        pr.a0 = k + (k & 1u);
        pr.a1 = k + ((k + 1u) & 1u);
    } else {
        pr.a0 = pr.a1 = k + ((shift && rem > half) ? 1u : 0u);
    }
    return true;
}

struct SeqItem {
    int cls;          // SEQSUM2_LITERAL or the binade of a run
    unsigned a0, a1;  // the run's composed pair
    int last;         // thread that closes the item (its own id for a literal thread)
};

struct SeqSum2Scratch {
    float *wsum;      // [32] warp totals -> exclusive warp prefixes
    SeqPair *wtail;   // [32] pair of the run that is open at the end of each warp
    int *wtail_f;     // [32] 1: that run started inside the warp
    int *wcls_last;   // [32] class of the warp's last thread
    int *wcls_first;  // [32] class of the warp's first thread
    int *wcnt;        // [32] items per warp -> exclusive offsets
    int *cls;         // [T]  class per thread (fallback walks back over it)
    SeqItem *items;   // [T]
    float *result;    // [1]
    int *info;        // [2] {items, fallbacks}
};
__host__ __device__ inline size_t seqsum2_scratch_bytes(int T = SEQSUM2_THREADS) { // T = threads that run the accumulator
    return 32 * 4 + 32 * sizeof(SeqPair) + 4 * 32 * 4 + (size_t)T * 4 + (size_t)T * sizeof(SeqItem) + 16 + 16;
}
__device__ __forceinline__ SeqSum2Scratch seqsum2_carve(unsigned char *p, int T = SEQSUM2_THREADS) { // p 16-byte aligned
    SeqSum2Scratch s;
    s.items = reinterpret_cast<SeqItem *>(p); p += (size_t)T * sizeof(SeqItem);
    s.wtail = reinterpret_cast<SeqPair *>(p); p += 32 * sizeof(SeqPair);
    s.cls = reinterpret_cast<int *>(p); p += (size_t)T * 4;
    s.wsum = reinterpret_cast<float *>(p); p += 32 * 4;
    s.wtail_f = reinterpret_cast<int *>(p); p += 32 * 4;
    s.wcls_last = reinterpret_cast<int *>(p); p += 32 * 4;
    s.wcls_first = reinterpret_cast<int *>(p); p += 32 * 4;
    s.wcnt = reinterpret_cast<int *>(p); p += 32 * 4;
    s.result = reinterpret_cast<float *>(p); p += 16;
    s.info = reinterpret_cast<int *>(p);
    return s;
}

// Segmented inclusive scan step set over one warp: f = 1 when the run containing this lane starts inside the covered range.
// (Code size matters more than instruction count here: these phases run once per call on a cold instruction cache, so every
// loop is kept rolled and the helpers out of line -- a taken branch into code that is not cached costs more than the loop.)
__device__ __noinline__ void seq2_warp_segscan(SeqPair &p, int &f, int lane) {
#pragma unroll 1
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned u0 = __shfl_up_sync(0xffffffffu, p.a0, d), u1 = __shfl_up_sync(0xffffffffu, p.a1, d);
        const int fu = __shfl_up_sync(0xffffffffu, f, d);
        if (lane >= d && !f) {
            SeqPair L;
            L.a0 = u0; L.a1 = u1;
            p = seq_compose(L, p);
            f = fu;
        }
    }
}

struct SeqSum2BlockSync {
    __device__ __forceinline__ void operator()() const { __syncthreads(); }
};

// Chunk stride that makes the 16-byte reads of consecutive threads hit distinct shared-memory banks (E = terms per thread):
// thread t's terms live at sq[t * S .. t * S + E).  E = 16 -> 20, 8 -> 12, 32 -> 36, 4 -> 4.
__host__ __device__ inline int seqsum2_stride(int E) { return (E % 4 == 0 && (E / 4) % 2 == 0) ? E + 4 : E; }

// literal adds of one thread's E terms (16-byte loads when the layout allows)
__device__ __noinline__ float seq2_literal(float s, const float *q, int E, bool vec) {
    int k = 0;
    if (vec) {
#pragma unroll 1
        for (; k + 4 <= E; k += 4) {
            const float4 v = *reinterpret_cast<const float4 *>(q + k);
            s = __fadd_rn(s, v.x); s = __fadd_rn(s, v.y); s = __fadd_rn(s, v.z); s = __fadd_rn(s, v.w);
        }
    }
#pragma unroll 1
    for (; k < E; k++) s = __fadd_rn(s, q[k]);
    return s;
}

// inclusive float prefix over the 32 lanes of a warp (predictor only: plain adds)
__device__ __noinline__ float seq2_warp_scan_f(float v, int lane) {
#pragma unroll 1
    for (int d = 1; d < 32; d <<= 1) {
        const float u = __shfl_up_sync(0xffffffffu, v, d);
        if (lane >= d) v += u;
    }
    return v;
}

// sq: n terms, thread t's E = ceil(n / T) consecutive terms at sq[t * S + k] (S >= E; S = E is the plain contiguous layout),
// zero-padded up to T whole chunks.  Exactly T threads (a multiple of 32, at most SEQSUM2_THREADS) call this with tid in
// [0, T); `sync` is a barrier over those T threads (the whole CTA, or a named barrier over a subset of its warps as in the
// persistent decode kernel).  When S and E are multiples of 4 and sq is 16-byte aligned the terms are read with 16-byte loads.
template <int T, class Sync>
__device__ float block_seqsum_exact_v2_t(const float *sq, int n, SeqSum2Scratch sc, int tid, Sync sync, int S = 0) {
    static_assert(T % 32 == 0 && T <= SEQSUM2_THREADS, "T threads = T/32 whole warps");
    constexpr int NW = T / 32;
    const int lane = tid & 31, warp = tid >> 5;
    const int E = (n + T - 1) / T;
    if (S == 0) S = E;
    const bool vec = ((E | S) & 3) == 0 && (reinterpret_cast<uintptr_t>(sq) & 15) == 0;
    const float *mine = sq + tid * S;

    // ---- 1. float prefix over per-thread sums
    float loc = 0.0f;
    {
        int k = 0;
        if (vec) {
#pragma unroll 1
            for (; k < E; k += 4) {
                const float4 v = *reinterpret_cast<const float4 *>(mine + k);
                loc += v.x; loc += v.y; loc += v.z; loc += v.w;
            }
        }
#pragma unroll 1
        for (; k < E; k++) loc += mine[k];
    }
    const float inc = seq2_warp_scan_f(loc, lane);
    if (lane == 31) sc.wsum[warp] = inc;
    sync();
    if (warp == 0) {
        const float w = lane < NW ? sc.wsum[lane] : 0.0f;
        const float v = seq2_warp_scan_f(w, lane);
        if (lane < NW) sc.wsum[lane] = v - w; // exclusive
    }
    sync();
    const float wex = sc.wsum[warp];
    const float p_end = wex + inc, p_start = wex + (inc - loc);

    // ---- 2. classify, compose the thread's own steps
    int cls = SEQSUM2_LITERAL;
    SeqPair pr;
    pr.a0 = pr.a1 = 0u;
    {
        const int e = f32_exponent(p_start);
        if (p_start > 0.0f && e > -100 && e < 128 && f32_exponent(p_end) == e) { // e == 128: inf/nan prefix -> literal adds
            const float b = __uint_as_float((unsigned)(e + 127) << 23);
            // margin 2^-9: the sequential sum deviates from any exact prefix by < n * 2^-24 relative (n <= 8192 -> 2^-11)
            if (p_start >= b * (1.0f + 0x1p-9f) && p_end <= 2.0f * b * (1.0f - 0x1p-9f)) {
                bool ok = true;
                int k = 0;
                if (vec)
#pragma unroll 1
                    for (; k < E; k += 4) { // four independent pair evaluations, composed as a tree: the dependent chain is E/4 + 2 composes, not E
                        const float4 v = *reinterpret_cast<const float4 *>(mine + k);
                        SeqPair q0, q1, q2, q3;
                        const bool o0 = seq_pair(v.x, e, q0), o1 = seq_pair(v.y, e, q1), o2 = seq_pair(v.z, e, q2), o3 = seq_pair(v.w, e, q3);
                        ok = ok && o0 && o1 && o2 && o3; // composing an invalid pair is harmless: the result is discarded
                        pr = seq_compose(pr, seq_compose(seq_compose(q0, q1), seq_compose(q2, q3)));
                    }
#pragma unroll 1
                for (; ok && k < E; k++) {
                    SeqPair q;
                    if (!seq_pair(mine[k], e, q)) { ok = false; break; }
                    pr = seq_compose(pr, q);
                }
                if (ok) cls = e;
            }
        }
    }
    sc.cls[tid] = cls;
    if (lane == 31) sc.wcls_last[warp] = cls;
    if (lane == 0) sc.wcls_first[warp] = cls;
    sync();

    // ---- 3. segmented scan over runs of clean threads with equal binade
    int prev_cls = __shfl_up_sync(0xffffffffu, cls, 1);
    if (lane == 0) prev_cls = warp ? sc.wcls_last[warp - 1] : SEQSUM2_LITERAL;
    int next_cls = __shfl_down_sync(0xffffffffu, cls, 1);
    if (lane == 31) next_cls = warp < NW - 1 ? sc.wcls_first[warp + 1] : SEQSUM2_LITERAL;
    const bool clean = cls != SEQSUM2_LITERAL;
    int f = (clean && prev_cls == cls) ? 0 : 1; // 1 = a run (or a literal thread) starts here
    seq2_warp_segscan(pr, f, lane);
    if (lane == 31) { sc.wtail[warp] = pr; sc.wtail_f[warp] = f; }
    sync();
    if (warp == 0) { // carry[w] = pair of the run that is still open when warp w begins (scan over the warp tails)
        SeqPair t;
        t.a0 = t.a1 = 0u;
        int tf = 1;
        if (lane < NW) { t = sc.wtail[lane]; tf = sc.wtail_f[lane]; }
        seq2_warp_segscan(t, tf, lane);
        if (lane < NW) sc.wtail[lane] = t; // inclusive: run open at the END of warp `lane`, composed from its true start
    }
    sync();
    if (!f && warp > 0) pr = seq_compose(sc.wtail[warp - 1], pr); // f == 0 in warp 0 cannot happen (thread 0 always starts a run)

    // ---- 4. item list
    const bool is_item = !clean || next_cls != cls;
    const unsigned bal = __ballot_sync(0xffffffffu, is_item);
    if (lane == 0) sc.wcnt[warp] = __popc(bal);
    sync();
    if (warp == 0) {
        const int c = lane < NW ? sc.wcnt[lane] : 0;
        int v = c;
#pragma unroll 1
        for (int d = 1; d < 32; d <<= 1) {
            const int u = __shfl_up_sync(0xffffffffu, v, d);
            if (lane >= d) v += u;
        }
        if (lane < NW) sc.wcnt[lane] = v - c;
        if (lane == 31) sc.info[0] = v;
    }
    sync();
    if (is_item) {
        SeqItem it;
        it.cls = cls; it.a0 = pr.a0; it.a1 = pr.a1; it.last = tid;
        sc.items[sc.wcnt[warp] + __popc(bal & ((1u << lane) - 1u))] = it;
    }
    sync();

    // ---- 5. resolver
    if (tid == 0) {
        const int n_items = sc.info[0];
        float s = 0.0f;
        int fallbacks = 0;
        SeqItem nxt = sc.items[0];
#pragma unroll 1
        for (int i = 0; i < n_items; i++) {
            const SeqItem it = nxt;
            if (i + 1 < n_items) nxt = sc.items[i + 1]; // in flight while this item is resolved
            if (it.cls == SEQSUM2_LITERAL) {
                s = seq2_literal(s, sq + it.last * S, E, vec);
                continue;
            }
            const unsigned sb = __float_as_uint(s);
            bool ok = f32_exponent(s) == it.cls && (sb >> 23) != 0u;
            if (ok) {
                const unsigned M = (sb & 0x7fffffu) | 0x800000u;
                const unsigned M2 = M + ((M & 1u) ? it.a1 : it.a0);
                if (M2 < (1u << 24)) s = __uint_as_float(((unsigned)(it.cls + 127) << 23) | (M2 & 0x7fffffu));
                else ok = false;
            }
            if (!ok) { // misprediction: replay the run literally (its first thread: walk back over equal classes)
                int first = it.last;
                while (first > 0 && sc.cls[first - 1] == it.cls) first--;
#pragma unroll 1
                for (int j = first; j <= it.last; j++) s = seq2_literal(s, sq + j * S, E, vec);
                fallbacks++;
            }
        }
        sc.result[0] = s;
        sc.info[1] = fallbacks;
    }
    sync();
    return sc.result[0];
}

// The whole-CTA form used by k_rmsnorm_quant: SEQSUM2_THREADS threads, __syncthreads.
__device__ __forceinline__ float block_seqsum_exact_v2(const float *sq, int n, SeqSum2Scratch sc) {
    return block_seqsum_exact_v2_t<SEQSUM2_THREADS>(sq, n, sc, (int)threadIdx.x, SeqSum2BlockSync());
}
