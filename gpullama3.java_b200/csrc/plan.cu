// plan.cu -- libb200llama.so: plan lifecycle, weight upload/repack, CUDA-graph capture and the
// C ABI declared in include/b200llama.h.  Plays the role of TornadoVMMasterPlan*.java +
// tornadovm/plan/** + tornadovm/layers/** of the reference (one native context and one CUDA
// graph per token instead of N+2 TaskGraph executions, TornadoVMMasterPlanSingleToken.java:68-95).
#include "../../include/b200llama.h"
#include "decode_kernels.cuh"
#include "prefill.cuh"
#include "stream_matvec.cuh"
#include "stream_matvec_f16.cuh"
#include "kquant.cuh"
#include "decode_persistent.cuh"
#include "sampler.cuh"

#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <chrono>
#include <string>
#include <thread>
#include <utility>
#include <vector>

namespace {

struct LayerW {
    DevMat qkv, wo, w1, w3, w2;
    TileMat tqkv{}, two{}, tgu{}, tw2{}; // tile-major copies for the streaming kernel (Q8_0)
    float *attn_norm = nullptr, *ffn_norm = nullptr, *q_norm = nullptr, *k_norm = nullptr;
};

} // namespace

// Weight upload pipeline (SURVEY 8f N1; replaces the reference's lazy FIRST_EXECUTION copy-in, LlamaQ8_0FFNLayers.java:122-132,
// timed by TornadoVMMasterPlanSingleToken.java:51-54): pageable/mmapped host bytes -> pinned double buffer (several host
// threads) -> async H2D on a copy stream -> device staging (double buffered) -> repack kernel on the plan's stream.  The host
// copy of chunk i+1, the DMA of chunk i and the repack of the previous matrix overlap; nothing synchronises per matrix.
struct Uploader {
    cudaStream_t copy = nullptr;
    unsigned char *pin[2] = {nullptr, nullptr};
    size_t pin_bytes = 0;
    cudaEvent_t pin_done[2] = {nullptr, nullptr};
    bool pin_used[2] = {false, false};
    int pi = 0;
    unsigned char *dst[2] = {nullptr, nullptr};
    size_t dst_bytes = 0;
    cudaEvent_t d_ready[2] = {nullptr, nullptr}, d_free[2] = {nullptr, nullptr};
    bool d_used[2] = {false, false};
    int di = 0;
    int threads = 4;
    double host_copy_s = 0.0, total_s = 0.0;
    int64_t h2d_bytes = 0;
};

// The kernels every decode matvec of a plan runs on, chosen once in build() from the weight type and the shapes:
// the Q8_0 tile stream (k_stream_matvec_q8), the Q8_0 row kernels (k_matvec_q8, k_gateup_q8), the FP16 per-warp rings
// (k_stream_matvec_f16) or the FP16 row kernels (k_matvec_f16, k_swiglu).  The row kernels serve the shapes the other
// two layouts do not fit.
enum MvPath { Q8_TILES, Q8_ROWS, F16_RINGS, F16_ROWS };

struct b200_plan {
    b200_config cfg{};
    Uploader up;
    int device = 0;
    int wtype = 0; // B200_GGML_Q8_0 or B200_GGML_F16 (matrix type)
    int qd = 0, kvd = 0;
    int prefill_batch = 0;
    cudaStream_t stream = nullptr;
    std::vector<void *> allocs;
    int64_t bytes = 0;
    std::string err;

    DevMat emb{}, out{};
    TileMat tout{};
    MvPath path = Q8_ROWS;
    // The tile stream and the rings launch with PDL, leave per-CTA argmax partials of the classifier and stamp trace records.
    bool streaming() const { return path == Q8_TILES || path == F16_RINGS; }
    int kflags = 0; // KF_* (common.cuh): what the attention prologues do for this architecture
    size_t kq_off = 0; // K-quant files: offset of the raw (K-quant bytes) area inside each staging buffer; 0 = no K-quant tensor in the file
    bool f16_copies = false; // Q8_0 plan that also holds f16 weight matrices for the tensor-core prefill
    int n_sms = 148;
    unsigned *blk_cnt = nullptr;
    float *part_val = nullptr;
    int *part_idx = nullptr;
    float *out_norm = nullptr;
    std::vector<LayerW> layers;
    float *rope_cr = nullptr, *rope_ci = nullptr;

    // activations
    float *x = nullptr, *xb = nullptr, *qkv = nullptr, *hb = nullptr, *hb2 = nullptr, *logits = nullptr;
    int8_t *xq = nullptr, *hq = nullptr;
    float *xs = nullptr, *hs = nullptr;
    float *key_cache = nullptr, *value_cache = nullptr;
    StepState *st = nullptr;
    int *seq_tokens = nullptr, *out_ids = nullptr;
    int seq_cap = 0;
    StepState *h_st = nullptr; // pinned
    int *h_ids = nullptr;      // pinned, seq_cap

    cudaGraphExec_t g_decode = nullptr, g_prefill = nullptr, g_trace = nullptr; // the multi-kernel decode graph (round 1)
    cudaGraphExec_t g_pdecode = nullptr, g_pprefill = nullptr, g_ptrace = nullptr; // one persistent kernel per token (decode_persistent.cuh)
    unsigned long long *trace_rec = nullptr;
    int decode_mode = B200_DECODE_GRAPH; // which of the two the forward entry points launch
    float *att_scratch = nullptr; // [heads][ctx] score rows when the context does not fit shared memory
    int *smp_indices = nullptr, *smp_out = nullptr; // device-side sampler scratch (sampler.cuh): candidate list, {id, info[4]}

    // tensor parallelism (tp.n == 1: single GPU).  *_l = this rank's share.
    TpCtx tp{};
    unsigned char *comm = nullptr; // IPC-exported communication buffer (x, gathered activations, flags)
    size_t comm_bytes = 0;
    bool attached = false;
    int nh_l = 0, nkv_l = 0, qd_l = 0, kvd_l = 0, hid_l = 0, dim_l = 0, voc_l = 0;
    int8_t *attq = nullptr; // gathered attention output (quantised) feeding the Wo matvec
    float *atts = nullptr;
    void *peer_open[TP_MAX] = {nullptr};
    int launches_decode = 0, launches_prefill = 0;
    float prefill_ms = 0.f; // device time of the last tensor-core prefill chunk
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;

    PrefillCtx prefill;
    // persistent decode kernel
    bool pd_ok = false;           // the plan fits the kernel's restrictions
    std::string pd_why;           // ... or why not
    PdSmem pd_L{};
    PdLayer *pd_layers = nullptr; // device copies of the per-layer descriptors
    unsigned *pd_sync = nullptr;  // epoch counters, ticks, error word
    unsigned *h_err = nullptr;    // mapped pinned host word written by a timed-out wait
    unsigned *d_err = nullptr;    // its device alias
    unsigned long long *pd_trace = nullptr;
    unsigned pd_flags_off = 0;
    bool pd_coop = true;          // launched with the cooperative attribute (co-residency guaranteed by the driver)
};

namespace {

int fail(b200_plan *p, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (p) p->err = buf;
    return code;
}

#define CK(call)                                                                                     \
    do {                                                                                             \
        cudaError_t e_ = (call);                                                                     \
        if (e_ != cudaSuccess)                                                                       \
            return fail(p, e_ == cudaErrorMemoryAllocation ? B200_ERR_OOM : B200_ERR_CUDA, "%s: %s (%s:%d)", #call, \
                        cudaGetErrorString(e_), __FILE__, __LINE__);                                 \
    } while (0)

// Largest dynamic shared memory a kernel may ask for = the device opt-in limit minus the kernel's own static shared memory.
template <typename K> cudaError_t set_max_dyn(K kern, int maxdyn) {
    cudaFuncAttributes fa;
    cudaError_t e = cudaFuncGetAttributes(&fa, kern);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, maxdyn - (int)fa.sharedSizeBytes);
}

template <typename T> int dalloc(b200_plan *p, T **ptr, size_t n_bytes) {
    void *d = nullptr;
    if (n_bytes == 0) n_bytes = 16;
    CK(cudaMalloc(&d, n_bytes));
    p->allocs.push_back(d);
    p->bytes += (int64_t)n_bytes;
    *ptr = reinterpret_cast<T *>(d);
    return B200_OK;
}

void par_memcpy(void *dst, const void *src, size_t n, int threads) {
    if (threads <= 1 || n < (size_t)(4u << 20)) { memcpy(dst, src, n); return; }
    std::vector<std::thread> th;
    const size_t per = ((n + threads - 1) / threads + 4095) & ~(size_t)4095;
    for (int i = 0; i < threads; i++) {
        const size_t o = (size_t)i * per;
        if (o >= n) break;
        const size_t m = n - o < per ? n - o : per;
        th.emplace_back([=] { memcpy((unsigned char *)dst + o, (const unsigned char *)src + o, m); });
    }
    for (auto &t : th) t.join();
}

int up_init(b200_plan *p, size_t dst_bytes) {
    Uploader &u = p->up;
    u.pin_bytes = (size_t)64 << 20;
    u.dst_bytes = dst_bytes;
    CK(cudaStreamCreateWithFlags(&u.copy, cudaStreamNonBlocking));
    for (int i = 0; i < 2; i++) {
        CK(cudaHostAlloc((void **)&u.pin[i], u.pin_bytes, cudaHostAllocDefault));
        CK(cudaMalloc((void **)&u.dst[i], dst_bytes));
        CK(cudaEventCreateWithFlags(&u.pin_done[i], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&u.d_ready[i], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&u.d_free[i], cudaEventDisableTiming));
    }
    return B200_OK;
}

void up_destroy(b200_plan *p) {
    Uploader &u = p->up;
    if (u.copy) cudaStreamSynchronize(u.copy);
    for (int i = 0; i < 2; i++) {
        if (u.pin[i]) cudaFreeHost(u.pin[i]);
        if (u.dst[i]) cudaFree(u.dst[i]);
        if (u.pin_done[i]) cudaEventDestroy(u.pin_done[i]);
        if (u.d_ready[i]) cudaEventDestroy(u.d_ready[i]);
        if (u.d_free[i]) cudaEventDestroy(u.d_free[i]);
        u.pin[i] = nullptr; u.dst[i] = nullptr; u.pin_done[i] = u.d_ready[i] = u.d_free[i] = nullptr;
    }
    if (u.copy) cudaStreamDestroy(u.copy);
    u.copy = nullptr;
}

// host bytes -> device, through the pinned double buffer, on the copy stream (asynchronous with respect to the caller except
// for the wait on a pinned buffer still in flight)
int up_h2d(b200_plan *p, void *dst, const void *src, size_t bytes) {
    Uploader &u = p->up;
    for (size_t o = 0; o < bytes; o += u.pin_bytes) {
        const size_t n = bytes - o < u.pin_bytes ? bytes - o : u.pin_bytes;
        const int i = u.pi;
        if (u.pin_used[i]) CK(cudaEventSynchronize(u.pin_done[i]));
        const auto t0 = std::chrono::steady_clock::now();
        par_memcpy(u.pin[i], (const unsigned char *)src + o, n, u.threads);
        u.host_copy_s += std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        CK(cudaMemcpyAsync((unsigned char *)dst + o, u.pin[i], n, cudaMemcpyHostToDevice, u.copy));
        CK(cudaEventRecord(u.pin_done[i], u.copy));
        u.pin_used[i] = true;
        u.pi ^= 1;
        u.h2d_bytes += (int64_t)n;
    }
    return B200_OK;
}
// device staging buffer protocol: begin (copy stream waits until the repack that last read this buffer is done) -> h2d... ->
// ready (plan stream waits for the copies) -> [repack kernel on the plan stream] -> release
int up_stage_begin(b200_plan *p, unsigned char **stage) {
    Uploader &u = p->up;
    if (u.d_used[u.di]) CK(cudaStreamWaitEvent(u.copy, u.d_free[u.di], 0));
    *stage = u.dst[u.di];
    return B200_OK;
}
int up_stage_ready(b200_plan *p) {
    Uploader &u = p->up;
    CK(cudaEventRecord(u.d_ready[u.di], u.copy));
    CK(cudaStreamWaitEvent(p->stream, u.d_ready[u.di], 0));
    return B200_OK;
}
int up_stage_release(b200_plan *p) {
    Uploader &u = p->up;
    CK(cudaEventRecord(u.d_free[u.di], p->stream));
    u.d_used[u.di] = true;
    u.di ^= 1;
    return B200_OK;
}

// GGUF Q8_0 blocks (f16 scale + 32 int8, 34 bytes, GGMLType.java:13) -> split planes.
// One thread per 16-bit word of the raw stream: word 0 of each block is the scale.
__global__ void k_repack_q8(const uint16_t *__restrict__ raw, uint16_t *__restrict__ qs, uint16_t *__restrict__ sc,
                            size_t n_words) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_words) return;
    size_t blk = i / 17;
    int w = (int)(i % 17);
    uint16_t v = raw[i];
    if (w == 0) sc[blk] = v;
    else qs[blk * 16 + (w - 1)] = v;
}

const b200_tensor *find(const b200_tensor *t, int n, const std::string &name) {
    for (int i = 0; i < n; i++)
        if (name == t[i].name) return &t[i];
    return nullptr;
}

int64_t n_elems(const b200_tensor *t) {
    int64_t n = 1;
    for (int i = 0; i < t->n_dims; i++) n *= t->dims[i];
    return n;
}

static inline int eff_type(int t) { return kq_is_kquant(t) ? B200_GGML_Q8_0 : t; } // AbstractModelLoader.effectiveGpuWeightType (:58-64)

// Upload rows [0, rows) of a [rows][cols] GGUF matrix into dst at row offset `row_off`.  K-quant sources are re-quantised to Q8_0 on
// the device (kquant.cuh) between the copy and the repack.
int upload_matrix(b200_plan *p, const b200_tensor *t, int rows, int cols, DevMat &dst, int row_off, int src_row = 0,
                  int src_full_rows = -1) { // rows [src_row, src_row + rows) of a source tensor with src_full_rows rows (Phi-3's fused wqkv / gate-up)
    if (!t) return fail(p, B200_ERR_BAD_ARG, "missing tensor");
    if (src_full_rows < 0) src_full_rows = rows;
    if (n_elems(t) != (int64_t)src_full_rows * cols || src_row < 0 || src_row + rows > src_full_rows)
        return fail(p, B200_ERR_BAD_ARG, "tensor %s has %lld elements, expected %lld", t->name, (long long)n_elems(t),
                    (long long)src_full_rows * cols);
    const size_t src_row_bytes = kq_is_kquant(t->ggml_type) ? (size_t)cols / 256 * kq_block_bytes(t->ggml_type)
                                 : t->ggml_type == B200_GGML_Q8_0 ? (size_t)cols / 32 * 34 : (size_t)cols * (t->ggml_type == B200_GGML_F16 ? 2 : 4);
    const unsigned char *tdata = (const unsigned char *)t->data + (size_t)src_row * src_row_bytes;
    if (eff_type(t->ggml_type) != dst.type)
        return fail(p, B200_ERR_UNSUPPORTED, "tensor %s has ggml type %d, plan weight type is %d", t->name, t->ggml_type,
                    dst.type);
    if (dst.type == B200_GGML_Q8_0) {
        const bool kq = kq_is_kquant(t->ggml_type);
        if (kq && (cols % 256 || !p->kq_off)) return fail(p, B200_ERR_BAD_ARG, "K-quant tensor %s: rows must be multiples of 256 elements", t->name);
        const size_t kb = kq ? (size_t)kq_block_bytes(t->ggml_type) : 0;
        size_t nblk = (size_t)rows * cols / 32;
        int8_t *qs = (int8_t *)dst.qs + (size_t)row_off * cols;
        __half *sc = (__half *)dst.sc + (size_t)row_off * (cols / 32);
        // chunked through the staging buffer (multiple of 34 bytes; of 8 blocks = one super-block for K-quants)
        const size_t q8_area = p->kq_off ? p->kq_off : p->up.dst_bytes;
        size_t blk_per_chunk = (q8_area / 34) & ~(size_t)7;
        for (size_t b0 = 0; b0 < nblk; b0 += blk_per_chunk) {
            size_t nb = nblk - b0 < blk_per_chunk ? nblk - b0 : blk_per_chunk;
            const unsigned char *hsrc = kq ? tdata + b0 / 8 * kb : tdata + b0 * 34;
            const size_t hbytes = kq ? nb / 8 * kb : nb * 34;
            int rc;
            unsigned char *stage = nullptr;
            if ((rc = up_stage_begin(p, &stage))) return rc;
            if ((rc = up_h2d(p, stage + (kq ? p->kq_off : 0), hsrc, hbytes))) return rc;
            if ((rc = up_stage_ready(p))) return rc;
            if (kq) CK(launch_requant_kquant(t->ggml_type, (const unsigned char *)stage + p->kq_off, (unsigned char *)stage, (long long)nb, p->stream));
            size_t words = nb * 17;
            k_repack_q8<<<(unsigned)((words + 255) / 256), 256, 0, p->stream>>>((const uint16_t *)stage, (uint16_t *)(qs + b0 * 32),
                                                                                  (uint16_t *)(sc + b0), words);
            CK(cudaGetLastError());
            if ((rc = up_stage_release(p))) return rc;
        }
    } else {
        size_t esz = dst.type == B200_GGML_F16 ? 2 : 4;
        return up_h2d(p, (uint8_t *)dst.qs + (size_t)row_off * cols * esz, tdata, (size_t)rows * cols * esz); // ordered by the final synchronize
    }
    return B200_OK;
}

// Upload up to three stacked GGUF Q8_0 matrices (or the gate/up pair) into tile-major layout.
int upload_tiles(b200_plan *p, const b200_tensor *t0, const b200_tensor *t1, const b200_tensor *t2, int r0, int r1, int r2, int cols,
                 bool gateup, TileMat &out, const int *row0 = nullptr, const int *full = nullptr) {
    const b200_tensor *ts[3] = {t0, t1, t2};
    int rs[3] = {r0, r1, r2};
    RepackSrc src;
    size_t off = 0;
    int rc;
    unsigned char *stage = nullptr;
    if ((rc = up_stage_begin(p, &stage))) return rc;
    const size_t stage_bytes = p->up.dst_bytes;
    const size_t q8_area = p->kq_off ? p->kq_off : stage_bytes;
    size_t roff = 0; // cursor inside the raw (K-quant) area
    struct Requant { int type; const unsigned char *raw; unsigned char *q8; long long nblk; } rq[3];
    int n_rq = 0;
    for (int k = 0; k < 3; k++) {
        src.raw[k] = nullptr;
        src.rows[k] = rs[k];
        src.row0[k] = 0; // only this rank's row range [row0, row0 + rows) crosses PCIe (rows are contiguous in GGUF)
        if (rs[k] == 0) continue;
        const int full_rows = full ? full[k] : rs[k];
        const int first = row0 ? row0[k] : 0;
        const b200_tensor *t = ts[k];
        if (!t) return fail(p, B200_ERR_BAD_ARG, "missing tensor");
        const bool kq = kq_is_kquant(t->ggml_type);
        if (t->ggml_type != B200_GGML_Q8_0 && !kq) return fail(p, B200_ERR_UNSUPPORTED, "tensor %s has ggml type %d, plan weight type is Q8_0", t->name, t->ggml_type);
        if (kq && (cols % 256 || !p->kq_off)) return fail(p, B200_ERR_BAD_ARG, "K-quant tensor %s: rows must be multiples of 256 elements", t->name);
        if (n_elems(t) != (int64_t)full_rows * cols) return fail(p, B200_ERR_BAD_ARG, "tensor %s has %lld elements, expected %lld", t->name, (long long)n_elems(t), (long long)full_rows * cols);
        if (first < 0 || first + rs[k] > full_rows) return fail(p, B200_ERR_BAD_ARG, "row range of tensor %s out of bounds", t->name);
        const size_t row_bytes = (size_t)cols / 32 * 34, nbytes = (size_t)rs[k] * row_bytes;
        if (off + nbytes > q8_area) return fail(p, B200_ERR_STATE, "staging buffer too small");
        if (kq) { // the K-quant bytes land in the raw area; the Q8_0 blocks are produced on the device once the copies are in
            const size_t raw_row = (size_t)cols / 256 * kq_block_bytes(t->ggml_type), raw_bytes = (size_t)rs[k] * raw_row;
            const unsigned char *hsrc = (const unsigned char *)t->data + (size_t)first * raw_row;
            if (p->kq_off + roff + raw_bytes > stage_bytes) return fail(p, B200_ERR_STATE, "staging buffer too small");
            unsigned char *rdst = stage + p->kq_off + roff;
            if ((rc = up_h2d(p, rdst, hsrc, raw_bytes))) return rc;
            rq[n_rq++] = Requant{t->ggml_type, rdst, stage + off, (long long)rs[k] * (cols / 32)};
            roff += (raw_bytes + 255) & ~(size_t)255;
        } else {
            const unsigned char *hsrc = (const unsigned char *)t->data + (size_t)first * row_bytes;
            if ((rc = up_h2d(p, stage + off, hsrc, nbytes))) return rc;
        }
        src.raw[k] = stage + off;
        off += (nbytes + 255) & ~(size_t)255;
    }
    if ((rc = up_stage_ready(p))) return rc;
    for (int i = 0; i < n_rq; i++) CK(launch_requant_kquant(rq[i].type, rq[i].raw, rq[i].q8, rq[i].nblk, p->stream));
    src.gateup = gateup ? 1 : 0;
    const int rows = gateup ? r0 + r1 : r0 + r1 + r2;
    out.rows = rows;
    out.cols = cols;
    out.nseg = smv_pick_nseg(cols);
    out.seg = cols / out.nseg;
    out.unit_bytes = smv_unit_bytes(out.seg);
    size_t total = (size_t)rows * out.nseg * out.unit_bytes;
    unsigned char *d;
    rc = dalloc(p, &d, total);
    if (rc) return rc;
    out.base = d;
    k_repack_tiles<<<(unsigned)((size_t)rows * out.nseg), 128, 0, p->stream>>>(src, d, rows, cols, out.seg, out.nseg, out.unit_bytes);
    CK(cudaGetLastError());
    return up_stage_release(p);
}

int alloc_matrix(b200_plan *p, DevMat &m, int rows, int cols, int type) {
    m.rows = rows;
    m.cols = cols;
    m.type = type;
    m.sc = nullptr;
    void *q = nullptr;
    int rc;
    if (type == B200_GGML_Q8_0) {
        if ((rc = dalloc(p, (int8_t **)&q, (size_t)rows * cols))) return rc;
        __half *s;
        if ((rc = dalloc(p, &s, (size_t)rows * (cols / 32) * 2))) return rc;
        m.sc = s;
    } else {
        if ((rc = dalloc(p, (uint8_t **)&q, (size_t)rows * cols * (type == B200_GGML_F16 ? 2 : 4)))) return rc;
    }
    m.qs = q;
    return B200_OK;
}

int upload_f32(b200_plan *p, const b200_tensor *t, int n, float **dst, const char *what) {
    if (!t) return fail(p, B200_ERR_BAD_ARG, "missing tensor %s", what);
    if (t->ggml_type != B200_GGML_F32) return fail(p, B200_ERR_UNSUPPORTED, "tensor %s must be F32", what);
    if (n_elems(t) != n) return fail(p, B200_ERR_BAD_ARG, "tensor %s has wrong size", what);
    int rc = dalloc(p, dst, (size_t)n * 4);
    if (rc) return rc;
    CK(cudaMemcpy(*dst, t->data, (size_t)n * 4, cudaMemcpyHostToDevice));
    return B200_OK;
}

template <int MODE> int launch_matvec_q8(b200_plan *p, const DevMat &m, const int8_t *xq, const float *xs, float *out) {
    int R = (m.rows % 4 == 0 && m.rows >= 32768) ? 4 : (m.rows % 2 == 0 ? 2 : 1);
    int warps = m.rows / R;
    int ctas = (warps + 7) / 8;
    size_t smem = q8_smem_bytes(m.cols, R, 8);
    const int8_t *qs = (const int8_t *)m.qs;
    if (R == 4) k_matvec_q8<4, MODE><<<ctas, 256, smem, p->stream>>>(qs, m.sc, xq, xs, m.rows, m.cols, out);
    else if (R == 2) k_matvec_q8<2, MODE><<<ctas, 256, smem, p->stream>>>(qs, m.sc, xq, xs, m.rows, m.cols, out);
    else k_matvec_q8<1, MODE><<<ctas, 256, smem, p->stream>>>(qs, m.sc, xq, xs, m.rows, m.cols, out);
    CK(cudaGetLastError());
    return B200_OK;
}

size_t f16_smem_bytes(int cols, int lanes) {
    int L = lanes > 0 ? lanes : 1;
    return (size_t)cols * 4 + (size_t)8 * (32 / L) * 256 * 2;
}

template <int MODE> int launch_matvec_f16(b200_plan *p, const DevMat &m, const float *x, float *out) {
    int L = p->cfg.fp16_lanes > 0 ? p->cfg.fp16_lanes : 1;
    int rw = 32 / L;
    int warps = (m.rows + rw - 1) / rw;
    int ctas = (warps + 7) / 8;
    k_matvec_f16<MODE><<<ctas, 256, f16_smem_bytes(m.cols, p->cfg.fp16_lanes), p->stream>>>((const __half *)m.qs, x, m.rows,
                                                                                            m.cols, p->cfg.fp16_lanes, out);
    CK(cudaGetLastError());
    return B200_OK;
}

// FP16 plans on the streaming path (stream_matvec_f16.cuh); m2 = ffn_up for SF_GATEUP.
template <typename... KA, typename... A> int launch_k(b200_plan *p, bool pdl, void (*kern)(KA...), dim3 grid, dim3 block, size_t smem, A... args);
int sf_grid(const b200_plan *p, int rows, int cols, bool gateup) { // CTAs of an FP16 streaming launch
    const int lanes = p->cfg.fp16_lanes;
    const SfLayout L = sf_layout(rows, cols, lanes, gateup);
    const int rw = 64 / lanes, mr = gateup ? rw / 2 : rw;
    const int grid = L.ctas_per_sm * p->n_sms;
    return grid > rows / mr ? rows / mr : grid;
}
template <int MODE> int launch_stream_f16(b200_plan *p, bool pdl, const DevMat &m, const DevMat *m2, const float *x, float *out, TraceBuf tr,
                                          bool argmax = false) {
    const int lanes = p->cfg.fp16_lanes;
    const SfLayout L = sf_layout(m.rows, m.cols, lanes, MODE == SF_GATEUP);
    if (!L.ok) return fail(p, B200_ERR_STATE, "f16 streaming layout does not fit %d x %d", m.rows, m.cols);
    SfArgs a;
    a.w0 = (const __half *)m.qs; a.w1 = m2 ? (const __half *)m2->qs : nullptr; a.x = x; a.out = out; a.rows = m.rows; a.cols = m.cols;
    a.seg = L.seg; a.nseg = L.nseg; a.stages = L.stages; a.tr = tr;
    a.part_val = argmax ? p->part_val : nullptr;
    a.part_idx = argmax ? p->part_idx : nullptr;
    const int grid = sf_grid(p, m.rows, m.cols, MODE == SF_GATEUP);
    if (lanes == 16) return launch_k(p, pdl, k_stream_matvec_f16<16, MODE>, dim3(grid), dim3(SF_THREADS), L.total, a);
    return launch_k(p, pdl, k_stream_matvec_f16<8, MODE>, dim3(grid), dim3(SF_THREADS), L.total, a);
}

// Kernel launch with the programmatic-dependent-launch attribute (captured into the CUDA graph as
// a programmatic edge): the kernel may become resident while its predecessor is still running.
template <typename... KA, typename... A>
int launch_k(b200_plan *p, bool pdl, void (*kern)(KA...), dim3 grid, dim3 block, size_t smem, A... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = p->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    CK(cudaLaunchKernelEx(&cfg, kern, static_cast<KA>(args)...));
    return B200_OK;
}

const size_t SMV_SMEM_BUDGET_MAX = 96 * 1024;
// Read ONCE per plan (b200_plan_create), never inside a launch helper.
void read_knobs(b200_plan *p) {
    const char *d = getenv("B200_DECODE");
    // default: the CUDA graph -- measured faster than the persistent kernel on the same box (profiles/r2_final_a.log: 313.6 vs 285.1 tok/s,
    // 8B Q8_0; under tensor parallelism by 10-21 %).  B200_DECODE=persistent or b200_set_decode_mode select the one-kernel-per-token path.
    p->decode_mode = (d && !strcmp(d, "persistent")) ? B200_DECODE_PERSISTENT : B200_DECODE_GRAPH;
    const char *t = getenv("B200_UPLOAD_THREADS"); // host threads filling the pinned upload buffers
    if (t) p->up.threads = atoi(t);
}

template <int MODE>
int launch_stream(b200_plan *p, bool pdl, const TileMat &W, const int8_t *xq, const float *xs, float *out, int8_t *hq, float *hs, bool argmax,
                  TraceBuf tr, int wait_slot = -1, unsigned wait_op = 0, int out_slot = -1, unsigned out_op = 0, int row_base = 0) {
    SmvSmem L = smv_layout(W.cols, W.seg, SMV_SMEM_BUDGET_MAX);
    SmvArgs a;
    a.W = W; a.xq = xq; a.xs = xs; a.out = out; a.hq = hq; a.hs = hs; a.blk_cnt = p->blk_cnt;
    a.part_val = argmax ? p->part_val : nullptr;
    a.part_idx = argmax ? p->part_idx : nullptr;
    a.tr = tr;
    a.tp = p->tp;
    a.wait_slot = wait_slot; a.wait_op = wait_op; a.out_slot = out_slot; a.out_op = out_op; a.row_base = row_base;
    return launch_k(p, pdl, k_stream_matvec_q8<MODE>, dim3(p->n_sms), dim3(SMV_THREADS), L.total, a, L);
}

bool stream_shape_ok(int rows, int cols) {
    if (rows % 4 || cols % 32) return false;
    int nseg = smv_pick_nseg(cols);
    if (!nseg) return false;
    return smv_layout(cols, cols / nseg, SMV_SMEM_BUDGET_MAX).stages >= 3;
}

bool gateup_fits(int hidden, int n_sms) { // epilogue buffer holds this CTA's hidden units
    return 2 * ((hidden / 2) / n_sms + 1) <= SMV_HVALS;
}

// k_attention's dynamic shared memory: q | k | out | score row (the row lives in a global scratch buffer for long contexts).
size_t att_smem_bytes(int head_size, int ctx, bool scratch) { return (size_t)(3 * head_size + (scratch ? 0 : ctx)) * 4; }

// The matrix roles of a decode step; the values are b200_time_kernel's kernel ids.
enum MvRole { MV_GATEUP, MV_W2, MV_QKV, MV_WO, MV_CLS };

// Launches matrix role `role` of layer l (the classifier ignores l) on the plan's path; returns how many kernels it launched,
// or a negative B200_ERR_*.  Under tensor parallelism a forward numbers its flag epochs op = 4*l + {0: attention out,
// 1: x after Wo, 2: hb, 3: x after W2}: the tile stream waits on the slot that carries its activation and publishes its output.
int launch_mv(b200_plan *p, MvRole role, int l, bool pdl, TraceBuf tr) {
    const b200_config &c = p->cfg;
    LayerW &L = p->layers[l];
    int rc = B200_OK, n = 1;
    if (p->path == Q8_TILES) {
        const bool tpar = p->tp.n > 1;
        const int slot_att = tpar ? TP_SLOT_ATT : -1, slot_x = tpar ? TP_SLOT_X : -1, slot_hq = tpar ? TP_SLOT_HQ : -1, rank = p->tp.rank;
        const unsigned op = 4u * l;
        switch (role) {
        case MV_QKV: rc = launch_stream<SMV_STORE>(p, pdl, L.tqkv, p->xq, p->xs, p->qkv, nullptr, nullptr, false, tr); break;
        case MV_WO: rc = launch_stream<SMV_RESID>(p, pdl, L.two, p->attq, p->atts, p->x, nullptr, nullptr, false, tr, slot_att, op + 0, slot_x, op + 1, rank * p->dim_l); break;
        case MV_GATEUP: rc = launch_stream<SMV_GATEUP>(p, pdl, L.tgu, p->xq, p->xs, p->hb, p->hq, p->hs, false, tr, -1, 0, slot_hq, op + 2, rank * p->hid_l); break;
        case MV_W2: rc = launch_stream<SMV_RESID>(p, pdl, L.tw2, p->hq, p->hs, p->x, nullptr, nullptr, false, tr, slot_hq, op + 2, slot_x, op + 3, rank * p->dim_l); break;
        case MV_CLS: rc = launch_stream<SMV_STORE>(p, pdl, p->tout, p->xq, p->xs, p->logits, nullptr, nullptr, true, tr, -1, 0, -1, 0, rank * p->voc_l); break;
        }
    } else if (p->path == Q8_ROWS) {
        switch (role) {
        case MV_QKV: rc = launch_matvec_q8<MODE_STORE>(p, L.qkv, p->xq, p->xs, p->qkv); break;
        case MV_WO: rc = launch_matvec_q8<MODE_RESID>(p, L.wo, p->xq, p->xs, p->x); break;
        case MV_GATEUP:
            k_gateup_q8<<<c.hidden_dim / 32, 256, q8_smem_bytes(c.dim, 4, 8), p->stream>>>(
                (const int8_t *)L.w1.qs, L.w1.sc, (const int8_t *)L.w3.qs, L.w3.sc, p->xq, p->xs, c.hidden_dim, c.dim, p->hq, p->hs, p->hb);
            CK(cudaGetLastError());
            break;
        case MV_W2: rc = launch_matvec_q8<MODE_RESID>(p, L.w2, p->hq, p->hs, p->x); break;
        case MV_CLS: rc = launch_matvec_q8<MODE_STORE>(p, p->out, p->xq, p->xs, p->logits); break;
        }
    } else if (p->path == F16_RINGS) {
        switch (role) {
        case MV_QKV: rc = launch_stream_f16<SF_STORE>(p, pdl, L.qkv, nullptr, p->xb, p->qkv, tr); break;
        case MV_WO: rc = launch_stream_f16<SF_RESID>(p, pdl, L.wo, nullptr, p->xb, p->x, tr); break;
        case MV_GATEUP: rc = launch_stream_f16<SF_GATEUP>(p, pdl, L.w1, &L.w3, p->xb, p->hb, tr); break; // gate, up and SwiGLU in one launch
        case MV_W2: rc = launch_stream_f16<SF_RESID>(p, pdl, L.w2, nullptr, p->hb, p->x, tr); break;
        case MV_CLS: rc = launch_stream_f16<SF_STORE>(p, pdl, p->out, nullptr, p->xb, p->logits, tr, true); break;
        }
    } else {
        switch (role) {
        case MV_QKV: rc = launch_matvec_f16<MODE_STORE>(p, L.qkv, p->xb, p->qkv); break;
        case MV_WO: rc = launch_matvec_f16<MODE_RESID>(p, L.wo, p->xb, p->x); break;
        case MV_GATEUP:
            if ((rc = launch_matvec_f16<MODE_STORE>(p, L.w1, p->xb, p->hb)) || (rc = launch_matvec_f16<MODE_STORE>(p, L.w3, p->xb, p->hb2))) break;
            k_swiglu<<<(c.hidden_dim + 255) / 256, 256, 0, p->stream>>>(p->hb, p->hb2, c.hidden_dim);
            CK(cudaGetLastError());
            n = 3;
            break;
        case MV_W2: rc = launch_matvec_f16<MODE_RESID>(p, L.w2, p->hb, p->x); break;
        case MV_CLS: rc = launch_matvec_f16<MODE_STORE>(p, p->out, p->xb, p->logits); break;
        }
    }
    return rc ? rc : n;
}

// Enqueue one single-token forward on p->stream (captured into a CUDA graph at creation).
// with_logits=false is the prefill variant (InferenceCoreBatchPrefillDecode.java:166-167).
int enqueue_forward(b200_plan *p, bool with_logits, int *launches, bool trace = false) {
    const b200_config &c = p->cfg;
    const bool q8 = p->wtype == B200_GGML_Q8_0, pdl = p->streaming();
    int n = 0;
    auto TR = [&](int id) { return TraceBuf{trace ? p->trace_rec : nullptr, n, id}; };
    const size_t norm_smem = norm_smem_bytes(c.dim);
    int8_t *xq = q8 ? p->xq : nullptr;
    float *xs = q8 ? p->xs : nullptr;
    float *xbf = q8 ? nullptr : p->xb;
    const size_t ctx_kv = (size_t)c.context_length * p->kvd_l;
    const int rank = p->tp.rank;
    auto norm = [&](bool embed, const float *w, int wait_op) {
        auto go = [&](auto kern) {
            return launch_k(p, pdl, kern, dim3(1), dim3(NORM_THREADS), norm_smem, p->x, (const StepState *)p->st, p->emb, w, c.rms_norm_eps, c.dim, xq, xs, xbf, TR(1), p->tp, wait_op);
        };
        return embed ? go(k_rmsnorm_quant<true>) : go(k_rmsnorm_quant<false>);
    };
    for (int l = 0; l < c.n_layers; l++) {
        LayerW &L = p->layers[l];
        int rc;
        // TP flag epochs: see launch_mv
        if ((rc = norm(l == 0, L.attn_norm, l == 0 ? -1 : 4 * (l - 1) + 3))) return rc;
        n++;
        if ((rc = launch_mv(p, MV_QKV, l, pdl, TR(2))) < 0) return rc;
        n += rc;
        float *kc = p->key_cache + (size_t)l * ctx_kv, *vc = p->value_cache + (size_t)l * ctx_kv;
        {
            const size_t att_smem = att_smem_bytes(c.head_size, c.context_length, p->att_scratch != nullptr);
            auto att = [&](auto kern) {
                return launch_k(p, pdl, kern, dim3(p->nh_l), dim3(ATT_THREADS), att_smem, p->qkv, kc, vc, (const StepState *)p->st,
                                (const float *)p->rope_cr, (const float *)p->rope_ci, p->nh_l, p->nkv_l, p->kflags, (const float *)L.q_norm,
                                (const float *)L.k_norm, c.rms_norm_eps, (float)sqrt((double)c.head_size), q8 ? p->attq : nullptr, q8 ? p->atts : nullptr, xbf, TR(4),
                                p->tp, (unsigned)(4 * l + 0), rank * p->nh_l, p->att_scratch, c.context_length);
            };
            if (c.head_size == 128) rc = att(k_attention<128>);
            else if (c.head_size == 64) rc = att(k_attention<64>);
            else if (c.head_size == 256) rc = att(k_attention<256>);
            else if (c.head_size == 96) rc = att(k_attention<96>);
            else rc = att(k_attention<32>);
            if (rc) return rc;
            n++;
        }
        if ((rc = launch_mv(p, MV_WO, l, pdl, TR(5))) < 0) return rc;
        n += rc;
        if ((rc = norm(false, L.ffn_norm, 4 * l + 1))) return rc;
        n++;
        if ((rc = launch_mv(p, MV_GATEUP, l, pdl, TR(6))) < 0) return rc;
        n += rc;
        if ((rc = launch_mv(p, MV_W2, l, pdl, TR(7))) < 0) return rc;
        n += rc;
    }
    const int last_x_op = 4 * (c.n_layers - 1) + 3;
    if (with_logits) {
        // rmsnorm(x, x, rms_final_weight) then wcls.matmul (InferenceCore.java:167-169)
        int rc;
        if ((rc = norm(false, p->out_norm, last_x_op))) return rc;
        n++;
        if ((rc = launch_mv(p, MV_CLS, 0, pdl, TR(8))) < 0) return rc;
        n += rc;
    }
    {
        int rc;
        // part_val / part_idx exist only on the streaming paths; the row kernels leave the whole argmax to this kernel
        if ((rc = launch_k(p, pdl, k_argmax_advance, dim3(1), dim3(1024), (size_t)0, (const float *)p->logits, c.vocab_size, p->st, (const int *)p->seq_tokens, p->out_ids, with_logits ? 1 : 0,
                           (const float *)p->part_val, (const int *)p->part_idx, p->path == F16_RINGS ? sf_grid(p, c.vocab_size, c.dim, false) : p->n_sms,
                           TR(9), p->tp, with_logits ? -1 : last_x_op))) return rc;
        n++;
    }
    if (launches) *launches = n;
    return B200_OK;
}

// ---- one persistent kernel per token (decode_persistent.cuh) ---------------------------------------------------------------
// Checks the kernel's restrictions and allocates its descriptors; never launches (the KV cache must stay zero-initialised).
// Leaves p->pd_ok / p->pd_why; a plan that does not fit simply keeps the multi-kernel graph.
int pd_prepare(b200_plan *p) {
    const b200_config &c = p->cfg;
    p->pd_ok = false;
    if (p->path != Q8_TILES) { p->pd_why = "the persistent decode kernel needs the Q8_0 streaming layout"; return B200_OK; }
    if (c.head_size != 64 && c.head_size != 128) { p->pd_why = "the persistent decode kernel supports head sizes 64 and 128"; return B200_OK; }
    if (p->nh_l > p->n_sms) { p->pd_why = "more attention heads than SMs"; return B200_OK; }
    if (!gateup_fits(p->hid_l, p->n_sms)) { p->pd_why = "hidden slice per CTA exceeds the epilogue buffer"; return B200_OK; }
    int max_seg = p->tout.seg;
    for (const LayerW &L : p->layers) {
        const int segs[4] = {L.tqkv.seg, L.two.seg, L.tgu.seg, L.tw2.seg};
        for (int k = 0; k < 4; k++) if (segs[k] > max_seg) max_seg = segs[k];
    }
    int maxdyn = 0;
    CK(cudaDeviceGetAttribute(&maxdyn, cudaDevAttrMaxSharedMemoryPerBlockOptin, p->device));
    const int att_floats = 3 * c.head_size + (p->att_scratch ? 0 : (c.context_length + PD_CT - 1) / PD_CT * PD_CT); // score row padded to whole accumulator chunks
    const PdSmem L = pd_layout(c.dim, p->qd, c.hidden_dim, c.head_size, att_floats, max_seg, (size_t)maxdyn);
    if (L.stages < 4) { p->pd_why = "shape leaves fewer than 4 ring stages of shared memory"; return B200_OK; }
    int rc;
    if (!p->pd_layers) {
        std::vector<PdLayer> h(c.n_layers);
        const size_t ctx_kv = (size_t)c.context_length * p->kvd_l;
        for (int l = 0; l < c.n_layers; l++) {
            const LayerW &W = p->layers[l];
            h[l].qkv = W.tqkv; h[l].wo = W.two; h[l].gu = W.tgu; h[l].w2 = W.tw2;
            h[l].attn_norm = W.attn_norm; h[l].ffn_norm = W.ffn_norm; h[l].q_norm = W.q_norm; h[l].k_norm = W.k_norm;
            h[l].kc = p->key_cache + (size_t)l * ctx_kv;
            h[l].vc = p->value_cache + (size_t)l * ctx_kv;
        }
        if ((rc = dalloc(p, &p->pd_layers, h.size() * sizeof(PdLayer)))) return rc;
        CK(cudaMemcpy(p->pd_layers, h.data(), h.size() * sizeof(PdLayer), cudaMemcpyHostToDevice));
        if ((rc = dalloc(p, &p->pd_trace, (size_t)p->n_sms * (c.n_layers + 1) * PD_STAMPS * 8))) return rc;
        CK(cudaMemset(p->pd_trace, 0, (size_t)p->n_sms * (c.n_layers + 1) * PD_STAMPS * 8));
    }
    CK(set_max_dyn(k_decode_persistent<128>, maxdyn));
    CK(set_max_dyn(k_decode_persistent<64>, maxdyn));
    p->pd_L = L;
    p->pd_ok = true;
    p->pd_why = "";
    return B200_OK;
}

int enqueue_persistent(b200_plan *p, bool with_logits, int *launches, bool trace) {
    const b200_config &c = p->cfg;
    PdArgs a;
    memset(&a, 0, sizeof a);
    a.layers = p->pd_layers; a.n_layers = c.n_layers; a.lm_head = p->tout; a.out_norm = p->out_norm; a.emb = p->emb;
    a.dim = c.dim; a.hidden = c.hidden_dim; a.qd = p->qd; a.n_heads = p->nh_l; a.n_kv_heads = p->nkv_l;
    a.head_size = c.head_size; a.arch = p->kflags; a.ctx = c.context_length;
    a.eps = c.rms_norm_eps; a.sqrt_hs = (float)sqrt((double)c.head_size);
    a.rope_cr = p->rope_cr; a.rope_ci = p->rope_ci;
    a.st = p->st; a.seq_tokens = p->seq_tokens; a.out_ids = p->out_ids;
    a.x = p->x; a.qkv = p->qkv; a.hb = p->hb; a.logits = p->logits;
    a.attq = p->attq; a.atts = p->atts; a.hq = p->hq; a.hs = p->hs; a.blk_cnt = p->blk_cnt;
    a.part_val = p->part_val; a.part_idx = p->part_idx; a.sync = p->pd_sync; a.host_err = p->d_err;
    a.att_scratch = p->att_scratch; a.trace = trace ? p->pd_trace : nullptr;
    a.with_logits = with_logits ? 1 : 0;
    a.tp = p->tp; a.pd_flags_off = p->pd_flags_off;
    a.head_base = p->tp.rank * p->nh_l; a.dim_base = p->tp.rank * p->dim_l; a.hid_base = p->tp.rank * p->hid_l; a.voc_base = p->tp.rank * p->voc_l;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(p->n_sms);
    cfg.blockDim = dim3(PD_THREADS);
    cfg.dynamicSmemBytes = p->pd_L.total;
    cfg.stream = p->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeCooperative; // every CTA spins on its peers: the driver must guarantee co-residency
    attr[0].val.cooperative = 1;
    cfg.attrs = attr;
    cfg.numAttrs = p->pd_coop ? 1 : 0;
    if (c.head_size == 128) CK(cudaLaunchKernelEx(&cfg, k_decode_persistent<128>, a, p->pd_L));
    else CK(cudaLaunchKernelEx(&cfg, k_decode_persistent<64>, a, p->pd_L));
    if (launches) *launches = 1;
    return B200_OK;
}

int capture(b200_plan *p, bool with_logits, cudaGraphExec_t *exec, int *launches, bool trace = false, bool persistent = false) {
    cudaGraph_t g = nullptr;
    CK(cudaStreamBeginCapture(p->stream, cudaStreamCaptureModeThreadLocal));
    int rc = persistent ? enqueue_persistent(p, with_logits, launches, trace) : enqueue_forward(p, with_logits, launches, trace);
    cudaError_t e = cudaStreamEndCapture(p->stream, &g);
    if (rc) { if (g) cudaGraphDestroy(g); return rc; }
    if (e != cudaSuccess) return fail(p, B200_ERR_CUDA, "cudaStreamEndCapture: %s", cudaGetErrorString(e));
    e = cudaGraphInstantiate(exec, g, 0);
    cudaGraphDestroy(g);
    if (e != cudaSuccess) return fail(p, B200_ERR_CUDA, "cudaGraphInstantiate: %s", cudaGetErrorString(e));
    return B200_OK;
}

// Both decode implementations are captured; b200_set_decode_mode picks which one the forward calls launch.
int capture_all(b200_plan *p) {
    int rc;
    if ((rc = capture(p, true, &p->g_decode, &p->launches_decode))) return rc;
    if ((rc = capture(p, false, &p->g_prefill, nullptr))) return rc;
    if (p->streaming()) {
        if ((rc = dalloc(p, &p->trace_rec, (size_t)(p->launches_decode + 8) * 32))) return rc;
        if ((rc = capture(p, true, &p->g_trace, nullptr, true))) return rc;
    }
    if ((rc = pd_prepare(p))) return rc;
    if (p->pd_ok) {
        // grid = one CTA per SM with (almost) all of its shared memory: co-resident on an idle GPU either way; the cooperative
        // attribute makes the driver check it.  Should a driver refuse cooperative kernel nodes in a graph, retry without.
        for (int attempt = 0; attempt < 2; attempt++) {
            p->pd_coop = attempt == 0;
            rc = capture(p, true, &p->g_pdecode, nullptr, false, true);
            if (!rc) rc = capture(p, false, &p->g_pprefill, nullptr, false, true);
            if (!rc) rc = capture(p, true, &p->g_ptrace, nullptr, true, true);
            if (!rc) break;
            cudaGetLastError();
            for (cudaGraphExec_t *g : {&p->g_pdecode, &p->g_pprefill, &p->g_ptrace})
                if (*g) { cudaGraphExecDestroy(*g); *g = nullptr; }
        }
        if (rc) { p->pd_ok = false; p->pd_why = "persistent decode kernel could not be captured: " + p->err; }
    }
    if (!p->pd_ok && p->decode_mode == B200_DECODE_PERSISTENT) p->decode_mode = B200_DECODE_GRAPH;
    return B200_OK;
}

// cudaFuncSetAttribute is per function and process-wide: every kernel gets the device opt-in maximum ONCE, so a later plan
// with a smaller context never lowers the limit under an earlier plan's instantiated graphs.
const int ATT_SMEM_FLOATS_MAX = 4096; // q|k|out|scores beyond this: the score row goes to a global scratch row

int set_smem_attrs(b200_plan *p) {
    const b200_config &c = p->cfg;
    int maxdyn = 0;
    CK(cudaDeviceGetAttribute(&maxdyn, cudaDevAttrMaxSharedMemoryPerBlockOptin, p->device));
    if (c.dim > 8192) return fail(p, B200_ERR_UNSUPPORTED, "dim > 8192 not supported by the RMSNorm kernel");
    size_t need_norm = norm_smem_bytes(c.dim);
    size_t need_att = att_smem_bytes(c.head_size, c.context_length, p->att_scratch != nullptr);
    int maxcols = c.hidden_dim > c.dim ? c.hidden_dim : c.dim;
    if (p->qd > maxcols) maxcols = p->qd;
    size_t need_mv = q8_smem_bytes(maxcols, 4, 8);
    size_t need_f16 = f16_smem_bytes(maxcols, p->cfg.fp16_lanes);
    if (need_norm > (size_t)maxdyn || need_att > (size_t)maxdyn || (p->wtype == B200_GGML_Q8_0 && need_mv > (size_t)maxdyn) ||
        (p->wtype == B200_GGML_F16 && need_f16 > (size_t)maxdyn))
        return fail(p, B200_ERR_UNSUPPORTED, "shape needs more shared memory than the device offers (%d bytes)", maxdyn);
    static bool done = false; // process-wide, like the attribute itself (plans are created from one thread at a time per process)
    if (done) return B200_OK;
    CK(set_max_dyn(k_rmsnorm_quant<true>, maxdyn));
    CK(set_max_dyn(k_rmsnorm_quant<false>, maxdyn));
    CK(set_max_dyn(k_attention<32>, maxdyn));
    CK(set_max_dyn(k_attention<64>, maxdyn));
    CK(set_max_dyn(k_attention<128>, maxdyn));
    CK(set_max_dyn(k_attention<96>, maxdyn));
    CK(set_max_dyn(k_attention<256>, maxdyn));
    CK(set_max_dyn(k_matvec_q8<1, MODE_STORE>, maxdyn));
    CK(set_max_dyn(k_matvec_q8<2, MODE_STORE>, maxdyn));
    CK(set_max_dyn(k_matvec_q8<4, MODE_STORE>, maxdyn));
    CK(set_max_dyn(k_matvec_q8<1, MODE_RESID>, maxdyn));
    CK(set_max_dyn(k_matvec_q8<2, MODE_RESID>, maxdyn));
    CK(set_max_dyn(k_matvec_q8<4, MODE_RESID>, maxdyn));
    CK(set_max_dyn(k_gateup_q8, maxdyn));
    CK(cudaFuncSetAttribute(k_stream_matvec_q8<SMV_STORE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMV_SMEM_BUDGET_MAX));
    CK(cudaFuncSetAttribute(k_stream_matvec_q8<SMV_RESID>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMV_SMEM_BUDGET_MAX));
    CK(cudaFuncSetAttribute(k_stream_matvec_q8<SMV_GATEUP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMV_SMEM_BUDGET_MAX));
    CK(set_max_dyn(k_matvec_f16<MODE_STORE>, maxdyn));
    CK(set_max_dyn(k_matvec_f16<MODE_RESID>, maxdyn));
    CK(set_max_dyn(k_stream_matvec_f16<16, SF_STORE>, maxdyn));
    CK(set_max_dyn(k_stream_matvec_f16<16, SF_RESID>, maxdyn));
    CK(set_max_dyn(k_stream_matvec_f16<16, SF_GATEUP>, maxdyn));
    CK(set_max_dyn(k_stream_matvec_f16<8, SF_STORE>, maxdyn));
    CK(set_max_dyn(k_stream_matvec_f16<8, SF_RESID>, maxdyn));
    CK(set_max_dyn(k_stream_matvec_f16<8, SF_GATEUP>, maxdyn));
    done = true;
    return B200_OK;
}

int prefill_init(b200_plan *p);

int build(b200_plan *p, const b200_tensor *tensors, int n_tensors) {
    const b200_config &c = p->cfg;
    if (c.arch != B200_ARCH_LLAMA && c.arch != B200_ARCH_QWEN3 && c.arch != B200_ARCH_PHI3) return fail(p, B200_ERR_UNSUPPORTED, "unknown arch %d", c.arch);
    p->kflags = c.arch == B200_ARCH_QWEN3 ? (KF_NEOX | KF_QKNORM) : c.arch == B200_ARCH_PHI3 ? KF_NEOX : 0;
    if (c.dim <= 0 || c.dim % 32 || c.hidden_dim % 32 || (c.head_size != 32 && c.head_size != 64 && c.head_size != 96 && c.head_size != 128 && c.head_size != 256) || c.n_heads % c.n_kv_heads ||
        c.n_layers <= 0 || c.vocab_size <= 0 || c.context_length <= 0)
        return fail(p, B200_ERR_BAD_ARG, "unsupported shape (dim/hidden must be multiples of 32, head_size one of 32/64/96/128/256)");
    if (c.fp16_lanes != 0 && c.fp16_lanes != 8 && c.fp16_lanes != 16 && c.fp16_lanes != 4 && c.fp16_lanes != 32)
        return fail(p, B200_ERR_BAD_ARG, "fp16_lanes must be 0, 4, 8, 16 or 32");
    p->qd = c.n_heads * c.head_size;
    p->kvd = c.n_kv_heads * c.head_size;
    if (c.arch != B200_ARCH_QWEN3 && p->qd != c.dim) return fail(p, B200_ERR_BAD_ARG, "llama / phi3: n_heads*head_size must equal dim");
    {
        const int tn = c.tp_size;
        if (tn < 1 || tn > TP_MAX || c.tp_rank < 0 || c.tp_rank >= tn) return fail(p, B200_ERR_BAD_ARG, "bad tp_rank/tp_size %d/%d", c.tp_rank, tn);
        if (tn > 1 && (c.n_heads % tn || c.n_kv_heads % tn || c.dim % (4 * tn) || c.hidden_dim % (32 * tn) || c.vocab_size % (4 * tn)))
            return fail(p, B200_ERR_UNSUPPORTED, "shape does not split %d ways (heads, kv heads, dim/4, hidden/32 and vocab/4 must be divisible)", tn);
        p->nh_l = c.n_heads / tn; p->nkv_l = c.n_kv_heads / tn;
        p->qd_l = p->nh_l * c.head_size; p->kvd_l = p->nkv_l * c.head_size;
        p->hid_l = c.hidden_dim / tn; p->dim_l = c.dim / tn; p->voc_l = c.vocab_size / tn;
        p->tp.rank = c.tp_rank; p->tp.n = 1; // n becomes tp_size once the peers are attached
        p->tp.ops_per_fwd = 4u * (unsigned)c.n_layers + 1u;
    }

    const b200_tensor *emb = find(tensors, n_tensors, "token_embd.weight");
    if (!emb) return fail(p, B200_ERR_BAD_ARG, "missing tensor token_embd.weight");
    const b200_tensor *wq0 = find(tensors, n_tensors, c.arch == B200_ARCH_PHI3 ? "blk.0.attn_qkv.weight" : "blk.0.attn_q.weight");
    if (!wq0) return fail(p, B200_ERR_BAD_ARG, "missing tensor blk.0.attn_q.weight (Phi-3: blk.0.attn_qkv.weight)");
    p->wtype = eff_type(wq0->ggml_type); // K-quant matrices become Q8_0 while they are uploaded (kquant.cuh)
    if (p->wtype != B200_GGML_Q8_0 && p->wtype != B200_GGML_F16)
        return fail(p, B200_ERR_UNSUPPORTED, "Type: %d currently not supported for B200 weights (Q8_0, F16 and the K-quants Q4_K/Q5_K/Q6_K only)", wq0->ggml_type);
    bool any_kq = false;
    for (int i = 0; i < n_tensors; i++) any_kq = any_kq || kq_is_kquant(tensors[i].ggml_type);

    CK(cudaSetDevice(p->device));
    read_knobs(p);
    CK(cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking));
    CK(cudaEventCreate(&p->ev0));
    CK(cudaEventCreate(&p->ev1));
    int rc;
    CK(cudaDeviceGetAttribute(&p->n_sms, cudaDevAttrMultiProcessorCount, p->device));
    if (p->wtype == B200_GGML_Q8_0) {
        const bool tiles = stream_shape_ok(p->qd_l + 2 * p->kvd_l, c.dim) && stream_shape_ok(p->dim_l, p->qd) && stream_shape_ok(2 * p->hid_l, c.dim) &&
                           stream_shape_ok(p->dim_l, c.hidden_dim) && stream_shape_ok(p->voc_l, c.dim) && gateup_fits(p->hid_l, p->n_sms);
        p->path = tiles ? Q8_TILES : Q8_ROWS;
    } else {
        const int lanes = c.fp16_lanes;
        const bool rings = sf_layout(p->qd + 2 * p->kvd, c.dim, lanes, false).ok && sf_layout(c.dim, p->qd, lanes, false).ok &&
                           sf_layout(c.hidden_dim, c.dim, lanes, true).ok && sf_layout(c.dim, c.hidden_dim, lanes, false).ok && sf_layout(c.vocab_size, c.dim, lanes, false).ok;
        p->path = rings ? F16_RINGS : F16_ROWS;
    }
    if (c.tp_size > 1 && p->path != Q8_TILES) return fail(p, B200_ERR_UNSUPPORTED, "tensor parallelism needs the Q8_0 streaming path");
    size_t stage_bytes = (size_t)34 * (8u << 20); // 8 Mi blocks = 272 MiB
    if (p->path == Q8_TILES) {
        size_t m1 = (size_t)c.vocab_size * c.dim, m2 = (size_t)2 * c.hidden_dim * c.dim, m3 = (size_t)(p->qd + 2 * p->kvd) * c.dim;
        size_t mx = m1 > m2 ? m1 : m2;
        if (m3 > mx) mx = m3;
        size_t need = mx / 32 * 34 + 4096;
        if (need > stage_bytes) stage_bytes = need;
    }
    if (any_kq) { // second half of each staging buffer receives the raw K-quant bytes (always fewer than their Q8_0 form)
        stage_bytes = (stage_bytes + 255) & ~(size_t)255;
        p->kq_off = stage_bytes;
        stage_bytes *= 2;
    }
    const auto t_up0 = std::chrono::steady_clock::now();
    if ((rc = up_init(p, stage_bytes))) return rc;
    struct UploadGuard { b200_plan *pl; ~UploadGuard() { up_destroy(pl); } } guard{p};

    // embedding table (+ tied classifier: AbstractModelLoader.java:186-195)
    if ((rc = alloc_matrix(p, p->emb, c.vocab_size, c.dim, eff_type(emb->ggml_type)))) return rc;
    if ((rc = upload_matrix(p, emb, c.vocab_size, c.dim, p->emb, 0))) return rc;
    const b200_tensor *outw = find(tensors, n_tensors, "output.weight");
    if (!outw && eff_type(emb->ggml_type) != p->wtype) return fail(p, B200_ERR_UNSUPPORTED, "tied output weight type differs from the matrix type");
    p->out = p->emb; // a tied classifier; replaced below when the file has its own and the row kernels or rings read it
    if (p->path == Q8_TILES) {
        const int r0[3] = {c.tp_rank * p->voc_l, 0, 0}, fu[3] = {c.vocab_size, 0, 0};
        if ((rc = upload_tiles(p, outw ? outw : emb, nullptr, nullptr, p->voc_l, 0, 0, c.dim, false, p->tout, r0, fu))) return rc;
        if ((rc = dalloc(p, &p->blk_cnt, (size_t)(c.hidden_dim / 32) * 4))) return rc;
        CK(cudaMemset(p->blk_cnt, 0, (size_t)(c.hidden_dim / 32) * 4));
    } else if (outw) {
        if ((rc = alloc_matrix(p, p->out, c.vocab_size, c.dim, p->wtype))) return rc;
        if ((rc = upload_matrix(p, outw, c.vocab_size, c.dim, p->out, 0))) return rc;
    }
    if (p->streaming()) { // per-CTA argmax partials of the classifier launch: one CTA per SM on the tile stream, at most 3 on the rings
        const size_t parts = (size_t)p->n_sms * (p->path == F16_RINGS ? 4 : 1);
        if ((rc = dalloc(p, &p->part_val, parts * 4))) return rc;
        if ((rc = dalloc(p, &p->part_idx, parts * 4))) return rc;
    }
    if ((rc = upload_f32(p, find(tensors, n_tensors, "output_norm.weight"), c.dim, &p->out_norm, "output_norm.weight"))) return rc;

    p->layers.resize(c.n_layers);
    for (int l = 0; l < c.n_layers; l++) {
        LayerW &L = p->layers[l];
        std::string pre = "blk." + std::to_string(l) + ".";
        auto T = [&](const char *s) { return find(tensors, n_tensors, pre + s); };
        if ((rc = upload_f32(p, T("attn_norm.weight"), c.dim, &L.attn_norm, "attn_norm.weight"))) return rc;
        if ((rc = upload_f32(p, T("ffn_norm.weight"), c.dim, &L.ffn_norm, "ffn_norm.weight"))) return rc;
        if (c.arch == B200_ARCH_QWEN3) {
            if ((rc = upload_f32(p, T("attn_q_norm.weight"), c.head_size, &L.q_norm, "attn_q_norm.weight"))) return rc;
            if ((rc = upload_f32(p, T("attn_k_norm.weight"), c.head_size, &L.k_norm, "attn_k_norm.weight"))) return rc;
        }
        // Phi-3 stores wqkv and gate|up fused (Phi3StandardWeights: attn_qkv.weight = [q; k; v] rows, ffn_up.weight = [gate; up] rows,
        // InferenceCore.java:718-724,779-781): the row ranges below address the same source tensor; rows are independent dot products, so
        // splitting a fused matrix by rows changes nothing in the arithmetic.
        const bool phi3 = c.arch == B200_ARCH_PHI3;
        const b200_tensor *tq = T(phi3 ? "attn_qkv.weight" : "attn_q.weight"), *tk = phi3 ? tq : T("attn_k.weight"), *tv = phi3 ? tq : T("attn_v.weight");
        const b200_tensor *tg = T(phi3 ? "ffn_up.weight" : "ffn_gate.weight"), *tu = T("ffn_up.weight");
        const int q_full = phi3 ? p->qd + 2 * p->kvd : p->qd, k_full = phi3 ? q_full : p->kvd, g_full = phi3 ? 2 * c.hidden_dim : c.hidden_dim;
        const int k_src = phi3 ? p->qd : 0, v_src = phi3 ? p->qd + p->kvd : 0, u_src = phi3 ? c.hidden_dim : 0;
        if (p->path == Q8_TILES) {
            const int rk = c.tp_rank;
            const int qr0[3] = {rk * p->qd_l, k_src + rk * p->kvd_l, v_src + rk * p->kvd_l}, qfu[3] = {q_full, k_full, k_full};
            if ((rc = upload_tiles(p, tq, tk, tv, p->qd_l, p->kvd_l, p->kvd_l, c.dim, false, L.tqkv, qr0, qfu))) return rc;
            const int dr0[3] = {rk * p->dim_l, 0, 0}, dfu[3] = {c.dim, 0, 0};
            if ((rc = upload_tiles(p, T("attn_output.weight"), nullptr, nullptr, p->dim_l, 0, 0, p->qd, false, L.two, dr0, dfu))) return rc;
            const int gr0[3] = {rk * p->hid_l, u_src + rk * p->hid_l, 0}, gfu[3] = {g_full, g_full, 0};
            if ((rc = upload_tiles(p, tg, tu, nullptr, p->hid_l, p->hid_l, 0, c.dim, true, L.tgu, gr0, gfu))) return rc;
            if ((rc = upload_tiles(p, T("ffn_down.weight"), nullptr, nullptr, p->dim_l, 0, 0, c.hidden_dim, false, L.tw2, dr0, dfu))) return rc;
            continue;
        }
        // fused [Wq; Wk; Wv] so one launch produces the packed q|k|v vector
        if ((rc = alloc_matrix(p, L.qkv, p->qd + 2 * p->kvd, c.dim, p->wtype))) return rc;
        if ((rc = upload_matrix(p, tq, p->qd, c.dim, L.qkv, 0, 0, q_full))) return rc;
        if ((rc = upload_matrix(p, tk, p->kvd, c.dim, L.qkv, p->qd, k_src, k_full))) return rc;
        if ((rc = upload_matrix(p, tv, p->kvd, c.dim, L.qkv, p->qd + p->kvd, v_src, k_full))) return rc;
        if ((rc = alloc_matrix(p, L.wo, c.dim, p->qd, p->wtype))) return rc;
        if ((rc = upload_matrix(p, T("attn_output.weight"), c.dim, p->qd, L.wo, 0))) return rc;
        if ((rc = alloc_matrix(p, L.w1, c.hidden_dim, c.dim, p->wtype))) return rc;
        if ((rc = upload_matrix(p, tg, c.hidden_dim, c.dim, L.w1, 0, 0, g_full))) return rc;
        if ((rc = alloc_matrix(p, L.w3, c.hidden_dim, c.dim, p->wtype))) return rc;
        if ((rc = upload_matrix(p, tu, c.hidden_dim, c.dim, L.w3, 0, u_src, g_full))) return rc;
        if ((rc = alloc_matrix(p, L.w2, c.dim, c.hidden_dim, p->wtype))) return rc;
        if ((rc = upload_matrix(p, T("ffn_down.weight"), c.dim, c.hidden_dim, L.w2, 0))) return rc;
    }

    // drain the pipeline: every copy and every repack has finished before the first forward
    CK(cudaStreamSynchronize(p->up.copy));
    CK(cudaStreamSynchronize(p->stream));
    p->up.total_s = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_up0).count();
    up_destroy(p); // pinned buffers and device staging are not needed any more (the timings survive)
    // RoPE table exactly as RoPE.precomputeFreqsCis (RoPE.java:6-37, ropeScaling=false):
    // freq = (float)(1.0 / Math.pow(theta, i / (double) headSize)); val = pos * freq (float);
    // cos/sin evaluated in double and narrowed.
    {
        int half = c.head_size / 2;
        std::vector<float> cr((size_t)c.context_length * half), ci((size_t)c.context_length * half);
        size_t k = 0;
        for (int pos = 0; pos < c.context_length; pos++)
            for (int i = 0; i < c.head_size; i += 2) {
                float freq = (float)(1.0 / pow((double)c.rope_theta, i / (double)c.head_size));
                float val = (float)pos * freq;
                cr[k] = (float)cos((double)val);
                ci[k] = (float)sin((double)val);
                k++;
            }
        if ((rc = dalloc(p, &p->rope_cr, cr.size() * 4))) return rc;
        if ((rc = dalloc(p, &p->rope_ci, ci.size() * 4))) return rc;
        CK(cudaMemcpy(p->rope_cr, cr.data(), cr.size() * 4, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(p->rope_ci, ci.data(), ci.size() * 4, cudaMemcpyHostToDevice));
    }

    int big = c.dim > p->qd ? c.dim : p->qd;
    if (c.tp_size > 1) {
        // one IPC-exportable allocation: x | attq | atts | hq | hs | argmax partials | flags | tick | done counters
        auto al = [](size_t v) { return (v + 255) & ~(size_t)255; };
        size_t o = 0;
        p->tp.off_x = (unsigned)o; o = al(o + (size_t)c.dim * 4);
        p->tp.off_attq = (unsigned)o; o = al(o + (size_t)p->qd);
        p->tp.off_atts = (unsigned)o; o = al(o + (size_t)(p->qd / 32) * 4);
        p->tp.off_hq = (unsigned)o; o = al(o + (size_t)c.hidden_dim);
        p->tp.off_hs = (unsigned)o; o = al(o + (size_t)(c.hidden_dim / 32) * 4);
        p->tp.off_pv = (unsigned)o; o = al(o + TP_MAX * 4);
        p->tp.off_pi = (unsigned)o; o = al(o + TP_MAX * 4);
        p->tp.off_flags = (unsigned)o; o = al(o + TP_SLOTS * TP_MAX * 4);
        p->tp.off_tick = (unsigned)o; o = al(o + 4);
        p->tp.off_done = (unsigned)o; o = al(o + TP_SLOTS * 4);
        p->pd_flags_off = (unsigned)o; o = al(o + PD_S_SLOTS * TP_MAX * 4); // epoch flags of the persistent decode kernel
        p->comm_bytes = o;
        if ((rc = dalloc(p, &p->comm, o))) return rc;
        CK(cudaMemset(p->comm, 0, o));
        p->x = reinterpret_cast<float *>(p->comm + p->tp.off_x);
    } else if ((rc = dalloc(p, &p->x, (size_t)c.dim * 4))) return rc;
    if ((rc = dalloc(p, &p->xb, (size_t)big * 4))) return rc;
    if ((rc = dalloc(p, &p->qkv, (size_t)(p->qd_l + 2 * p->kvd_l) * 4))) return rc;
    if ((rc = dalloc(p, &p->hb, (size_t)c.hidden_dim * 4))) return rc;
    if ((rc = dalloc(p, &p->hb2, (size_t)c.hidden_dim * 4))) return rc;
    if ((rc = dalloc(p, &p->logits, (size_t)sampler_padded(c.vocab_size) * 4))) return rc; // zero pad: the sampler's exact sum runs over whole thread chunks
    if ((rc = dalloc(p, &p->xq, (size_t)big))) return rc;
    if ((rc = dalloc(p, &p->xs, (size_t)(big / 32) * 4))) return rc;
    if (c.tp_size > 1) {
        p->hq = reinterpret_cast<int8_t *>(p->comm + p->tp.off_hq);
        p->hs = reinterpret_cast<float *>(p->comm + p->tp.off_hs);
        p->attq = reinterpret_cast<int8_t *>(p->comm + p->tp.off_attq);
        p->atts = reinterpret_cast<float *>(p->comm + p->tp.off_atts);
    } else {
        if ((rc = dalloc(p, &p->hq, (size_t)c.hidden_dim))) return rc;
        if ((rc = dalloc(p, &p->hs, (size_t)(c.hidden_dim / 32) * 4))) return rc;
        p->attq = p->xq; // the attention output is the activation of the Wo matvec
        p->atts = p->xs;
    }
    size_t kv_bytes = (size_t)c.n_layers * c.context_length * p->kvd_l * 4;
    if ((rc = dalloc(p, &p->key_cache, kv_bytes))) return rc;
    if ((rc = dalloc(p, &p->value_cache, kv_bytes))) return rc;
    CK(cudaMemset(p->key_cache, 0, kv_bytes));
    CK(cudaMemset(p->value_cache, 0, kv_bytes));
    CK(cudaMemset(p->logits, 0, (size_t)sampler_padded(c.vocab_size) * 4));
    if ((rc = dalloc(p, &p->smp_indices, (size_t)c.vocab_size * 4))) return rc;
    if ((rc = dalloc(p, &p->smp_out, 8 * 4))) return rc;
    p->seq_cap = c.context_length + 8;
    if ((rc = dalloc(p, &p->st, sizeof(StepState)))) return rc;
    if ((rc = dalloc(p, &p->seq_tokens, (size_t)p->seq_cap * 4))) return rc;
    if ((rc = dalloc(p, &p->out_ids, (size_t)p->seq_cap * 4))) return rc;
    CK(cudaMemset(p->st, 0, sizeof(StepState)));
    CK(cudaMemset(p->seq_tokens, 0, (size_t)p->seq_cap * 4));
    CK(cudaMallocHost(&p->h_st, sizeof(StepState)));
    CK(cudaMallocHost(&p->h_ids, (size_t)p->seq_cap * 4));

    // epoch counters of the persistent kernel + the error word every bounded device-side wait reports through
    if ((rc = dalloc(p, &p->pd_sync, PD_S_WORDS * 4))) return rc;
    CK(cudaMemset(p->pd_sync, 0, PD_S_WORDS * 4));
    CK(cudaHostAlloc(&p->h_err, 64, cudaHostAllocMapped));
    *p->h_err = 0u;
    CK(cudaHostGetDevicePointer((void **)&p->d_err, p->h_err, 0));
    p->tp.err = p->pd_sync + PD_S_ERR;
    p->tp.host_err = p->d_err;
    if (3 * c.head_size + c.context_length > ATT_SMEM_FLOATS_MAX) { // long context: score rows in global memory
        if ((rc = dalloc(p, &p->att_scratch, (size_t)p->nh_l * ((c.context_length + PD_CT - 1) / PD_CT * PD_CT) * 4))) return rc;
    }
    if ((rc = set_smem_attrs(p))) return rc;
    if (c.tp_size > 1) { CK(cudaStreamSynchronize(p->stream)); return B200_OK; } // graphs are captured by b200_tp_attach
    if ((rc = capture_all(p))) return rc;
    if (p->prefill_batch > 1)
        if ((rc = prefill_init(p))) return rc;
    CK(cudaStreamSynchronize(p->stream));
    return B200_OK;
}

// ---- batched prefill on the tensor cores (prefill.cuh) -------------------------------------------
int prefill_init(b200_plan *p) {
    PrefillCtx &c = p->prefill;
    const b200_config &g = p->cfg;
    c.batch = p->prefill_batch;
    c.ready = false;
    c.mode = 0;
    const int kv_mul = g.n_heads / g.n_kv_heads, nqkv = p->qd + 2 * p->kvd;
    if (p->wtype != B200_GGML_F16 && !p->f16_copies) {
        c.why = p->path == Q8_TILES ? "Q8_0 plan: the tensor-core prefill is opt-in (b200_set_prefill_mode builds f16 twins of the weight matrices, +2 bytes per weight)"
                                    : "tensor-core prefill needs FP16 weight matrices or a Q8_0 plan on the streaming path";
        return B200_OK;
    }
    if (g.tp_size > 1) { c.why = "tensor-core prefill is single-GPU"; return B200_OK; }
    if (g.head_size != 64 && g.head_size != 128) { c.why = "tensor-core prefill supports head sizes 64 and 128"; return B200_OK; }
    if (kv_mul > 64 || (kv_mul & (kv_mul - 1))) { c.why = "tensor-core prefill needs a power-of-two GQA ratio <= 64"; return B200_OK; }
    if (g.dim % 128 || p->qd % 128 || nqkv % 128 || g.hidden_dim % 64) { c.why = "tensor-core prefill needs dim, q width and q+k+v width multiples of 128, hidden a multiple of 64"; return B200_OK; }
    if (!pg::encode_fn()) { c.why = "cuTensorMapEncodeTiled not available from the driver"; return B200_OK; }
    c.bpad = (c.batch + 511) / 512 * 512; // a whole number of 256-row CTA-pair tiles
    int rc;
    if ((rc = dalloc(p, &c.X, (size_t)c.bpad * g.dim * 4))) return rc;
    if ((rc = dalloc(p, &c.QKV, (size_t)c.bpad * nqkv * 4))) return rc;
    if ((rc = dalloc(p, &c.A16, (size_t)c.bpad * g.dim * 2))) return rc;
    if ((rc = dalloc(p, &c.ATT16, (size_t)c.bpad * p->qd * 2))) return rc;
    if ((rc = dalloc(p, &c.H16, (size_t)c.bpad * g.hidden_dim * 2))) return rc;
    if ((rc = dalloc(p, &c.tok, (size_t)c.bpad * 4))) return rc;
    if ((rc = dalloc(p, &c.KH, (size_t)g.context_length * p->kvd * 2))) return rc; // f16 K / V of the layer being processed
    if ((rc = dalloc(p, &c.VH, (size_t)g.context_length * p->kvd * 2))) return rc;
    CK(cudaMemset(c.X, 0, (size_t)c.bpad * g.dim * 4));
    CK(cudaMemset(c.QKV, 0, (size_t)c.bpad * nqkv * 4));
    CK(cudaMemset(c.A16, 0, (size_t)c.bpad * g.dim * 2));
    CK(cudaMemset(c.ATT16, 0, (size_t)c.bpad * p->qd * 2));
    CK(cudaMemset(c.H16, 0, (size_t)c.bpad * g.hidden_dim * 2));
    CK(cudaMemset(c.tok, 0, (size_t)c.bpad * 4));
    bool ok = pg::make_map(&c.mA, c.A16, c.bpad, g.dim, pg::BM) == 0 && pg::make_map(&c.mATT, c.ATT16, c.bpad, p->qd, pg::BM) == 0 &&
              pg::make_map(&c.mH, c.H16, c.bpad, g.hidden_dim, pg::BM) == 0 && pg::make_map_c(&c.mX, c.X, c.bpad, g.dim) == 0 &&
              pg::make_map_c(&c.mQKV, c.QKV, c.bpad, nqkv) == 0;
    c.pair = nqkv % 256 == 0 && g.dim % 256 == 0 && g.hidden_dim % 128 == 0; // the GEMMs divide into 256-wide pair tiles
    const int gu_box = c.pair ? 128 : pg::BN / 2; // gate/up tile: 128 + 128 weight rows on a CTA pair, 64 + 64 on one CTA
    c.maps.resize(g.n_layers);
    for (int l = 0; ok && l < g.n_layers; l++) {
        const LayerW &L = p->layers[l];
        PrefillLayerMaps &m = c.maps[l];
        ok = pg::make_map(&m.qkv, L.qkv.qs, nqkv, g.dim, pg::BN) == 0 && pg::make_map(&m.wo, L.wo.qs, g.dim, p->qd, pg::BN) == 0 &&
             pg::make_map(&m.w1, L.w1.qs, g.hidden_dim, g.dim, gu_box) == 0 && pg::make_map(&m.w3, L.w3.qs, g.hidden_dim, g.dim, gu_box) == 0 &&
             pg::make_map(&m.w2, L.w2.qs, g.dim, g.hidden_dim, pg::BN) == 0;
    }
    if (!ok) { c.why = "cuTensorMapEncodeTiled rejected a tensor map"; return B200_OK; }
    if (g.head_size == 128) CK(cudaFuncSetAttribute(k_pf_attention_mma<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pm_smem_bytes<128>()));
    else CK(cudaFuncSetAttribute(k_pf_attention_mma<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pm_smem_bytes<64>()));
    c.ready = true;
    c.mode = 1;
    c.why = "";
    return B200_OK;
}

// Q8_0 plan: f16 twins of the weight matrices, dequantised on the device from the tile-major stream (value = f16(q * scale),
// Q8_0FloatTensor.getFloat rounded once) -- the B operands of the tensor-core GEMMs; the reference's Q8_0 MMA prefill also
// feeds FP16 tiles (LlamaQ8_0LayersBatchPrefillMMA.java).  Built on the first b200_set_prefill_mode(TENSOR_CORE).
int build_f16_twins(b200_plan *p) {
    const b200_config &c = p->cfg;
    if (p->f16_copies) return B200_OK;
    if (p->path != Q8_TILES || c.tp_size > 1) return fail(p, B200_ERR_UNSUPPORTED, "f16 twins need a single-GPU Q8_0 plan on the streaming path");
    for (int l = 0; l < c.n_layers; l++) {
        LayerW &L = p->layers[l];
        int rc;
        if ((rc = alloc_matrix(p, L.qkv, p->qd + 2 * p->kvd, c.dim, B200_GGML_F16))) return rc;
        if ((rc = alloc_matrix(p, L.wo, c.dim, p->qd, B200_GGML_F16))) return rc;
        if ((rc = alloc_matrix(p, L.w1, c.hidden_dim, c.dim, B200_GGML_F16))) return rc;
        if ((rc = alloc_matrix(p, L.w3, c.hidden_dim, c.dim, B200_GGML_F16))) return rc;
        if ((rc = alloc_matrix(p, L.w2, c.dim, c.hidden_dim, B200_GGML_F16))) return rc;
        auto run = [&](const TileMat &t, int gateup, const DevMat &o0, const DevMat &o1) {
            k_tiles_to_f16<<<(unsigned)((size_t)t.rows * t.nseg), 128, 0, p->stream>>>(t, gateup, (__half *)o0.qs, (__half *)o1.qs);
        };
        run(L.tqkv, 0, L.qkv, L.qkv);
        run(L.two, 0, L.wo, L.wo);
        run(L.tgu, 1, L.w1, L.w3);
        run(L.tw2, 0, L.w2, L.w2);
        CK(cudaGetLastError());
    }
    CK(cudaStreamSynchronize(p->stream));
    p->f16_copies = true;
    return B200_OK;
}

// One prefill GEMM over n tokens: C[n][N] (MODE: =, += or gate/up SwiGLU) from the A activations and the B (and B2) weight maps, K deep.
// CTA pairs (c.pair): M in 256-row pair tiles; QKV and gate/up on the persistent kernel, the x += A W^T GEMMs split K so that the
// grid fills the SMs -- every split reduce-adds its partial product through TMA.  Single CTAs: a GEMM that fits one wave has one
// CTA per SM anyway and gets the deep ring; otherwise two CTAs share an SM.  A gate/up tile covers half as many output columns.
template <int MODE>
int pf_gemm(b200_plan *p, int n, const CUtensorMap &a, const CUtensorMap &b, const CUtensorMap &b2, const CUtensorMap &c_map, void *C, int N, int K) {
    const int gu = MODE == pg::GEMM_GATEUP ? 2 : 1;
    cudaStream_t s = p->stream;
    if (p->prefill.pair) {
        const int mt2 = (n + 255) / 256 * 2, nt = N * gu / 256;
        if constexpr (MODE == pg::GEMM_RESID) {
            const int ctas = mt2 * nt, nk = K / pg::BK;
            int splits = p->n_sms / ctas;
            if (splits > 4) splits = 4;
            while (splits > 1 && nk / splits < 8) splits--;
            return pg::gemm2_launch<256, pg::GEMM2_STAGES_256>(a, b, c_map, n, mt2, nt, K, s, splits < 1 ? 1 : splits);
        } else {
            return pg::gemm2_persist_launch<MODE, 256, pg::GEMM2_PERSIST_STAGES_256>(a, b, b2, c_map, C, N, n, mt2, nt, K, p->n_sms, s);
        }
    }
    const int mt = (n + pg::BM - 1) / pg::BM, nt = N * gu / pg::BN;
    if (mt * nt <= p->n_sms) return pg::gemm_launch<MODE, pg::GEMM_STAGES_DEEP>(a, b, b2, c_map, C, N, n, mt, nt, K, s);
    return pg::gemm_launch<MODE, pg::GEMM_STAGES>(a, b, b2, c_map, C, N, n, mt, nt, K, s);
}

// n tokens already in c.tok (device), positions start_pos .. start_pos + n - 1
int prefill_forward(b200_plan *p, int n, int start_pos, int *launches) {
    PrefillCtx &c = p->prefill;
    const b200_config &g = p->cfg;
    cudaStream_t s = p->stream;
    const int nqkv = p->qd + 2 * p->kvd, kv_mul = g.n_heads / g.n_kv_heads;
    const size_t ctx_kv = (size_t)g.context_length * p->kvd;
    const float inv_sqrt_hs = (float)(1.0 / sqrt((double)g.head_size));
    int nl = 0;
    k_pf_embed<<<n, 256, 0, s>>>(c.tok, p->emb, c.X, g.dim); nl++;
    for (int l = 0; l < g.n_layers; l++) {
        const LayerW &L = p->layers[l];
        const PrefillLayerMaps &m = c.maps[l];
        float *kc = p->key_cache + (size_t)l * ctx_kv, *vc = p->value_cache + (size_t)l * ctx_kv;
        k_pf_rmsnorm_f16<<<n, 256, 0, s>>>(c.X, L.attn_norm, g.rms_norm_eps, g.dim, c.A16); nl++;
        if (pf_gemm<pg::GEMM_F32>(p, n, c.mA, m.qkv, m.qkv, c.mQKV, c.QKV, nqkv, g.dim)) return fail(p, B200_ERR_CUDA, "QKV GEMM launch failed");
        nl++;
        const int qt = PM_ROWS / kv_mul;
        const dim3 ag((n + qt - 1) / qt, g.n_kv_heads);
        if (start_pos > 0) { // rows written by earlier chunks / decode steps
            const size_t n4 = (size_t)start_pos * p->kvd / 4;
            k_pf_kv_to_f16<<<(unsigned)((n4 + 255) / 256 < 1184 ? (n4 + 255) / 256 : 1184), 256, 0, s>>>(kc, vc, c.KH, c.VH, n4);
            nl++;
        }
        if (g.head_size == 128) {
            k_pf_rope_kv<128><<<n, 256, 0, s>>>(c.QKV, nqkv, kc, vc, c.KH, c.VH, p->kvd, g.n_heads, g.n_kv_heads, p->kflags, L.q_norm, L.k_norm, g.rms_norm_eps, p->rope_cr, p->rope_ci, start_pos);
            k_pf_attention_mma<128><<<ag, PM_THREADS, pm_smem_bytes<128>(), s>>>(c.QKV, nqkv, c.KH, c.VH, p->kvd, kv_mul, n, start_pos, inv_sqrt_hs, c.ATT16, p->qd);
        } else {
            k_pf_rope_kv<64><<<n, 256, 0, s>>>(c.QKV, nqkv, kc, vc, c.KH, c.VH, p->kvd, g.n_heads, g.n_kv_heads, p->kflags, L.q_norm, L.k_norm, g.rms_norm_eps, p->rope_cr, p->rope_ci, start_pos);
            k_pf_attention_mma<64><<<ag, PM_THREADS, pm_smem_bytes<64>(), s>>>(c.QKV, nqkv, c.KH, c.VH, p->kvd, kv_mul, n, start_pos, inv_sqrt_hs, c.ATT16, p->qd);
        }
        nl += 2;
        if (pf_gemm<pg::GEMM_RESID>(p, n, c.mATT, m.wo, m.wo, c.mX, c.X, g.dim, p->qd)) return fail(p, B200_ERR_CUDA, "Wo GEMM launch failed");
        nl++;
        k_pf_rmsnorm_f16<<<n, 256, 0, s>>>(c.X, L.ffn_norm, g.rms_norm_eps, g.dim, c.A16); nl++;
        if (pf_gemm<pg::GEMM_GATEUP>(p, n, c.mA, m.w1, m.w3, c.mX, c.H16, g.hidden_dim, g.dim)) return fail(p, B200_ERR_CUDA, "gate/up GEMM launch failed");
        nl++;
        if (pf_gemm<pg::GEMM_RESID>(p, n, c.mH, m.w2, m.w2, c.mX, c.X, g.dim, g.hidden_dim)) return fail(p, B200_ERR_CUDA, "W2 GEMM launch failed");
        nl++;
    }
    CK(cudaGetLastError());
    if (launches) *launches = nl;
    return B200_OK;
}

cudaGraphExec_t decode_graph(b200_plan *p) { return p->decode_mode == B200_DECODE_PERSISTENT && p->g_pdecode ? p->g_pdecode : p->g_decode; }
cudaGraphExec_t prefill_graph(b200_plan *p) { return p->decode_mode == B200_DECODE_PERSISTENT && p->g_pprefill ? p->g_pprefill : p->g_prefill; }

// After a synchronize: did a device-side wait of the persistent kernel (or a tensor-parallel flag wait) give up?
int check_device_error(b200_plan *p) {
    if (p->h_err && *reinterpret_cast<volatile unsigned *>(p->h_err)) {
        const unsigned code = *reinterpret_cast<volatile unsigned *>(p->h_err);
        return fail(p, B200_ERR_STATE, "a device-side wait timed out (code %u: 1+phase of the persistent decode kernel, 100+slot of a tensor-parallel flag): a peer "
                                       "rank is missing or the ranks' call sequences diverged; the plan must be freed", code);
    }
    return B200_OK;
}

int set_state(b200_plan *p, int token, int pos, int n_seq, int feedback) {
    StepState *h = p->h_st;
    h->token = token; h->pos = pos; h->step = 0; h->n_seq = n_seq; h->feedback = feedback;
    CK(cudaMemcpyAsync(p->st, h, sizeof(StepState), cudaMemcpyHostToDevice, p->stream));
    return B200_OK;
}

int check_pos(b200_plan *p, int token, int pos) {
    if (token < 0 || token >= p->cfg.vocab_size) return fail(p, B200_ERR_BAD_ARG, "token %d out of range", token);
    if (pos < 0 || pos >= p->cfg.context_length) return fail(p, B200_ERR_BAD_ARG, "position %d outside the KV cache (%d)", pos, p->cfg.context_length);
    return B200_OK;
}

} // namespace

extern "C" {

int b200_plan_create(const b200_config *cfg, const b200_tensor *tensors, int32_t n_tensors, int32_t prefill_batch_size,
                     int32_t device, b200_plan **out, char *err, size_t err_len) {
    if (out) *out = nullptr;
    if (!cfg || !tensors || !out || n_tensors <= 0) {
        if (err && err_len) snprintf(err, err_len, "null argument");
        return B200_ERR_BAD_ARG;
    }
    b200_plan *p = new b200_plan();
    p->cfg = *cfg;
    if (p->cfg.tp_size <= 0) p->cfg.tp_size = 1;
    p->device = device;
    p->prefill_batch = prefill_batch_size;
    int rc = build(p, tensors, n_tensors);
    if (rc != B200_OK) {
        if (err && err_len) snprintf(err, err_len, "%s", p->err.c_str());
        b200_plan_free(p);
        return rc;
    }
    *out = p;
    return B200_OK;
}

int b200_forward_decode(b200_plan *p, int32_t token, int32_t position, float *logits, int32_t *argmax) {
    if (!p) return B200_ERR_BAD_ARG;
    if (!p->g_decode) return fail(p, B200_ERR_STATE, "tensor-parallel plan: call b200_tp_attach on every rank first");
    if (logits && p->tp.n > 1) return fail(p, B200_ERR_UNSUPPORTED, "full logits are not gathered under tensor parallelism (argmax is)");
    int rc;
    if ((rc = check_pos(p, token, position))) return rc;
    CK(cudaSetDevice(p->device));
    if ((rc = set_state(p, token, position, 0, 0))) return rc;
    CK(cudaGraphLaunch(decode_graph(p), p->stream));
    if (argmax) CK(cudaMemcpyAsync(p->h_ids, p->out_ids, 4, cudaMemcpyDeviceToHost, p->stream));
    if (logits) CK(cudaMemcpyAsync(logits, p->logits, (size_t)p->cfg.vocab_size * 4, cudaMemcpyDeviceToHost, p->stream));
    CK(cudaStreamSynchronize(p->stream));
    if ((rc = check_device_error(p))) return rc;
    if (argmax) *argmax = p->h_ids[0];
    return B200_OK;
}

int b200_forward_decode_sample(b200_plan *p, int32_t token, int32_t position, float temperature, float topp, float uniform01, int32_t *token_out, int32_t *info) {
    if (!p || !token_out) return B200_ERR_BAD_ARG;
    if (!p->g_decode) return fail(p, B200_ERR_STATE, "tensor-parallel plan: call b200_tp_attach on every rank first");
    if (p->tp.n > 1) return fail(p, B200_ERR_UNSUPPORTED, "the device-side temperature/top-p sampler needs the whole logits row on one GPU (tensor-parallel plans sample greedily)");
    if (!(temperature >= 0.0f) || !(uniform01 >= 0.0f && uniform01 < 1.0f)) return fail(p, B200_ERR_BAD_ARG, "temperature must be >= 0 and the uniform number in [0, 1)");
    int rc;
    if ((rc = check_pos(p, token, position))) return rc;
    CK(cudaSetDevice(p->device));
    if ((rc = set_state(p, token, position, 0, 0))) return rc;
    CK(cudaGraphLaunch(decode_graph(p), p->stream));
    const bool greedy = temperature == 0.0f; // Sampler.selectSampler: temperature 0 -> FloatTensor.argmax, already computed by the forward
    if (!greedy) {
        static bool attr = false;
        if (!attr) { CK(cudaFuncSetAttribute(k_sample, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sampler_smem_bytes())); attr = true; }
        SamplerArgs a;
        a.logits = p->logits; a.n = p->cfg.vocab_size; a.temperature = temperature; a.topp = topp; a.r01 = uniform01;
        a.indices = p->smp_indices; a.out_id = p->smp_out; a.info = p->smp_out + 1;
        k_sample<<<1, SAMPLER_THREADS, sampler_smem_bytes(), p->stream>>>(a);
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(p->h_ids, p->smp_out, 5 * 4, cudaMemcpyDeviceToHost, p->stream));
    } else CK(cudaMemcpyAsync(p->h_ids, p->out_ids, 4, cudaMemcpyDeviceToHost, p->stream));
    CK(cudaStreamSynchronize(p->stream));
    if ((rc = check_device_error(p))) return rc;
    *token_out = p->h_ids[0];
    if (info) for (int k = 0; k < 4; k++) info[k] = greedy ? 0 : p->h_ids[1 + k];
    return B200_OK;
}

int b200_forward_prefill(b200_plan *p, int32_t token, int32_t position) {
    if (!p) return B200_ERR_BAD_ARG;
    if (!p->g_prefill) return fail(p, B200_ERR_STATE, "tensor-parallel plan: call b200_tp_attach on every rank first");
    int rc;
    if ((rc = check_pos(p, token, position))) return rc;
    CK(cudaSetDevice(p->device));
    if ((rc = set_state(p, token, position, 0, 0))) return rc;
    CK(cudaGraphLaunch(prefill_graph(p), p->stream));
    CK(cudaStreamSynchronize(p->stream));
    return check_device_error(p);
}

int b200_forward_batch_prefill(b200_plan *p, const int32_t *tokens, int32_t n, int32_t start_pos) {
    if (!p || !tokens) return B200_ERR_BAD_ARG;
    if (n <= 0) return B200_OK;
    if (!p->g_prefill) return fail(p, B200_ERR_STATE, "tensor-parallel plan: call b200_tp_attach on every rank first");
    if (p->prefill_batch > 1 && n > p->prefill_batch) return fail(p, B200_ERR_BAD_ARG, "chunk of %d tokens exceeds prefill_batch_size %d", n, p->prefill_batch);
    if (start_pos < 0 || start_pos + n > p->cfg.context_length) return fail(p, B200_ERR_BAD_ARG, "positions %d..%d outside the KV cache", start_pos, start_pos + n - 1);
    for (int i = 0; i < n; i++)
        if (tokens[i] < 0 || tokens[i] >= p->cfg.vocab_size) return fail(p, B200_ERR_BAD_ARG, "token %d out of range", tokens[i]);
    CK(cudaSetDevice(p->device));
    if (p->prefill.ready && p->prefill.mode == 1) { // tensor-core GEMM path (prefill.cuh)
        memcpy(p->h_ids, tokens, (size_t)n * 4);
        CK(cudaMemcpyAsync(p->prefill.tok, p->h_ids, (size_t)n * 4, cudaMemcpyHostToDevice, p->stream));
        CK(cudaEventRecord(p->ev0, p->stream));
        int rc2 = prefill_forward(p, n, start_pos, &p->launches_prefill);
        if (rc2) return rc2;
        CK(cudaEventRecord(p->ev1, p->stream));
        CK(cudaStreamSynchronize(p->stream));
        CK(cudaEventElapsedTime(&p->prefill_ms, p->ev0, p->ev1));
        return B200_OK;
    }
    // Exact path: the prefill graph token by token (bit-identical KV cache to the CPU
    // batchForwardJavaPrefill, InferenceCoreBatchPrefillDecode.java:62-168).
    if (n > p->seq_cap) return fail(p, B200_ERR_BAD_ARG, "chunk too long");
    memcpy(p->h_ids, tokens, (size_t)n * 4);
    CK(cudaMemcpyAsync(p->seq_tokens, p->h_ids, (size_t)n * 4, cudaMemcpyHostToDevice, p->stream));
    int rc;
    if ((rc = set_state(p, tokens[0], start_pos, n, 0))) return rc;
    for (int i = 0; i < n; i++) CK(cudaGraphLaunch(prefill_graph(p), p->stream));
    CK(cudaStreamSynchronize(p->stream));
    return check_device_error(p);
}

int b200_decode_sequence(b200_plan *p, const int32_t *tokens, int32_t n, int32_t start_pos, int32_t feedback,
                         int32_t *out_ids, float *device_ms) {
    if (!p || !tokens) return B200_ERR_BAD_ARG;
    if (n <= 0) return B200_OK;
    if (!p->g_decode) return fail(p, B200_ERR_STATE, "tensor-parallel plan: call b200_tp_attach on every rank first");
    if (n > p->seq_cap) return fail(p, B200_ERR_BAD_ARG, "sequence of %d steps exceeds capacity %d", n, p->seq_cap);
    if (start_pos < 0 || start_pos + n > p->cfg.context_length) return fail(p, B200_ERR_BAD_ARG, "positions %d..%d outside the KV cache (%d)", start_pos, start_pos + n - 1, p->cfg.context_length);
    int nt = feedback ? 1 : n;
    for (int i = 0; i < nt; i++)
        if (tokens[i] < 0 || tokens[i] >= p->cfg.vocab_size) return fail(p, B200_ERR_BAD_ARG, "token %d out of range", tokens[i]);
    CK(cudaSetDevice(p->device));
    memcpy(p->h_ids, tokens, (size_t)nt * 4);
    CK(cudaMemcpyAsync(p->seq_tokens, p->h_ids, (size_t)nt * 4, cudaMemcpyHostToDevice, p->stream));
    int rc;
    if ((rc = set_state(p, tokens[0], start_pos, nt, feedback))) return rc;
    CK(cudaEventRecord(p->ev0, p->stream));
    for (int i = 0; i < n; i++) CK(cudaGraphLaunch(decode_graph(p), p->stream));
    CK(cudaEventRecord(p->ev1, p->stream));
    if (out_ids) CK(cudaMemcpyAsync(p->h_ids, p->out_ids, (size_t)n * 4, cudaMemcpyDeviceToHost, p->stream));
    CK(cudaStreamSynchronize(p->stream));
    if ((rc = check_device_error(p))) return rc;
    if (out_ids) memcpy(out_ids, p->h_ids, (size_t)n * 4);
    if (device_ms) CK(cudaEventElapsedTime(device_ms, p->ev0, p->ev1));
    return B200_OK;
}

int b200_set_decode_mode(b200_plan *p, int32_t mode) {
    if (!p || (mode != B200_DECODE_GRAPH && mode != B200_DECODE_PERSISTENT)) return B200_ERR_BAD_ARG;
    if (!p->g_decode) return fail(p, B200_ERR_STATE, "tensor-parallel plan: call b200_tp_attach on every rank first");
    if (mode == B200_DECODE_PERSISTENT && !p->pd_ok) return fail(p, B200_ERR_UNSUPPORTED, "%s", p->pd_why.c_str());
    p->decode_mode = mode;
    return B200_OK;
}

int b200_decode_info(b200_plan *p, int32_t *mode, int32_t *launches, int32_t *ring_stages, int32_t *smem_bytes) {
    if (!p) return B200_ERR_BAD_ARG;
    const bool pers = p->decode_mode == B200_DECODE_PERSISTENT && p->g_pdecode;
    if (mode) *mode = pers ? B200_DECODE_PERSISTENT : B200_DECODE_GRAPH;
    if (launches) *launches = pers ? 1 : p->launches_decode;
    if (ring_stages) *ring_stages = p->pd_ok ? p->pd_L.stages : 0;
    if (smem_bytes) *smem_bytes = p->pd_ok ? (int32_t)p->pd_L.total : 0;
    return B200_OK;
}

int b200_trace_persistent(b200_plan *p, int32_t token, int32_t position, uint64_t *stamps, int64_t cap, int32_t *n_ctas, int32_t *n_rows, int32_t *n_stamps) {
    if (!p || !stamps) return B200_ERR_BAD_ARG;
    if (!p->g_ptrace) return fail(p, B200_ERR_UNSUPPORTED, "%s", p->pd_ok ? "no traced persistent graph" : p->pd_why.c_str());
    int rc;
    if ((rc = check_pos(p, token, position))) return rc;
    CK(cudaSetDevice(p->device));
    const size_t words = (size_t)p->n_sms * (p->cfg.n_layers + 1) * PD_STAMPS;
    if ((size_t)cap < words) return fail(p, B200_ERR_BAD_ARG, "stamp buffer too small: need %zu uint64", words);
    CK(cudaMemsetAsync(p->pd_trace, 0, words * 8, p->stream));
    if ((rc = set_state(p, token, position, 0, 0))) return rc;
    CK(cudaGraphLaunch(p->g_ptrace, p->stream));
    CK(cudaStreamSynchronize(p->stream));
    if ((rc = check_device_error(p))) return rc;
    CK(cudaMemcpy(stamps, p->pd_trace, words * 8, cudaMemcpyDeviceToHost));
    if (n_ctas) *n_ctas = p->n_sms;
    if (n_rows) *n_rows = p->cfg.n_layers + 1;
    if (n_stamps) *n_stamps = PD_STAMPS;
    return B200_OK;
}

int b200_set_prefill_mode(b200_plan *p, int32_t mode) {
    if (!p || (mode != B200_PREFILL_EXACT && mode != B200_PREFILL_TENSOR_CORE)) return B200_ERR_BAD_ARG;
    if (mode == B200_PREFILL_TENSOR_CORE && !p->prefill.ready && p->prefill_batch > 1 && p->path == Q8_TILES && p->cfg.tp_size == 1) {
        CK(cudaSetDevice(p->device)); // opt-in on a Q8_0 plan: build the f16 twins, then the GEMM context
        int rc = build_f16_twins(p);
        if (rc) return rc;
        if ((rc = prefill_init(p))) return rc;
    }
    if (mode == B200_PREFILL_TENSOR_CORE && !p->prefill.ready) return fail(p, B200_ERR_UNSUPPORTED, "%s", p->prefill.why);
    p->prefill.mode = mode;
    return B200_OK;
}

int b200_prefill_info(b200_plan *p, int32_t *mode, int32_t *launches, float *device_ms) {
    if (!p) return B200_ERR_BAD_ARG;
    if (mode) *mode = p->prefill.ready ? p->prefill.mode : B200_PREFILL_EXACT;
    if (launches) *launches = p->launches_prefill;
    if (device_ms) *device_ms = p->prefill_ms;
    return B200_OK;
}

int b200_kv_reset(b200_plan *p) {
    if (!p) return B200_ERR_BAD_ARG;
    CK(cudaSetDevice(p->device));
    size_t kv_bytes = (size_t)p->cfg.n_layers * p->cfg.context_length * p->kvd_l * 4;
    CK(cudaMemsetAsync(p->key_cache, 0, kv_bytes, p->stream));
    CK(cudaMemsetAsync(p->value_cache, 0, kv_bytes, p->stream));
    CK(cudaStreamSynchronize(p->stream));
    return B200_OK;
}

int b200_read_buffer(b200_plan *p, const char *name, int32_t layer, void *dst, size_t bytes) {
    if (!p || !name || !dst) return B200_ERR_BAD_ARG;
    const b200_config &c = p->cfg;
    const void *src = nullptr;
    size_t sz = 0;
    std::string s = name;
    size_t ctx_kv = (size_t)c.context_length * p->kvd_l;
    if (s == "x") { src = p->x; sz = (size_t)c.dim * 4; }
    else if (s == "xb") { src = p->xb; sz = (size_t)(c.dim > p->qd ? c.dim : p->qd) * 4; }
    else if (s == "q" || s == "qkv") { src = p->qkv; sz = (size_t)(p->qd_l + 2 * p->kvd_l) * 4; }
    else if (s == "hb") { src = p->hb; sz = (size_t)c.hidden_dim * 4; }
    else if (s == "logits") { src = p->logits; sz = (size_t)c.vocab_size * 4; }
    else if (s == "xq") { src = p->xq; sz = (size_t)(c.dim > p->qd ? c.dim : p->qd); }
    else if (s == "xs") { src = p->xs; sz = (size_t)((c.dim > p->qd ? c.dim : p->qd) / 32) * 4; }
    else if (s == "hq") { src = p->hq; sz = (size_t)c.hidden_dim; }
    else if (s == "hs") { src = p->hs; sz = (size_t)(c.hidden_dim / 32) * 4; }
    else if (s == "key_cache" || s == "value_cache") {
        if (layer < 0 || layer >= c.n_layers) return fail(p, B200_ERR_BAD_ARG, "layer out of range");
        src = (s == "key_cache" ? p->key_cache : p->value_cache) + (size_t)layer * ctx_kv;
        sz = ctx_kv * 4;
    } else return fail(p, B200_ERR_BAD_ARG, "unknown buffer %s", name);
    if (bytes < sz) sz = bytes;
    CK(cudaSetDevice(p->device));
    CK(cudaStreamSynchronize(p->stream));
    CK(cudaMemcpy(dst, src, sz, cudaMemcpyDeviceToHost));
    return B200_OK;
}

int b200_time_kernel(b200_plan *p, int32_t which, int32_t reps, float *avg_ms, int64_t *algorithmic_bytes) {
    if (!p || !avg_ms || reps <= 0) return B200_ERR_BAD_ARG;
    if (p->cfg.tp_size > 1) return fail(p, B200_ERR_UNSUPPORTED, "b200_time_kernel is single-GPU only");
    if (which < MV_GATEUP || which > MV_CLS) return fail(p, B200_ERR_BAD_ARG, "unknown kernel id %d", which);
    const b200_config &c = p->cfg;
    const MvRole role = (MvRole)which;
    CK(cudaSetDevice(p->device));
    std::vector<float> save(c.dim);
    CK(cudaStreamSynchronize(p->stream));
    CK(cudaMemcpy(save.data(), p->x, (size_t)c.dim * 4, cudaMemcpyDeviceToHost));
    // stand-alone launches (no PDL overlap), one per layer
    int rc;
    for (int l = 0; l < c.n_layers; l++) if ((rc = launch_mv(p, role, l, false, TraceBuf{nullptr, 0, 0})) < 0) return rc; // warm-up pass (also defeats L2 for pass 1)
    CK(cudaEventRecord(p->ev0, p->stream));
    for (int r = 0; r < reps; r++)
        for (int l = 0; l < c.n_layers; l++) if ((rc = launch_mv(p, role, l, false, TraceBuf{nullptr, 0, 0})) < 0) return rc;
    CK(cudaEventRecord(p->ev1, p->stream));
    CK(cudaStreamSynchronize(p->stream));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, p->ev0, p->ev1));
    *avg_ms = ms / (reps * c.n_layers);
    if (algorithmic_bytes) { // the weight bytes one launch streams
        const int64_t rows[5] = {2LL * c.hidden_dim, c.dim, p->qd + 2LL * p->kvd, c.dim, c.vocab_size}, cols[5] = {c.dim, c.hidden_dim, c.dim, p->qd, c.dim};
        const int64_t e = rows[role] * cols[role];
        *algorithmic_bytes = p->wtype == B200_GGML_Q8_0 ? e / 32 * 34 : e * 2;
    }
    CK(cudaMemcpy(p->x, save.data(), (size_t)c.dim * 4, cudaMemcpyHostToDevice));
    return B200_OK;
}

int b200_tp_handle(b200_plan *p, void *handle64) {
    if (!p || !handle64) return B200_ERR_BAD_ARG;
    if (p->cfg.tp_size <= 1 || !p->comm) return fail(p, B200_ERR_STATE, "not a tensor-parallel plan");
    CK(cudaSetDevice(p->device));
    cudaIpcMemHandle_t h;
    CK(cudaIpcGetMemHandle(&h, p->comm));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    memcpy(handle64, &h, 64);
    return B200_OK;
}

int b200_tp_attach(b200_plan *p, const void *handles, int32_t n) {
    if (!p || !handles) return B200_ERR_BAD_ARG;
    if (p->cfg.tp_size <= 1 || !p->comm) return fail(p, B200_ERR_STATE, "not a tensor-parallel plan");
    if (n != p->cfg.tp_size) return fail(p, B200_ERR_BAD_ARG, "expected %d handles, got %d", p->cfg.tp_size, n);
    if (p->attached) return fail(p, B200_ERR_STATE, "already attached");
    CK(cudaSetDevice(p->device));
    for (int k = 0; k < n; k++) {
        if (k == p->cfg.tp_rank) { p->tp.peer[k] = p->comm; continue; }
        cudaIpcMemHandle_t h;
        memcpy(&h, (const unsigned char *)handles + (size_t)k * 64, 64);
        void *ptr = nullptr;
        CK(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
        p->peer_open[k] = ptr;
        p->tp.peer[k] = (unsigned char *)ptr;
    }
    p->tp.n = n;
    p->attached = true;
    int rc;
    if ((rc = capture_all(p))) return rc;
    CK(cudaStreamSynchronize(p->stream));
    return B200_OK;
}

int b200_trace_decode(b200_plan *p, int32_t token, int32_t position, uint64_t *records, int32_t cap, int32_t *n_out) {
    if (!p || !records || !n_out) return B200_ERR_BAD_ARG;
    if (!p->g_trace) return fail(p, B200_ERR_UNSUPPORTED, "tracing needs a streaming path (Q8_0 tiles or the FP16 rings)");
    int rc;
    if ((rc = check_pos(p, token, position))) return rc;
    CK(cudaSetDevice(p->device));
    int n = p->launches_decode;
    std::vector<unsigned long long> init((size_t)n * 4);
    for (int i = 0; i < n; i++) { init[i * 4] = 0; init[i * 4 + 1] = ~0ull; init[i * 4 + 2] = 0; init[i * 4 + 3] = 0; }
    CK(cudaMemcpyAsync(p->trace_rec, init.data(), init.size() * 8, cudaMemcpyHostToDevice, p->stream));
    if ((rc = set_state(p, token, position, 0, 0))) return rc;
    CK(cudaGraphLaunch(p->g_trace, p->stream));
    CK(cudaStreamSynchronize(p->stream));
    int m = n < cap ? n : cap;
    CK(cudaMemcpy(records, p->trace_rec, (size_t)m * 32, cudaMemcpyDeviceToHost));
    *n_out = m;
    return B200_OK;
}

static int run_seqsum_hook(const float *terms, int32_t n, int threads, float *out, int32_t *info) {
    if (!terms || !out || n <= 0 || n > 8192) return B200_ERR_BAD_ARG;
    if (threads != 256 && threads != 512 && threads != 1024) return B200_ERR_BAD_ARG;
    float *d = nullptr, *o = nullptr;
    if (cudaMalloc(&d, (size_t)n * 4) != cudaSuccess) return B200_ERR_OOM;
    if (cudaMalloc(&o, 16) != cudaSuccess) { cudaFree(d); return B200_ERR_OOM; }
    cudaError_t e = cudaMemcpy(d, terms, (size_t)n * 4, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        if (threads == 1024) {
            const size_t smem = (size_t)1024 * ((n + 1023) / 1024) * 4 + seqsum2_scratch_bytes(1024);
            e = cudaFuncSetAttribute(k_test_seqsum2<1024>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e == cudaSuccess) k_test_seqsum2<1024><<<1, 1024, smem>>>(d, n, o, reinterpret_cast<int *>(o) + 1);
        } else if (threads == 512) {
            const size_t smem = (size_t)512 * ((n + 511) / 512) * 4 + seqsum2_scratch_bytes(512);
            e = cudaFuncSetAttribute(k_test_seqsum2<512>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e == cudaSuccess) k_test_seqsum2<512><<<1, 512, smem>>>(d, n, o, reinterpret_cast<int *>(o) + 1);
        } else {
            const size_t smem = (size_t)256 * ((n + 255) / 256) * 4 + seqsum2_scratch_bytes(256);
            e = cudaFuncSetAttribute(k_test_seqsum2<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e == cudaSuccess) k_test_seqsum2<256><<<1, 256, smem>>>(d, n, o, reinterpret_cast<int *>(o) + 1);
        }
    }
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    int32_t host[3] = {0, 0, 0};
    if (e == cudaSuccess) e = cudaMemcpy(host, o, 12, cudaMemcpyDeviceToHost);
    memcpy(out, host, 4);
    if (info) { info[0] = host[1]; info[1] = host[2]; }
    cudaFree(d);
    cudaFree(o);
    return e == cudaSuccess ? B200_OK : B200_ERR_CUDA;
}

int b200_test_seqsum2(const float *terms, int32_t n, int32_t threads, float *out, int32_t *info) { return run_seqsum_hook(terms, n, threads, out, info); }

int b200_requant_kquant(int32_t ggml_type, const void *src, int64_t n_elems, void *dst_q8_0) {
    if (!src || !dst_q8_0 || n_elems <= 0 || n_elems % 256 || !kq_is_kquant(ggml_type)) return B200_ERR_BAD_ARG;
    const size_t raw = (size_t)(n_elems / 256) * kq_block_bytes(ggml_type), q8 = (size_t)(n_elems / 32) * 34;
    unsigned char *ds = nullptr, *dd = nullptr;
    int rc = B200_OK;
    auto ok = [&](cudaError_t e) { if (e != cudaSuccess && rc == B200_OK) rc = e == cudaErrorMemoryAllocation ? B200_ERR_OOM : B200_ERR_CUDA; return rc == B200_OK; };
    if (ok(cudaMalloc(&ds, raw)) && ok(cudaMalloc(&dd, q8)) && ok(cudaMemcpy(ds, src, raw, cudaMemcpyHostToDevice)) &&
        ok(launch_requant_kquant(ggml_type, ds, dd, n_elems / 32, 0)) && ok(cudaDeviceSynchronize()))
        ok(cudaMemcpy(dst_q8_0, dd, q8, cudaMemcpyDeviceToHost));
    cudaFree(ds); cudaFree(dd);
    return rc;
}

int b200_gemm_f16(const uint16_t *a, const uint16_t *b, float *c, int32_t m, int32_t n, int32_t k, int32_t iters, float *ms, int32_t stages,
                  int32_t resid, int32_t two_cta) {
    if (!a || !b || !c || m <= 0 || n <= 0 || k <= 0 || m % 128 || n % 128 || k % 64) return B200_ERR_BAD_ARG;
    // only the kernels the prefill launches (pg::gemm_f16); with resid, C starts at 0 and accumulates over the timed launches
    if (resid < 0 || (two_cta ? two_cta != (resid ? 256 : 1256) : (stages != 0 && stages != 3 && stages != 6))) return B200_ERR_BAD_ARG;
    __half *da = nullptr, *db = nullptr;
    float *dc = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    int rc = B200_OK;
    auto ok = [&](cudaError_t e) { if (e != cudaSuccess && rc == B200_OK) rc = e == cudaErrorMemoryAllocation ? B200_ERR_OOM : B200_ERR_CUDA; return rc == B200_OK; }; // first failure wins
    if (ok(cudaMalloc(&da, (size_t)m * k * 2)) && ok(cudaMalloc(&db, (size_t)n * k * 2)) && ok(cudaMalloc(&dc, (size_t)m * n * 4)) &&
        ok(cudaMemcpy(da, a, (size_t)m * k * 2, cudaMemcpyHostToDevice)) && ok(cudaMemcpy(db, b, (size_t)n * k * 2, cudaMemcpyHostToDevice)) &&
        ok(cudaMemset(dc, resid ? 0 : 0xFF, (size_t)m * n * 4))) {
        if (pg::gemm_f16(da, db, dc, m, n, k, stages, resid, two_cta, 0)) rc = B200_ERR_CUDA;
        ok(cudaDeviceSynchronize());
        if (rc == B200_OK && iters > 0 && ms && ok(cudaEventCreate(&e0)) && ok(cudaEventCreate(&e1)) && ok(cudaEventRecord(e0, 0))) {
            for (int i = 0; i < iters && rc == B200_OK; i++)
                if (pg::gemm_f16(da, db, dc, m, n, k, stages, resid, two_cta, 0)) rc = B200_ERR_CUDA;
            float t = 0.f;
            if (ok(cudaEventRecord(e1, 0)) && ok(cudaEventSynchronize(e1)) && ok(cudaEventElapsedTime(&t, e0, e1))) *ms = t / iters;
            if (rc == B200_OK && resid) { // C accumulated 1 + iters products: return exactly one
                if (ok(cudaMemset(dc, 0, (size_t)m * n * 4)) && pg::gemm_f16(da, db, dc, m, n, k, stages, resid, two_cta, 0)) rc = B200_ERR_CUDA;
                ok(cudaDeviceSynchronize());
            }
        }
        if (rc == B200_OK) ok(cudaMemcpy(c, dc, (size_t)m * n * 4, cudaMemcpyDeviceToHost));
    }
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
    cudaFree(da); cudaFree(db); cudaFree(dc);
    return rc;
}

int b200_upload_info(b200_plan *p, double *seconds, double *host_copy_seconds, int64_t *h2d_bytes) {
    if (!p) return B200_ERR_BAD_ARG;
    if (seconds) *seconds = p->up.total_s;
    if (host_copy_seconds) *host_copy_seconds = p->up.host_copy_s;
    if (h2d_bytes) *h2d_bytes = p->up.h2d_bytes;
    return B200_OK;
}

int b200_launches_per_decode(b200_plan *p) {
    if (!p) return 0;
    return (p->decode_mode == B200_DECODE_PERSISTENT && p->g_pdecode) ? 1 : p->launches_decode;
}
int64_t b200_device_bytes(b200_plan *p) { return p ? p->bytes : 0; }

void b200_plan_free(b200_plan *p) {
    if (!p) return;
    cudaSetDevice(p->device);
    if (p->stream) cudaStreamSynchronize(p->stream);
    prefill_free(p->prefill);
    if (p->g_decode) cudaGraphExecDestroy(p->g_decode);
    if (p->g_prefill) cudaGraphExecDestroy(p->g_prefill);
    if (p->g_trace) cudaGraphExecDestroy(p->g_trace);
    if (p->g_pdecode) cudaGraphExecDestroy(p->g_pdecode);
    if (p->g_pprefill) cudaGraphExecDestroy(p->g_pprefill);
    if (p->g_ptrace) cudaGraphExecDestroy(p->g_ptrace);
    if (p->h_err) cudaFreeHost(p->h_err);
    for (int k = 0; k < TP_MAX; k++) if (p->peer_open[k]) cudaIpcCloseMemHandle(p->peer_open[k]);
    for (void *d : p->allocs) cudaFree(d);
    if (p->h_st) cudaFreeHost(p->h_st);
    if (p->h_ids) cudaFreeHost(p->h_ids);
    if (p->ev0) cudaEventDestroy(p->ev0);
    if (p->ev1) cudaEventDestroy(p->ev1);
    if (p->stream) cudaStreamDestroy(p->stream);
    delete p;
}

const char *b200_last_error(b200_plan *p) { return p ? p->err.c_str() : "null plan"; }
const char *b200_version(void) { return "b200llama 0.1 sm_100a"; }

} // extern "C"
