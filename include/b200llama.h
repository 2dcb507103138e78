/*
 * b200llama.h -- C ABI of libb200llama.so: the B200-native replacement for the
 * TornadoVM execution-plan layer of beehive-lab/GPULlama3.java.
 *
 * One `b200_plan` plays the role of one `TornadoVMMasterPlan` instance
 * (reference: src/main/java/org/beehive/gpullama3/tornadovm/TornadoVMMasterPlan.java:30-85).
 * It owns the device copies of the weights (repacked from GGUF block layout at
 * creation), the FP32 KV cache ([layer][ctx][kvDim], LlamaState.java:46-47,69-70) and all
 * activation buffers.  Plain pointers and sizes only; no C++/torch types.
 *
 * Threading: a plan is single-owner (one thread at a time, like the reference where the
 * server serialises on a lock, InferenceService.java:31,58).  Several plans may coexist;
 * there is no process-global state.
 *
 * Errors: every entry point returns B200_OK (0) or a negative B200_ERR_* code;
 * b200_last_error(plan) gives the message.  The Java shim maps B200_ERR_UNSUPPORTED to
 * UnsupportedOperationException (ForwardPlanFactory.java:84-87) and B200_ERR_OOM to the
 * reference's out-of-memory error (README.md:262-265).
 */
#ifndef B200LLAMA_H
#define B200LLAMA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200_OK 0
#define B200_ERR_BAD_ARG (-1)
#define B200_ERR_UNSUPPORTED (-2)
#define B200_ERR_OOM (-3)
#define B200_ERR_CUDA (-4)
#define B200_ERR_NCCL (-5)
#define B200_ERR_STATE (-6)

#define B200_ARCH_LLAMA 0 /* InferenceCore.forwardJava,      InferenceCore.java:50-172  */
#define B200_ARCH_QWEN3 1 /* InferenceCore.forwardJavaQwen3, InferenceCore.java:565-697 */
#define B200_ARCH_PHI3 2  /* InferenceCore.forwardJavaPhi3,  InferenceCore.java:699-800: fused blk.N.attn_qkv.weight ([q; k; v] rows) and
                           * blk.N.ffn_up.weight ([gate; up] rows), NeoX-pair RoPE without q/k norm; n_heads * head_size == dim */

/* GGML tensor type ids accepted for weights (tensor/GGMLType.java:5-20) */
#define B200_GGML_F32 0
#define B200_GGML_F16 1
#define B200_GGML_Q8_0 8
/* K-quants are accepted for weight matrices and the embedding table of a Q8_0 plan: they are re-quantised to Q8_0 on the device while
 * the upload pipeline streams them in, byte-identical to ModelLoader.dequantizeToQ8_0TornadoTensor (model/loader/ModelLoader.java:163,
 * 173-224); the plan then computes exactly as for a Q8_0 file (AbstractModelLoader.java:45-59). */
#define B200_GGML_Q4_K 12
#define B200_GGML_Q5_K 13
#define B200_GGML_Q6_K 14

/* Model configuration: the fields of Configuration the forward pass reads
 * (LlamaModelLoader.java:47-63, Qwen3ModelLoader.java:48-74). */
typedef struct b200_config {
    int32_t arch;           /* B200_ARCH_* */
    int32_t dim;            /* embedding_length */
    int32_t hidden_dim;     /* feed_forward_length */
    int32_t n_layers;       /* block_count */
    int32_t n_heads;        /* attention.head_count */
    int32_t n_kv_heads;     /* attention.head_count_kv */
    int32_t head_size;      /* dim/n_heads (Llama) or attention.key_length (Qwen3) */
    int32_t vocab_size;
    int32_t context_length; /* KV-cache positions to allocate (Options.maxTokens) */
    float rms_norm_eps;
    float rope_theta;
    int32_t fp16_lanes;     /* FP16 weights only: lane count of the CPU path's vector species the
                               results are pinned to (FP16FloatTensor.java:62-110, FloatTensor.java:21);
                               8, 16 or 0 (scalar).  Ignored for Q8_0. */
    int32_t tp_rank;        /* tensor-parallel rank of this process, 0 when tp_size == 1 */
    int32_t tp_size;        /* 1, 2, 4 or 8 */
} b200_config;

/* One named GGUF tensor: raw host bytes exactly as mapped from the file
 * (GGUF.loadTensorsStandard, GGUF.java:105-137).  dims[0] is the innermost dimension. */
typedef struct b200_tensor {
    const char *name; /* GGUF name, e.g. "blk.0.attn_q.weight" (LlamaModelLoader.java:78-99) */
    const void *data;
    int32_t ggml_type;
    int32_t n_dims;
    int64_t dims[4];
} b200_tensor;

typedef struct b200_plan b200_plan;

/* TornadoVMMasterPlan.initializeTornadoVMPlan(state, model) (TornadoVMMasterPlan.java:55-70)
 * + forceCopyInReadOnlyData (TornadoVMMasterPlanSingleToken.java:100-117): copies/repacks every
 * tensor to `device`, allocates KV cache and activations, captures the decode CUDA graph.
 * The host pointers are not retained.  prefill_batch_size mirrors -Dllama.prefillBatchSize
 * (TornadoVMMasterPlan.java:41); 0/1 = no batched-prefill buffers.
 * On failure *out is NULL and err (if non-NULL) receives the message. */
int b200_plan_create(const b200_config *cfg, const b200_tensor *tensors, int32_t n_tensors,
                     int32_t prefill_batch_size, int32_t device, b200_plan **out, char *err, size_t err_len);

/* TornadoVMMasterPlan.tornadoVMForwardDecode(position) with the embedding gather moved
 * device-side (replaces InferenceCore.forwardTornadoVM, InferenceCore.java:956-980, which copies
 * the embedding row H2D every token).  Runs one single-token forward at `position`.
 * logits (vocab_size floats, host) may be NULL: then only 4 bytes cross PCIe.
 * argmax (host) may be NULL; otherwise receives FloatTensor.argmax semantics
 * (first strict maximum, FloatTensor.java:138-151), computed on the device. */
int b200_forward_decode(b200_plan *plan, int32_t token, int32_t position, float *logits, int32_t *argmax);

/* b200_forward_decode + Sampler.sampleToken on the DEVICE (inference/sampler/Sampler.java:74-122, CategoricalSampler.java:28-40,
 * ToppSampler.java:62-156): the reference copies the whole logits row to the host whenever temperature > 0; here 4 bytes go in
 * (the uniform number the host-side Java RNG produced for this token, in [0,1)) and 4 bytes come out.  temperature == 0 is
 * FloatTensor.argmax; otherwise logits/temperature, softmax, then categorical sampling (topp <= 0 or >= 1) or top-p.  Every
 * float is evaluated in the reference's order (csrc/sampler.cuh), so the same uniform number yields the same token id.
 * info (nullable, 4 ints): {top-p candidates after the cutoff, tokens kept, items / fallbacks of the exact softmax sum}.
 * Single-GPU plans only (B200_ERR_UNSUPPORTED under tensor parallelism). */
int b200_forward_decode_sample(b200_plan *plan, int32_t token, int32_t position, float temperature, float topp, float uniform01,
                               int32_t *token_out, int32_t *info);

/* TornadoVMMasterPlanPrefillDecode.tornadoVMForwardPrefill(position)
 * (TornadoVMMasterPlanPrefillDecode.java:116): single-token forward that only fills the KV
 * cache -- final norm, lm_head and argmax are skipped. */
int b200_forward_prefill(b200_plan *plan, int32_t token, int32_t position);

/* TornadoVMMasterPlanBatchPrefillDecode.tornadoVMForwardBatchPrefill()
 * (TornadoVMMasterPlanBatchPrefillDecode.java:107-123) with explicit arguments instead of
 * state.embeddingXBatch/batchStartPosHolder: tokens[b] is processed at start_pos+b,
 * n <= prefill_batch_size.  KV cache only, no logits (InferenceCoreBatchPrefillDecode.java:166-167). */
int b200_forward_batch_prefill(b200_plan *plan, const int32_t *tokens, int32_t n, int32_t start_pos);

/* How b200_forward_batch_prefill computes (the reference has the same two families:
 * LlamaFP16LayersBatchPrefill vs ...BatchPrefillMMA, selected by TensorCoreSupport.java):
 *   B200_PREFILL_EXACT       the single-token prefill graph per token: KV cache bit-identical to the CPU path;
 *   B200_PREFILL_TENSOR_CORE TMA + tcgen05 GEMMs over the whole chunk, FP16 operands / FP32 accumulation:
 *                            KV cache within FP16 tolerance of the CPU path.  Default for FP16 plans created
 *                            with prefill_batch_size > 1.  Opt-in for single-GPU Q8_0 plans: the first call
 *                            dequantises f16 twins of the weight matrices on the device (+2 bytes/weight);
 *                            there the CPU path additionally rounds activations to int8, so agreement is
 *                            percent-level, not FP16-level -- hence not the default.  Returns
 *                            B200_ERR_UNSUPPORTED with the reason in b200_last_error when unavailable. */
#define B200_PREFILL_EXACT 0
#define B200_PREFILL_TENSOR_CORE 1
int b200_set_prefill_mode(b200_plan *plan, int32_t mode);

/* Active mode, kernels launched and device milliseconds of the last tensor-core chunk (any pointer may be NULL). */
int b200_prefill_info(b200_plan *plan, int32_t *mode, int32_t *launches, float *device_ms);

/* How the single-token forwards (b200_forward_decode / _prefill / b200_decode_sequence) run.  Both replace
 * TornadoVMMasterPlanSingleToken.tornadoVMForwardDecode's N+2 TaskGraph executions
 * (TornadoVMMasterPlanSingleToken.java:68-95) and produce bit-identical results:
 *   B200_DECODE_GRAPH       one CUDA graph of ~7 kernels per layer with programmatic-dependent-launch edges (the default:
 *                           measured 3.19 ms vs 3.51 ms per token on Llama-3-8B Q8_0, profiles/r2_final_a.log);
 *   B200_DECODE_PERSISTENT  ONE persistent kernel per token (csrc/decode_persistent.cuh): one CTA per SM streams the
 *                           weights of every matrix through a shared-memory ring while epoch counters order the phases.
 *                           Available when the plan fits (Q8_0 streaming layout, head size 64/128); the environment
 *                           variable B200_DECODE=persistent selects it at creation.
 * Returns B200_ERR_UNSUPPORTED with the reason in b200_last_error when the plan cannot run the requested mode.
 * Under tensor parallelism every rank must switch at the same point of the call sequence. */
#define B200_DECODE_GRAPH 0
#define B200_DECODE_PERSISTENT 1
int b200_set_decode_mode(b200_plan *plan, int32_t mode);

/* Active decode mode, kernels per decode step, and the persistent kernel's ring depth / shared memory (0 if unsupported). */
int b200_decode_info(b200_plan *plan, int32_t *mode, int32_t *launches, int32_t *ring_stages, int32_t *smem_bytes);

/* Device-resident token loop (what LlamaBench.runTest times, LlamaBench.java:234-254, and the
 * greedy generation loop InferenceEngine.java:96-145 with the sampler on the device):
 * runs n single-token forwards at positions start_pos..start_pos+n-1 without host round trips.
 * feedback == 0: step i consumes tokens[i] (n entries).  feedback != 0: step 0 consumes
 * tokens[0], step i>0 consumes the argmax of step i-1 (greedy generation).
 * out_ids (n ints, may be NULL) receives each step's argmax.  device_ms (may be NULL)
 * receives the CUDA-event time of the n steps on the plan's stream. */
int b200_decode_sequence(b200_plan *plan, const int32_t *tokens, int32_t n, int32_t start_pos,
                         int32_t feedback, int32_t *out_ids, float *device_ms);

/* Zero the KV cache (a fresh State in the reference: Java arrays start zeroed,
 * LlamaState.java:46-47; matters because the Qwen3 loop skips a position,
 * InferenceEngine.java:175-225). */
int b200_kv_reset(b200_plan *plan);

/* Test/diagnostic read-back of a named device buffer into host memory.  Names:
 * "x","xb","q","k","v","hb","logits","key_cache","value_cache","xq","xs".  `layer` selects the
 * layer for the KV caches (ignored otherwise).  Copies min(bytes, buffer size). */
int b200_read_buffer(b200_plan *plan, const char *name, int32_t layer, void *dst, size_t bytes);

/* Measurement hook for bench.py's roofline line: launches ONE kernel family of the decode step
 * stand-alone, `reps` times per layer, cycling over all layers so every launch streams weights
 * that are not L2-resident, and returns the average duration of one launch (CUDA events on the
 * plan's stream).  which: 0 = fused gate/up+SwiGLU, 1 = down projection (+residual),
 * 2 = fused QKV, 3 = attention output projection (+residual), 4 = lm_head.  Each id launches what the
 * decode step launches for that matrix, without programmatic dependent launch (on the FP16 row
 * kernels gate/up is three launches: w1, w3 and the SwiGLU).
 * The residual stream is restored afterwards; the KV cache is not touched. */
int b200_time_kernel(b200_plan *plan, int32_t which, int32_t reps, float *avg_ms, int64_t *algorithmic_bytes);

/* ---- tensor parallelism (one process per GPU; cfg.tp_size in {2,4,8}) ----------------------------
 * Nothing like this exists in the reference (docs/GPULlama3_ROADMAP.md:21 lists multi-GPU as open).
 * Every rank holds ROWS of every matrix (its query/KV heads, its slice of the FFN and of the
 * vocabulary), so each dot product keeps the reference's summation order and the tokens stay
 * bit-identical to the single-GPU path; slices are all-gathered by the kernels themselves through
 * peer-mapped buffers.  Protocol: every rank calls b200_plan_create (with the FULL tensors; the
 * library uploads only its share), then b200_tp_handle; the 64-byte handles are exchanged by the
 * host (torch.distributed / MPI / anything), then every rank calls b200_tp_attach with the n handles
 * in rank order.  After that all ranks must issue the same forward calls with the same arguments.
 * Under TP b200_forward_decode returns the argmax only (logits must be NULL). */
int b200_tp_handle(b200_plan *plan, void *handle64);
int b200_tp_attach(b200_plan *plan, const void *handles, int32_t n);

/* Diagnostic: runs ONE decode step through a traced copy of the decode graph (same kernels, same
 * programmatic-dependent-launch edges) and returns one record per kernel launch, in launch order:
 * {kernel id, earliest CTA entry, latest dependency-wait return, latest CTA exit}, the times in
 * %globaltimer nanoseconds.  ids: 1 rmsnorm, 2 qkv, 3 rope+kv, 4 attention, 5 attn-out, 6 gate/up,
 * 7 down, 8 lm_head, 9 argmax/advance.  records holds 4*cap uint64. */
int b200_trace_decode(b200_plan *plan, int32_t token, int32_t position, uint64_t *records, int32_t cap, int32_t *n_out);

/* Diagnostic: ONE decode step through the persistent kernel with phase stamps: stamps[cta][row][k] (uint64, %globaltimer ns),
 * rows 0..n_layers-1 = layers with k = {0 layer start, 1 attn norm done, 2 QKV rows done, 3 attention gathered, 4 Wo rows done,
 * 5 x gathered, 6 ffn norm done, 7 gate/up done, 8 hidden activation gathered+staged, 9 W2 rows done, 10/11 attn norm: squares staged /
 * exact sum done, 12-15 (head CTAs) attention: QKV gathered / scores+max / softmax / output quantised}; row n_layers = lm_head
 * {0 start, 1 final norm done, 2 lm_head rows done, 3 (CTA 0) step advanced}.  cap = capacity of stamps in uint64. */
int b200_trace_persistent(b200_plan *plan, int32_t token, int32_t position, uint64_t *stamps, int64_t cap, int32_t *n_ctas, int32_t *n_rows, int32_t *n_stamps);

/* Test hook for the exact parallel evaluation of the reference's sequential float sum (csrc/seqsum2.cuh; the RMSNorm
 * accumulator of InferenceCore.java:39-48): sums n <= 8192 non-negative host floats on the device exactly as
 * `for (i) s += t[i]` would, run by `threads` = 1024 (the RMSNorm kernel's form), 512 (the persistent decode kernel's form)
 * or 256 threads; info = {items walked, fallbacks}. */
int b200_test_seqsum2(const float *terms, int32_t n, int32_t threads, float *out, int32_t *info /* nullable */);

/* Test hook for the device-side K-quant -> Q8_0 re-quantiser the upload pipeline applies to Q4_K / Q5_K / Q6_K tensors (csrc/kquant.cuh;
 * replaces ModelLoader.dequantizeToQ8_0TornadoTensor, model/loader/ModelLoader.java:173-224): host K-quant blocks in, host GGUF Q8_0
 * blocks (34 bytes per 32 elements) out, byte-identical to the reference's.  n_elems % 256 == 0. */
int b200_requant_kquant(int32_t ggml_type, const void *src, int64_t n_elems, void *dst_q8_0);

/* Batched-prefill GEMM building block (csrc/prefill_gemm.cuh; replaces the reference's mma.sync GEMMs
 * gemmMMA / gemmMMAQKV / gemmMMAGateUp, TransformerBatchPrefillKernels.java:792-1132) exposed for
 * tests and measurement: C[m][n] (f32) = A[m][k] (f16 bits) x B[n][k]^T (f16 bits) on tcgen05 tensor
 * cores, FP32 accumulation in TMEM.  Host pointers; m % 128 == n % 128 == k % 64 == 0.
 * The kernel is one the prefill launches, chosen by two_cta: 0 = single-CTA (C = A B^T, or C += A B^T with resid = 1;
 * stages 3 or 6, 0 = 3), 256 = CTA-pair C += A B^T split `resid` ways over k (needs resid >= 1), 1256 = persistent CTA-pair
 * C = A B^T (needs resid == 0); CTA-pair kernels need m % 256 == n % 256 == 0.  Any other combination returns B200_ERR_BAD_ARG.
 * iters > 0 additionally times `iters` back-to-back launches (device events) into *ms. */
int b200_gemm_f16(const uint16_t *a, const uint16_t *b, float *c, int32_t m, int32_t n, int32_t k, int32_t iters, float *ms /* nullable */,
                  int32_t stages, int32_t resid, int32_t two_cta);

/* Weight upload of b200_plan_create (the counterpart of the reference's load-time metrics, ModelLoader.java:102-106 and the
 * copy-in timing of TornadoVMMasterPlanSingleToken.java:51-54): wall seconds from the first tensor to the last repack kernel,
 * seconds the host spent copying mapped/pageable bytes into the pinned double buffer, and bytes sent over PCIe (a tensor-parallel
 * rank sends only its row ranges).  The pipeline: pinned double buffer filled by several host threads -> async H2D on a copy
 * stream -> double-buffered device staging -> repack kernel on the plan's stream. */
int b200_upload_info(b200_plan *plan, double *seconds, double *host_copy_seconds, int64_t *h2d_bytes);

/* Number of kernels one decode step launches (bench.py's gpu_launches). */
int b200_launches_per_decode(b200_plan *plan);

/* Bytes of device memory held by the plan (weights + KV + activations). */
int64_t b200_device_bytes(b200_plan *plan);

/* TornadoVMMasterPlan.freeTornadoExecutionPlan() */
void b200_plan_free(b200_plan *plan);

const char *b200_last_error(b200_plan *plan);

/* Library build id, e.g. "b200llama 0.1 sm_100a". */
const char *b200_version(void);

#ifdef __cplusplus
}
#endif
#endif /* B200LLAMA_H */
