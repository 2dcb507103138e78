"""GPU tests of the tensor-core batched prefill (csrc/prefill.cuh, csrc/prefill_gemm.cuh) through the C ABI.

Tolerances (this is the one floating-point path that is NOT bit-exact, by design -- activations are rounded to
FP16 before each GEMM, as in the reference's MMA prefill, TransformerBatchPrefillKernels.java:61,792-915):
  * GEMM building block vs an fp32 matmul of the same fp16 operands: |err| <= 2^-14 * K^(1/2) * max|ref|-ish;
    asserted as max|err| <= 1e-4 * max|ref| (measured 8e-6 .. 2e-5; only the fp32 summation order differs);
  * KV cache after prefill and the logits of the following decode step vs the CPU oracle:
    max|err| <= 2^-8 * max|ref| (SURVEY.md 8d "FP16-scale tolerance"; measured 2e-4 .. 1.2e-3)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

FP16_TOL = 2.0 ** -8
Q8_NOISE_TOL = 0.03  # Q8_0 model vs the CPU path itself: the CPU path's own int8 activation rounding (measured 0.5-2.5 %), reported, not the parity bar


@pytest.mark.parametrize("m,n,k", [(128, 128, 64), (256, 384, 512), (384, 1024, 2240)])
def test_gemm_tcgen05_matches_fp32(pkg, m, n, k):
    rng = np.random.default_rng(m + n + k)
    a = (rng.standard_normal((m, k)) * 0.5).astype(np.float16)
    b = (rng.standard_normal((n, k)) * 0.5).astype(np.float16)
    ref = a.astype(np.float32) @ b.astype(np.float32).T
    for kw in ({}, {"resid": 1}, {"stages": 6}):
        c, ms = pkg.native.gemm_f16(a, b, iters=2, **kw)
        assert np.max(np.abs(c - ref)) <= 1e-4 * np.max(np.abs(ref)), kw
        assert ms > 0


def test_gemm_rejects_ragged_shapes(pkg):
    a = np.zeros((100, 64), dtype=np.float16)
    b = np.zeros((128, 64), dtype=np.float16)
    with pytest.raises(Exception):
        pkg.native.gemm_f16(a, b)


def _prefill_and_compare(pkg, orc, m, n_tok, batch, tol=FP16_TOL):
    c = m.configuration
    plan = pkg.B200MasterPlan.initialize_plan(m, prefill_batch_size=batch)
    om = orc.OracleModel(m)
    try:
        assert plan.prefill_info()[0] == plan.PREFILL_TENSOR_CORE  # default for FP16 plans created with a batch size
        toks = orc.bench_tokens(c.vocab_size, n_tok + 1)
        for off in range(0, n_tok, batch):
            plan.forward_batch_prefill(toks[off:min(off + batch, n_tok)], off)
        assert plan.prefill_info()[1] > 0
        for pos in range(n_tok):
            om.forward(int(toks[pos]), pos, want_logits=False)
        nv = n_tok * c.kv_dim
        for l in range(c.n_layers):
            nkv = c.context_length * c.kv_dim
            for name, ref in (("key_cache", om.key_cache(l)), ("value_cache", om.value_cache(l))):
                got = plan.read_buffer(name, nkv, layer=l)
                err = np.max(np.abs(got[:nv] - ref[:nv])) / np.max(np.abs(ref[:nv]))
                assert err <= tol, f"{name} layer {l}: rel err {err:.2e}"
                assert not np.any(got[nv:]), f"{name} layer {l}: rows past the prompt were written"
        lg, _ = plan.forward_decode(int(toks[n_tok]), n_tok)
        ref = om.forward(int(toks[n_tok]), n_tok)
        err = np.max(np.abs(lg - ref)) / np.max(np.abs(ref))
        assert err <= tol, f"logits after prefill: rel err {err:.2e}"
        # the exact mode of the same plan stays bit-identical to the CPU path
        plan.set_prefill_mode("exact")
        plan.kv_reset()
        for off in range(0, n_tok, batch):
            plan.forward_batch_prefill(toks[off:min(off + batch, n_tok)], off)
        k = plan.read_buffer("key_cache", c.context_length * c.kv_dim, layer=c.n_layers - 1)
        assert np.array_equal(k.view(np.uint32)[:nv], om.key_cache(c.n_layers - 1).view(np.uint32)[:nv])
    finally:
        plan.free()
        om.close()


@pytest.mark.parametrize("shape,n_tok,batch", [("tiny-llama", 50, 32), ("tiny-qwen3", 37, 16), ("tiny-llama-tied", 130, 130), ("tiny-llama", 300, 300),
                                               ("tiny-qwen3", 520, 512), ("tiny-phi3-gqa", 45, 32), ("tiny-llama-384", 150, 100)])
def test_tensor_core_prefill_within_fp16_tolerance(pkg, orc, make_model, shape, n_tok, batch):
    """Chunks that start at position > 0, a ragged last chunk, a chunk longer than one 128-row GEMM tile, chunks
    longer than 256 rows (two CTA-pair tiles per pair, ragged and full, then an 8-token tail at position 512),
    Llama (interleaved RoPE), Qwen3 (q/k norm + NeoX RoPE, q width != dim) and Phi-3 (fused qkv / gate-up source tensors, NeoX RoPE without norm).
    tiny-llama-384 runs the single-CTA GEMMs: the CTA pairs need dim to be a multiple of 256, and 384 is not."""
    m = make_model(shape, pkg.gguf.GGMLType.F16, n_tok + 8)
    _prefill_and_compare(pkg, orc, m, n_tok, batch)


def test_tensor_core_prefill_mid_llama(pkg, orc):
    """The real Llama-3-8B layer geometry (2 layers): 136 tokens in chunks of 128 (split-K residual GEMMs, an 8-token tail)."""
    sh = pkg.synth.SHAPES["mid-llama"]
    F16 = pkg.gguf.GGMLType.F16
    m = pkg.loader.model_from_tensors(sh, F16, pkg.synth.build_tensors_fast(sh, F16, seed=1234), 144)
    _prefill_and_compare(pkg, orc, m, 136, 128)


def _dequantised_f16_twin(pkg, m):
    """The model the Q8_0 tensor-core prefill actually computes with: every matrix replaced by f16(q * scale) (Q8_0FloatTensor.getFloat
    rounded once, as k_tiles_to_f16 does on the device), norms untouched, embedding kept in Q8_0 (the gather dequantises in fp32)."""
    G = pkg.gguf.GGMLType
    tensors = {}
    for name, (tt, dims, raw) in m.tensors.items():
        if tt == G.Q8_0 and name != "token_embd.weight":
            blocks = np.ascontiguousarray(raw).reshape(-1, 34)
            d = blocks[:, :2].copy().view("<f2").astype(np.float32)
            q = blocks[:, 2:].view(np.int8).astype(np.float32)
            tensors[name] = (G.F16, dims, (q * d).astype(np.float16).view(np.uint8).reshape(-1))
        else:
            tensors[name] = (tt, dims, raw)
    cfg = m.configuration
    twin = pkg.loader.Model(None, type(cfg)(**{**cfg.__dict__, "quantization": "FP16"}), m.model_type, tensors)
    return twin


@pytest.mark.parametrize("shape", ["tiny-llama", "tiny-qwen3"])
def test_tensor_core_prefill_q8_model(pkg, orc, make_model, shape):
    """Opt-in on a Q8_0 plan: f16 twins of the matrices are dequantised on the device for the GEMMs (the reference's Q8_0 MMA prefill
    feeds FP16 tiles the same way, TransformerBatchPrefillKernels.java:1563-1574).  PARITY BAR: the KV cache must agree at FP16
    tolerance (2^-8) with the CPU oracle evaluated on exactly those dequantised FP16 weights -- that is what this path computes.
    Against the CPU path of the Q8_0 model itself the difference is the CPU path's own int8 activation rounding, which the tensor-core
    path (like the reference's GPU prefill) does not apply: percent-level, bounded loosely and reported, which is why this mode is not
    the default for Q8_0 plans."""
    m = make_model(shape, pkg.gguf.GGMLType.Q8_0, 48)
    c = m.configuration
    n_tok, batch = 40, 16
    plan = pkg.B200MasterPlan.initialize_plan(m, prefill_batch_size=batch)
    om_twin = orc.OracleModel(_dequantised_f16_twin(pkg, m))
    om_q8 = orc.OracleModel(m)
    try:
        assert plan.prefill_info()[0] == plan.PREFILL_EXACT  # Q8_0 plans default to the exact path
        plan.set_prefill_mode("tensor_core")
        toks = orc.bench_tokens(c.vocab_size, n_tok + 1)
        for off in range(0, n_tok, batch):
            plan.forward_batch_prefill(toks[off:min(off + batch, n_tok)], off)
        for pos in range(n_tok):
            om_twin.forward(int(toks[pos]), pos, want_logits=False)
            om_q8.forward(int(toks[pos]), pos, want_logits=False)
        nv = n_tok * c.kv_dim
        worst_twin = worst_q8 = 0.0
        for l in range(c.n_layers):
            nkv = c.context_length * c.kv_dim
            for name in ("key_cache", "value_cache"):
                got = plan.read_buffer(name, nkv, layer=l)[:nv]
                rt = (om_twin.key_cache(l) if name == "key_cache" else om_twin.value_cache(l))[:nv]
                rq = (om_q8.key_cache(l) if name == "key_cache" else om_q8.value_cache(l))[:nv]
                worst_twin = max(worst_twin, float(np.max(np.abs(got - rt)) / np.max(np.abs(rt))))
                worst_q8 = max(worst_q8, float(np.max(np.abs(got - rq)) / np.max(np.abs(rq))))
        assert worst_twin <= FP16_TOL, f"vs the oracle on the dequantised FP16 weights: rel err {worst_twin:.2e}"
        assert worst_q8 <= Q8_NOISE_TOL, f"vs the CPU path of the Q8_0 model (its int8 activation rounding): rel err {worst_q8:.2e}"
        print(f"q8 tensor-core prefill {shape}: {worst_twin:.2e} vs dequantised-FP16 oracle, {worst_q8:.2e} vs the Q8_0 CPU path")
        # the exact mode of the same plan stays bit-identical to the CPU path of the Q8_0 model
        plan.set_prefill_mode("exact")
        plan.kv_reset()
        for off in range(0, n_tok, batch):
            plan.forward_batch_prefill(toks[off:min(off + batch, n_tok)], off)
        k = plan.read_buffer("key_cache", c.context_length * c.kv_dim, layer=c.n_layers - 1)
        assert np.array_equal(k.view(np.uint32)[:nv], om_q8.key_cache(c.n_layers - 1).view(np.uint32)[:nv])
    finally:
        plan.free()
        om_twin.close()
        om_q8.close()


def test_tensor_core_prefill_unsupported_is_loud(pkg, make_model):
    """A plan created without a prefill batch size keeps the exact path and says why the tensor-core one is unavailable."""
    m = make_model("tiny-llama", pkg.gguf.GGMLType.F16, 32)
    plan = pkg.B200MasterPlan.initialize_plan(m, prefill_batch_size=0)
    try:
        assert plan.prefill_info()[0] == plan.PREFILL_EXACT
        with pytest.raises(Exception, match="prefill batch size"):
            plan.set_prefill_mode("tensor_core")
        plan.set_prefill_mode("exact")
    finally:
        plan.free()
