"""GPU parity tests: the CUDA path, called through the C ABI (ctypes -> libb200llama.so), against
the CPU oracle on the same seeded synthetic GGUF models.  Bar: logits BIT-EXACT (uint32 view
equal) and greedy token ids identical for both Q8_0 and FP16 weights -- the kernels reproduce
the CPU path's float evaluation order (DESIGN.md "Exactness"), so no tolerance is needed."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def assert_bit_equal(a, b, what):
    a, b = np.asarray(a, dtype=np.float32), np.asarray(b, dtype=np.float32)
    if not np.array_equal(bits(a), bits(b)):
        bad = np.flatnonzero(bits(a) != bits(b))
        i = bad[0]
        raise AssertionError(f"{what}: {len(bad)}/{a.size} elements differ; first at {i}: gpu={a[i]!r} oracle={b[i]!r} "
                             f"max|d|={np.abs(a - b).max():.3e}")


MODES = ["graph", "persistent"]  # the CUDA graph of ~7 kernels per layer / one persistent kernel per token


def set_mode(pkg, plan, mode):
    """Select the decode implementation; a plan that cannot run the persistent kernel (FP16 weights) skips that case."""
    try:
        plan.set_decode_mode(mode)
    except pkg.native.UnsupportedOperation as e:
        plan.free()
        pytest.skip(str(e))
    assert plan.decode_info()[0] == {"graph": 0, "persistent": 1}[mode]


def run_stream(pkg, orc, model, lanes, n, check_kv=True, prefill_first=0, mode="graph", launches=None):
    plan = pkg.B200MasterPlan.initialize_plan(model, fp16_lanes=lanes)
    set_mode(pkg, plan, mode)
    if launches is not None:  # kernels per decode step: tells the decode paths apart
        assert plan.launches_per_decode == launches, plan.launches_per_decode
    om = orc.OracleModel(model, lanes=lanes)
    c = model.configuration
    stream = orc.bench_tokens(c.vocab_size, n)
    try:
        for pos in range(n):
            tok = int(stream[pos])
            if pos < prefill_first:
                plan.forward_prefill(tok, pos)
                om.forward(tok, pos, want_logits=False)
                continue
            lg, am = plan.forward_decode(tok, pos)
            ref = om.forward(tok, pos)
            assert_bit_equal(lg, ref, f"logits pos {pos}")
            assert am == orc.argmax(ref), f"argmax pos {pos}"
        if check_kv:
            for l in range(c.n_layers):
                nkv = c.context_length * c.kv_dim
                assert_bit_equal(plan.read_buffer("key_cache", nkv, layer=l), om.key_cache(l), f"key cache layer {l}")
                assert_bit_equal(plan.read_buffer("value_cache", nkv, layer=l), om.value_cache(l), f"value cache layer {l}")
    finally:
        plan.free()
        om.close()


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("shape", ["tiny-llama", "tiny-llama-tied", "tiny-qwen3", "tiny-llama-odd-vocab"])
def test_decode_q8_bit_exact(pkg, orc, make_model, shape, mode):
    """tiny-llama-odd-vocab: its 510-row classifier does not fit the tile stream, so the plan runs the Q8_0 row kernels, and the
    persistent kernel, which reads the tile stream, is refused."""
    m = make_model(shape, pkg.gguf.GGMLType.Q8_0, 24)
    if shape == "tiny-llama-odd-vocab":
        plan = pkg.B200MasterPlan.initialize_plan(m)
        try:
            with pytest.raises(pkg.native.UnsupportedOperation, match="streaming layout"):
                plan.set_decode_mode("persistent")
        finally:
            plan.free()
        if mode == "persistent":
            return
    run_stream(pkg, orc, m, 16, 20, mode=mode)


@pytest.mark.parametrize("shape,lanes", [("tiny-llama", 16), ("tiny-llama-tied", 8), ("tiny-llama", 0), ("tiny-qwen3", 16)])
def test_decode_f16_bit_exact(pkg, orc, make_model, shape, lanes):
    m = make_model(shape, pkg.gguf.GGMLType.F16, 24)
    run_stream(pkg, orc, m, lanes, 12)


@pytest.mark.parametrize("shape,lanes", [("mid-llama-1b", 16), ("mid-llama", 16), ("mid-llama", 8), ("mid-qwen3-4b", 16)])
def test_decode_mid_geometries_f16(pkg, orc, shape, lanes):
    """FP16 plans on the per-warp bulk-copy rings (csrc/stream_matvec_f16.cuh) at the real layer geometries, bit-exact vs the oracle:
    Llama-3.2-1B (BASELINE config 1: dim 2048, hidden 8192, tied classifier), Llama-3-8B (config 3: hidden 14336 -> a 57 KB activation
    next to the rings), Qwen3-4B (dim 2560 -> 256-column segments).  A warp laps its ring many times per matvec; the 8-lane species
    puts four rows (two gate + two up) into one warp."""
    sh = pkg.synth.SHAPES[shape]
    F16 = pkg.gguf.GGMLType.F16
    m = pkg.loader.model_from_tensors(sh, F16, pkg.synth.build_tensors_fast(sh, F16, seed=7), 16)
    run_stream(pkg, orc, m, lanes, 4, check_kv=True)


@pytest.mark.parametrize("shape,quant,mode", [("tiny-phi3", "Q8_0", "graph"), ("tiny-phi3", "F16", "graph"), ("tiny-phi3-gqa", "Q8_0", "graph"),
                                              ("tiny-phi3-gqa", "Q8_0", "persistent"), ("tiny-phi3-gqa", "F16", "graph")])
def test_decode_phi3_bit_exact(pkg, orc, make_model, shape, quant, mode):
    """Phi-3 (InferenceCore.forwardJavaPhi3, InferenceCore.java:699-800): fused attn_qkv / gate-up tensors split by rows at upload,
    NeoX-pair RoPE without q/k norm.  Mini-like (multi-head, head size 96: graph only, FP16 through the round-1 kernels since dim 384
    is not a multiple of 256) and medium-like (GQA, head size 128: also the persistent kernel and the FP16 rings)."""
    m = make_model(shape, getattr(pkg.gguf.GGMLType, quant), 24)
    assert m.model_type == "PHI_3" and m.configuration.arch == 2
    run_stream(pkg, orc, m, 16, 14, mode=mode)


@pytest.mark.parametrize("quant", ["Q8_0", "F16"])
def test_decode_phi3_mini_geometry(pkg, orc, quant):
    """The Phi-3-mini layer geometry (dim 3072, hidden 8192, 32 heads of 96, fused 9216-row qkv and 16384-row gate-up), 2 layers."""
    sh = pkg.synth.SHAPES["mid-phi3-mini"]
    tt = getattr(pkg.gguf.GGMLType, quant)
    m = pkg.loader.model_from_tensors(sh, tt, pkg.synth.build_tensors_fast(sh, tt, seed=9), 16)
    run_stream(pkg, orc, m, 16, 4, check_kv=True)


def test_decode_f16_round1_kernels_still_exact(pkg, orc, make_model):
    """The round-1 launches (k_matvec_f16 + separate SwiGLU), the fallback for shapes the rings do not fit: dim 384 is not a
    multiple of the rings' 256-column segments.  They issue 9 launches per layer where the rings issue 7."""
    m = make_model("tiny-llama-384", pkg.gguf.GGMLType.F16, 24)
    run_stream(pkg, orc, m, 16, 8, launches=9 * m.configuration.n_layers + 3)


@pytest.mark.parametrize("mode", MODES)
def test_decode_small_llama_q8(pkg, orc, make_model, mode):
    """dim 1536 (not a multiple of 512: exercises the column tail), 12 heads / 4 KV heads, 3 layers."""
    m = make_model("small-llama", pkg.gguf.GGMLType.Q8_0, 40)
    run_stream(pkg, orc, m, 16, 36, check_kv=False, mode=mode)


_mid_cache = {}


def mid_model(pkg, name, ctx):
    if name not in _mid_cache:
        sh = pkg.synth.SHAPES[name]
        _mid_cache[name] = (sh, pkg.synth.build_tensors_fast(sh, pkg.gguf.GGMLType.Q8_0, seed=5))
    sh, tensors = _mid_cache[name]
    return pkg.loader.model_from_tensors(sh, pkg.gguf.GGMLType.Q8_0, tensors, ctx)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("shape", ["mid-llama", "mid-qwen3-4b", "mid-llama-1b", "mid-llama-70b"])
def test_decode_mid_geometries_q8(pkg, orc, shape, mode):
    """2-layer cuts of the BASELINE geometries, bit-exact vs the oracle: Llama-3-8B (dim 4096, hidden 14336 = 7 column segments,
    32/8 heads), Qwen3-4B (dim 2560 / hidden 9728 / q width 4096: three different segment widths, q/k norm, NeoX rope),
    Llama-3.2-1B (head 64, tied classifier), Llama-3-70B (dim 8192 / hidden 28672 / 64 heads).  The ring laps many times per matvec."""
    m = mid_model(pkg, shape, 16)
    run_stream(pkg, orc, m, 16, 5, check_kv=True, mode=mode)


@pytest.mark.parametrize("mode", MODES)
def test_prefill_graph_then_decode(pkg, orc, make_model, mode):
    """forward_prefill (no logits) fills the same KV cache as a full forward."""
    m = make_model("tiny-llama", pkg.gguf.GGMLType.Q8_0, 24)
    run_stream(pkg, orc, m, 16, 16, prefill_first=9, mode=mode)


@pytest.mark.parametrize("mode", MODES)
def test_batch_prefill_matches_oracle(pkg, orc, make_model, mode):
    m = make_model("tiny-llama", pkg.gguf.GGMLType.Q8_0, 32)
    c = m.configuration
    plan = pkg.B200MasterPlan.initialize_plan(m, prefill_batch_size=8)
    set_mode(pkg, plan, mode)
    plan.set_prefill_mode("exact")  # the token-by-token graph; the tensor-core mode is covered by test_gpu_prefill.py
    om = orc.OracleModel(m)
    stream = orc.bench_tokens(c.vocab_size, 20)
    for off in range(0, 16, 8):
        plan.forward_batch_prefill(stream[off:off + 8], off)
    for pos in range(16):
        om.forward(int(stream[pos]), pos, want_logits=False)
    for l in range(c.n_layers):
        nkv = c.context_length * c.kv_dim
        assert_bit_equal(plan.read_buffer("key_cache", nkv, layer=l), om.key_cache(l), f"key cache layer {l}")
        assert_bit_equal(plan.read_buffer("value_cache", nkv, layer=l), om.value_cache(l), f"value cache layer {l}")
    lg, am = plan.forward_decode(int(stream[16]), 16)
    assert_bit_equal(lg, om.forward(int(stream[16]), 16), "decode after batched prefill")
    plan.free()


@pytest.mark.parametrize("mode", MODES)
def test_decode_sequence_device_loop(pkg, orc, make_model, mode):
    """The device-resident loop (tokens and argmax never leave the GPU) equals step-by-step calls,
    in both teacher-forced (LlamaBench) and greedy-feedback modes."""
    m = make_model("tiny-llama", pkg.gguf.GGMLType.Q8_0, 40)
    c = m.configuration
    plan = pkg.B200MasterPlan.initialize_plan(m)
    set_mode(pkg, plan, mode)
    om = orc.OracleModel(m)
    stream = orc.bench_tokens(c.vocab_size, 24)
    ids, ms = plan.decode_sequence(stream, 24, 0, feedback=False)
    ref = [orc.argmax(om.forward(int(stream[p]), p)) for p in range(24)]
    assert list(ids) == ref and ms > 0
    plan.kv_reset()
    om.reset()
    ids, _ = plan.decode_sequence(stream[:1], 16, 0, feedback=True)
    tok, ref = int(stream[0]), []
    for p in range(16):
        tok = orc.argmax(om.forward(tok, p))
        ref.append(tok)
    assert list(ids) == ref
    plan.free()


@pytest.mark.parametrize("mode", MODES)
def test_generation_loops_match_oracle(pkg, orc, make_model, mode):
    """The reference's loop conventions end to end: Llama (BOS at pos 0 and 1) and Qwen3 (skipped
    position, which reads the zero-initialised KV row)."""
    for shape, loop in (("tiny-llama", "llama"), ("tiny-qwen3", "qwen3")):
        m = make_model(shape, pkg.gguf.GGMLType.Q8_0, 32)
        plan = pkg.B200MasterPlan.initialize_plan(m)
        set_mode(pkg, plan, mode)
        om = orc.OracleModel(m)
        prompt = [int(t) for t in orc.bench_tokens(m.configuration.vocab_size, 6)]
        fn = pkg.engine.generate_tokens_llama if loop == "llama" else pkg.engine.generate_tokens_qwen3
        got = fn(lambda t, p: plan.forward_decode(t, p, logits=False)[1], prompt[0], 0, prompt, [], 20, 32)
        ref = fn(lambda t, p: om.forward_argmax(t, p), prompt[0], 0, prompt, [], 20, 32)
        assert got == ref and len(got) > 8
        plan.free()


def test_batch_prefill_generation_loop(pkg, orc, make_model):
    m = make_model("tiny-llama", pkg.gguf.GGMLType.Q8_0, 32)
    plan = pkg.B200MasterPlan.initialize_plan(m, prefill_batch_size=4)
    plan.set_prefill_mode("exact")
    om = orc.OracleModel(m)
    prompt = [int(t) for t in orc.bench_tokens(m.configuration.vocab_size, 7)]
    got = pkg.engine.generate_tokens_llama_batch_prefill(plan, prompt[0], 0, prompt, [], 20, 32, 4)
    ref = pkg.engine.generate_tokens_llama(lambda t, p: om.forward_argmax(t, p), prompt[0], 0, prompt, [], 20, 32)
    assert got == ref
    plan.free()


def test_mistral_named_model_runs_the_llama_path(pkg, orc, tmp_path):
    """SURVEY 8(f) N4: Mistral = the Llama forward through the same kernels (Mistral.java -> InferenceCore.forwardJava)."""
    path = str(tmp_path / "mistral.gguf")
    pkg.synth.write_model(path, "tiny-llama", pkg.gguf.GGMLType.Q8_0, seed=11, display_name="Mistral-7B-Instruct synthetic")
    m = pkg.load_model(path, 24)
    assert m.model_type == "MISTRAL"
    for mode in MODES:
        run_stream(pkg, orc, m, 16, 12, mode=mode)


def test_modes_interleave(pkg, orc, make_model):
    """Both decode implementations share the KV cache and the step state: switching between them mid-stream changes nothing."""
    m = make_model("tiny-llama", pkg.gguf.GGMLType.Q8_0, 24)
    plan = pkg.B200MasterPlan.initialize_plan(m)
    om = orc.OracleModel(m)
    stream = orc.bench_tokens(m.configuration.vocab_size, 16)
    for pos in range(16):
        plan.set_decode_mode("persistent" if (pos // 3) % 2 == 0 else "graph")
        lg, am = plan.forward_decode(int(stream[pos]), pos)
        assert_bit_equal(lg, om.forward(int(stream[pos]), pos), f"logits pos {pos}")
    plan.free()


def test_long_context_score_row_in_global_memory(pkg, orc, make_model):
    """A context too long for the shared-memory score row (ADVICE r1: real checkpoints default to 131072) builds a plan and stays bit-exact."""
    m = make_model("tiny-llama", pkg.gguf.GGMLType.Q8_0, 20000)
    for mode in MODES:
        run_stream(pkg, orc, m, 16, 6, check_kv=False, mode=mode)


@pytest.mark.parametrize("shape,quant,ctx,mode", [("tiny-llama", "Q8_0", 704, "graph"), ("tiny-llama", "Q8_0", 704, "persistent"),
                                                  ("tiny-qwen3", "Q8_0", 704, "graph"), ("tiny-qwen3", "Q8_0", 704, "persistent"),
                                                  ("tiny-phi3", "Q8_0", 704, "graph"), ("tiny-llama", "F16", 704, "graph"),
                                                  ("tiny-llama", "Q8_0", 20000, "graph"), ("tiny-qwen3", "Q8_0", 20000, "persistent")])
def test_deep_context_bit_exact(pkg, orc, make_model, shape, quant, ctx, mode):
    """Depth: 700 positions.  Past 128 keys the attention kernel's score and weighted-sum loops run several software-pipelined passes
    (next pass's K / V rows in flight during the current chain), from 512 keys on the softmax sum is the exact parallel accumulator, the
    K/V rows are bulk-prefetched into L2 ahead of the dependency wait; with a 20000-token context the score row lives in global memory.
    Logits are compared on both sides of every switch-over (127|128|129 keys, 255|256|257, 511|512|513, ...) and at the end; the KV cache
    of all 700 positions must be bit-equal.  Head sizes 64 (Llama), 128 (Qwen3: q/k norm, NeoX), 96 (Phi-3)."""
    m = make_model(shape, getattr(pkg.gguf.GGMLType, quant), ctx)
    c = m.configuration
    plan = pkg.B200MasterPlan.initialize_plan(m)
    set_mode(pkg, plan, mode)
    om = orc.OracleModel(m, lanes=16)
    n = 700
    check = {0, 1, 126, 127, 128, 129, 254, 255, 256, 257, 383, 384, 510, 511, 512, 513, 639, 640, 641, 698, 699}
    toks = orc.bench_tokens(c.vocab_size, n)
    try:
        for pos in range(n):
            tok = int(toks[pos])
            if pos in check:
                lg, am = plan.forward_decode(tok, pos)
                ref = om.forward(tok, pos)
                assert_bit_equal(lg, ref, f"logits at position {pos}")
                assert am == orc.argmax(ref)
            else:
                plan.forward_prefill(tok, pos)
                om.forward(tok, pos, want_logits=False)
        nkv = n * c.kv_dim
        for l in range(c.n_layers):
            assert_bit_equal(plan.read_buffer("key_cache", c.context_length * c.kv_dim, layer=l)[:nkv], om.key_cache(l)[:nkv], f"key cache layer {l}")
            assert_bit_equal(plan.read_buffer("value_cache", c.context_length * c.kv_dim, layer=l)[:nkv], om.value_cache(l)[:nkv], f"value cache layer {l}")
    finally:
        plan.free()
        om.close()


@pytest.mark.parametrize("mode", MODES)
def test_kv_reset_and_determinism(pkg, orc, make_model, mode):
    m = make_model("tiny-qwen3", pkg.gguf.GGMLType.Q8_0, 24)
    plan = pkg.B200MasterPlan.initialize_plan(m)
    set_mode(pkg, plan, mode)
    stream = orc.bench_tokens(m.configuration.vocab_size, 10)
    a = [plan.forward_decode(int(stream[p]), p)[0] for p in range(10)]
    plan.kv_reset()
    b = [plan.forward_decode(int(stream[p]), p)[0] for p in range(10)]
    for x, y in zip(a, b):
        assert_bit_equal(x, y, "rerun after kv_reset")
    plan.free()


def test_error_conventions(pkg, make_model):
    m = make_model("tiny-llama", pkg.gguf.GGMLType.Q8_0, 16)
    plan = pkg.B200MasterPlan.initialize_plan(m)
    with pytest.raises(pkg.native.B200Error):
        plan.forward_decode(10 ** 6, 0)  # token out of range
    with pytest.raises(pkg.native.B200Error):
        plan.forward_decode(1, 16)  # position outside the KV cache
    plan.free()
    # unsupported quantisation -> UnsupportedOperation (ForwardPlanFactory.java:84-87)
    bad = dict(m.tensors)
    tt, dims, raw = bad["blk.0.attn_q.weight"]
    bad["blk.0.attn_q.weight"] = (2, dims, raw)  # Q4_0
    m.tensors = bad
    with pytest.raises(pkg.native.UnsupportedOperation):
        pkg.B200MasterPlan(m)


def _seq(t):
    return np.add.accumulate(np.asarray(t, dtype=np.float32), dtype=np.float32)[-1]


@pytest.mark.parametrize("threads", [1024, 512, 256])
def test_exact_parallel_sequential_sum(pkg, threads):
    """csrc/seqsum2.cuh (1024 = the norm kernel's form, 512 = the persistent decode kernel's form, 256 = a narrower
    one): the parallel emulation of `for (i) s += t[i]` in float32 must equal the
    literal chain bit for bit, on benign and adversarial inputs (ties, binade edges, zeros,
    huge dynamic range, sums parked next to a power of two, forced fallbacks)."""
    rng = np.random.default_rng(0)
    cases = []
    for trial in range(120):
        n = int(rng.choice([33, 64, 256, 1000, 1536, 2560, 4096, 8192]))
        kind = trial % 10
        if kind == 0: x = rng.standard_normal(n)
        elif kind == 1: x = rng.standard_normal(n) * 10.0 ** rng.integers(-6, 6)
        elif kind == 2: x = rng.standard_cauchy(n)
        elif kind == 3: x = np.full(n, rng.standard_normal())
        elif kind == 4: x = 2.0 ** rng.integers(-10, 10, n)
        elif kind == 5:
            x = rng.standard_normal(n); x[rng.integers(0, n, n // 4)] = 0
        elif kind == 6: x = rng.standard_normal(n) * np.exp(rng.standard_normal(n) * 3)
        elif kind == 7: x = np.round(rng.standard_normal(n) * 8) / 8
        elif kind == 8:
            x = np.zeros(n); x[n // 2:] = rng.standard_normal(n - n // 2)  # all-zero head -> literal path
        else:
            x = rng.standard_normal(n) * 1e-3; x[rng.integers(min(40, n - 1), n)] = 1e3  # one huge term: multi-binade jump
        cases.append((x.astype(np.float32) ** 2).astype(np.float32))
    # sums parked right below / at / above a power of two (prediction least certain)
    for n in (512, 4096):
        for eps in (-3e-7, -1e-7, 0.0, 1e-7, 3e-7):
            t = np.full(n, (1.0 + eps) / n, dtype=np.float64).astype(np.float32)
            cases.append(t)
            cases.append(np.concatenate([t, t]).astype(np.float32)[: min(2 * n, 8192)])
    # more segments than the entry list holds -> sequential fallback must still be exact
    cases.append((4.0 ** (np.arange(300) % 150 - 75)).astype(np.float32))
    cases.append(np.array([1.0] * 40 + [np.inf] + [1.0] * 40, dtype=np.float32))
    for t in cases:
        got = np.float32(pkg.native.test_seqsum(t, threads=threads))
        ref = _seq(t)
        assert got.view(np.uint32) == ref.view(np.uint32) or (np.isnan(got) and np.isnan(ref)), (len(t), got, ref)
