"""GPU tests of the K-quant load path (csrc/kquant.cuh inside the upload pipeline, SURVEY 8(f) N4) through the C ABI.

Bar: byte-exact.  The device re-quantiser must produce the very Q8_0 blocks ModelLoader.dequantizeToQ8_0TornadoTensor builds on the host
(model/loader/ModelLoader.java:173-224, restated in oracle/oracle.c and pinned against gguf-py in tests/test_kquants.py), and a plan
created from K-quant tensors must then decode bit-identically to the oracle running on those re-quantised Q8_0 tensors."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name", ["Q4_K", "Q5_K", "Q6_K"])
def test_device_requantiser_is_byte_exact(pkg, orc, name):
    G = pkg.gguf.GGMLType
    tt = getattr(G, name)
    rng = np.random.Generator(np.random.PCG64(7 + tt))
    n = 256 * 4099  # not a multiple of the launch width
    raw = pkg.synth.random_kquant(tt, n, rng, zero_blocks=5)
    got = pkg.native.requant_kquant(tt, raw, n)
    ref = orc.kquant_to_q8_0(tt, raw, n)
    bad = np.nonzero(got != ref)[0]
    assert bad.size == 0, f"{name}: {bad.size} bytes differ, first at block {bad[0] // 34} byte {bad[0] % 34}"
    # arbitrary bit patterns in every field (finite FP16 scales)
    ts = G.SIZES[tt][0]
    wild = rng.integers(0, 256, size=(2048, ts), dtype=np.uint8)
    for col in ((0, 2) if tt != G.Q6_K else (208,)):
        hi = wild[:, col + 1]
        wild[:, col + 1] = np.where((hi & 0x7C) == 0x7C, hi & 0xBF, hi)
    got = pkg.native.requant_kquant(tt, wild.reshape(-1), 2048 * 256)
    assert np.array_equal(got, orc.kquant_to_q8_0(tt, wild.reshape(-1), 2048 * 256)), name


def _requantised_twin(pkg, orc, m):
    """The Q8_0 model the reference's accelerator path would hold after loading this K-quant model."""
    G = pkg.gguf.GGMLType
    tensors = {}
    for name, (tt, dims, raw) in m.tensors.items():
        if tt in G.K_QUANTS:
            tensors[name] = (G.Q8_0, dims, orc.kquant_to_q8_0(tt, np.asarray(raw), int(np.prod(dims))))
        else:
            tensors[name] = (tt, dims, raw)
    return pkg.loader.Model(None, m.configuration, m.model_type, tensors)


def _decode_matches(pkg, orc, m, n_tok, mode=None, rows=False):
    c = m.configuration
    plan = pkg.B200MasterPlan.initialize_plan(m)
    om = orc.OracleModel(_requantised_twin(pkg, orc, m))
    try:
        if rows:  # the Q8_0 row kernels: the plan has no tile-major stream, so the persistent kernel is unavailable
            with pytest.raises(pkg.native.UnsupportedOperation, match="streaming layout"):
                plan.set_decode_mode("persistent")
        if mode:
            plan.set_decode_mode(mode)
        toks = orc.bench_tokens(c.vocab_size, n_tok)
        for pos in range(n_tok):
            lg, am = plan.forward_decode(int(toks[pos]), pos)
            ref = om.forward(int(toks[pos]), pos)
            assert np.array_equal(lg.view(np.uint32), ref.view(np.uint32)), f"logits differ at position {pos}"
            assert am == orc.argmax(ref)
        nkv = c.context_length * c.kv_dim
        k = plan.read_buffer("key_cache", nkv, layer=c.n_layers - 1)
        assert np.array_equal(k.view(np.uint32), om.key_cache(c.n_layers - 1).view(np.uint32))
    finally:
        plan.free()
        om.close()


@pytest.mark.parametrize("shape,mix", [("tiny-llama", "Q4_K_M"), ("tiny-llama-tied", "Q6_K"), ("tiny-qwen3", "Q5_K"), ("tiny-qwen3", "Q4_K_M")])
def test_kquant_model_decodes_like_its_q8_0_twin(pkg, orc, shape, mix):
    """Mixed-format files (Q4_K matrices, Q6_K attn_v / ffn_down / classifier / embedding, Q5_K attention output), single-format files,
    a tied classifier (the K-quant embedding table doubles as lm_head), Llama and Qwen3."""
    sh = pkg.synth.SHAPES[shape]
    m = pkg.loader.model_from_tensors(sh, pkg.gguf.GGMLType.Q8_0, pkg.synth.build_tensors_kquant(sh, seed=11, mix=mix), 24)
    _decode_matches(pkg, orc, m, 10)


def test_kquant_model_other_paths(pkg, orc):
    """The persistent decode kernel and the Q8_0 row kernels (a 510-row classifier does not fit the tile stream, so every matrix
    goes through the chunked split-plane upload) see the same re-quantised weights."""
    for shape, mode, rows in (("tiny-llama", "persistent", False), ("tiny-llama-odd-vocab", None, True)):
        sh = pkg.synth.SHAPES[shape]
        tensors = pkg.synth.build_tensors_kquant(sh, seed=12)
        m = pkg.loader.model_from_tensors(sh, pkg.gguf.GGMLType.Q8_0, tensors, 24)
        _decode_matches(pkg, orc, m, 6, mode=mode, rows=rows)


def test_kquant_real_geometry(pkg, orc):
    """Llama-3-8B layer geometry (2 layers, Q4_K_M mix): 14336-wide rows = 56 super-blocks, three source formats inside one fused QKV /
    gate-up tile group, a 128 Mi-element classifier through the staging buffers."""
    sh = pkg.synth.SHAPES["mid-llama"]
    m = pkg.loader.model_from_tensors(sh, pkg.gguf.GGMLType.Q8_0, pkg.synth.build_tensors_kquant(sh, seed=13), 16)
    _decode_matches(pkg, orc, m, 4)
    info = None
    plan = pkg.B200MasterPlan.initialize_plan(m)
    try:
        info = plan.upload_info()
    finally:
        plan.free()
    q8_bytes = sum(int(np.prod(d)) // 32 * 34 for _, (t, d, _) in m.tensors.items() if t in pkg.gguf.GGMLType.K_QUANTS)
    assert 0 < info["h2d_bytes"] < 0.75 * q8_bytes  # the K-quant bytes crossed PCIe, not their Q8_0 expansion


def test_kquant_rejects_ragged_rows(pkg):
    """Rows that are not whole 256-element super-blocks cannot be K-quant tensors (GGUF forbids it too): loud error, no fallback."""
    G = pkg.gguf.GGMLType
    sh = pkg.synth.SHAPES["tiny-llama"]
    tensors = pkg.synth.build_tensors_kquant(sh, seed=14)
    tt, dims, raw = tensors["blk.0.attn_q.weight"]
    tensors["blk.0.attn_q.weight"] = (tt, dims, raw[:-144])
    m = pkg.loader.model_from_tensors(sh, G.Q8_0, tensors, 16)
    with pytest.raises(Exception):
        pkg.B200MasterPlan.initialize_plan(m)
