"""Seeded synthetic GGUF models in the BASELINE shapes (no real checkpoints are available
offline; SURVEY.md section 8d).  Tensor names/types are exactly what the reference loaders
expect (``model/loader/LlamaModelLoader.java:78-99``, ``Qwen3ModelLoader.java:98-124``):
norm weights F32, matrices and the embedding table in the model quantisation, metadata keys
per ``LlamaModelLoader.java:47-63`` / ``Qwen3ModelLoader.java:48-74``.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from .gguf import GGMLType, write_gguf


@dataclass(frozen=True)
class Shape:
    arch: str  # "llama" | "qwen3" | "phi3"
    dim: int
    hidden: int
    n_layers: int
    n_heads: int
    n_kv_heads: int
    head_size: int
    vocab: int
    tied: bool
    rope_theta: float
    eps: float
    model_ctx: int = 8192

    @property
    def q_dim(self):
        return self.n_heads * self.head_size

    @property
    def kv_dim(self):
        return self.n_kv_heads * self.head_size

    def matmul_elements(self) -> int:
        """Weight elements streamed per decoded token (SURVEY.md 8d)."""
        per_layer = 2 * self.q_dim * self.dim + 2 * self.kv_dim * self.dim + 3 * self.hidden * self.dim
        return self.n_layers * per_layer + self.vocab * self.dim

    def matmul_elements_no_head(self) -> int:
        """Weight elements a prefill token multiplies (no lm_head: prefill skips logits)."""
        return self.matmul_elements() - self.vocab * self.dim


SHAPES = {
    # tiny parity shapes (oracle finishes in milliseconds)
    "tiny-llama": Shape("llama", 256, 512, 2, 4, 2, 64, 512, False, 500000.0, 1e-5),
    "tiny-llama-tied": Shape("llama", 256, 512, 2, 4, 2, 64, 512, True, 500000.0, 1e-5),
    "tiny-qwen3": Shape("qwen3", 256, 768, 2, 4, 2, 128, 640, True, 1000000.0, 1e-6),
    # shapes the fast decode layouts do not fit: a classifier of 510 rows (not a multiple of 4) keeps a Q8_0 plan off the tile
    # stream; dim 384 (not a multiple of 256) keeps an FP16 plan off the rings and its prefill off the CTA-pair GEMMs
    "tiny-llama-odd-vocab": Shape("llama", 256, 512, 2, 4, 2, 64, 510, False, 500000.0, 1e-5),
    "tiny-llama-384": Shape("llama", 384, 1024, 2, 6, 3, 64, 512, False, 500000.0, 1e-5),
    # Phi-3 (forwardJavaPhi3: fused attn_qkv / gate-up tensors, NeoX-pair RoPE): mini-like (multi-head, head size 96) and medium-like (GQA, 128)
    "tiny-phi3": Shape("phi3", 384, 768, 2, 4, 4, 96, 512, False, 10000.0, 1e-5, 4096),
    "tiny-phi3-gqa": Shape("phi3", 512, 1024, 2, 4, 2, 128, 512, False, 10000.0, 1e-5, 4096),
    "mid-phi3-mini": Shape("phi3", 3072, 8192, 2, 32, 32, 96, 8192, False, 10000.0, 1e-5, 4096),  # Phi-3-mini-4k layer geometry
    # mid shape: exercises column tails (dim not a multiple of 512) and several row tiles
    "small-llama": Shape("llama", 1536, 4096, 3, 12, 4, 128, 4096, False, 500000.0, 1e-5),
    # the real Llama-3-8B layer geometry (7 column segments in the down projection, 4 KB rows) with 2 layers / small vocab
    "mid-llama": Shape("llama", 4096, 14336, 2, 32, 8, 128, 8192, False, 500000.0, 1e-5),
    # 2-layer cuts of the other BASELINE geometries (parity tests at the real row/segment shapes, small vocabulary)
    "mid-qwen3-4b": Shape("qwen3", 2560, 9728, 2, 32, 8, 128, 8192, True, 1000000.0, 1e-6, 40960),
    "mid-llama-1b": Shape("llama", 2048, 8192, 2, 32, 8, 64, 8192, True, 500000.0, 1e-5, 131072),
    "mid-llama-70b": Shape("llama", 8192, 28672, 2, 64, 8, 128, 8192, False, 500000.0, 1e-5),
    # BASELINE.json shapes
    "llama-3.2-1b": Shape("llama", 2048, 8192, 16, 32, 8, 64, 128256, True, 500000.0, 1e-5, 131072),
    "llama-3-8b": Shape("llama", 4096, 14336, 32, 32, 8, 128, 128256, False, 500000.0, 1e-5),
    "qwen3-4b": Shape("qwen3", 2560, 9728, 36, 32, 8, 128, 151936, True, 1000000.0, 1e-6, 40960),
    "llama-3-70b": Shape("llama", 8192, 28672, 80, 64, 8, 128, 128256, False, 500000.0, 1e-5),
}


def quantize_q8_0(x: np.ndarray) -> np.ndarray:
    """ggml reference Q8_0 quantiser (amax/127, roundf = half away from zero, f16 scale).
    Returns raw block bytes, 34 per 32 elements."""
    x = np.ascontiguousarray(x, dtype=np.float32).reshape(-1, 32)
    amax = np.abs(x).max(axis=1)
    d = (amax / np.float32(127.0)).astype(np.float32)
    with np.errstate(divide="ignore"):
        inv = np.where(d != 0, np.float32(1.0) / d, np.float32(0.0)).astype(np.float32)
    s = x * inv[:, None]
    q = np.trunc(s + np.copysign(np.float32(0.5), s)).astype(np.int8)
    out = np.empty((x.shape[0], 34), dtype=np.uint8)
    out[:, 0:2] = d.astype(np.float16).view(np.uint8).reshape(-1, 2)
    out[:, 2:] = q.view(np.uint8)
    return out.reshape(-1)


def encode(x: np.ndarray, ggml_type: int) -> np.ndarray:
    if ggml_type == GGMLType.F32:
        return np.ascontiguousarray(x, dtype="<f4").view(np.uint8).reshape(-1)
    if ggml_type == GGMLType.F16:
        return np.ascontiguousarray(x, dtype=np.float32).astype("<f2").view(np.uint8).reshape(-1)
    if ggml_type == GGMLType.Q8_0:
        return quantize_q8_0(x)
    raise ValueError(ggml_type)


# ---- synthetic byte-level BPE vocabulary (no real tokenizer files offline) --------------------------------------
_CORPUS = ("the quick brown fox jumps over the lazy dog. she sells sea shells by the sea shore; it's what they've done, "
           "isn't it? numbers 12345 and 2024-09-24, prices $3.50 or 100%. GPU kernels stream weights: decode, prefill, "
           "attention! Grüße aus München, naïve café, 東京 こんにちは, emoji 🙂🚀. user system assistant\n\ttabs and  double  spaces ")

LLAMA_SPECIALS = ["<|begin_of_text|>", "<|end_of_text|>", "<|reserved_special_token_0|>", "<|reserved_special_token_1|>", "<|finetune_right_pad_id|>",
                  "<|reserved_special_token_2|>", "<|start_header_id|>", "<|end_header_id|>", "<|eom_id|>", "<|eot_id|>", "<|python_tag|>"]
QWEN3_SPECIALS = ["<|endoftext|>", "<|im_start|>", "<|im_end|>", "<|object_ref_start|>", "<|object_ref_end|>", "<|box_start|>", "<|box_end|>",
                  "<tool_call>", "</tool_call>", "<think>", "</think>"]


def gpt2_byte_symbols() -> list[str]:
    """The 256 single-symbol tokens, indexed by byte value (the GPT-2 bytes_to_unicode table, LlamaTokenizer.java:98-116)."""
    keep = set(range(ord("!"), ord("~") + 1)) | set(range(0xA1, 0xAD)) | set(range(0xAE, 0x100))
    out, n = [], 0
    for b in range(256):
        if b in keep:
            out.append(chr(b))
        else:
            out.append(chr(256 + n))
            n += 1
    return out


def build_vocab(vocab_size: int, arch: str = "llama", seed: int = 1234):
    """(tokens, merge_lines, token_types, base_tokens): 256 byte symbols, BPE merges trained on a small fixed corpus
    (ids in merge order, so the vocabulary is a consistent BPE vocabulary), padding tokens, then the special tokens."""
    specials = QWEN3_SPECIALS if arch == "qwen3" else LLAMA_SPECIALS
    n_merges = vocab_size - 256 - len(specials)
    if n_merges < 0:
        raise ValueError("vocabulary too small for the byte symbols and the special tokens")
    sym = gpt2_byte_symbols()
    rng = np.random.default_rng(seed)
    words_src = _CORPUS.split(" ")
    text = " ".join(words_src[i] for i in rng.integers(0, len(words_src), 4000))
    words: dict[tuple, int] = {}
    for w in text.split(" "):
        key = tuple(sym[b] for b in (" " + w).encode("utf-8"))
        words[key] = words.get(key, 0) + 1
    tokens, merges = list(sym), []
    have = set(tokens)
    while len(merges) < n_merges:
        counts: dict[tuple, int] = {}
        for w, c in words.items():
            for a, b in zip(w, w[1:]):
                counts[(a, b)] = counts.get((a, b), 0) + c
        cand = [(c, p) for p, c in counts.items() if p[0] + p[1] not in have]
        if not cand:
            break
        _, (a, b) = max(cand, key=lambda t: (t[0], t[1]))
        merges.append(f"{a} {b}")
        tokens.append(a + b)
        have.add(a + b)
        new_words = {}
        for w, c in words.items():
            out, i = [], 0
            while i < len(w):
                if i + 1 < len(w) and w[i] == a and w[i + 1] == b:
                    out.append(a + b)
                    i += 2
                else:
                    out.append(w[i])
                    i += 1
            new_words[tuple(out)] = new_words.get(tuple(out), 0) + c
        words = new_words
    pad = 0
    while len(tokens) < vocab_size - len(specials):  # corpus exhausted: unused filler tokens (type 5 = unused)
        tokens.append(f"[PAD{pad}]")
        pad += 1
    base = len(tokens)
    tokens += specials
    types = [1] * base + [3] * len(specials)  # 1 normal, 3 control
    for i in range(base - pad, base):
        types[i] = 5
    if arch == "qwen3":
        for t in ("<think>", "</think>", "<tool_call>", "</tool_call>"):
            types[tokens.index(t)] = 4  # user defined: displayed (Qwen3Tokenizer.shouldDisplayToken)
    return tokens, merges, types, base


def metadata_for(shape: Shape, quant: int, name: str) -> dict:
    a = shape.arch
    md = {
        "general.architecture": a,
        "general.name": name,  # ModelLoader.detectModelType keys on this substring (ModelLoader.java:57-80)
        "general.file_type": 7 if quant == GGMLType.Q8_0 else 1,  # AbstractModelLoader.java:40-50
        f"{a}.embedding_length": shape.dim,
        f"{a}.feed_forward_length": shape.hidden,
        f"{a}.block_count": shape.n_layers,
        f"{a}.attention.head_count": shape.n_heads,
        f"{a}.attention.head_count_kv": shape.n_kv_heads,
        f"{a}.context_length": shape.model_ctx,
        f"{a}.attention.layer_norm_rms_epsilon": float(shape.eps),
        f"{a}.rope.freq_base": float(shape.rope_theta),
        f"{a}.vocab_size": shape.vocab,
    }
    if a == "qwen3":
        md["qwen3.attention.key_length"] = shape.head_size
        md["qwen3.attention.value_length"] = shape.head_size
    if shape.vocab <= 4096:  # tokenizer section (GGUF keys the loaders read: tokenizer.ggml.tokens / merges / token_type)
        tokens, merges, types, base = build_vocab(shape.vocab, a)
        md["tokenizer.ggml.model"] = "gpt2"
        md["tokenizer.ggml.tokens"] = tokens
        md["tokenizer.ggml.merges"] = merges
        md["tokenizer.ggml.token_type"] = types
        md["b200.synthetic.base_tokens"] = base  # the reference hard-codes 128000 for Llama-3 (LlamaTokenizer.java:45)
    return md


def tensor_plan(shape: Shape, quant: int):
    """[(name, ggml_type, dims(ne0 innermost), kind)] in file order."""
    t = [("token_embd.weight", quant, (shape.dim, shape.vocab), "w")]
    for i in range(shape.n_layers):
        p = f"blk.{i}."
        if shape.arch == "phi3":  # Phi3ModelLoader.java:107-113: fused [q; k; v] and [gate; up] tensors
            t += [
                (p + "attn_norm.weight", GGMLType.F32, (shape.dim,), "n"),
                (p + "attn_qkv.weight", quant, (shape.dim, shape.q_dim + 2 * shape.kv_dim), "w"),
                (p + "attn_output.weight", quant, (shape.q_dim, shape.dim), "w"),
                (p + "ffn_norm.weight", GGMLType.F32, (shape.dim,), "n"),
                (p + "ffn_down.weight", quant, (shape.hidden, shape.dim), "w"),
                (p + "ffn_up.weight", quant, (shape.dim, 2 * shape.hidden), "w"),
            ]
            continue
        t += [
            (p + "attn_norm.weight", GGMLType.F32, (shape.dim,), "n"),
            (p + "attn_q.weight", quant, (shape.dim, shape.q_dim), "w"),
            (p + "attn_k.weight", quant, (shape.dim, shape.kv_dim), "w"),
            (p + "attn_v.weight", quant, (shape.dim, shape.kv_dim), "w"),
            (p + "attn_output.weight", quant, (shape.q_dim, shape.dim), "w"),
        ]
        if shape.arch == "qwen3":
            t += [(p + "attn_q_norm.weight", GGMLType.F32, (shape.head_size,), "n"),
                  (p + "attn_k_norm.weight", GGMLType.F32, (shape.head_size,), "n")]
        t += [
            (p + "ffn_norm.weight", GGMLType.F32, (shape.dim,), "n"),
            (p + "ffn_gate.weight", quant, (shape.dim, shape.hidden), "w"),
            (p + "ffn_down.weight", quant, (shape.hidden, shape.dim), "w"),
            (p + "ffn_up.weight", quant, (shape.dim, shape.hidden), "w"),
        ]
    t.append(("output_norm.weight", GGMLType.F32, (shape.dim,), "n"))
    if not shape.tied:
        t.append(("output.weight", quant, (shape.dim, shape.vocab), "w"))
    return t


def build_tensors(shape: Shape, quant: int, seed: int = 1234, w_std: float = 0.02):
    """Seeded tensors: matrices N(0, w_std) (scaled so activations stay O(1) through the
    stack), norm weights 1 + N(0, 0.02).  Returns [(name, type, dims, raw uint8)]."""
    rng = np.random.Generator(np.random.PCG64(seed))
    out = []
    for name, tt, dims, kind in tensor_plan(shape, quant):
        n = int(np.prod(dims))
        if kind == "n":
            x = (1.0 + 0.02 * rng.standard_normal(n, dtype=np.float32)).astype(np.float32)
        else:
            # fan-in scaled so that W.x of a unit-RMS vector is O(1): keeps logits in a sane range
            std = w_std if w_std > 0 else 1.0 / np.sqrt(dims[0])
            x = rng.standard_normal(n, dtype=np.float32) * np.float32(std)
        out.append((name, tt, dims, encode(x, tt)))
    return out


def random_kquant(ggml_type: int, n_elems: int, rng, zero_blocks: int = 0) -> np.ndarray:
    """Random but well-formed K-quant super-blocks (Q4_K / Q5_K / Q6_K): uniform random quants, sub-block scales and mins, and FP16 block
    scales sized so the dequantised weights stay O(1/sqrt(fan-in))-ish.  There is no K-quant QUANTISER here (the hot path only ever reads
    these formats); the test models need valid bytes, not a faithful compression of given floats.  `zero_blocks` leading super-blocks get
    d = dmin = 0 (an all-zero Q8_0 block: scale 0, the re-quantiser's division guard)."""
    ts, bs = GGMLType.SIZES[ggml_type]
    assert ggml_type in GGMLType.K_QUANTS and n_elems % bs == 0
    nb = n_elems // bs
    raw = rng.integers(0, 256, size=(nb, ts), dtype=np.uint8)
    if ggml_type == GGMLType.Q6_K:
        d = rng.uniform(2e-5, 6e-5, nb).astype(np.float16)   # x int8 scale (<= 127) x 6-bit quant (<= 32)
        d[:zero_blocks] = 0
        raw[:, 208:210] = d.view(np.uint8).reshape(nb, 2)
    else:
        d = rng.uniform(1e-4, 4e-4, nb).astype(np.float16)   # x 6-bit scale (<= 63) x 4/5-bit quant (<= 15 / 31)
        dmin = rng.uniform(1e-4, 4e-4, nb).astype(np.float16) * np.float16(4 if ggml_type == GGMLType.Q4_K else 8)
        d[:zero_blocks] = 0
        dmin[:zero_blocks] = 0
        raw[:, 0:2] = d.view(np.uint8).reshape(nb, 2)
        raw[:, 2:4] = dmin.view(np.uint8).reshape(nb, 2)
    return raw.reshape(-1)


def build_tensors_kquant(shape: Shape, seed: int = 1234, mix: str = "Q4_K_M") -> dict:
    """{name: (ggml_type, dims, raw)} of a K-quant file in the layout llama.cpp's mixes use: "Q4_K_M" = Q4_K matrices with Q6_K for
    attn_v / ffn_down / the classifier and a Q5_K attention output (to touch all three formats), "Q6_K" / "Q5_K" / "Q4_K" = one format
    throughout.  Norms are F32 as always."""
    rng = np.random.Generator(np.random.PCG64(seed))
    pure = {"Q4_K": GGMLType.Q4_K, "Q5_K": GGMLType.Q5_K, "Q6_K": GGMLType.Q6_K}.get(mix)

    def pick(name):
        if pure is not None:
            return pure
        if "attn_v" in name or "ffn_down" in name or name in ("output.weight", "token_embd.weight"):
            return GGMLType.Q6_K
        return GGMLType.Q5_K if "attn_output" in name else GGMLType.Q4_K
    out = {}
    for name, _, dims, kind in tensor_plan(shape, GGMLType.Q8_0):
        n = int(np.prod(dims))
        if kind == "n":
            out[name] = (GGMLType.F32, dims, (1.0 + 0.02 * rng.standard_normal(n, dtype=np.float32)).astype(np.float32).view(np.uint8))
        else:
            tt = pick(name)
            out[name] = (tt, dims, random_kquant(tt, n, rng, zero_blocks=1 if "attn_q" in name else 0))
    return out


def write_model(path: str, shape_name: str, quant: int, seed: int = 1234, w_std: float = 0.0,
                display_name: str | None = None):
    shape = SHAPES[shape_name]
    name = display_name or {"llama": "Llama synthetic ", "qwen3": "Qwen3 synthetic ", "phi3": "Phi3 synthetic "}[shape.arch] + shape_name
    write_gguf(path, metadata_for(shape, quant, name), build_tensors(shape, quant, seed, w_std))
    return shape


def tp_row_ranges(shape: Shape, tp_rank: int, tp_size: int) -> dict:
    """Row range [r0, r1) of every sharded matrix that tensor-parallel rank `tp_rank` uploads (mirrors plan.tp_shard_plan /
    csrc/plan.cu); tensors not listed (embedding table, norms) are needed whole."""
    r, n = tp_rank, tp_size
    qd_l, kvd_l = shape.q_dim // n, shape.kv_dim // n
    hid_l, dim_l, voc_l = shape.hidden // n, shape.dim // n, shape.vocab // n
    out = {}
    for i in range(shape.n_layers):
        p = f"blk.{i}."
        out[p + "attn_q.weight"] = (r * qd_l, (r + 1) * qd_l)
        out[p + "attn_k.weight"] = (r * kvd_l, (r + 1) * kvd_l)
        out[p + "attn_v.weight"] = (r * kvd_l, (r + 1) * kvd_l)
        out[p + "attn_output.weight"] = (r * dim_l, (r + 1) * dim_l)
        out[p + "ffn_gate.weight"] = (r * hid_l, (r + 1) * hid_l)
        out[p + "ffn_up.weight"] = (r * hid_l, (r + 1) * hid_l)
        out[p + "ffn_down.weight"] = (r * dim_l, (r + 1) * dim_l)
    if not shape.tied:
        out["output.weight"] = (r * voc_l, (r + 1) * voc_l)
    return out


def build_tensors_fast(shape: Shape, quant: int, seed: int = 1234, device: str | None = None, tp_rank: int = 0, tp_size: int = 1):
    """Same tensor set as build_tensors, generated with torch (on the GPU when there is one) so an
    8B/70B-shaped model takes seconds, not minutes.  Data plumbing only -- not on the hot path.
    Returns {name: (ggml_type, dims, uint8 ndarray in GGUF layout)} (host memory).

    tp_size > 1: every value is generated (same seeded stream, so the model is identical for every world size) but only the rows
    this rank uploads are copied to the host; the arrays keep their full size (untouched pages are never committed), because the
    C ABI takes whole-tensor descriptors and reads only the rank's row range.  A 70B-shaped model then costs each of 8 ranks
    ~10 GB of host memory instead of 74 GB."""
    import torch

    dev = torch.device(device or ("cuda" if torch.cuda.is_available() else "cpu"))
    gen = torch.Generator(device=dev)
    gen.manual_seed(seed)
    out = {}
    chunk = 1 << 26
    ranges = tp_row_ranges(shape, tp_rank, tp_size) if tp_size > 1 else {}
    for name, tt, dims, kind in tensor_plan(shape, quant):
        n = int(np.prod(dims))
        if kind == "n":
            x = 1.0 + 0.02 * torch.randn(n, device=dev, generator=gen)
            out[name] = (tt, dims, x.float().cpu().numpy().view(np.uint8).reshape(-1))
            continue
        std = 1.0 / float(np.sqrt(dims[0]))
        nbytes = GGMLType.byte_size_for(tt, n)
        host = np.empty(nbytes, dtype=np.uint8)
        cols = int(dims[0])
        row_bytes = GGMLType.byte_size_for(tt, cols)
        keep = ranges.get(name)  # None: the whole tensor
        ho = 0
        for o in range(0, n, chunk):
            m = min(chunk, n - o)
            x = torch.randn(m, device=dev, generator=gen) * std
            cb = GGMLType.byte_size_for(tt, m)
            lo, hi = ho, ho + cb  # byte range of this chunk in the tensor
            if keep is not None:
                lo, hi = max(lo, keep[0] * row_bytes), min(hi, keep[1] * row_bytes)
            if lo < hi:
                if tt == GGMLType.F16:
                    b = x.half().view(torch.uint8)
                elif tt == GGMLType.Q8_0:
                    xb = x.view(-1, 32)
                    d = xb.abs().amax(dim=1) / 127.0
                    inv = torch.where(d != 0, 1.0 / d, torch.zeros_like(d))
                    sc = xb * inv[:, None]
                    q = torch.trunc(sc + torch.copysign(torch.full_like(sc, 0.5), sc)).to(torch.int8)
                    blk = torch.empty((xb.shape[0], 34), dtype=torch.uint8, device=dev)
                    blk[:, 0:2] = d.half().view(torch.uint8).view(-1, 2)
                    blk[:, 2:] = q.view(torch.uint8)
                    b = blk.view(-1)
                else:
                    b = x.float().view(torch.uint8)
                host[lo:hi] = b[lo - ho:hi - ho].cpu().numpy().reshape(-1)
            ho += cb
        assert ho == nbytes
        out[name] = (tt, dims, host)
    return out
