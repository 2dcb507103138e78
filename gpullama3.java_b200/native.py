"""ctypes binding of libb200llama.so (the C ABI in include/b200llama.h).

There is deliberately NO fallback: if the CUDA library is missing or a call fails, this
module raises.  Nothing here (or anywhere in the package) touches ``oracle/``.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libb200llama.so")

B200_OK = 0
ERRORS = {-1: "BAD_ARG", -2: "UNSUPPORTED", -3: "OOM", -4: "CUDA", -5: "NCCL", -6: "STATE"}


class B200Error(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"b200llama error {ERRORS.get(code, code)}: {msg}")
        self.code = code


class UnsupportedOperation(B200Error):
    """Counterpart of the reference's UnsupportedOperationException (ForwardPlanFactory.java:84-87)."""


class Config(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("arch", "dim", "hidden_dim", "n_layers", "n_heads", "n_kv_heads", "head_size",
                                        "vocab_size", "context_length")] + \
               [("rms_norm_eps", C.c_float), ("rope_theta", C.c_float), ("fp16_lanes", C.c_int32),
                ("tp_rank", C.c_int32), ("tp_size", C.c_int32)]


class Tensor(C.Structure):
    _fields_ = [("name", C.c_char_p), ("data", C.c_void_p), ("ggml_type", C.c_int32), ("n_dims", C.c_int32),
                ("dims", C.c_int64 * 4)]


EXPORTS = ["b200_plan_create", "b200_forward_decode", "b200_forward_prefill", "b200_forward_batch_prefill", "b200_set_prefill_mode", "b200_prefill_info",
           "b200_set_decode_mode", "b200_decode_info", "b200_trace_persistent", "b200_test_seqsum2", "b200_forward_decode_sample", "b200_upload_info", "b200_requant_kquant",
           "b200_decode_sequence", "b200_time_kernel", "b200_tp_handle", "b200_tp_attach", "b200_trace_decode", "b200_gemm_f16", "b200_kv_reset", "b200_read_buffer", "b200_launches_per_decode",
           "b200_device_bytes", "b200_plan_free", "b200_last_error", "b200_version"]

_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, i32 = C.c_void_p, C.c_int32
    L.b200_plan_create.argtypes = [C.POINTER(Config), C.POINTER(Tensor), i32, i32, i32, C.POINTER(vp), C.c_char_p, C.c_size_t]
    L.b200_forward_decode.argtypes = [vp, i32, i32, vp, C.POINTER(i32)]
    L.b200_forward_prefill.argtypes = [vp, i32, i32]
    L.b200_forward_decode_sample.argtypes = [vp, i32, i32, C.c_float, C.c_float, C.c_float, C.POINTER(i32), C.POINTER(i32)]
    L.b200_forward_batch_prefill.argtypes = [vp, vp, i32, i32]
    L.b200_decode_sequence.argtypes = [vp, vp, i32, i32, i32, vp, C.POINTER(C.c_float)]
    L.b200_kv_reset.argtypes = [vp]
    L.b200_trace_decode.argtypes = [vp, i32, i32, vp, i32, C.POINTER(i32)]
    L.b200_tp_handle.argtypes = [vp, vp]
    L.b200_tp_attach.argtypes = [vp, vp, i32]
    L.b200_set_prefill_mode.argtypes = [vp, i32]
    L.b200_set_decode_mode.argtypes = [vp, i32]
    L.b200_decode_info.argtypes = [vp, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]
    L.b200_trace_persistent.argtypes = [vp, i32, i32, vp, C.c_int64, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]
    L.b200_test_seqsum2.argtypes = [vp, i32, i32, C.POINTER(C.c_float), C.POINTER(i32)]
    L.b200_prefill_info.argtypes = [vp, C.POINTER(i32), C.POINTER(i32), C.POINTER(C.c_float)]
    L.b200_gemm_f16.argtypes = [vp, vp, vp, i32, i32, i32, i32, C.POINTER(C.c_float), i32, i32, i32]
    L.b200_time_kernel.argtypes = [vp, i32, i32, C.POINTER(C.c_float), C.POINTER(C.c_int64)]
    L.b200_read_buffer.argtypes = [vp, C.c_char_p, i32, vp, C.c_size_t]
    L.b200_upload_info.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int64)]
    L.b200_launches_per_decode.argtypes = [vp]
    L.b200_device_bytes.argtypes = [vp]
    L.b200_device_bytes.restype = C.c_int64
    L.b200_plan_free.argtypes = [vp]
    L.b200_plan_free.restype = None
    L.b200_last_error.argtypes = [vp]
    L.b200_last_error.restype = C.c_char_p
    L.b200_version.restype = C.c_char_p
    _lib = L
    return L


def _raise(code: int, msg: str):
    if code == -2:
        raise UnsupportedOperation(code, msg)
    raise B200Error(code, msg)


def test_seqsum(terms, want_info: bool = False, threads: int = 1024):
    """seqsum2.cuh run by threads = 1024 (the norm kernel's form), 512 (the persistent decode kernel's form) or 256."""
    t = np.ascontiguousarray(terms, dtype=np.float32)
    out = C.c_float(0)
    info = (C.c_int32 * 2)()
    rc = lib().b200_test_seqsum2(t.ctypes.data, len(t), threads, C.byref(out), info)
    if rc != B200_OK:
        _raise(rc, "b200_test_seqsum2 failed")
    return (out.value, info[0], info[1]) if want_info else out.value


def requant_kquant(ggml_type: int, raw, n_elems: int) -> np.ndarray:
    """Device K-quant (Q4_K = 12 / Q5_K = 13 / Q6_K = 14) -> GGUF Q8_0 bytes (csrc/kquant.cuh; ModelLoader.java:173-224)."""
    raw = np.ascontiguousarray(raw, dtype=np.uint8)
    out = np.empty(n_elems // 32 * 34, dtype=np.uint8)
    lib().b200_requant_kquant.argtypes = [C.c_int32, C.c_void_p, C.c_int64, C.c_void_p]
    rc = lib().b200_requant_kquant(int(ggml_type), raw.ctypes.data, int(n_elems), out.ctypes.data)
    if rc != B200_OK:
        _raise(rc, "b200_requant_kquant failed")
    return out


def gemm_f16(a, b, iters: int = 0, stages: int = 0, resid: int = 0, two_cta: int = 0):
    """C = A @ B.T on the tcgen05 prefill GEMM (A [m,k], B [n,k] float16) -> (C float32, ms per launch or None).
    stages / resid / two_cta pick the prefill kernel as include/b200llama.h documents for b200_gemm_f16."""
    a = np.ascontiguousarray(a, dtype=np.float16)
    b = np.ascontiguousarray(b, dtype=np.float16)
    m, k = a.shape
    n, k2 = b.shape
    if k != k2:
        raise ValueError("inner dimensions differ")
    c = np.empty((m, n), dtype=np.float32)
    ms = C.c_float(0)
    rc = lib().b200_gemm_f16(a.ctypes.data, b.ctypes.data, c.ctypes.data, m, n, k, iters, C.byref(ms), stages, resid, two_cta)
    if rc != B200_OK:
        _raise(rc, "b200_gemm_f16 failed")
    return c, (ms.value if iters > 0 else None)


GGML_SIZES = {0: (4, 1), 1: (2, 1), 8: (34, 32), 12: (144, 256), 13: (176, 256), 14: (210, 256)}  # (bytes, elements) per block, GGMLType.java:5-20


class NativePlan:
    """Owns one ``b200_plan*``."""

    def __init__(self, cfg: Config, tensors: dict, prefill_batch_size: int = 0, device: int = 0):
        L = lib()
        arr = (Tensor * len(tensors))()
        self._keep = []
        for i, (name, (tt, dims, raw)) in enumerate(tensors.items()):
            raw = np.ascontiguousarray(raw)
            ts_bs = GGML_SIZES.get(int(tt))
            n_el = int(np.prod(dims))
            if ts_bs is not None and (n_el % ts_bs[1] or raw.nbytes != n_el // ts_bs[1] * ts_bs[0]):
                # the C ABI takes plain pointers: a short buffer would be read past its end on the device side of the upload
                raise B200Error(-1, f"tensor {name}: {raw.nbytes} bytes do not hold {n_el} elements of ggml type {int(tt)}")
            self._keep.append(raw)
            arr[i].name = name.encode()
            arr[i].data = raw.ctypes.data
            arr[i].ggml_type = int(tt)
            arr[i].n_dims = len(dims)
            for k, d in enumerate(dims):
                arr[i].dims[k] = int(d)
        out = C.c_void_p()
        err = C.create_string_buffer(512)
        rc = L.b200_plan_create(C.byref(cfg), arr, len(tensors), prefill_batch_size, device, C.byref(out), err, 512)
        self._keep = None  # the library never touches the host pointers again
        if rc != B200_OK:
            _raise(rc, err.value.decode())
        self._p = out
        self.cfg = cfg

    def _ck(self, rc: int):
        if rc != B200_OK:
            _raise(rc, lib().b200_last_error(self._p).decode())

    def forward_decode(self, token: int, position: int, want_logits: bool = True, want_argmax: bool = True):
        logits = np.empty(self.cfg.vocab_size, dtype=np.float32) if want_logits else None
        am = C.c_int32(-1)
        self._ck(lib().b200_forward_decode(self._p, token, position, logits.ctypes.data if want_logits else None,
                                           C.byref(am) if want_argmax else None))
        return logits, (am.value if want_argmax else None)

    def forward_decode_sample(self, token: int, position: int, temperature: float, topp: float, uniform01: float, want_info: bool = False):
        out = C.c_int32(-1)
        info = (C.c_int32 * 4)()
        self._ck(lib().b200_forward_decode_sample(self._p, token, position, temperature, topp, uniform01, C.byref(out), info))
        return (out.value, list(info)) if want_info else out.value

    def forward_prefill(self, token: int, position: int):
        self._ck(lib().b200_forward_prefill(self._p, token, position))

    def set_prefill_mode(self, mode: int):
        self._ck(lib().b200_set_prefill_mode(self._p, mode))

    def set_decode_mode(self, mode: int):
        self._ck(lib().b200_set_decode_mode(self._p, mode))

    def decode_info(self):
        """(mode, kernels per decode step, ring stages, shared-memory bytes of the persistent kernel)."""
        a, b, c, d = C.c_int32(0), C.c_int32(0), C.c_int32(0), C.c_int32(0)
        self._ck(lib().b200_decode_info(self._p, C.byref(a), C.byref(b), C.byref(c), C.byref(d)))
        return a.value, b.value, c.value, d.value

    def trace_persistent(self, token: int, position: int) -> np.ndarray:
        """uint64 %globaltimer stamps [cta][row][k] of one traced step of the persistent decode kernel."""
        cap = 200 * (self.cfg.n_layers + 1) * 32
        buf = np.zeros(cap, dtype=np.uint64)
        a, b, c = C.c_int32(0), C.c_int32(0), C.c_int32(0)
        self._ck(lib().b200_trace_persistent(self._p, token, position, buf.ctypes.data, cap, C.byref(a), C.byref(b), C.byref(c)))
        return buf[: a.value * b.value * c.value].reshape(a.value, b.value, c.value)

    def prefill_info(self):
        mode, launches, ms = C.c_int32(0), C.c_int32(0), C.c_float(0)
        self._ck(lib().b200_prefill_info(self._p, C.byref(mode), C.byref(launches), C.byref(ms)))
        return mode.value, launches.value, ms.value

    def forward_batch_prefill(self, tokens, start_pos: int):
        t = np.ascontiguousarray(tokens, dtype=np.int32)
        self._ck(lib().b200_forward_batch_prefill(self._p, t.ctypes.data, len(t), start_pos))

    def decode_sequence(self, tokens, n: int, start_pos: int, feedback: bool = False):
        t = np.ascontiguousarray(tokens, dtype=np.int32)
        out = np.empty(n, dtype=np.int32)
        ms = C.c_float(0)
        self._ck(lib().b200_decode_sequence(self._p, t.ctypes.data, n, start_pos, 1 if feedback else 0, out.ctypes.data, C.byref(ms)))
        return out, ms.value

    def time_kernel(self, which: int, reps: int = 3):
        ms, nbytes = C.c_float(0), C.c_int64(0)
        self._ck(lib().b200_time_kernel(self._p, which, reps, C.byref(ms), C.byref(nbytes)))
        return ms.value, nbytes.value

    def tp_handle(self) -> bytes:
        buf = C.create_string_buffer(64)
        self._ck(lib().b200_tp_handle(self._p, buf))
        return buf.raw

    def tp_attach(self, handles: list):
        blob = b"".join(handles)
        self._ck(lib().b200_tp_attach(self._p, blob, len(handles)))

    def trace_decode(self, token: int, position: int):
        cap = self.launches_per_decode + 8
        rec = np.zeros((cap, 4), dtype=np.uint64)
        n = C.c_int32(0)
        self._ck(lib().b200_trace_decode(self._p, token, position, rec.ctypes.data, cap, C.byref(n)))
        return rec[: n.value]

    def kv_reset(self):
        self._ck(lib().b200_kv_reset(self._p))

    def read_buffer(self, name: str, n: int, dtype=np.float32, layer: int = 0) -> np.ndarray:
        out = np.empty(n, dtype=dtype)
        self._ck(lib().b200_read_buffer(self._p, name.encode(), layer, out.ctypes.data, out.nbytes))
        return out

    def upload_info(self) -> dict:
        a, b, c = C.c_double(0), C.c_double(0), C.c_int64(0)
        self._ck(lib().b200_upload_info(self._p, C.byref(a), C.byref(b), C.byref(c)))
        return {"seconds": a.value, "host_copy_seconds": b.value, "h2d_bytes": c.value,
                "GB/s": (c.value / a.value / 1e9) if a.value > 0 else None}

    @property
    def launches_per_decode(self) -> int:
        return lib().b200_launches_per_decode(self._p)

    @property
    def device_bytes(self) -> int:
        return lib().b200_device_bytes(self._p)

    def free(self):
        if self._p:
            lib().b200_plan_free(self._p)
            self._p = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass
