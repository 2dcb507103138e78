#!/usr/bin/env python
"""bench.py -- Llama-3-8B Q8_0 single-stream decode (tg) on B200, the BASELINE.json headline.

A "step" is one single-token decode forward (all layers + lm_head + on-device argmax) at a
growing KV position, on the LlamaBench synthetic token stream (`new Random(42).nextInt(vocab)`,
LlamaBench.java:188-193) over a seeded synthetic GGUF-layout model of the real Llama-3-8B shape.

  value        tok/s with tokens already resident in HBM (device loop b200_decode_sequence,
               CUDA-event time on the plan's stream, max over ranks)
  e2e          tok/s through the reference-facing call b200_forward_decode with HOST buffers:
               every step copies the token/position H2D and the argmax D2H inside the timed region
  roofline     the WHOLE decode step (default: one CUDA graph of 227 kernels per token; --decode-mode persistent: one kernel):
               achieved = algorithmic bytes per token / device time per token, peak = MEASURED_PEAKS.json
               hbm_gbs; per launch = per token / kernels per token; the stand-alone streaming matvecs (the dominant
               kernels by bytes and time, timed live with CUDA events on the plan's stream) are listed under
               roofline.other_kernels; traffic = measured DRAM bytes per launch from the committed ncu capture
  cpu_baseline the oracle (CPU restatement of the reference's onGPU=false path) on this box's
               host cores, bounded sample
  parity       in the same run: greedy ids of the first steps GPU == oracle, max|dlogit| of step 0
               (BASELINE.md section 3); a mismatch exits non-zero
`--impl reference` times only that CPU restatement (the reference itself needs a JDK + TornadoVM,
neither is installable here; see DESIGN.md).
`--dump-outputs DIR` writes what the timed device loop computed (ids.npy: the greedy id of every timed step;
logits.npy: the logits of the last timed step, single GPU only) so that two builds can be compared output
for output: the model and the token stream are seeded, so the same arguments give the same inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import __graft_entry__ as ge  # noqa: E402

WORKLOAD = "llama-3-8b"
QUANT = "q8_0"
FALLBACK_HBM_GBS = 6650.0


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    return FALLBACK_HBM_GBS, "fallback"


FALLBACK_TENSOR_TFLOPS = 2250.0  # nominal dense bf16/fp16


def tensor_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            j = json.load(f)
        return float(j["bf16_tflops"]), float(j.get("bf16_tflops_sustained", j["bf16_tflops"])), "measured (cuBLAS bf16 8192^3; fp16 shares the rate)"
    return FALLBACK_TENSOR_TFLOPS, FALLBACK_TENSOR_TFLOPS, "fallback (nominal)"


def prefill_leg(pkg, lb, local: int, n: int, reps: int):
    """BASELINE config 3: Llama-3-8B FP16, --batch-prefill-size 512, pp512 from depth 0 (LlamaBench `pp`
    semantics: forward only, no logits).  Tensor-core path: TMA + tcgen05 GEMMs, csrc/prefill*.cuh."""
    shape = pkg.synth.SHAPES[WORKLOAD]
    F16 = pkg.gguf.GGMLType.F16
    model = pkg.loader.model_from_tensors(shape, F16, pkg.synth.build_tensors_fast(shape, F16, seed=1234, device=f"cuda:{local}"), n + 8)
    plan = pkg.B200MasterPlan.initialize_plan(model, prefill_batch_size=n, device=local)
    toks = np.asarray(lb.synthetic_tokens(shape.vocab, n), dtype=np.int32)
    mode = plan.prefill_info()[0]
    dev, wall = [], []
    for r in range(3 + reps):  # 3 untimed warm-up chunks
        t0 = time.perf_counter()
        plan.forward_batch_prefill(toks, 0)  # host tokens in, synchronous: the e2e call
        t1 = time.perf_counter()
        if r >= 3:
            dev.append(plan.prefill_info()[2])
            wall.append((t1 - t0) * 1e3)
    launches = plan.prefill_info()[1]
    plan.free()
    d, w = float(np.mean(dev)), float(np.mean(wall))
    gemm = 2.0 * shape.matmul_elements_no_head() * n
    att = 4.0 * shape.q_dim * shape.n_layers * (n * (n + 1) / 2.0)
    burst, sustained, src = tensor_peak()
    tf = (gemm + att) / (d * 1e-3) / 1e12
    return {"metric": "prefill_tokens_per_s", "value": n / d * 1e3, "unit": "tok/s", "ms_per_chunk": d, "reps": reps, "dtype": "f16 operands, f32 accumulate (TMEM)",
            "e2e": {"value": n / w * 1e3, "unit": "tok/s", "h2d_bytes_per_step": 4 * n, "d2h_bytes_per_step": 0},
            "gpu_launches": launches, "mode": "tensor_core" if mode == 1 else "exact",
            "config": {"workload": f"Llama-3-8B-shaped synthetic GGUF, FP16, pp{n} in one chunk (--batch-prefill-size {n}) from depth 0, KV cache only (no logits)",
                       "l2": "inputs larger than L2 (15.0 GB of FP16 weights per chunk)"},
            "roofline": {"kernel": "whole prefill chunk (k_gemm_f16_tcgen05 = 85 % of it, profiles/)", "bound": "tensor", "achieved": tf, "peak": burst, "peak_sustained": sustained,
                         "peak_source": src, "unit": "TFLOP/s", "frac": tf / burst, "flop_per_chunk": {"gemm": gemm, "attention": att}, "traffic": None}}


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "samples": len(sm), "reasons": sorted(reasons)}


def algorithmic_bytes_per_token(shape, quant_q8: bool, ctx_avg_pos: float) -> dict:
    """SURVEY.md 8(d): matmul weights read once + F32 norm weights + FP32 KV reads."""
    elems = shape.matmul_elements()
    w = elems // 32 * 34 if quant_q8 else elems * 2
    norms = (2 * shape.n_layers + 1) * shape.dim * 4
    kv = 2 * shape.n_layers * (ctx_avg_pos + 1) * shape.kv_dim * 4
    return {"weights": w, "norms": norms, "kv": kv, "total": w + norms + kv}


def build_model(pkg, ctx: int, device: str | None, tp_rank: int = 0, tp_size: int = 1):
    shape = pkg.synth.SHAPES[WORKLOAD]
    quant = pkg.gguf.GGMLType.Q8_0 if QUANT == "q8_0" else pkg.gguf.GGMLType.F16
    t0 = time.time()
    tensors = pkg.synth.build_tensors_fast(shape, quant, seed=1234, device=device, tp_rank=tp_rank, tp_size=tp_size)
    model = pkg.loader.model_from_tensors(shape, quant, tensors, ctx)
    return shape, model, time.time() - t0


def cpu_leg(orc, model, tokens, budget_s: float, max_tokens: int):
    """Times the CPU restatement (per-row activation quantisation exactly as the reference does,
    Q8_0FloatTensor.java:100-117; rows over all host cores like Parallel.parallelFor) on the bench's own
    token stream from position 0, and keeps what the parity gate needs: step 0's logits, every step's argmax."""
    cores = orc.use_all_cores()  # torchrun exports OMP_NUM_THREADS=1: set the thread count explicitly
    om = orc.OracleModel(model, per_row_quant=True)
    lg0 = om.forward(int(tokens[0]), 0).copy()  # untimed warm-up (page-in); position 0 of the stream
    ids = [orc.argmax(lg0)]
    n, t0 = 0, time.perf_counter()
    while n < max_tokens:
        ids.append(orc.argmax(om.forward(int(tokens[1 + n]), 1 + n)))
        n += 1
        if time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    om.close()
    return n / dt, n, dt, cores, {"logits0": lg0, "ids": ids}


def parity_gate(plan, tokens, ref, want_logits: bool):
    """BASELINE.md section 3: the GPU path on the same tokens/positions the oracle just ran.  Teacher-forced (LlamaBench's
    token stream), so every step is an independent check of logits -> argmax at a growing KV depth."""
    plan.kv_reset()
    n = len(ref["ids"])
    got, dmax = [], None
    for i in range(n):
        lg, am = plan.forward_decode(int(tokens[i]), i, logits=want_logits and i == 0)
        got.append(int(am))
        if want_logits and i == 0:
            dmax = float(np.abs(lg - ref["logits0"]).max())
            bit_equal = bool(np.array_equal(lg.view(np.uint32), ref["logits0"].view(np.uint32)))
    out = {"steps": n, "ids_equal": got == [int(v) for v in ref["ids"]], "against": "oracle (CPU restatement of InferenceCore.forwardJava), same tokens and positions"}
    if dmax is not None:
        out["max_abs_dlogit"] = dmax
        out["logits_bit_equal"] = bit_equal
        out["tolerance"] = "0 (decode reproduces the CPU path's float order; FP16-scale 2^-8*max|logit| would be the north-star bound)"
    return out


def dump_outputs(d: str, ids, logits):
    """What the timed device loop hands its caller (the greedy ids) plus the last step's logits (tensor-parallel ranks
    hold only their slice of the vocabulary, so those are written only on one GPU)."""
    os.makedirs(d, exist_ok=True)
    np.save(os.path.join(d, "ids.npy"), np.asarray(ids, dtype=np.float64))
    if logits is not None:
        np.save(os.path.join(d, "logits.npy"), np.asarray(logits, dtype=np.float32))


def main():
    global WORKLOAD, QUANT
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=128)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-budget", type=float, default=20.0, help="seconds of CPU-baseline work")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--no-pp", action="store_true", help="skip the pp512 tensor-core prefill leg")
    ap.add_argument("--decode-mode", default="default", choices=["default", "persistent", "graph"],
                    help="decode implementation: one persistent kernel per token, or the round-1 CUDA graph of ~7 kernels per layer")
    ap.add_argument("--quant", default="q8_0", choices=["q8_0", "f16"], help="weight type of the synthetic model (f16: the exact lane-order FP16 matvec path, graph mode)")
    ap.add_argument("--depth", type=int, default=-1, help="LlamaBench -d: KV positions filled before the timed steps (default: the warm-up steps)")
    ap.add_argument("--workload", default=WORKLOAD, choices=["llama-3-8b", "llama-3-70b", "llama-3.2-1b", "qwen3-4b"],
                    help="shape of the synthetic model (default: the BASELINE headline, Llama-3-8B; 70B is BASELINE config 5, meant for --gpus 2/4/8)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps write DIR/ids.npy (float64, greedy id of every timed step) and, on one GPU, "
                         "DIR/logits.npy (float32, logits of the last timed step)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the timed GPU path; --impl reference times a bounded CPU sample")
    K, W = args.steps, max(args.warmup, 3)
    WORKLOAD = args.workload
    QUANT = args.quant
    pretty = {"llama-3-8b": "Llama-3-8B", "llama-3-70b": "Llama-3-70B", "llama-3.2-1b": "Llama-3.2-1B", "qwen3-4b": "Qwen3-4B"}[WORKLOAD]

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    pkg = ge.import_package()
    lb = pkg.llama_bench
    shape = pkg.synth.SHAPES[WORKLOAD]
    D = max(W, args.depth)  # LlamaBench -d: positions filled before the timed steps; the fill doubles as the warm-up
    ctx = D + K + 8  # LlamaBench: depth + tokens + 8 (LlamaBench.java:174)
    tokens = np.asarray(lb.synthetic_tokens(shape.vocab, D + K), dtype=np.int32)
    qname = "Q8_0" if QUANT == "q8_0" else "FP16"
    config = {"workload": f"{pretty}-shaped synthetic GGUF, {qname}, tg{K} single-stream decode from depth {D}",
              "weights": "seeded N(0,1/sqrt(fan_in)) quantised with the ggml Q8_0 rule; tokens java.util.Random(42)",
              "context": ctx, "l2": f"inputs larger than L2 ({(shape.matmul_elements() // 32 * 34 if QUANT == 'q8_0' else shape.matmul_elements() * 2) / 1e9:.2f} GB of weights stream per step vs 126 MB L2)"}

    if args.impl == "reference":
        if world > 1 and rank != 0:
            return 0
        orc = ge.import_oracle()
        _, model, _ = build_model(pkg, ctx, None)
        budget = max(10.0, min(120.0, 8.0 * (K + W)))  # bounded sample: the whole run ends within minutes
        tps, n, dt, cores, _ = cpu_leg(orc, model, tokens, budget, max(1, min(K, D + K - 1)))
        line = {"metric": "decode_tokens_per_s", "value": tps, "unit": "tok/s", "n_gpus": args.gpus, "steps": K, "warmup": W,
                "ms_per_step": 1e3 / tps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "q8_0xq8_0->int32, f32 accumulate",
                "data": "synthetic", "impl": "reference", "config": config,
                "cpu_baseline": {"value": tps, "unit": "tok/s", "cores": cores, "kind": "port",
                                 "sample": f"{n} decode steps of the same workload in {dt:.1f} s (C restatement of InferenceCore.forwardJava, -O2, OpenMP rows)"},
                "e2e": {"value": tps, "unit": "tok/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    import torch
    import torch.distributed as dist

    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    torch.cuda.set_device(local)
    # a rank that never runs the oracle keeps only the rows it uploads on the host (70B: ~10 GB instead of 74 GB per rank)
    shard_host = world > 1 and (rank != 0 or args.no_cpu)
    shape, model, gen_s = build_model(pkg, ctx, f"cuda:{local}", rank if shard_host else 0, world if shard_host else 1)
    t0 = time.time()
    plan = pkg.B200MasterPlan.initialize_plan(model, device=local, tp_rank=rank, tp_size=world)
    load_s = time.time() - t0

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if args.decode_mode != "default":
        plan.set_decode_mode(args.decode_mode)
    dmode, launches_per_step, ring_stages, pd_smem = plan.decode_info()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()  # nvidia-smi forks BEFORE the barrier: no rank waits on it inside the timed region
    # ---- value: device loop, tokens resident in HBM ------------------------------------------
    plan.decode_sequence(tokens[:D], D, 0)  # D >= W untimed warm-up steps (positions 0..D-1)
    barrier()
    ids, ms = plan.decode_sequence(tokens[D:D + K], K, D)
    barrier()
    if args.dump_outputs and rank == 0:  # read back before the e2e leg and the kernel timings overwrite the logits buffer
        dump_outputs(args.dump_outputs, ids, plan.read_buffer("logits", shape.vocab) if world == 1 else None)
    ms_rank = [ms]
    if world > 1:
        t = torch.tensor([ms], device=f"cuda:{local}")
        allt = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        ms_rank = [float(v.item()) for v in allt]
        ms = max(ms_rank)
    value = K / (ms / 1e3)  # one stream; under --gpus N the model is tensor-parallel over N ranks (strong scaling)

    # ---- e2e: reference-facing call, host token in / host argmax out every step ----------------
    plan.kv_reset()
    if D > W:
        plan.decode_sequence(tokens[:D - W], D - W, 0)
    for i in range(D - W, D):  # W untimed warm-up calls through the same entry point
        plan.forward_decode(int(tokens[i]), i, logits=False)
    barrier()
    t0 = time.perf_counter()
    e2e_ids = []
    for i in range(K):
        _, am = plan.forward_decode(int(tokens[D + i]), D + i, logits=False)
        e2e_ids.append(am)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device=f"cuda:{local}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    clocks = sampler.stop() if rank == 0 else None
    assert list(ids) == e2e_ids, "device loop and per-step API disagree"

    if rank != 0:
        if not args.no_cpu:  # tensor-parallel parity gate: rank 0 runs the oracle, every rank issues the same forwards
            box = [None]
            dist.broadcast_object_list(box, src=0)
            n_par = int(box[0])
            plan.kv_reset()
            for i in range(n_par):
                plan.forward_decode(int(tokens[i]), i, logits=False)
        plan.free()
        dist.barrier()
        dist.destroy_process_group()
        return 0

    # ---- roofline: the whole decode step (in persistent mode it is ONE kernel launch) ------------------
    peak, peak_src = peaks()
    ab = algorithmic_bytes_per_token(shape, QUANT == "q8_0", D + (K - 1) / 2.0)
    step_bytes = ab["total"] / world                 # algorithmic bytes one GPU must read per token
    step_gbs = step_bytes * value / 1e9              # ... x tok/s
    per_kernel = {}
    if world == 1:  # the stand-alone streaming matvecs of the graph path, for context (b200_time_kernel, PDL off)
        for which, name in ((0, "gate_up"), (1, "down_proj"), (2, "qkv"), (3, "attn_out"), (4, "lm_head")):
            m, b = plan.time_kernel(which, reps=3 if which != 4 else 1)
            per_kernel[name] = {"ms": m, "GB/s": b / (m / 1e3) / 1e9, "bytes": b, "frac": b / (m / 1e3) / 1e9 / peak}
    persistent = dmode == 1
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "r2_decode_traffic.json")  # dram bytes per launch from the committed ncu --set full capture
    if world == 1 and WORKLOAD == "llama-3-8b" and QUANT == "q8_0" and os.path.exists(tpath):
        with open(tpath) as f:
            traffic = json.load(f).get("persistent" if persistent else "graph")
    line = {
        "metric": "decode_tokens_per_s", "value": value, "unit": "tok/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak" if world == 1 else "strong", "vs_baseline": None,
        "dtype": "q8_0xq8_0->int32, f32 accumulate" if QUANT == "q8_0" else "f16 weights x f32 activations, f32 fma chains (16 lanes)", "data": "synthetic", "config": config,
        "parallelism": "single GPU" if world == 1 else f"tp{world}: row-sharded weights, in-kernel all-gather over NVLink peer memory (bit-exact with tp1)",
        "decode_mode": "persistent (1 kernel per token)" if persistent else f"graph ({launches_per_step} kernels per token)",
        "e2e": {"value": K / e2e_s, "unit": "tok/s", "h2d_bytes_per_step": 32, "d2h_bytes_per_step": 4},
        "gpu_launches": launches_per_step * K,
        "clocks": clocks,
        "ms_per_step_by_rank": [m / K for m in ms_rank],
        "roofline": {"kernel": ("k_decode_persistent: the whole token (all layers + lm_head + argmax) in one launch; " if persistent else "whole decode step (CUDA graph); ")
                               + ("per GPU" if world > 1 else "single GPU"),
                     "bound": "hbm", "achieved": step_gbs, "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": step_gbs / peak,
                     "bytes_per_launch": step_bytes if persistent else step_bytes / launches_per_step, "ms_per_launch": ms / K if persistent else ms / K / launches_per_step,
                     "algorithmic_bytes_per_token": ab, "traffic": traffic,
                     "persistent_kernel": {"ring_stages": ring_stages, "smem_bytes": pd_smem} if persistent else None,
                     "dominant_kernel": ({"name": ("k_stream_matvec_q8<GATEUP>" if QUANT == "q8_0" else "k_stream_matvec_f16<GATEUP>") + " (gate/up + SwiGLU: the largest share of the step's bytes and time), stand-alone, CUDA events on the plan's stream",
                                          "achieved": per_kernel["gate_up"]["GB/s"], "peak": peak, "unit": "GB/s", "frac": per_kernel["gate_up"]["frac"],
                                          "bytes_per_launch": per_kernel["gate_up"]["bytes"], "ms_per_launch": per_kernel["gate_up"]["ms"]} if "gate_up" in per_kernel else None),
                     "other_kernels": per_kernel},
        "load": {"synthesise_s": gen_s, "upload_repack_s": load_s, "device_bytes": plan.device_bytes, "pipeline": plan.upload_info()},
    }
    if not args.no_cpu:
        orc = ge.import_oracle()
        # N = 1: the reported CPU baseline (bounded sample).  N > 1: a short run, only to carry driver-visible TP parity.
        tps, n, dt, cores, ref = cpu_leg(orc, model, tokens, args.cpu_budget if world == 1 else 6.0, 16 if world == 1 else 4)
        if world == 1:
            line["cpu_baseline"] = {"value": tps, "unit": "tok/s", "cores": cores, "kind": "port",
                                    "sample": f"{n} decode steps of the same workload in {dt:.1f} s (C restatement of InferenceCore.forwardJava, -O2, OpenMP rows)"}
        if world > 1:  # the other ranks wait here, then run the same parity calls (TP: every rank issues the same forwards)
            dist.broadcast_object_list([len(ref["ids"])], src=0)
        line["parity"] = parity_gate(plan, tokens, ref, want_logits=world == 1)
    plan.free()
    if not args.no_pp and world == 1 and WORKLOAD == "llama-3-8b" and QUANT == "q8_0":  # BASELINE config 3 is the 8B FP16 model
        del model, plan
        line["pp512"] = prefill_leg(pkg, lb, local, 512, 5)
    print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if "parity" in line and not line["parity"]["ids_equal"]:
        sys.stderr.write("PARITY FAILURE: GPU greedy ids differ from the oracle\n")
        return 3
    return 0


if __name__ == "__main__":
    sys.exit(main())
