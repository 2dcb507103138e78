#!/usr/bin/env python
"""SURVEY 8(f) N1: time the load of a model FROM A GGUF FILE ON DISK through the upload pipeline (the counterpart of the
reference's load-time metric, ModelLoader.java:102-106, and its first-execution copy-in, TornadoVMMasterPlanSingleToken.java:51-54).

    python tools/load_bench.py [workload] [dir]   ->  gpurun_out/load_bench_<workload>.json

Writes a seeded synthetic GGUF of the real shape (no checkpoints offline), drops it from the process (the page cache may still hold it:
reported as "warm"), then: parse + mmap (gguf.GGUFFile) and b200_plan_create (pinned double buffer -> copy stream -> device staging ->
repack kernels), with the default and with 8 host copy threads."""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as ge  # noqa: E402


def main():
    workload = sys.argv[1] if len(sys.argv) > 1 else "llama-3-8b"
    d = sys.argv[2] if len(sys.argv) > 2 else "/tmp"
    pkg = ge.import_package()
    shape = pkg.synth.SHAPES[workload]
    Q = pkg.gguf.GGMLType.Q8_0
    path = os.path.join(d, f"{workload}-q8_0-synthetic.gguf")
    t0 = time.time()
    tensors = pkg.synth.build_tensors_fast(shape, Q, seed=1234, device="cuda:0")
    plan_order = [(name, tt, dims, tensors[name][2]) for name, tt, dims, _ in pkg.synth.tensor_plan(shape, Q)]
    gen_s = time.time() - t0
    t0 = time.time()
    pkg.gguf.write_gguf(path, pkg.synth.metadata_for(shape, Q, "Llama synthetic " + workload), plan_order)
    write_s = time.time() - t0
    size = os.path.getsize(path)
    del tensors, plan_order
    out = {"workload": workload, "file_bytes": size, "synthesise_s": gen_s, "write_s": write_s, "runs": []}
    for label, env in (("pipelined", {}), ("pipelined, 8 host threads", {"B200_UPLOAD_THREADS": "8"})):
        os.environ.update(env)
        try:
            t0 = time.time()
            model = pkg.load_model(path, 64)
            parse_s = time.time() - t0
            t0 = time.time()
            plan = pkg.B200MasterPlan.initialize_plan(model)
            create_s = time.time() - t0
            info = plan.upload_info()
            _, am = plan.forward_decode(1, 0, logits=False)
            plan.free()
            out["runs"].append({"path": label, "parse_mmap_s": parse_s, "plan_create_s": create_s, "upload": info, "first_argmax": int(am),
                                "file_GB_per_s_end_to_end": size / (parse_s + create_s) / 1e9})
        finally:
            for k in env:
                del os.environ[k]
    os.remove(path)
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    with open(os.path.join(ROOT, "gpurun_out", f"load_bench_{workload}.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
