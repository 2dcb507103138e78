"""Checks the tcgen05 prefill GEMM against an fp32 matmul of the same fp16 operands and times it.
usage: python tools/gemm_check.py [--big] [--stages 3|6] [--resid R] [--two-cta 0|256|1256] [--out-dir DIR]"""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from __graft_entry__ import import_package  # noqa: E402

pkg = import_package()
from gpullama3_java_b200 import native  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--big", action="store_true")
ap.add_argument("--stages", type=int, default=3, help="single-CTA ring depth: 3 or 6")
ap.add_argument("--resid", type=int, default=0, help="C += A B^T; with --two-cta 256 the number of K splits")
# 0: single-CTA kernel; 256: CTA-pair residual GEMM (needs --resid >= 1); 1256: persistent pair kernel
ap.add_argument("--two-cta", type=int, default=0)
ap.add_argument("--out-dir", default=".", help="directory for gemm_check_s<stages>_2cta<two-cta>_r<resid>.json")
args = ap.parse_args()
two = args.two_cta

rng = np.random.default_rng(7)
out = []
shapes = [(128, 128, 64), (256, 384, 512), (512, 4096, 4096)]
if args.big:
    shapes += [(512, 6144, 4096), (512, 28672, 4096), (512, 4096, 14336), (4096, 4096, 4096), (8192, 8192, 8192)]
for (m, n, k) in shapes:
    if two and (m % 256 or n % 256):
        continue
    a = (rng.standard_normal((m, k)) * 0.5).astype(np.float16)
    b = (rng.standard_normal((n, k)) * 0.5).astype(np.float16)
    c, ms = native.gemm_f16(a, b, iters=20, stages=args.stages, resid=args.resid, two_cta=two)
    if m * n * k <= 512 * 4096 * 4096:
        ref = a.astype(np.float32) @ b.astype(np.float32).T
        err = float(np.max(np.abs(c - ref)))
        scale = float(np.max(np.abs(ref)))
    else:  # spot check 64 rows
        rows = rng.integers(0, m, 64)
        ref = a[rows].astype(np.float32) @ b.astype(np.float32).T
        err = float(np.max(np.abs(c[rows] - ref)))
        scale = float(np.max(np.abs(ref)))
    rec = {"two_cta": two, "resid": str(args.resid), "stages": str(args.stages), "m": m, "n": n, "k": k, "max_abs_err": err, "ref_max": scale, "ms": ms, "tflops": 2.0 * m * n * k / (ms * 1e-3) / 1e12}
    print(json.dumps(rec), flush=True)
    out.append(rec)
os.makedirs(args.out_dir, exist_ok=True)
json.dump(out, open(os.path.join(args.out_dir, "gemm_check_s%d_2cta%d_r%d.json" % (args.stages, two, args.resid)), "w"), indent=1)
