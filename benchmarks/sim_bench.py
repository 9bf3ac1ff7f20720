#!/usr/bin/env python
"""The tcgen05 similarity / InfoNCE kernel alone: ONE launch (cor_sim_lse_parts, engine umma) after an L2 flush, CUDA
events, median of --iters; log-sum-exp checked against an fp32 torch restatement on the same bf16 operands.

    python benchmarks/sim_bench.py [--shapes 1024x102400,16x102400,256x4096]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from cor_b200 import _lib as L  # noqa: E402
from cor_b200 import ops  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--iters", type=int, default=15)
ap.add_argument("--shapes", default="1024x102400,256x102400,16x102400,256x4096")
ap.add_argument("--tag", default=os.environ.get("COR_B200_LIB", "default"))
args = ap.parse_args()
pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
HBM, TCB = pk.get("hbm_gbs", 6650.0), pk.get("bf16_tflops", 1590.0)
flush = torch.zeros(64 << 20, dtype=torch.float32, device="cuda")
g = torch.Generator(device="cuda").manual_seed(0)
D, inv_tau = 256, 1 / 0.07
for shp in args.shapes.split(","):
    Nq, Nr = (int(v) for v in shp.split("x"))
    R = torch.nn.functional.normalize(torch.randn(Nr, D, device="cuda", generator=g), dim=-1).bfloat16()
    Q = torch.nn.functional.normalize(torch.randn(Nq, D, device="cuda", generator=g), dim=-1).bfloat16()
    _, lse = ops._sim_forward(R, Q, inv_tau, False, True, "umma")
    ref = torch.logsumexp((Q.float() @ R.float().t()) * inv_tau, dim=1)
    err = float((lse - ref).abs().max())
    for _ in range(3):
        ops._sim_lse_parts(R, Q, inv_tau, "umma")
    ts = []
    for _ in range(args.iters):
        flush.add_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        ops._sim_lse_parts(R, Q, inv_tau, "umma")
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    ts.sort()
    t = ts[len(ts) // 2] * 1e-3
    flops, byts = 2.0 * Nq * Nr * D, (Nq + Nr) * D * 2
    print(json.dumps({"lib": args.tag, "case": f"sim_umma lse {Nq}x{Nr}x{D}", "us": round(t * 1e6, 2), "us_best": round(ts[0] * 1e3, 2),
                      "tflops": round(flops / t / 1e12, 1), "tc_frac_burst": round(flops / t / 1e12 / TCB, 3),
                      "gbs": round(byts / t / 1e9, 1), "hbm_frac": round(byts / t / 1e9 / HBM, 3), "lse_max_abs_err": err}), flush=True)
