"""Top-k retrieval: the fused path (cor_topk_select, candidates kept inside the tensor-core similarity kernel, S never
written) against the S route (cor_sim_umma_fwd writes S [Nq, Nr] fp32, cor_topk selects from it), alternated in one run.

Workloads (unit rows generated on the device from a seed, bf16, D = 256):
    256 x 4 096    k 10        BASELINE config 3 (bench.py's topk_256x4096_k10); gallery 2 MB and S 4 MB fit the 126 MB L2
    256 x 1 M      k 10, 256   gallery 512 MB, S 1 GB: neither fits L2
    4 096 x 1 M    k 10, 256   S 16 GB
    256 x 4 M      k 10, 256   gallery 2 GB, S 4 GB
Each arm is timed with CUDA events over `--iters` back-to-back calls after `--warmup` calls, the two arms interleaved
`--rounds` times.  Both arms start from the bf16 rows (no cast copy) and their outputs are checked equal.  The S route's
time includes allocating S.  Bytes per call computed from shapes: the fused path reads the gallery once (per query tile
of 256); the S route also writes S once and reads it five times (four radix passes, one collect).  Prints one JSON line
per measurement and writes them to `--out`, then the GPU name and power limit.

    python benchmarks/topk_bench.py [--rounds 3] [--iters 10] [--out profiles/r06_topk_bench.log]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

L2_BYTES = 126 * 1024 * 1024
WORKLOADS = [(256, 4096, (10,)), (256, 1 << 20, (10, 256)), (4096, 1 << 20, (10, 256)), (256, 1 << 22, (10, 256))]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:                 # the timing stands without it; say why it is missing
        out = f"nvidia-smi unavailable: {e}"
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": out}


def rows(seed, n, D, dev):
    g = torch.Generator(device=dev).manual_seed(seed)
    return torch.nn.functional.normalize(torch.randn(n, D, device=dev, generator=g), dim=-1).bfloat16()


def s_route(r16, q16, k):
    from cor_b200 import ops
    Nr, D = r16.shape
    Nq = q16.shape[0]
    S, _ = ops._sim_forward(r16, q16, 1.0, True, False, "umma")
    idx = torch.empty((Nq, k), dtype=torch.int64, device=r16.device)
    score = torch.empty((Nq, k), dtype=torch.float32, device=r16.device)
    ops._call("cor_topk", r16.device, ops.ptr(S), ops.ptr(r16), ops.ptr(q16), Nr, Nq, D, k, ops.ptr(idx), ops.ptr(score))
    return idx, score


def fused(r16, q16, k):
    from cor_b200 import ops
    return ops._topk_select(r16, q16, k)


def time_ms(fn, iters, warmup):
    for _ in range(warmup):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join("profiles", "r06_topk_bench.log"))
    a = ap.parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("topk_bench.py measures on a GPU; none is visible")
    from cor_b200 import _lib
    dev = torch.device("cuda:0")
    D = 256
    lines = []

    def emit(rec):
        print(json.dumps(rec), flush=True)
        lines.append(rec)

    for Nq, Nr, ks in WORKLOADS:
        r16, q16 = rows(1, Nr, D, dev), rows(2, Nq, D, dev)
        gallery, s_bytes = Nr * D * 2, Nq * Nr * 4
        for k in ks:
            fi, fs = fused(r16, q16, k)
            si, ss = s_route(r16, q16, k)
            equal = bool(torch.equal(fi, si) and torch.equal(fs, ss))
            del fi, fs, si, ss
            work = _lib.load().cor_topk_select_work_bytes(Nq, Nr, D, k)
            for rnd in range(a.rounds):
                for arm, fn in (("fused", fused), ("s_route", s_route)):
                    ms = time_ms(lambda: fn(r16, q16, k), a.iters, a.warmup)
                    qtiles = (Nq + 255) // 256
                    alg = gallery * qtiles + (0 if arm == "fused" else 6 * s_bytes)
                    emit({"what": "topk", "arm": arm, "round": rnd, "Nq": Nq, "Nr": Nr, "D": D, "k": k, "ms": round(ms, 4),
                          "algorithmic_bytes": alg, "gallery_fits_l2": gallery <= L2_BYTES,
                          "s_fits_l2": s_bytes <= L2_BYTES, "work_bytes": work if arm == "fused" else s_bytes,
                          "outputs_equal": equal})
        del r16, q16
        torch.cuda.empty_cache()
    info = gpu_info()
    emit(info)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for rec in lines:
            f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
