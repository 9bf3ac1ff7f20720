"""A/B of the cross-batch region memory against no memory, alternated in one run, and the memory kernels' own times.

Step: the benchmark's shape (16 triplets x 64 masks, C = 256, bf16 features, fp32 masks), each arm captured once in a
CUDA graph and replayed; ms/step from CUDA events over `--steps` replays, the arms interleaved `--rounds` times:
    none      region_step(tau=0.07)                                    (no memory)
    mem8192   region_step(..., memory=m), m full with K =  8 192 rows  (each replay scans, then enqueues the batch)
    mem65536  region_step(..., memory=m), m full with K = 65 536 rows
Kernels (CUDA events around `--iters` back-to-back launches, 16 queries, D = 256): the scan (cor_memory_scan), the
memory dQ (cor_memory_dq, queries' gradient only) at K = 65 536 (33.5 MB bank, resident in the 126 MB L2 after the
first pass) and K = 262 144 (134 MB, more than L2), and the enqueue of one step's 1 024 fp32 rows.  Achieved rates are
computed from shapes: the scan does 2 Nq K D flop and reads K D bf16; the dQ 4 Nq K D flop (two GEMMs) over the same
bank; the enqueue reads n C fp32 and writes n C bf16 (its eager time includes the host cost of each call).  Prints one
JSON line per measurement, then the GPU name and power limit.

    python benchmarks/memory_ab.py [--steps 200] [--rounds 3] [--iters 50]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:                 # the timing stands without it; say why it is missing
        out = f"nvidia-smi unavailable: {e}"
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": out}


def time_replays(bufs, steps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        bufs.replay()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def time_us(fn, iters):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e3 / iters


def full_memory(K, C, dev, seed):
    from cor_b200 import region
    m = region.RegionMemory(K, C, dev)
    g = torch.Generator(device=dev).manual_seed(seed)
    for i in range(0, K, 8192):
        n = min(8192, K - i)
        m.enqueue(torch.nn.functional.normalize(torch.randn(n, C, device=dev, generator=g), dim=-1))
    return m


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--iters", type=int, default=50)
    args = ap.parse_args()
    import bench
    from cor_b200 import ops, region
    dev = torch.device("cuda:0")
    cfg = dict(bench.CFG)
    inp = bench.device_inputs(dev, 1234, cfg, "f32")
    arms = {"none": None, "mem8192": full_memory(8192, cfg["C"], dev, 1), "mem65536": full_memory(65536, cfg["C"], dev, 2)}
    bufs = {}
    for name, mem in arms.items():
        b = region.StepBuffers(cfg["B"], cfg["M"], cfg["C"], cfg["h"], cfg["w"], cfg["H"], cfg["W"], cfg["hp"], cfg["wp"], device=dev,
                               emb_dtype=torch.bfloat16, mask_dtype=inp["masks"].dtype)
        b.load(inp)
        kw = dict(memory=mem) if mem is not None else {}
        b.capture(backward=True, emb_grad=True, warmup=2, tau=cfg["tau"], gather=False, **kw)
        bufs[name] = b
    for b in bufs.values():
        time_replays(b, 20)
    for r in range(args.rounds):
        for name, b in bufs.items():
            ms = time_replays(b, args.steps)
            print(json.dumps({"what": "step", "arm": name, "round": r, "ms_per_step": round(ms, 4),
                              "launches_per_step": b.launches_per_step}), flush=True)
    del bufs, arms
    torch.cuda.empty_cache()

    Nq, D = 16, cfg["C"]
    g = torch.Generator(device=dev).manual_seed(7)
    q16 = torch.nn.functional.normalize(torch.randn(Nq, D, device=dev, generator=g), dim=-1).bfloat16()
    g_loss = torch.ones(1, device=dev)
    for K in (65536, 262144):
        m = full_memory(K, D, dev, 3)
        work = ops._memory_scan_work(m, Nq, D, dev)
        lse = torch.full((Nq,), 30.0, device=dev)
        gq = torch.zeros(Nq, D, device=dev)
        us = time_us(lambda: ops._memory_scan(m, q16, 1.0 / cfg["tau"], None, work), args.iters)
        bank_bytes = K * D * 2
        print(json.dumps({"what": "memory_scan", "Nq": Nq, "K": K, "D": D, "us": round(us, 2), "tflops": round(2 * Nq * K * D / us / 1e6, 2),
                          "gbps": round(bank_bytes / us / 1e3, 1)}), flush=True)
        us = time_us(lambda: ops._memory_dq(m, q16, lse, 1.0 / cfg["tau"], None, g_loss, 1.0, gq, None), args.iters)
        print(json.dumps({"what": "memory_dq", "Nq": Nq, "K": K, "D": D, "us": round(us, 2), "tflops": round(4 * Nq * K * D / us / 1e6, 2),
                          "gbps": round(bank_bytes / us / 1e3, 1), "launches": 2}), flush=True)
        del m, work
        torch.cuda.empty_cache()
    m = region.RegionMemory(65536, D, dev)
    rows = torch.randn(cfg["B"] * cfg["M"], D, device=dev, generator=g)
    us = time_us(lambda: m.enqueue(rows), args.iters)
    n = rows.shape[0]
    print(json.dumps({"what": "memory_enqueue", "n": n, "C": D, "us": round(us, 2), "gbps": round(n * D * 6 / us / 1e3, 1)}), flush=True)
    print(json.dumps(gpu_info()), flush=True)


if __name__ == "__main__":
    main()
