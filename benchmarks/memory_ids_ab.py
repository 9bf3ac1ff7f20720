"""A/B of the region memory's row ids (``query_ids=``, ``enqueue(ids=)``) against the memory without them, alternated in
one run, and the kernels the ids add or replace.

Step: the benchmark's shape (16 triplets x 64 masks, C = 256, bf16 features, fp32 masks) with a full K = 65 536 memory,
each arm captured once in a CUDA graph and replayed; ms/step from CUDA events over `--steps` replays, the arms
interleaved `--rounds` times:
    mem           region_step(memory=m), as without ids                 (scan, dQ; the enqueue writes -1 ids)
    mem+ids       StepBuffers(ids=True) with query ids -1: the exclusion mask is built and read every step, no row matches
    mem+ids hit   StepBuffers(ids=True) with query ids 0..15; the memory starts with one row of each id at a random slot,
                  and every replay pushes its ground-truth rows with those ids, so a query's matches grow by one a step
                  while that step's rows stay in the ring (reported as `matched_rows_per_query` after the arm's last round)
Kernels (CUDA events around a CUDA graph of `--iters` back-to-back calls, so that the host's per-call cost is not timed;
16 queries, D = 256, K = 65 536, the 33.5 MB bank resident in L2 after the first pass): the mask (cor_memory_exclude),
the scan without and with a mask (cor_memory_scan, cor_memory_scan_x), the dQ without and with a mask (cor_memory_dq,
cor_memory_dq_x, queries' gradient only); the masked kernels once with no bit set and once with one matching row per
query.  Prints one JSON line per measurement, then the
GPU name and power limit.

    python benchmarks/memory_ids_ab.py [--steps 200] [--rounds 3] [--iters 50]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

K = 65536


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
    """Device time per call: `iters` calls captured into one CUDA graph, replayed three times after a warm-up."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for _ in range(iters):
            fn()
    graph.replay()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(3):
        graph.replay()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e3 / (3 * iters)


def full_memory(C, dev, seed, ids=None):
    """A full memory of unit rows; ids: None (every row -1) or a function (n, generator) -> int64 ids of a batch."""
    from cor_b200 import region
    m = region.RegionMemory(K, C, dev)
    g = torch.Generator(device=dev).manual_seed(seed)
    for i in range(0, K, 8192):
        n = min(8192, K - i)
        rows = torch.nn.functional.normalize(torch.randn(n, C, device=dev, generator=g), dim=-1)
        m.enqueue(rows, ids=None if ids is None else ids(n, g))
    return m


def one_hit_memory(C, dev, seed, nq):
    """A full memory whose ids are >= 1000 except one row of each id 0 .. nq-1, at random slots."""
    m = full_memory(C, dev, seed, ids=lambda n, g: torch.randint(1000, 1 << 40, (n,), device=dev, generator=g))
    g = torch.Generator(device=dev).manual_seed(seed + 1)
    m.ids[torch.randperm(K, device=dev, generator=g)[:nq]] = torch.arange(nq, device=dev)
    return m


def matched_per_query(m, qids):
    ids = m.row_ids()
    return float(sum(int((ids == q).sum()) for q in qids.tolist() if q >= 0)) / len(qids)


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
    B, C = cfg["B"], cfg["C"]
    inp = bench.device_inputs(dev, 1234, cfg, "f32")
    hit_ids = torch.arange(B, device=dev)
    arms = {
        "mem": (full_memory(C, dev, 2), None),
        "mem+ids": (full_memory(C, dev, 2, ids=lambda n, g: torch.randint(0, 1 << 40, (n,), device=dev, generator=g)),
                    torch.full((B,), -1, dtype=torch.int64, device=dev)),
        "mem+ids hit": (one_hit_memory(C, dev, 2, B), hit_ids),
    }
    print(json.dumps({"what": "start", "matched_rows_per_query": {k: matched_per_query(m, q) for k, (m, q) in arms.items() if q is not None}}),
          flush=True)
    bufs = {}
    for name, (mem, qids) in arms.items():
        b = region.StepBuffers(cfg["B"], cfg["M"], cfg["C"], cfg["h"], cfg["w"], cfg["H"], cfg["W"], cfg["hp"], cfg["wp"], device=dev,
                               emb_dtype=torch.bfloat16, mask_dtype=inp["masks"].dtype, ids=qids is not None)
        b.load(dict(inp, ids=qids) if qids is not None else inp)
        b.capture(backward=True, emb_grad=True, warmup=2, tau=cfg["tau"], gather=False, memory=mem)
        bufs[name] = b
    for b in bufs.values():
        time_replays(b, 20)
    for r in range(args.rounds):
        for name, b in bufs.items():
            ms = time_replays(b, args.steps)
            print(json.dumps({"what": "step", "arm": name, "round": r, "ms_per_step": round(ms, 4),
                              "launches_per_step": b.launches_per_step}), flush=True)
    print(json.dumps({"what": "end", "matched_rows_per_query": {k: matched_per_query(m, q) for k, (m, q) in arms.items() if q is not None}}),
          flush=True)
    del bufs, arms
    torch.cuda.empty_cache()

    Nq, D = 16, C
    g = torch.Generator(device=dev).manual_seed(7)
    q16 = torch.nn.functional.normalize(torch.randn(Nq, D, device=dev, generator=g), dim=-1).bfloat16()
    g_loss = torch.ones(1, device=dev)
    lse = torch.full((Nq,), 30.0, device=dev)
    gq = torch.zeros(Nq, D, device=dev)
    inv_tau = 1.0 / cfg["tau"]
    m = one_hit_memory(D, dev, 3, Nq)
    work = ops._memory_scan_work(m, Nq, D, dev)
    masks = {"none": ops._memory_exclude(m, torch.full((Nq,), -1, dtype=torch.int64, device=dev)),
             "one_hit": ops._memory_exclude(m, torch.arange(Nq, device=dev))}
    torch.cuda.synchronize()
    bits = {k: int(sum(bin(int(w) & 0xFFFFFFFF).count("1") for w in v.view(torch.int32).cpu().tolist())) for k, v in masks.items()}
    qids = torch.arange(Nq, device=dev)
    xw = ops._memory_exclude_work(m, Nq, dev)
    us = time_us(lambda: ops._memory_exclude(m, qids, xw), args.iters)
    print(json.dumps({"what": "memory_exclude", "Nq": Nq, "K": K, "us": round(us, 2), "mask_bytes": Nq * K // 8}), flush=True)
    us = time_us(lambda: ops._memory_scan(m, q16, inv_tau, None, work), args.iters)
    print(json.dumps({"what": "memory_scan", "Nq": Nq, "K": K, "D": D, "us": round(us, 2)}), flush=True)
    for k, x in masks.items():
        us = time_us(lambda: ops._memory_scan(m, q16, inv_tau, None, work, x), args.iters)
        print(json.dumps({"what": "memory_scan_x", "mask": k, "excluded_pairs": bits[k], "Nq": Nq, "K": K, "D": D, "us": round(us, 2)}),
              flush=True)
    us = time_us(lambda: ops._memory_dq(m, q16, lse, inv_tau, None, g_loss, 1.0, gq, None), args.iters)
    print(json.dumps({"what": "memory_dq", "Nq": Nq, "K": K, "D": D, "us": round(us, 2), "launches": 2}), flush=True)
    for k, x in masks.items():
        us = time_us(lambda: ops._memory_dq(m, q16, lse, inv_tau, None, g_loss, 1.0, gq, None, x), args.iters)
        print(json.dumps({"what": "memory_dq_x", "mask": k, "excluded_pairs": bits[k], "Nq": Nq, "K": K, "D": D, "us": round(us, 2),
                          "launches": 2}), flush=True)
    print(json.dumps(gpu_info()), flush=True)


if __name__ == "__main__":
    main()
