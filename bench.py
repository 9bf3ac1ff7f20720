#!/usr/bin/env python
"""bench.py -- region-scored triplets/s for CORE's region pooling / scoring / loss path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one forward + backward of the region path over one batch of synthetic triplets
(BASELINE.json config[1]: 16 triplets x 64 candidate 1024x1024 masks per GPU, bf16 features):
mask resample + validity sums, region pooling (fg, bg and all candidates), L2-normalise, fg/bg
cosine losses, region x query InfoNCE (negatives all-gathered across ranks), segmentation loss,
and the backward of all of it.  Prints ONE JSON line (see README / DESIGN.md for the keys).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "region_scored_triplets_per_sec"
UNIT = "triplets/s"
CFG = dict(B=16, M=64, C=256, h=64, w=64, H=1024, W=1024, hp=256, wp=256, tau=0.07)


def traffic_from_profiles(cfg, mask_dtype, kernel="mask_prep"):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, READ AT RUN TIME from the newest
    committed `ncu --set full` summary under profiles/ whose name carries this configuration's key
    (`..._B{B}_M{M}_{dtype}...csv`); the round-1 capture (no key in its name) is config 2 with fp32 masks.  None when no
    capture of this configuration is committed -- a stale constant could not reveal a regression."""
    import csv
    import glob
    key = f"_B{cfg['B']}_M{cfg['M']}_{mask_dtype}"
    cands = sorted(glob.glob(os.path.join(ROOT, "profiles", f"r*ncu_full*{key}*.csv")), reverse=True)
    if not cands and (cfg["B"], cfg["M"], mask_dtype) == (16, 64, "f32"):
        cands = [os.path.join(ROOT, "profiles", "r01_step_kernels_ncu_full_summary.csv")]
    for path in cands:
        try:
            with open(path, newline="") as f:
                for row in csv.DictReader(f):
                    if kernel not in row.get("Kernel Name", ""):
                        continue
                    tot = 0.0
                    for col, val in row.items():
                        for name in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                            if col.startswith(name):
                                unit = col[col.find("[") + 1:col.find("]")].lower() if "[" in col else "byte"
                                mul = {"byte": 1.0, "kbyte": 1e3, "mbyte": 1e6, "gbyte": 1e9}.get(unit, 1.0)
                                tot += float(val) * mul
                    if tot > 0:
                        return int(tot), os.path.relpath(path, ROOT)
        except Exception:
            continue
    return None, None


_T0 = time.perf_counter()


def trace(msg):
    """Stage markers on stderr (COR_BENCH_TRACE=1): locate a stall without a debugger."""
    if os.environ.get("COR_BENCH_TRACE"):
        print(f"[bench +{time.perf_counter() - _T0:7.2f}s rank {os.environ.get('RANK', '0')}] {msg}", file=sys.stderr, flush=True)


def peaks():
    """(HBM GB/s, bf16 TFLOP/s sustained, bf16 TFLOP/s burst, source)."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        burst = float(p.get("bf16_tflops", 1590.0))
        return float(p["hbm_gbs"]), float(p.get("bf16_tflops_sustained", burst)), burst, "measured"
    return 6650.0, 1590.0, 1590.0, "fallback"


# ------------------------------------------------------------------------------------------ inputs
def device_inputs(dev, seed, cfg, mask_dtype):
    """Seeded synthetic triplets generated on the device (SURVEY 8d recipe: union of rectangles and
    an ellipse per mask, 1 in 32 empty, 1 in 256 full; mask 0 of every image is the GT)."""
    B, M, H, W = cfg["B"], cfg["M"], cfg["H"], cfg["W"]
    g = torch.Generator(device=dev).manual_seed(seed)
    emb = torch.randn(B, cfg["C"], cfg["h"], cfg["w"], device=dev, generator=g).bfloat16()
    comb = torch.nn.functional.normalize(torch.randn(B, 1, cfg["C"], device=dev, generator=g), dim=-1)
    pred = torch.nn.functional.avg_pool2d(2 * torch.randn(B, 1, cfg["hp"] + 4, cfg["wp"] + 4, device=dev, generator=g), 5, 1) * 5
    pred = pred.bfloat16()
    masks = torch.empty(B, M, H, W, device=dev, dtype=torch.float32)
    yy = torch.arange(H, device=dev, dtype=torch.float32).view(1, H, 1)
    xx = torch.arange(W, device=dev, dtype=torch.float32).view(1, 1, W)
    r = torch.rand(B, M, 8, device=dev, generator=g)
    idx = torch.arange(B * M, device=dev).view(B, M)
    side = torch.sqrt(0.005 + 0.295 * r[..., 0])
    rh = torch.clamp((H * side * (0.4 + 0.6 * r[..., 1])).floor(), min=2)
    rw = torch.clamp((W * side * (0.4 + 0.6 * r[..., 2])).floor(), min=2)
    y0, x0 = (r[..., 3] * (H - rh)).floor(), (r[..., 4] * (W - rw)).floor()
    cy, cx = (0.2 + 0.6 * r[..., 5]) * H, (0.2 + 0.6 * r[..., 6]) * W
    ry, rx = torch.clamp(H * side * 0.4, min=2.0), torch.clamp(W * side * 0.4, min=2.0)
    v = lambda t, b_: t[b_].view(M, 1, 1)
    for b_ in range(B):       # one image at a time: [M,H,W] temporaries stay at 256 MB
        rect = (yy >= v(y0, b_)) & (yy < v(y0 + rh, b_)) & (xx >= v(x0, b_)) & (xx < v(x0 + rw, b_))
        ell = ((yy - v(cy, b_)) / v(ry, b_)) ** 2 + ((xx - v(cx, b_)) / v(rx, b_)) ** 2 <= 1.0
        m = (rect | ell).float()
        m[idx[b_] % 32 == 31] = 0.0
        m[idx[b_] % 256 == 129] = 1.0
        masks[b_] = m
    if mask_dtype == "u8":
        masks = (masks * 255).to(torch.uint8)
    return {"pred": pred, "emb": emb, "comb": comb, "masks": masks}


# -------------------------------------------------------------------------------------- clock probe
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.stop_flag, self.thread = index, [], threading.Event(), None

    def _run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.splitlines()[0].split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def __enter__(self):
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()
        return self

    def __exit__(self, *a):
        self.stop_flag.set()
        self.thread.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows)}


# ---------------------------------------------------------------------------------- CPU baseline leg
def cpu_kind():
    """"reference": oracle/_ref holds the reference's own modules (oracle/build_ref.py copied them, sha256 verified);
    "port": it does not travel with this snapshot and the ATen port stands in."""
    from oracle import ref_step
    return "reference" if (ref_step.available() and ref_step.verified()) else "port"


def cpu_port_step(sample, tau, kind=None):
    """One fwd+bwd of the same step on the host cores: through the reference's own functions (oracle/_ref) when they are
    there, else through the ATen port of the reference."""
    p, e, c = (sample[k].detach().clone().requires_grad_(True) for k in ("pred", "emb", "comb"))
    if (kind or cpu_kind()) == "reference" and not p.is_cuda:
        from oracle import ref_step
        loss, _ = ref_step.region_step_loss(p, e, c, sample["masks"], tau=tau)
    else:
        from oracle import aten_port as ap
        loss, _ = ap.region_step_loss(p, e, c, sample["masks"], tau=tau)
    loss.backward()
    return float(loss.detach())


def cpu_what(kind):
    return ("reference functions utils/loss_func.py (oracle/_ref, unmodified copy) + Class-N InfoNCE restatement" if kind == "reference"
            else "oracle/aten_port.py = reference ATen op sequence (oracle/_ref absent: build() copies the reference's modules there "
                 "only when COR_REFERENCE names a reference checkout)")


def cpu_baseline(inputs_cpu, cfg, triplets, iters, warm=1):
    cores = len(os.sched_getaffinity(0))
    torch.set_num_threads(cores)
    sample = {k: (v[:triplets].float() if v.is_floating_point() else v[:triplets].float() / 255.0) for k, v in inputs_cpu.items()}
    for _ in range(warm):
        cpu_port_step(sample, cfg["tau"])
    ts = []
    for _ in range(iters):
        t0 = time.perf_counter()
        cpu_port_step(sample, cfg["tau"])
        ts.append(time.perf_counter() - t0)
    med = sorted(ts)[len(ts) // 2]
    kind = cpu_kind()
    return {"value": triplets / med, "unit": UNIT, "cores": cores, "kind": kind,
            "sample": f"{triplets} triplets x {cfg['M']} masks {cfg['H']}x{cfg['W']} fp32, fwd+bwd, median of {iters} after {warm} warm-up "
                      f"({med * 1e3:.0f} ms/step); {cpu_what(kind)}"}, med


def torch_eager_gpu_baseline(inp, cfg, iters=5, warm=2):
    """SURVEY.md 8d: the reference's op sequence (oracle/aten_port.py) run by PyTorch eager ON THE SAME B200, full batch,
    fp32 and under bf16 autocast (how the reference trains, utils/trainer_v3_g.py:51) - the fair same-box bar next to the
    CPU baseline.  Checker code used as a baseline only; nothing of it is on the product path."""
    out = {}
    sample = {k: (v.float() if v.is_floating_point() else v.float() / 255.0) for k, v in inp.items()}
    for name, autocast in (("f32", False), ("bf16_autocast", True)):
        try:
            def one():
                with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
                    return cpu_port_step(sample, cfg["tau"])
            for _ in range(warm):
                one()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(iters):
                one()
            b.record()
            torch.cuda.synchronize()
            ms = a.elapsed_time(b) / iters
            out[name] = {"value": cfg["B"] / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "steps": iters}
        except Exception as e:  # noqa: BLE001 - a baseline must never take the bench down
            out[name] = {"error": f"{type(e).__name__}: {e}"[:200]}
        torch.cuda.empty_cache()
    out["what"] = ("reference ATen op sequence (oracle/aten_port.py, multi-mask recipe of SURVEY 8c) under PyTorch eager on this GPU, "
                   f"full batch of {cfg['B']} triplets x {cfg['M']} masks, fwd+bwd, device-resident inputs; includes float(loss)")
    return out


def run_reference(args, cfg):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    triplets = min(args.cpu_triplets, cfg["B"])
    host = device_inputs(torch.device("cpu"), 1234, dict(cfg, B=triplets), "f32")
    cores = len(os.sched_getaffinity(0))
    torch.set_num_threads(cores)
    kind = cpu_kind()
    sample = {k: v.float() for k, v in host.items()}
    for _ in range(args.warmup):
        cpu_port_step(sample, cfg["tau"])
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_port_step(sample, cfg["tau"])
    dt = (time.perf_counter() - t0) / args.steps
    val = triplets / dt
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": workload_config(cfg, args, sample_triplets=triplets),
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind,
                             "sample": (f"each step = the whole {cfg['B']}-triplet batch x {cfg['M']} masks" if triplets == cfg["B"] else
                                        f"each step = {triplets} triplets x {cfg['M']} masks (bounded sample of the {cfg['B']}-triplet batch)")
                                       + f", fwd+bwd; {cpu_what(kind)}"},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    emit_result(line)


def _negatives_note():
    """Where the InfoNCE negatives come from (same text on both arms of the bench)."""
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        return ("regions of all ranks: gathered / gradient reduced by our NVLink peer-memory kernels (csrc/peer.cu) on one node, "
                "NCCL all-gather / reduce-scatter with COR_PEER=0")
    return "all regions of the batch (single rank)"


def workload_config(cfg, args, sample_triplets=None):
    c = {"workload": f"CORE fwd+bwd region path, batch {cfg['B']} triplets x {cfg['M']} masks per GPU, "
                     f"{cfg['H']}x{cfg['W']} {args.mask_dtype} masks, bf16 features [B,{cfg['C']},{cfg['h']},{cfg['w']}], "
                     f"logits [B,1,{cfg['hp']},{cfg['wp']}] (BASELINE.json configs[1])",
         "triplets_per_gpu": cfg["B"], "masks_per_triplet": cfg["M"], "feature_map": [cfg["C"], cfg["h"], cfg["w"]],
         "mask_size": [cfg["H"], cfg["W"]], "mask_dtype": args.mask_dtype, "tau": cfg["tau"], "backward": True,
         "emb_grad": True, "negatives": _negatives_note(),
         "l2": "inputs (>= 1 GiB of masks per step) exceed the 126 MB L2; no explicit flush"}
    if sample_triplets is not None and sample_triplets != cfg["B"]:
        c["cpu_sample_triplets"] = sample_triplets
    return c


# --------------------------------------------------------------------------------------------- main
def _parse_cpulist(text):
    cpus = set()
    for part in text.strip().split(","):
        if not part:
            continue
        lo, _, hi = part.partition("-")
        cpus.update(range(int(lo), int(hi or lo) + 1))
    return cpus


def bind_to_gpu_numa(local):
    """Multi-rank e2e leg: run this rank (and first-touch its pinned staging buffers, which are allocated AFTER this call)
    on the CPUs local to its GPU, so that eight ranks do not all push their H2D copies through one socket.  The CPU set
    comes from NVML's affinity mask, else from sysfs (/sys/bus/pci/devices/<bdf>/{local_cpulist,numa_node}).  Returns
    a dict {"cpus": n bound to (None = unchanged), "numa_node": node or None, "how": source}."""
    info = {"cpus": None, "numa_node": None, "how": None}
    if os.environ.get("COR_BENCH_NUMA", "1") == "0":
        return info
    allowed = os.sched_getaffinity(0)
    local_cpus = set()
    bdf = None
    try:
        pr = torch.cuda.get_device_properties(local)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
    except Exception:
        pass
    try:
        import pynvml
        pynvml.nvmlInit()
        try:
            h = pynvml.nvmlDeviceGetHandleByPciBusId(("0000" + bdf).encode()) if bdf else pynvml.nvmlDeviceGetHandleByIndex(local)
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(local)
        n = os.cpu_count() or 1
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, (n + 63) // 64)
        local_cpus = {i for i in range(n) if (mask[i // 64] >> (i % 64)) & 1}
        info["how"] = "nvml"
    except Exception:
        local_cpus = set()
    if bdf:
        base = f"/sys/bus/pci/devices/{bdf}"
        try:
            node = int(open(base + "/numa_node").read().strip())
            info["numa_node"] = node if node >= 0 else None
        except Exception:
            pass
        if not local_cpus or local_cpus >= allowed:
            try:
                local_cpus = _parse_cpulist(open(base + "/local_cpulist").read())
                info["how"] = "sysfs local_cpulist"
            except Exception:
                pass
        if (not local_cpus or local_cpus >= allowed) and info["numa_node"] is not None:
            try:
                local_cpus = _parse_cpulist(open(f"/sys/devices/system/node/node{info['numa_node']}/cpulist").read())
                info["how"] = "sysfs node cpulist"
            except Exception:
                pass
    use = local_cpus & allowed
    if not use or use == allowed:
        return info
    try:
        os.sched_setaffinity(0, use)
        info["cpus"] = len(use)
    except Exception:
        pass
    return info


def pcie_h2d_gbs(dev, nbytes=1 << 30, copies=8):
    """Bare pinned-host -> device cudaMemcpyAsync: `copies` back-to-back copies of `nbytes` timed as ONE interval with
    CUDA events (after one warm-up copy), i.e. the SUSTAINED rate while every other rank does the same (the caller
    barriers first) -- the platform ceiling of the e2e leg.  (A best-of-N of single copies, as in round 1's first
    version of this probe, lets each rank catch a moment when the GPU sharing its PCIe uplink is idle and reads high.)"""
    src = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    src.fill_(1)                       # first touch on this rank's (NUMA-bound) CPUs
    dst = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    dst.copy_(src, non_blocking=True)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(copies):
        dst.copy_(src, non_blocking=True)
    b.record()
    torch.cuda.synchronize()
    gbs = copies * nbytes / (a.elapsed_time(b) * 1e-3) / 1e9
    del src, dst
    return gbs


def l2_flush(buf):
    buf.add_(1)                         # 256 MiB read + written: nothing of the previous launch stays in the 126 MB L2


def secondary_tensor_lines(dev, tc_burst, hbm_peak, iters=10):
    """Driver-run lines for the kernels the 16-query step does not exercise at their design point (VERDICT r1 item 2):
    the tcgen05 similarity / InfoNCE kernel at config 4's global shape (1024 queries x 102 400 regions x 256), its
    few-query shape (16 x 102 400, HBM-bound), InfoNCE forward+backward at the global shape, and config 3's top-k
    (256 x 4096, k = 10).  CUDA events around each launch, L2 flushed before every timed launch."""
    from cor_b200 import ops
    out = {}
    g = torch.Generator(device=dev).manual_seed(99)
    Nr, D = 102400, 256
    r32 = torch.nn.functional.normalize(torch.randn(Nr, D, device=dev, generator=g), dim=-1)
    r16 = r32.bfloat16()
    flush = torch.zeros(64 << 20, dtype=torch.float32, device=dev)

    def timed(fn, n=iters):
        ts = []
        for i in range(n + 2):
            l2_flush(flush)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            if i >= 2:
                ts.append(a.elapsed_time(b))
        ts.sort()
        return ts[len(ts) // 2], ts[0]

    for Nq in (1024, 16):
        q16 = torch.nn.functional.normalize(torch.randn(Nq, D, device=dev, generator=g), dim=-1).bfloat16()
        try:
            med, best = timed(lambda: ops._sim_lse_parts(r16, q16, 1.0 / 0.07, "umma"))
            flops = 2.0 * Nq * Nr * D
            byts = (Nq + Nr) * D * 2
            tf_s = flops / (med * 1e-3) / 1e12
            gb_s = byts / (med * 1e-3) / 1e9
            bound = "tensor" if Nq >= 256 else "hbm"
            out[f"sim_umma_kernel_{Nq}x{Nr}"] = {
                "what": "similarity + online log-sum-exp (InfoNCE forward), S never written; one launch", "bound": bound, "ms": med, "ms_best": best,
                "flops": flops, "algorithmic_bytes": byts, "achieved_tflops": tf_s, "achieved_gbs": gb_s,
                "peak": tc_burst if bound == "tensor" else hbm_peak, "unit": "TFLOP/s" if bound == "tensor" else "GB/s",
                "frac": (tf_s / tc_burst) if bound == "tensor" else (gb_s / hbm_peak),
                "peak_source": "MEASURED_PEAKS.json bf16_tflops (burst: kernel timed alone)" if bound == "tensor" else "MEASURED_PEAKS.json hbm_gbs"}
        except Exception as e:  # noqa: BLE001
            out[f"sim_umma_kernel_{Nq}x{Nr}"] = {"error": f"{type(e).__name__}: {e}"[:200]}
    try:
        Nq = 1024
        q32 = torch.nn.functional.normalize(torch.randn(Nq, D, device=dev, generator=g), dim=-1)
        tg = (torch.arange(Nq, device=dev) * 97) % Nr

        def fwd_bwd():
            r = r32.detach().requires_grad_(True)
            q = q32.detach().requires_grad_(True)
            ops.infonce_loss(r, q, tg, tau=0.07, regions_bf16=r16).backward()

        med, best = timed(fwd_bwd, n=5)
        out["infonce_fwd_bwd_1024x102400"] = {"what": "InfoNCE value + dQ + dR through the public op (includes its bf16 casts and launches)",
                                              "ms": med, "ms_best": best, "flops": 8.0 * Nq * Nr * D,
                                              "achieved_tflops": 8.0 * Nq * Nr * D / (med * 1e-3) / 1e12}
    except Exception as e:  # noqa: BLE001
        out["infonce_fwd_bwd_1024x102400"] = {"error": f"{type(e).__name__}: {e}"[:200]}
    try:   # the tensor-core backward alone (dQ and dR launches of csrc/nce_bwd_umma.cu), bare C-ABI call
        from cor_b200 import _lib as L
        lib = L.load()
        Nq = 1024
        q16 = torch.nn.functional.normalize(torch.randn(Nq, D, device=dev, generator=g), dim=-1).bfloat16()
        tg = (torch.arange(Nq, device=dev) * 97) % Nr
        _, lse = ops._sim_forward(r16, q16, 1.0 / 0.07, False, True, "umma")
        gl = torch.ones(1, device=dev)
        gq, gr = torch.empty(Nq, D, device=dev), torch.empty(Nr, D, device=dev)
        work = ops._work(lib.cor_infonce_bwd_umma_work_bytes(Nq, Nr, D), dev)
        med, best = timed(lambda: ops._call("cor_infonce_bwd_umma", dev, ops.ptr(r16), ops.ptr(q16), Nr, Nq, D, ops._f(1.0 / 0.07), ops.ptr(lse),
                                            ops.ptr(tg), ops.ptr(gl), ops._f(1.0), ops.ptr(gr), ops.ptr(gq), ops.ptr(work)), n=5)
        fl = 8.0 * Nq * Nr * D           # S recomputed for each product + the two products
        out["nce_bwd_umma_kernel_1024x102400"] = {"what": "InfoNCE backward dQ + dR on tcgen05: S tile recomputed, P formed in registers and fed back through "
                                                          "shared memory; no S, no P in HBM, no library GEMM", "bound": "tensor", "ms": med, "ms_best": best,
                                                  "flops": fl, "achieved_tflops": fl / (med * 1e-3) / 1e12, "peak": tc_burst, "unit": "TFLOP/s",
                                                  "frac": fl / (med * 1e-3) / 1e12 / tc_burst}
        del gq, gr, work
    except Exception as e:  # noqa: BLE001
        out["nce_bwd_umma_kernel_1024x102400"] = {"error": f"{type(e).__name__}: {e}"[:200]}
    try:   # the segmentation loss alone (what train_stage calls every step, utils/loss_func.py:5-32), CUDA-graph replay
        for Bs in (16, 128):
            pred = torch.randn(Bs, 1, 256, 256, device=dev, generator=g).bfloat16()
            mask = (torch.rand(Bs, 1, 1024, 1024, device=dev, generator=g) > 0.5).float()
            for _ in range(3):
                ops.seg_loss(pred, mask)
            torch.cuda.synchronize()
            gph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gph):
                ops.seg_loss(pred, mask)
            med, best = timed(gph.replay)
            alg, sect = Bs * 65536 * 18, Bs * 65536 * 34
            out[f"seg_loss_fwd_B{Bs}"] = {"what": "wbce_with_wiou_loss forward incl. the 1024->256 target resample: strip kernel + finalize (+ the wrapper's two "
                                                  "8-float copies), one graph replay", "bound": "hbm", "ms": med, "ms_best": best, "algorithmic_bytes": alg,
                                          "sector_floor_bytes": sect, "achieved_gbs": alg / (med * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                          "frac": alg / (med * 1e-3) / 1e9 / hbm_peak, "frac_of_sector_floor": sect / (med * 1e-3) / 1e9 / hbm_peak}
            del gph, pred, mask
    except Exception as e:  # noqa: BLE001
        out["seg_loss_fwd"] = {"error": f"{type(e).__name__}: {e}"[:200]}
    try:
        gal = r32[:4096].contiguous()
        qs = torch.nn.functional.normalize(torch.randn(256, D, device=dev, generator=g), dim=-1)
        med, best = timed(lambda: ops.topk_retrieve(gal, qs, 10))
        out["topk_256x4096_k10"] = {"what": "BASELINE configs[2]: similarity + radix select + exact re-score + sort (public op)", "ms": med,
                                    "ms_best": best, "queries_per_s": 256 / (med * 1e-3)}
    except Exception as e:  # noqa: BLE001
        out["topk_256x4096_k10"] = {"error": f"{type(e).__name__}: {e}"[:200]}
    del flush
    torch.cuda.empty_cache()
    return out


_RESULT_FD = None


def quiet_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner on stdout when
    NCCL_DEBUG=VERSION comes from the environment or from /etc/nccl.conf), so file descriptor 1 is pointed at stderr for
    the whole run and the result line goes to the saved descriptor."""
    global _RESULT_FD
    if _RESULT_FD is None:
        sys.stdout.flush()
        _RESULT_FD = os.dup(1)
        os.dup2(2, 1)


def emit_result(line):
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    if _RESULT_FD is None:
        os.write(1, data)
    else:
        os.write(_RESULT_FD, data)


DUMP_SAMPLE = 1 << 20      # elements kept of an output larger than this: a fixed, seeded sample (bounds the dump to a few 4 MB files)


def dump_outputs(out_dir, loss, grads):
    """What one timed step hands its caller -- the loss and the gradients of pred, comb and emb -- as float32
    DIR/<name>.npy, so that two builds can be compared output for output on the same seeded inputs.  An output with
    more than DUMP_SAMPLE elements is stored as the flat sample at sorted indices drawn once from a generator seeded
    with 0: the same positions in every run of the same configuration."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": loss.detach().float().reshape(1)}
    arrays.update({f"grad_{k}": g.detach().float() for k, g in sorted(grads.items()) if g is not None})
    for name, t in arrays.items():
        a = t.cpu().numpy()
        if a.size > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(0).choice(a.size, DUMP_SAMPLE, replace=False))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float32))
        print(f"[bench] {name}: {tuple(t.shape)} -> {out_dir}/{name}.npy {a.shape}", file=sys.stderr)


def main():
    quiet_stdout()
    ap_ = argparse.ArgumentParser()
    ap_.add_argument("--gpus", type=int, default=1)
    ap_.add_argument("--steps", type=int, default=20)
    ap_.add_argument("--warmup", type=int, default=3)
    ap_.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap_.add_argument("--mask-dtype", default="f32", choices=["f32", "u8"])
    ap_.add_argument("--batch", type=int, default=CFG["B"])
    ap_.add_argument("--masks", type=int, default=CFG["M"])
    ap_.add_argument("--cpu-triplets", type=int, default=16, help="triplets per CPU-baseline step (default: the whole 16-triplet batch)")
    ap_.add_argument("--cpu-iters", type=int, default=3)
    ap_.add_argument("--no-cpu-baseline", action="store_true")
    ap_.add_argument("--no-e2e", action="store_true", help="profiling runs only: skip the host-buffer leg")
    ap_.add_argument("--no-graph", action="store_true", help="time eager launches instead of the captured CUDA graph")
    ap_.add_argument("--no-u8-variant", action="store_true", help="skip the extra uint8-mask leg reported under 'variants'")
    ap_.add_argument("--no-secondary", action="store_true", help="skip the extra tensor-core / top-k kernel lines (N=1 only)")
    ap_.add_argument("--pool-engine", default="auto")
    ap_.add_argument("--sim-engine", default="auto")
    ap_.add_argument("--dump-outputs", metavar="DIR", help="write the loss and gradients of the last timed step as DIR/<name>.npy "
                                                           "(rank 0; outputs above 2^20 elements as a fixed, seeded sample).  --impl ours "
                                                           "only: the reference arm draws its inputs on the host, from another generator and "
                                                           "in fp32, so its outputs would not line up element for element with these")
    args = ap_.parse_args()
    if args.steps < 1:
        ap_.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap_.error("--dump-outputs writes what --impl ours computed (the reference arm's inputs differ; see --help)")
    cfg = dict(CFG, B=args.batch, M=args.masks)
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args, cfg)

    import torch.distributed as dist
    from cor_b200 import ops, region

    rank, world, local = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a B200: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"      # keep NCCL's banner off stdout (env beats /etc/nccl.conf)
        dist.init_process_group("nccl", device_id=dev)
    trace("init done")
    hbm_peak, tc_peak, tc_burst, peak_kind = peaks()

    inp = device_inputs(dev, 1234 + rank, cfg, args.mask_dtype)
    trace("inputs ready")
    kw = dict(tau=cfg["tau"], gather=world > 1, pool_engine=args.pool_engine, sim_engine=args.sim_engine)
    bufs = region.StepBuffers(cfg["B"], cfg["M"], cfg["C"], cfg["h"], cfg["w"], cfg["H"], cfg["W"], cfg["hp"], cfg["wp"], device=dev,
                              mask_dtype=inp["masks"].dtype)
    bufs.load(inp)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- CPU baseline first (rank 0, N=1 only), on a bounded sample of the same tensors
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        host_small = {k: v[:args.cpu_triplets].cpu() for k, v in inp.items()}
        cpu, _ = cpu_baseline(host_small, cfg, args.cpu_triplets, args.cpu_iters)

    trace("eager warm-up")
    # ---- warm-up (eager), then capture fwd+bwd of the step into one CUDA graph
    for _ in range(args.warmup):
        bufs._step(True, True, kw)
    barrier()
    trace("capture")
    graphed = False
    if not args.no_graph:
        try:
            bufs.capture(backward=True, emb_grad=True, warmup=1, **kw)
            graphed = True
        except Exception as e:  # e.g. a collective that cannot be captured: stay eager, say so
            print(f"[bench] CUDA-graph capture failed ({type(e).__name__}: {e}); timing eager launches", file=sys.stderr)
            bufs.graph = None
            torch.cuda.synchronize()

    def eager_step():
        bufs.loss, bufs.grads = bufs._step(True, True, kw)
        return bufs.loss

    step = bufs.replay if graphed else eager_step
    for _ in range(2):
        step()
    barrier()

    trace("timed loop")
    # ---- device-resident throughput: EXACTLY K steps between events, max over ranks
    n0 = ops.LAUNCHES["count"]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.profiler.start()     # ncu --profile-from-start off captures only the timed region
    clk = ClockSampler(local)       # samples nvidia-smi every 200 ms from here to the end of the e2e leg (GPU busy throughout)
    clk.__enter__()
    e0.record()
    for _ in range(args.steps):
        loss = step()
    e1.record()
    barrier()
    torch.cuda.profiler.stop()
    launches = ops.LAUNCHES["count"] - n0
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_step = float(ms) / args.steps
    value = cfg["B"] * world / (ms_step * 1e-3)
    if args.dump_outputs and rank == 0:     # before any later leg replays the step into the same buffers
        dump_outputs(args.dump_outputs, loss, bufs.grads)

    trace("events pass")
    # ---- per-kernel durations: the same K steps once more, eager, with CUDA events around every C-ABI call
    #      (single stream: COR_STEP_OVERLAP=0 keeps the segmentation-loss branch from running underneath the kernels being
    #      timed, so every duration is that kernel alone; the timed region above runs with the branch overlapped)
    ops.TIMING["events"] = {}
    prev_overlap = os.environ.get("COR_STEP_OVERLAP")
    os.environ["COR_STEP_OVERLAP"] = "0"
    for _ in range(args.steps):
        bufs._step(True, True, kw)
    barrier()
    if prev_overlap is None:
        os.environ.pop("COR_STEP_OVERLAP")
    else:
        os.environ["COR_STEP_OVERLAP"] = prev_overlap
    events, ops.TIMING["events"] = ops.TIMING["events"], None
    per_kernel = {k: sum(a.elapsed_time(b) for a, b in v) / args.steps for k, v in events.items()}   # ms per step
    calls = {k: len(v) // args.steps for k, v in events.items()}

    # ---- roofline of the dominant kernel (mask_prep: one pass over the full-resolution masks)
    esz = 4 if args.mask_dtype == "f32" else 1
    n_masks, P = cfg["B"] * cfg["M"], cfg["h"] * cfg["w"]
    prep_bytes = n_masks * cfg["H"] * cfg["W"] * esz + n_masks * P * (2 + 4) + n_masks * 16   # masks in; bf16 + f32 weights, stats out
    dom = max(per_kernel, key=per_kernel.get)
    prep_ms = per_kernel.get("cor_mask_prep", 0.0) / max(1, calls.get("cor_mask_prep", 1))
    achieved = prep_bytes / (prep_ms * 1e-3) / 1e9 if prep_ms > 0 else 0.0
    traffic, traffic_src = traffic_from_profiles(cfg, args.mask_dtype)
    roofline = {"kernel": "mask_prep_kernel (cor_mask_prep)", "bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                "frac": achieved / hbm_peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": f"{peak_kind} (MEASURED_PEAKS.json hbm_gbs)",
                "algorithmic_bytes_per_launch": prep_bytes, "ms_per_launch": prep_ms,
                "share_of_kernel_time": per_kernel.get("cor_mask_prep", 0.0) / max(1e-9, sum(per_kernel.values())),
                "dominant_by_events": dom, "timed": "CUDA events around the C-ABI call, eager pass over the same K steps"}
    pool_ms = per_kernel.get("cor_pool_umma_fwd", 0.0)
    pool_bytes = cfg["B"] * (cfg["C"] * P * 2 + (cfg["M"] + 16) // 16 * 16 * P * 2)
    secondary = {"pool_umma_kernel": {"bound": "hbm", "algorithmic_bytes": pool_bytes, "ms": pool_ms,
                                      "achieved_gbs": pool_bytes / (pool_ms * 1e-3) / 1e9 if pool_ms > 0 else None,
                                      "flops": 2.0 * cfg["B"] * cfg["M"] * P * cfg["C"]}}

    if args.no_e2e:
        clk.__exit__()
        if rank == 0:
            emit_result({"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "ms_per_step": ms_step, "e2e": None,
                              "roofline": roofline, "kernel_ms_per_step": per_kernel, "gpu_launches": launches, "graphed": graphed,
                              "note": "profiling run"})
        if world > 1:
            bufs.graph = None
            barrier()
            os._exit(0)
        return

    trace("e2e")
    # ---- end to end through the public API with host buffers (H2D of the step's inputs + D2H of the loss)
    numa = bind_to_gpu_numa(local) if world > 1 else {"cpus": None, "numa_node": None, "how": None}
    # platform ceiling of this leg: a bare pinned H2D copy on every GPU at once (same NUMA binding, same moment)
    barrier()
    pcie = torch.tensor([pcie_h2d_gbs(dev)], device=dev)
    pcie_all = [pcie.clone() for _ in range(world)]
    if world > 1:
        dist.all_gather(pcie_all, pcie)
    pcie_all = [round(float(x), 2) for x in pcie_all]
    host = {k: torch.empty(v.shape, dtype=v.dtype, pin_memory=True) for k, v in inp.items()}
    for k in host:
        host[k].copy_(inp[k])
    torch.cuda.synchronize()
    e2e_steps = max(3, min(args.steps, 10))
    for _ in range(2):
        bufs.run(host, **kw)
    barrier()
    t0 = time.perf_counter()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    marks = [torch.cuda.Event(enable_timing=True) for _ in range(e2e_steps + 1)]
    s0.record()
    marks[0].record()
    for i in range(e2e_steps):
        bufs.run(host, **kw)
        marks[i + 1].record()
    s1.record()
    barrier()
    wall = (time.perf_counter() - t0) / e2e_steps
    per_step = [round(marks[i].elapsed_time(marks[i + 1]), 2) for i in range(e2e_steps)]      # diagnosis only: the value is the mean
    # how much of a step is the copy: the same loads alone, events around them (max over ranks)
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    for _ in range(3):
        bufs.load(host)
    c1.record()
    barrier()
    h2d_t = torch.tensor([c0.elapsed_time(c1) / 3], device=dev)
    if world > 1:
        dist.all_reduce(h2d_t, op=dist.ReduceOp.MAX)
    h2d_ms = float(h2d_t)
    e2e_ms = torch.tensor([max(s0.elapsed_time(s1) / e2e_steps, wall * 1e3)], device=dev)
    if world > 1:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_val = cfg["B"] * world / (float(e2e_ms) * 1e-3)
    clk.__exit__()

    # ---- variant (reported, not the headline): the same masks shipped as uint8 -- bit-identical values after the
    #      kernel's /255 (what an 8-bit PNG holds before ToTensor, utils/dataloader.py:190), a quarter of the bytes
    variants = {}
    if args.mask_dtype == "f32" and not args.no_u8_variant:     # every rank runs it symmetrically (the step gathers negatives at N > 1)
        try:
            inp8 = dict(inp, masks=(inp["masks"] * 255).to(torch.uint8))
            b8 = region.StepBuffers(cfg["B"], cfg["M"], cfg["C"], cfg["h"], cfg["w"], cfg["H"], cfg["W"], cfg["hp"], cfg["wp"], device=dev,
                                    mask_dtype=torch.uint8)
            b8.load(inp8)
            b8.capture(backward=True, emb_grad=True, warmup=2, **kw)
            torch.cuda.synchronize()
            barrier()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            for _ in range(args.steps):
                b8.replay()
            a1.record()
            barrier()
            ms8 = torch.tensor([a0.elapsed_time(a1) / args.steps], device=dev)
            host8 = {k: torch.empty(v.shape, dtype=v.dtype, pin_memory=True).copy_(v) for k, v in inp8.items()}
            torch.cuda.synchronize()
            b8.run(host8, **kw)
            barrier()
            t8 = time.perf_counter()
            for _ in range(e2e_steps):
                b8.run(host8, **kw)
            barrier()
            w8 = torch.tensor([(time.perf_counter() - t8) / e2e_steps], device=dev)
            if world > 1:
                dist.all_reduce(ms8, op=dist.ReduceOp.MAX)
                dist.all_reduce(w8, op=dist.ReduceOp.MAX)
            ms8, w8 = float(ms8), float(w8)
            variants["u8_masks"] = {"what": "same step, masks shipped as uint8 (the 8-bit PNG bytes before ToTensor, utils/dataloader.py:187-197); "
                                            "the kernel's x/255 reproduces ToTensor bit for bit",
                                    "value": cfg["B"] * world / (ms8 * 1e-3), "ms_per_step": ms8,
                                    "e2e": {"value": cfg["B"] * world / w8, "unit": UNIT, "h2d_bytes_per_step": b8.h2d_bytes,
                                            "d2h_bytes_per_step": 4, "ms_per_step": w8 * 1e3}}
            b8.graph = None
            del b8, host8, inp8
        except Exception as e:   # the variant must never take the headline down with it
            variants["u8_masks"] = {"error": f"{type(e).__name__}: {e}"}

    eager_gpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        trace("torch eager on the GPU")
        eager_gpu = torch_eager_gpu_baseline(inp, cfg)
    if rank == 0 and world == 1 and not args.no_secondary:
        trace("secondary kernel lines")
        del inp
        torch.cuda.empty_cache()
        secondary.update(secondary_tensor_lines(dev, tc_burst, hbm_peak))

    trace("done")
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
                "data": "synthetic", "config": workload_config(cfg, args), "clocks": clk.summary(),
                "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": bufs.h2d_bytes, "d2h_bytes_per_step": 4,
                        "ms_per_step": float(e2e_ms), "steps": e2e_steps, "numa_local_cpus": numa["cpus"], "numa_node": numa["numa_node"],
                        "numa_how": numa["how"], "pcie_gbs_per_gpu": pcie_all,
                        "pcie_note": "8 back-to-back pinned cudaMemcpyAsync H2D copies of 1 GiB on every GPU at once, timed as one interval: the "
                                     "sustained platform ceiling of this leg (GPUs that share a PCIe uplink halve each other)",
                        "h2d_ms_per_step": h2d_ms, "per_step_ms_rank0": per_step, "frac_of_pcie_bound": (bufs.h2d_bytes / (min(pcie_all) * 1e9) * 1e3) / float(e2e_ms),
                        "pcie_bound_ms_per_step": bufs.h2d_bytes / (min(pcie_all) * 1e9) * 1e3},
                "gpu_launches": launches, "graphed": graphed, "roofline": roofline, "secondary_kernels": secondary, "variants": variants,
                "kernel_ms_per_step": {k: round(v, 4) for k, v in sorted(per_kernel.items(), key=lambda kv: -kv[1])},
                "loss": float(loss.detach())}
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if eager_gpu is not None:
            line["torch_eager_gpu"] = eager_gpu
        emit_result(line)
    if world > 1:
        # NCCL communicators captured in a CUDA graph can stall destroy_process_group(): release the
        # graph first, drain, and leave without the collective teardown.
        bufs.graph = None
        barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
