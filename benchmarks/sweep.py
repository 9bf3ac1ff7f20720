#!/usr/bin/env python
"""Per-kernel sweep on one B200 (BASELINE.json configs 3-5): CUDA-event time of ONE call after an L2 flush,
median of `--iters`, against the measured HBM / bf16 peaks.  Prints one JSON object per case.

    python benchmarks/sweep.py > profiles/rNN_sweep.jsonl
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from cor_b200 import ops, region  # noqa: E402


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), float(d["bf16_tflops"]), float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), "measured"
    return 6650.0, 1590.0, 1400.0, "fallback"


HBM, TC_BURST, TC_SUST, KIND = peaks()
FLUSH = None


def timeit(fn, iters, flush=True):
    global FLUSH
    if FLUSH is None:
        FLUSH = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        if flush:
            FLUSH.fill_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    ts.sort()
    return ts[len(ts) // 2] * 1e-3


def emit(name, t, bytes_=None, flops=None, **extra):
    d = {"case": name, "us": round(t * 1e6, 2)}
    if bytes_ is not None:
        d.update(bytes=int(bytes_), gbs=round(bytes_ / t / 1e9, 1), hbm_frac=round(bytes_ / t / 1e9 / HBM, 3))
    if flops is not None:
        d.update(flops=int(flops), tflops=round(flops / t / 1e12, 2), tc_frac_burst=round(flops / t / 1e12 / TC_BURST, 3))
    d.update(extra)
    d["peaks"] = KIND
    print(json.dumps(d), flush=True)


def unit(n, d, g):
    return torch.nn.functional.normalize(torch.randn(n, d, device="cuda", generator=g), dim=-1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=11)
    ap.add_argument("--only", default="")
    a = ap.parse_args()
    g = torch.Generator(device="cuda").manual_seed(0)
    want = lambda k: not a.only or a.only in k

    # ---- region pooling on tensor cores: masks/image 16-255, maps 64^2-128^2, C 256-1152 (config 5)
    if want("pool"):
        for (B, M, C, hw) in [(16, 16, 256, 64), (16, 64, 256, 64), (16, 100, 256, 64), (16, 256, 256, 64), (16, 64, 1152, 64),
                              (16, 64, 256, 128), (16, 256, 1152, 128), (10, 1, 256, 64)]:
            feat = torch.randn(B, C, hw, hw, device="cuda", generator=g).bfloat16()
            masks = (torch.rand(B, M, hw, hw, device="cuda", generator=g) > 0.7).to(torch.bfloat16)
            P = hw * hw
            eng = "umma" if M >= 16 else "stream"
            Rp = (M + 15) // 16 * 16          # no ones row: foreground rows only
            lib = ops.L.load()
            if eng == "umma":
                w16 = ops._umma_weight_buffer(feat.device, B, Rp, M, P, ones_row=False)
                ops.mask_prep(masks.reshape(B * M, hw, hw), (hw, hw), ops.W_CLAMP, want_f32=False, bf16_out=w16, group=M, group_stride=Rp * P)
                ks = lib.cor_pool_umma_ksplit(B, C, P)
                part = torch.empty((ks, B, Rp, C), dtype=torch.float32, device="cuda")
                fn = lambda: ops._call("cor_pool_umma_fwd", feat.device, ops.ptr(feat), ops.ptr(w16), B, C, P, Rp, ops.ptr(part))
                t = timeit(fn, a.iters)
                emit(f"pool_umma B{B} M{M} C{C} {hw}x{hw}", t, bytes_=B * (C * P * 2 + Rp * P * 2) + ks * B * Rp * C * 4,
                     flops=2.0 * B * Rp * P * C, ksplit=ks)
            else:
                w32, _ = ops.mask_prep(masks.reshape(B * M, hw, hw), (hw, hw), ops.W_CLAMP)
                fg = torch.empty(B, M, C, device="cuda")
                bg = torch.empty(B, M, C, device="cuda")
                fn = lambda: ops._call("cor_pool_stream_fwd", feat.device, ops.ptr(feat), ops.BF16, ops.ptr(w32), ops._ll(P), B, C, P, M,
                                       ops.W_CLAMP, ops.ptr(fg), ops.ptr(bg))
                t = timeit(fn, a.iters)
                emit(f"pool_stream(fg+bg) B{B} M{M} C{C} {hw}x{hw}", t, bytes_=B * (C * P * 2 + M * P * 4))
            del feat, masks

    # ---- similarity / InfoNCE / top-k (configs 3 and 4)
    if want("sim"):
        for (Nq, Nr, D, what) in [(256, 4096, 256, "S"), (256, 4096, 256, "lse"), (16, 102400, 256, "lse"), (1024, 102400, 256, "lse"),
                                  (128, 102400, 256, "lse"), (1024, 102400, 256, "S")]:
            R = unit(Nr, D, g).bfloat16()
            Q = unit(Nq, D, g).bfloat16()
            for eng in (["umma", "stream"] if Nq <= 16 else ["umma"]):
                fn = lambda: ops._sim_forward(R, Q, 1 / 0.07, what == "S", what == "lse", eng)
                t = timeit(fn, a.iters)
                by = (Nq + Nr) * D * 2 + (Nq * Nr * 4 if what == "S" else 0)
                emit(f"sim_{eng} {what} Nq{Nq} Nr{Nr} D{D}", t, bytes_=by, flops=2.0 * Nq * Nr * D)
        R = unit(4096, 256, g)
        Q = unit(256, 256, g)
        for k in (1, 10, 50):
            t = timeit(lambda: ops.topk_retrieve(R, Q, k), a.iters)
            emit(f"topk_retrieve (sim+select+rerank) Nq256 Nr4096 k{k}", t)

    # ---- InfoNCE forward + backward: tensor-core backward (nce_bwd_umma: coefficients formed in registers, no S / P written,
    #      no library GEMM) vs streaming backward
    if want("nce"):
        for (Nq, Nr, D) in [(256, 4096, 256), (1024, 102400, 256)]:
            R = unit(Nr, D, g).requires_grad_(True)
            Q = unit(Nq, D, g).requires_grad_(True)
            tg = (torch.arange(Nq, device="cuda") * 7) % Nr
            for eng in ("auto", "stream"):
                if eng == "stream" and Nq * Nr > (1 << 24):
                    iters = 3                      # the streaming backward takes milliseconds here
                else:
                    iters = a.iters

                def fn():
                    R.grad = Q.grad = None
                    ops.infonce_loss(R, Q, tg, tau=0.07, engine=eng).backward()
                t = timeit(fn, iters)
                emit(f"infonce fwd+bwd ({'dense' if eng == 'auto' else 'streaming'} backward) Nq{Nq} Nr{Nr} D{D}", t, flops=6.0 * Nq * Nr * D)

    # ---- segmentation loss, validation post-process
    if want("seg"):
        for B in (16, 128):
            pred = torch.randn(B, 1, 256, 256, device="cuda", generator=g).bfloat16()
            mask = (torch.rand(B, 1, 1024, 1024, device="cuda", generator=g) > 0.5).float()
            t = timeit(lambda: ops.seg_loss(pred, mask), a.iters)
            emit(f"seg_loss_fwd B{B} 256^2 <- 1024^2 f32 mask", t, bytes_=B * 256 * 256 * (2 + 16))
            pr = pred.clone().requires_grad_(True)
            loss = ops.seg_loss(pr, mask)
            t = timeit(lambda: loss.backward(retain_graph=True), a.iters)
            emit(f"seg_loss_bwd B{B}", t, bytes_=B * 256 * 256 * (2 + 4 + 4 + 2))
        pred = torch.randn(16, 1, 256, 256, device="cuda", generator=g).bfloat16()
        t = timeit(lambda: ops.val_postprocess(pred, size=(1024, 1024), want_hard=True), a.iters)
        emit("val_post B16 256^2 -> 1024^2 (f32 map + u8 mask)", t, bytes_=16 * 1024 * 1024 * 5)

    # ---- mask resample + sums at config-2 size
    if want("prep"):
        for dt, es in ((torch.float32, 4), (torch.uint8, 1)):
            n = 1024
            masks = (torch.rand(n, 1024, 1024, device="cuda", generator=g) > 0.5).to(dt)
            t = timeit(lambda: ops.mask_prep(masks, (64, 64), ops.W_CLAMP), a.iters, flush=False)
            emit(f"mask_prep n{n} 1024^2 {str(dt).split('.')[-1]} -> 64^2", t, bytes_=n * 1024 * 1024 * es + n * 4096 * 4)
            del masks


if __name__ == "__main__":
    main()
