"""A/B of the learnable InfoNCE logit scale against the float temperature, alternated in one run.

Step: the benchmark's shape (16 triplets x 64 masks, C = 256, bf16 features, fp32 masks), each arm captured once in a
CUDA graph and replayed; ms/step from CUDA events over `--steps` replays, the three arms interleaved `--rounds` times:
    tau      region_step(tau=0.07)                          (the float path)
    ls       region_step(logit_scale=s), s without grad
    ls_grad  region_step(logit_scale=s), s with grad        (gradient in grads["logit_scale"])
InfoNCE: ops.infonce_loss forward + backward at 1024 queries x 102 400 regions x 256 (the tensor-core forward and
backward), with tau, and with a scale with and without its gradient.  Prints one JSON line per measurement, then the GPU
name and power limit.

    python benchmarks/logit_scale_ab.py [--steps 200] [--rounds 3]
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    import bench
    from cor_b200 import ops, region
    dev = torch.device("cuda:0")
    cfg = dict(bench.CFG)
    inp = bench.device_inputs(dev, 1234, cfg, "f32")
    s = torch.tensor(1.0 / cfg["tau"], dtype=torch.float32, device=dev)
    arms = {"tau": dict(tau=cfg["tau"]), "ls": dict(logit_scale=s), "ls_grad": dict(logit_scale=s)}
    bufs = {}
    for name, kw in arms.items():
        b = region.StepBuffers(cfg["B"], cfg["M"], cfg["C"], cfg["h"], cfg["w"], cfg["H"], cfg["W"], cfg["hp"], cfg["wp"], device=dev,
                               emb_dtype=torch.bfloat16, mask_dtype=inp["masks"].dtype)
        b.load(inp)
        if name == "ls":
            # the scale without grad: StepBuffers always asks for its gradient, so this arm runs its own step body
            def _no_grad_scale(backward, emb_grad, kw, _b=b):
                kw = dict(kw)
                sc = kw.pop("logit_scale")
                pred = _b.d["pred"].detach().requires_grad_(backward)
                comb = _b.d["comb"].detach().requires_grad_(backward)
                emb = _b.d["emb"].detach().requires_grad_(backward and emb_grad)
                out = region.region_step(pred, emb, comb, _b.d["masks"], logit_scale=sc.detach(), **kw)
                if backward:
                    out.loss.backward(gradient=_b._seed)
                return out.loss.detach(), {"pred": pred.grad, "comb": comb.grad, "emb": emb.grad}
            b._step = _no_grad_scale
        b.capture(backward=True, emb_grad=True, warmup=2, gather=False, **kw)
        bufs[name] = b
    for name, b in bufs.items():
        time_replays(b, 20)
    launches = {name: b.launches_per_step for name, b in bufs.items()}
    for r in range(args.rounds):
        for name, b in bufs.items():
            ms = time_replays(b, args.steps)
            print(json.dumps({"what": "step", "arm": name, "round": r, "ms_per_step": round(ms, 4), "launches_per_step": launches[name],
                              "grads": sorted(k for k, v in b.grads.items() if v is not None)}), flush=True)
    del bufs
    torch.cuda.empty_cache()
    # ops.infonce_loss at 1024 x 102 400 x 256
    g = torch.Generator(device=dev).manual_seed(7)
    Nq, Nr, D = 1024, 102400, 256
    R = torch.nn.functional.normalize(torch.randn(Nr, D, device=dev, generator=g), dim=-1)
    Q = torch.nn.functional.normalize(torch.randn(Nq, D, device=dev, generator=g), dim=-1)
    T = torch.randint(0, Nr, (Nq,), device=dev, generator=g)
    r16 = R.bfloat16()

    def nce(kind):
        r, q = R.detach().requires_grad_(True), Q.detach().requires_grad_(True)
        if kind == "tau":
            loss = ops.infonce_loss(r, q, T, tau=0.07, regions_bf16=r16)
        else:
            sc = s.detach().requires_grad_(kind == "ls_grad")
            loss = ops.infonce_loss(r, q, T, regions_bf16=r16, logit_scale=sc)
        loss.backward()

    kinds = ("tau", "ls", "ls_grad")
    for k in kinds:
        for _ in range(3):
            nce(k)
    torch.cuda.synchronize()
    for r in range(args.rounds):
        for k in kinds:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(10):
                nce(k)
            b.record()
            torch.cuda.synchronize()
            print(json.dumps({"what": "infonce_fwd_bwd_1024x102400x256", "arm": k, "round": r, "ms": round(a.elapsed_time(b) / 10, 4)}),
                  flush=True)
    print(json.dumps(gpu_info()), flush=True)


if __name__ == "__main__":
    main()
