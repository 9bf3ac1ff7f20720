"""Per-kernel device time of the benched step (bench.py's batch, eager launches) from torch.profiler's CUDA activity.

    python benchmarks/step_profile.py [--steps 20] [--out profiles/<name>.csv]

Prints (and writes as CSV) microseconds per step for every kernel name, in order of first launch, plus the kernel count.
Run once per setting of a COR_* knob to compare two kernel chains; the tracing slows the host, so take step times from
bench.py, not from here."""
import argparse
import collections
import csv
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out")
    a = ap.parse_args()
    import bench
    from cor_b200 import region
    cfg = dict(bench.CFG)
    dev = torch.device("cuda:0")
    inp = bench.device_inputs(dev, 1234, cfg, "f32")
    bufs = region.StepBuffers(cfg["B"], cfg["M"], cfg["C"], cfg["h"], cfg["w"], cfg["H"], cfg["W"], cfg["hp"], cfg["wp"], device=dev,
                              mask_dtype=inp["masks"].dtype)
    bufs.load(inp)
    kw = dict(tau=cfg["tau"], gather=False)
    for _ in range(3):
        bufs._step(True, True, kw)
    torch.cuda.synchronize()
    acts = [torch.profiler.ProfilerActivity.CUDA]
    with torch.profiler.profile(activities=acts) as prof:
        for _ in range(a.steps):
            bufs._step(True, True, kw)
        torch.cuda.synchronize()
    dur, cnt = collections.OrderedDict(), collections.Counter()
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA or ev.name.startswith(("Memcpy", "Memset")):
            continue
        name = ev.name.split("(")[0].replace("void ", "").replace("cor::", "")[:80]
        dur[name] = dur.get(name, 0.0) + ev.device_time
        cnt[name] += 1
    rows = [(k, v / a.steps, cnt[k] / a.steps) for k, v in dur.items()]
    tot = sum(r[1] for r in rows)
    print(f"COR_STEP_TAIL={os.environ.get('COR_STEP_TAIL', '1')} {torch.cuda.get_device_name(0)}")
    for k, us, n in rows:
        print(f"{us:9.1f} us/step  x{n:.0f}  {k}")
    print(f"{tot:9.1f} us/step total, {sum(r[2] for r in rows):.0f} kernels/step")
    if a.out:
        with open(a.out, "w", newline="") as f:
            w = csv.writer(f)
            w.writerow(["kernel", "us_per_step", "launches_per_step"])
            for k, us, n in rows:
                w.writerow([k, f"{us:.2f}", f"{n:.0f}"])


if __name__ == "__main__":
    main()
