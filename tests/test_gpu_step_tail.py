"""The fused step's one-launch region tail (csrc/step_tail.cu, ``COR_STEP_TAIL=1``, the default) against the kernel chain
it replaces (``COR_STEP_TAIL=0``) on the same inputs: the benchmark's own batch, a single triplet with an odd mask count
and C = 128, an empty ground-truth mask, an upstream gradient other than 1, inputs without gradients -- and which cases
keep the old chain."""
import pytest
import torch


def dev():
    return torch.device("cuda:0")


def relnorm(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def _step(inp, monkeypatch, tail, seed=1.0, grad=("pred", "emb", "comb"), bg_mode=0):
    """One region_step forward + backward; returns (loss parts, grads, names of the library calls made)."""
    from cor_b200 import ops, region
    monkeypatch.setenv("COR_STEP_TAIL", "1" if tail else "0")
    calls = []
    real = ops._call

    def spy(name, *a):
        calls.append(name)
        return real(name, *a)

    monkeypatch.setattr(ops, "_call", spy)
    t = {k: inp[k].clone().requires_grad_(k in grad) for k in ("pred", "emb", "comb")}
    out = region.region_step(t["pred"], t["emb"], t["comb"], inp["masks"], tau=0.07, gather=False, bg_mode=bg_mode)
    out.loss.backward(torch.tensor(seed, device=dev()))
    torch.cuda.synchronize()
    monkeypatch.setattr(ops, "_call", real)
    parts = {k: getattr(out, k).detach().clone() for k in ("loss", "seg", "fg", "bg", "nce")}
    parts["regions"] = out.regions.detach().clone()
    return parts, {k: t[k].grad for k in t}, calls


def _bench_inputs():
    import bench
    return bench.device_inputs(dev(), 1234, dict(bench.CFG), "f32")


def _synth_inputs(B, M, C, empty_gt=None):
    from cor_b200 import synth
    d = synth.make_triplets(83 + M, B=B, M=M, C=C, h=16, w=16, H=64, W=64, hp=32, wp=32, degenerate=False)
    if empty_gt is not None:
        d["masks"][empty_gt, 0] = 0.0
    t = {k: torch.from_numpy(v).to(dev()) for k, v in d.items()}
    t["emb"] = t["emb"].bfloat16()
    return t


def _compare(a, b):
    (pa, ga, _), (pb, gb, _) = a, b
    lo = float(pb["loss"])
    assert abs(float(pa["loss"]) - lo) <= 1e-6 * abs(lo), (float(pa["loss"]), lo)
    for k in ("seg", "fg", "bg", "nce"):
        assert abs(float(pa[k]) - float(pb[k])) <= 1e-6 * abs(float(pb[k])) + 1e-7, k
    assert relnorm(pa["regions"], pb["regions"]) < 1e-6
    if ga["pred"] is not None:
        assert torch.equal(ga["pred"], gb["pred"])
    if ga["comb"] is not None:
        assert relnorm(ga["comb"], gb["comb"]) <= 1e-5, relnorm(ga["comb"], gb["comb"])
    if ga["emb"] is not None:
        assert relnorm(ga["emb"].float(), gb["emb"].float()) <= 1e-3, relnorm(ga["emb"].float(), gb["emb"].float())


@pytest.mark.gpu
def test_bench_batch_tail_matches_kernel_chain_and_is_deterministic(monkeypatch):
    inp = _bench_inputs()
    new = _step(inp, monkeypatch, True)
    old = _step(inp, monkeypatch, False)
    assert "cor_step_tail_fwd" in new[2] and "cor_step_tail_bwd" in new[2]
    assert "cor_step_tail_fwd" not in old[2] and "cor_infonce_tail" in old[2]
    assert len(new[2]) < len(old[2])
    _compare(new, old)
    again = _step(inp, monkeypatch, True)
    for k in new[0]:
        assert torch.equal(new[0][k], again[0][k]), k
    for k in new[1]:
        assert torch.equal(new[1][k], again[1][k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("case", [(1, 17, 128, None, 1.0), (3, 20, 128, 1, 2.5), (4, 64, 256, 0, -0.75), (16, 255, 128, 5, 1.0)])
def test_small_shapes_tail_matches_kernel_chain(monkeypatch, case):
    B, M, C, empty_gt, seed = case
    inp = _synth_inputs(B, M, C, empty_gt)
    new = _step(inp, monkeypatch, True, seed=seed)
    old = _step(inp, monkeypatch, False, seed=seed)
    assert "cor_step_tail_bwd" in new[2]
    _compare(new, old)


@pytest.mark.gpu
@pytest.mark.parametrize("grad", [("pred", "comb"), ("pred", "emb"), ("pred",)])
def test_tail_without_emb_or_comb_gradients(monkeypatch, grad):
    inp = _synth_inputs(3, 20, 256, 1)
    new = _step(inp, monkeypatch, True, seed=1.5, grad=grad)
    old = _step(inp, monkeypatch, False, seed=1.5, grad=grad)
    for k in ("pred", "emb", "comb"):
        assert (new[1][k] is None) == (k not in grad)
    _compare(new, old)


@pytest.mark.gpu
def test_paired_bg_mode_keeps_the_kernel_chain(monkeypatch):
    inp = _synth_inputs(3, 20, 128, 1)
    _, _, calls = _step(inp, monkeypatch, True, bg_mode=1)
    assert not any(c.startswith("cor_step_tail") for c in calls)
    assert "cor_infonce_tail" in calls


def test_tail_eligibility(monkeypatch):
    """Host-side choice only: multi-rank gathering, bg_mode 1, more than 16 queries, wide rows, a forced tensor-core
    similarity and the knob keep today's kernels."""
    from cor_b200 import region
    monkeypatch.delenv("COR_STEP_TAIL", raising=False)
    assert region._step_tail_ok(16, 64, 256, False, 0, "auto")
    assert region._step_tail_ok(1, 17, 128, False, 0, "stream")
    assert not region._step_tail_ok(16, 64, 256, True, 0, "auto")
    assert not region._step_tail_ok(16, 64, 256, False, 1, "auto")
    assert not region._step_tail_ok(17, 64, 256, False, 0, "auto")
    assert not region._step_tail_ok(16, 64, 384, False, 0, "auto")
    assert not region._step_tail_ok(16, 64, 256, False, 0, "umma")
    assert not region._step_tail_ok(16, 1024, 256, False, 0, "auto")      # 16 384 rows: the tensor-core similarity's regime
    monkeypatch.setenv("COR_STEP_TAIL", "0")
    assert not region._step_tail_ok(16, 64, 256, False, 0, "auto")
