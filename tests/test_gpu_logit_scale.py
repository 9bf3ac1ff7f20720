"""Learnable InfoNCE logit scale (``logit_scale=``): a 0-dim fp32 device tensor read by the kernels in place of 1/tau.

* The same fp32 value through the tensor gives the float path's results bit for bit, on every path of the step
  (one-launch tail, kernel chain, bg_mode 1, modular fp32 path) and of ``ops.infonce_loss`` (streaming, tensor-core).
* d loss / d s matches autograd through the fp64 oracle (``oracle.aten_port.infonce`` with a tensor temperature 1/s).
* It is right when nothing else needs a gradient, deterministic, and a captured graph picks up a new value per replay.
* The fused gather + similarity kernel gives the float entry's partials with a device scale (one-GPU lock-step).
* On >= 2 GPUs, the fused step's scale gradient on each rank matches the rank-local oracle (worker script)."""
import os
import socket
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TAU = 0.07


def dev():
    return torch.device("cuda:0")


def _bench_inputs():
    import bench
    return bench.device_inputs(dev(), 1234, dict(bench.CFG), "f32")


def _step(inp, monkeypatch, tail=True, tau=None, scale=None, scale_grad=False, seed=1.0, nce_weight=1.0,
          grad=("pred", "emb", "comb"), bg_mode=0, emb_dtype=None):
    """One region_step forward + backward: (loss parts, grads incl. "logit_scale", names of the library calls made)."""
    from cor_b200 import ops, region
    monkeypatch.setenv("COR_STEP_TAIL", "1" if tail else "0")
    calls = []
    real = ops._call

    def spy(name, *a):
        calls.append(name)
        return real(name, *a)

    monkeypatch.setattr(ops, "_call", spy)
    t = {k: inp[k].clone().requires_grad_(k in grad) for k in ("pred", "emb", "comb")}
    if emb_dtype is not None:
        t["emb"] = inp["emb"].to(emb_dtype).requires_grad_("emb" in grad)
    s = None
    if scale is not None:
        s = torch.tensor(scale, dtype=torch.float32, device=dev()).requires_grad_(scale_grad)
    kw = dict(logit_scale=s) if s is not None else dict(tau=tau)
    out = region.region_step(t["pred"], t["emb"], t["comb"], inp["masks"], gather=False, bg_mode=bg_mode, nce_weight=nce_weight, **kw)
    out.loss.backward(torch.tensor(seed, device=dev()))
    torch.cuda.synchronize()
    monkeypatch.setattr(ops, "_call", real)
    parts = {k: getattr(out, k).detach().clone() for k in ("loss", "seg", "fg", "bg", "nce")}
    parts["regions"] = out.regions.detach().clone()
    grads = {k: t[k].grad for k in t}
    grads["logit_scale"] = s.grad if s is not None else None
    return parts, grads, calls


def _oracle_scale_grad(regions, comb, s, g, nce_weight):
    """d (g * nce_weight * nce) / d s by autograd through the fp64 oracle, operands bf16-rounded as the kernels see them."""
    from oracle import aten_port as ap
    B, M, C = regions.shape
    R = regions.reshape(B * M, C).double().cpu()
    Q = comb.reshape(B, C).double().cpu()
    st = torch.tensor(float(s), dtype=torch.float64, requires_grad=True)
    nce = ap.infonce(R, Q, torch.arange(B) * M, tau=1.0 / st)
    (g * nce_weight * nce).backward()
    return float(st.grad)


# path name -> region_step options; every one keeps the step's own kernels for the InfoNCE
PATHS = {"tail": dict(tail=True), "chain": dict(tail=False), "bg_mode1": dict(bg_mode=1), "fp32_modular": dict(emb_dtype=torch.float32)}


@pytest.mark.parametrize("path", list(PATHS))
def test_same_value_same_bits(path, monkeypatch):
    inp = _bench_inputs()
    a = _step(inp, monkeypatch, tau=TAU, **PATHS[path])
    b = _step(inp, monkeypatch, scale=1.0 / TAU, **PATHS[path])
    import ctypes
    assert ctypes.c_float(1.0 / TAU).value == float(torch.tensor(1.0 / TAU, dtype=torch.float32))    # the same fp32 value
    for k in a[0]:
        assert torch.equal(a[0][k], b[0][k]), k
    for k in ("pred", "emb", "comb"):
        assert torch.equal(a[1][k], b[1][k]), k
    # same kernels, same launch counts: only the suffix of the InfoNCE entries differs
    assert [n[:-3] if n.endswith("_ls") else n for n in b[2]] == a[2]
    if path == "tail":
        assert "cor_step_tail_fwd_ls" in b[2] and "cor_step_tail_bwd_ls" in b[2]


@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("s", [1.0 / TAU, 5.0, 50.0])
def test_scale_gradient_matches_the_oracle(path, s, monkeypatch):
    inp = _bench_inputs()
    g, w = 0.7, 1.3
    p, gr, _ = _step(inp, monkeypatch, scale=s, scale_grad=True, seed=g, nce_weight=w, **PATHS[path])
    ref = _oracle_scale_grad(p["regions"], inp["comb"], s, g, w)
    got = float(gr["logit_scale"])
    assert abs(got - ref) <= 1e-3 * abs(ref), (got, ref)
    # the other gradients do not depend on whether the scale wants one
    _, g0, _ = _step(inp, monkeypatch, scale=s, scale_grad=False, seed=g, nce_weight=w, **PATHS[path])
    for k in ("pred", "emb", "comb"):
        assert torch.equal(gr[k], g0[k]), k


@pytest.mark.parametrize("path", ["tail", "chain"])
def test_only_the_scale_needs_a_gradient_and_runs_repeat(path, monkeypatch):
    inp = _bench_inputs()
    full = _step(inp, monkeypatch, scale=12.0, scale_grad=True, **PATHS[path])[1]["logit_scale"]
    only = [_step(inp, monkeypatch, scale=12.0, scale_grad=True, grad=(), **PATHS[path]) for _ in range(2)]
    assert torch.equal(only[0][1]["logit_scale"], only[1][1]["logit_scale"]), "two runs differ"
    assert torch.equal(only[0][1]["logit_scale"], full)
    if path == "tail":
        assert "cor_step_tail_bwd_ls" in only[0][2]


def _nce_case(Nq, Nr, D, seed):
    g = torch.Generator(device=dev()).manual_seed(seed)
    R = torch.nn.functional.normalize(torch.randn(Nr, D, device=dev(), generator=g), dim=-1)
    Q = torch.nn.functional.normalize(torch.randn(Nq, D, device=dev(), generator=g), dim=-1)
    T = torch.randint(0, Nr, (Nq,), device=dev(), generator=g)
    return R, Q, T


# (engine, Nq, Nr, D): the streaming backward, and a shape the dense tensor-core backward takes
NCE = {"stream": ("stream", 16, 4096, 256), "umma": ("umma", 256, 8192, 256)}


def _nce(case, tau=None, scale=None, scale_grad=False, need=(True, True), g=1.0):
    from cor_b200 import ops
    eng, Nq, Nr, D = NCE[case]
    R, Q, T = _nce_case(Nq, Nr, D, 5)
    r, q = R.clone().requires_grad_(need[0]), Q.clone().requires_grad_(need[1])
    s = torch.tensor(scale, dtype=torch.float32, device=dev()).requires_grad_(scale_grad) if scale is not None else None
    loss = ops.infonce_loss(r, q, T, tau=tau, engine=eng, logit_scale=s)
    loss.backward(torch.tensor(g, device=dev()))
    torch.cuda.synchronize()
    return loss.detach(), r.grad, q.grad, (s.grad if s is not None else None), (R, Q, T)


@pytest.mark.parametrize("case", list(NCE))
def test_infonce_loss_scale(case):
    from cor_b200 import ops
    eng, Nq, Nr, D = NCE[case]
    assert ops._infonce_bwd_dense(Nq, Nr, D, eng) == (case == "umma")
    a = _nce(case, tau=TAU)
    b = _nce(case, scale=1.0 / TAU)
    for x, y, nm in zip(a[:3], b[:3], ("loss", "g_regions", "g_queries")):
        assert torch.equal(x, y), nm
    from oracle import aten_port as ap
    R, Q, T = a[4]
    for s in (1.0 / TAU, 5.0, 50.0):
        c = _nce(case, scale=s, scale_grad=True, g=0.7)
        st = torch.tensor(s, dtype=torch.float64, requires_grad=True)
        (0.7 * ap.infonce(R.double().cpu(), Q.double().cpu(), T.cpu(), tau=1.0 / st)).backward()
        ref = float(st.grad)
        assert abs(float(c[3]) - ref) <= 1e-3 * abs(ref), (s, float(c[3]), ref)
        d = _nce(case, scale=s, g=0.7)
        assert torch.equal(c[1], d[1]) and torch.equal(c[2], d[2]), "region / query gradients changed"
    # only the scale wants a gradient (the dense backward then runs the dQ GEMM without storing it); deterministic
    e = [_nce(case, scale=20.0, scale_grad=True, need=(False, False)) for _ in range(2)]
    f = _nce(case, scale=20.0, scale_grad=True)
    assert torch.equal(e[0][3], e[1][3]) and torch.equal(e[0][3], f[3])


def test_graph_replay_reads_the_scale_every_replay():
    """Capture once with logit_scale=s, then s.fill_(v) + replay for two values: bit-equal to an eager step at v."""
    from cor_b200 import region
    import bench
    cfg = bench.CFG
    inp = _bench_inputs()
    mk = lambda: region.StepBuffers(cfg["B"], cfg["M"], cfg["C"], cfg["h"], cfg["w"], cfg["H"], cfg["W"], cfg["hp"], cfg["wp"],
                                    device=dev(), emb_dtype=torch.bfloat16)
    ref_bufs = mk()
    ref_bufs.load(inp)
    ref_bufs.capture(tau=TAU, gather=False)
    bufs = mk()
    bufs.load(inp)
    s = torch.tensor(1.0 / TAU, dtype=torch.float32, device=dev())
    bufs.capture(logit_scale=s, gather=False)
    assert bufs.launches_per_step == ref_bufs.launches_per_step
    ref_bufs.replay()
    bufs.replay()
    torch.cuda.synchronize()
    assert torch.equal(bufs.loss, ref_bufs.loss)             # the same value as the float path's capture, bit for bit
    for k in ("pred", "comb", "emb"):
        assert torch.equal(bufs.grads[k], ref_bufs.grads[k]), k
    got = {}
    for v in (9.0, 31.0):
        s.fill_(v)
        bufs.replay()
        torch.cuda.synchronize()
        got[v] = (bufs.loss.clone(), {k: t.clone() for k, t in bufs.grads.items()})
    for v, (loss, grads) in got.items():
        loss_e, grads_e = bufs._step(True, True, dict(logit_scale=torch.tensor(v, dtype=torch.float32, device=dev()), gather=False))
        torch.cuda.synchronize()
        assert torch.equal(loss.reshape(()), loss_e.reshape(())), v
        assert set(grads) == {"pred", "comb", "emb", "logit_scale"}
        for k in grads:
            assert torch.equal(grads[k], grads_e[k]), (v, k)
    assert not torch.equal(got[9.0][1]["logit_scale"], got[31.0][1]["logit_scale"])


def test_peer_gather_sim_with_a_device_scale():
    """Lock-step emulation of two ranks on one GPU (as tests/test_gpu_peer.py): the _ls entry, given the same value
    through device memory, leaves the same gathered rows and bit-equal log-sum-exp partials as the float entry."""
    import ctypes as C_
    from cor_b200 import _lib as L, ops
    from test_gpu_peer import _VirtualRank
    lib = L.load()
    os.environ.setdefault("COR_PEER_TIMEOUT_S", "5")
    world, n, Cc = 2, 96, 64
    flags = [torch.zeros(lib.cor_peer_flag_bytes() // 4, dtype=torch.int32, device=dev()) for _ in range(world)]
    pubs = [torch.zeros(n, Cc, dtype=torch.bfloat16, device=dev()) for _ in range(world)]
    galls = [torch.zeros(world * n, Cc, dtype=torch.float32, device=dev()) for _ in range(world)]
    ranks = [_VirtualRank(r, world, n, Cc, flags, pubs, galls) for r in range(world)]
    g = torch.Generator(device=dev()).manual_seed(7)
    rows = [torch.randn(n, Cc, device=dev(), generator=g).bfloat16() for _ in range(world)]
    q16 = torch.nn.functional.normalize(torch.randn(11, Cc, device=dev(), generator=g), dim=-1).bfloat16()
    scale = torch.tensor(1.0 / TAU, dtype=torch.float32, device=dev())
    results = []
    for it, use_scale in enumerate((False, True)):
        for r in ranks:
            if it > 0:
                r.ctl("cor_peer_wait_exit", 0)           # the same channel twice in a row
            r.pub.copy_(rows[r.rank])
            r.ctl("cor_peer_signal", 0)
        epoch = []
        for r in ranks:
            out = torch.empty((world * n, Cc), dtype=torch.bfloat16, device=dev())
            work = torch.zeros(lib.cor_peer_gather_sim_work_bytes() // 4, dtype=torch.float32, device=dev())
            nparts = C_.c_int(0)
            name, ta = ops._tau_arg("cor_peer_gather_sim", 1.0 / TAU, scale if use_scale else None)
            ops._call(name, dev(), ops.ptr(r.pub_ptrs), ops.ptr(out), ops._ll(n), Cc, ops.ptr(q16), int(q16.shape[0]), ta, ops.ptr(work),
                      C_.byref(nparts), ops.ptr(r.flag_ptrs), ops.ptr(r.state), r.rank, world, 0)
            epoch.append((out, work[:nparts.value * 16 * 2].clone()))
        results.append(epoch)
    torch.cuda.synchronize()
    for r in ranks:
        assert int(r.state[r.err_word].item()) == 0, "a wait expired"
    for (o0, p0), (o1, p1) in zip(*results):
        assert torch.equal(o0, o1) and torch.equal(p0, p1)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_multi_rank_scale_gradient_is_rank_local():
    n = min(torch.cuda.device_count(), 8)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "_logit_scale_worker.py")]
    r = subprocess.run(cmd, cwd=ROOT, env=dict(os.environ, NCCL_DEBUG="WARN"), capture_output=True, text=True, timeout=240)
    assert r.returncode == 0 and "LOGIT_SCALE_OK" in r.stdout, r.stdout[-3000:] + "\n" + r.stderr[-3000:]
