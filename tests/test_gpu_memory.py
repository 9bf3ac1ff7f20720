"""Cross-batch region memory (``region.RegionMemory``, ``memory=``): memory rows join every query's InfoNCE negatives.

* The ring: enqueue writes bf16 rows at (head + i) mod K and advances {head, count} exactly, across a wrap mid-batch.
* An empty memory changes no bit of the loss or any gradient, on ``ops.infonce_loss``, the one-launch tail and the chain.
* A filled memory matches the same call on cat(regions, memory rows) and an fp64 oracle (loss, queries, regions, scale).
* ``region_step`` with a full memory keeps its fused tail; the parts the memory does not touch are bit-equal.
* A backward after an enqueue raises; a captured graph replays eager steps bit for bit; two runs are bit-identical.
* On >= 2 GPUs each rank's loss and gradients match the rank-local oracle (worker script)."""
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


def _unit(n, D, g):
    return torch.nn.functional.normalize(torch.randn(n, D, device=dev(), generator=g), dim=-1)


def _filled(K, D, n_rows, seed=3):
    """A memory of capacity K after pushing n_rows unit rows in batches of at most K // 2 + 1 (wraps when n_rows > K)."""
    from cor_b200 import region
    m = region.RegionMemory(K, D, dev())
    g = torch.Generator(device=dev()).manual_seed(seed)
    left = n_rows
    while left > 0:
        n = min(left, max(1, K // 2 + 1))
        m.enqueue(_unit(n, D, g))
        left -= n
    return m


def oracle_nce(R, Q, T, mem, s, g=1.0):
    """fp64: mean_q (logsumexp_{r in R u mem} s <q, r> - s <q, R[t(q)]>) and its gradients (queries, regions, s); operands
    rounded to bf16 as the kernels see them, memory rows constant."""
    R64 = R.bfloat16().double().cpu().requires_grad_(True)
    Q64 = Q.bfloat16().double().cpu().requires_grad_(True)
    M64 = mem.double().cpu()
    st = torch.tensor(float(s), dtype=torch.float64, requires_grad=True)
    logits = st * (Q64 @ torch.cat([R64, M64]).t())
    loss = (torch.logsumexp(logits, 1) - logits[torch.arange(Q.shape[0]), T.cpu()]).mean()
    (g * loss).backward()
    return float(loss), Q64.grad, R64.grad, float(st.grad)


def rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).norm() / b.norm())


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_ring_slots_head_and_count(dtype):
    from cor_b200 import region
    K, C, n = 1000, 128, 384
    m = region.RegionMemory(K, C, dev())
    g = torch.Generator(device=dev()).manual_seed(1)
    ref = torch.zeros(K, C, dtype=torch.bfloat16, device=dev())
    head = count = 0
    for _ in range(5):
        rows = torch.randn(n, C, device=dev(), generator=g).to(dtype)
        m.enqueue(rows.view(3, n // 3, C))                  # any [..., C] shape
        slots = (head + torch.arange(n, device=dev())) % K   # the third and fifth batches wrap mid-batch
        ref[slots] = rows.to(torch.bfloat16)
        head, count = (head + n) % K, min(count + n, K)
        torch.cuda.synchronize()
        assert torch.equal(m.bank, ref)
        assert m.state[:2].tolist() == [head, count]
    assert m.count() == K
    assert torch.equal(m.rows(), torch.cat([ref[head:], ref[:head]]))
    m.reset()
    assert m.count() == 0 and m.rows().shape == (0, C)


def _nce(R, Q, T, memory=None, scale=None, g=1.0, engine="auto"):
    from cor_b200 import ops
    r, q = R.clone().requires_grad_(True), Q.clone().requires_grad_(True)
    s = torch.tensor(scale, dtype=torch.float32, device=dev(), requires_grad=True) if scale is not None else None
    kw = dict(logit_scale=s) if s is not None else dict(tau=TAU)
    loss = ops.infonce_loss(r, q, T, engine=engine, memory=memory, **kw)
    loss.backward(torch.tensor(g, device=dev()))
    torch.cuda.synchronize()
    return loss.detach(), r.grad, q.grad, (s.grad if s is not None else None)


@pytest.mark.parametrize("Nq,Nr,engine", [(16, 4096, "stream"), (256, 8192, "umma")])
def test_empty_memory_is_bit_equal_on_infonce_loss(Nq, Nr, engine):
    from cor_b200 import region
    g = torch.Generator(device=dev()).manual_seed(5)
    R, Q = _unit(Nr, 256, g), _unit(Nq, 256, g)
    T = torch.randint(0, Nr, (Nq,), device=dev(), generator=g)
    m = region.RegionMemory(4096, 256, dev())
    for scale in (None, 1.0 / TAU):
        a = _nce(R, Q, T, None, scale, engine=engine)
        b = _nce(R, Q, T, m, scale, engine=engine)
        for x, y in zip(a, b):
            assert (x is None and y is None) or torch.equal(x, y)


# (Nq, K, rows pushed): full, partly full, and full after a wrap (the head mid-ring)
FILL = [(Nq, K, n) for Nq in (1, 16, 64) for K, n in ((1, 1), (127, 127), (8192, 8192), (65536, 65536))]
FILL += [(16, 127, 60), (16, 8192, 5000), (64, 65536, 40000), (16, 8192, 8192 + 3000), (1, 127, 200)]


@pytest.mark.parametrize("Nq,K,n_rows", FILL)
def test_filled_memory_against_concatenation_and_oracle(Nq, K, n_rows):
    from cor_b200 import ops
    D, Nr = 256, 1024
    g = torch.Generator(device=dev()).manual_seed(11)
    R, Q = _unit(Nr, D, g), _unit(Nq, D, g)
    T = torch.randint(0, Nr, (Nq,), device=dev(), generator=g)
    m = _filled(K, D, n_rows)
    mem = m.rows()
    assert mem.shape[0] == min(K, n_rows)
    got = _nce(R, Q, T, m, scale=1.0 / TAU, g=0.7)
    # the same call on the concatenation (the memory rows exactly as stored); its region gradient's first Nr rows
    rc = torch.cat([R.bfloat16().float(), mem.float()])
    cat = _nce(rc, Q, T, None, scale=1.0 / TAU, g=0.7)
    loss, gq, gr, gs = oracle_nce(R, Q, T, mem, 1.0 / TAU, g=0.7)
    assert abs(float(got[0]) - loss) <= 1e-3 * abs(loss)
    assert abs(float(got[0]) - float(cat[0])) <= 1e-3 * abs(float(cat[0]))
    assert rel(got[2], gq) < 4e-3 and rel(got[2], cat[2]) < 4e-3
    assert rel(got[1], gr) < 4e-3 and rel(got[1], cat[1][:Nr]) < 4e-3
    assert abs(float(got[3]) - gs) <= 1e-3 * abs(gs)


@pytest.mark.parametrize("s", [1.0 / TAU, 50.0])
def test_scale_gradient_with_memory(s):
    g = torch.Generator(device=dev()).manual_seed(13)
    R, Q = _unit(1024, 256, g), _unit(16, 256, g)
    T = torch.arange(16, device=dev()) * 64
    m = _filled(8192, 256, 8192)
    got = _nce(R, Q, T, m, scale=s, g=0.7)
    ref = oracle_nce(R, Q, T, m.rows(), s, g=0.7)[3]
    assert abs(float(got[3]) - ref) <= 1e-3 * abs(ref), (float(got[3]), ref)


def _step(inp, monkeypatch, memory=None, tail=True, bg_mode=0, scale=None, seed=0.7):
    """region_step forward + backward at the bench shape: (parts, grads, library calls)."""
    from cor_b200 import ops, region
    monkeypatch.setenv("COR_STEP_TAIL", "1" if tail else "0")
    calls = []
    real = ops._call

    def spy(name, *a, **k):
        calls.append(name)
        return real(name, *a, **k)

    monkeypatch.setattr(ops, "_call", spy)
    t = {k: inp[k].clone().requires_grad_(True) for k in ("pred", "emb", "comb")}
    s = torch.tensor(scale, dtype=torch.float32, device=dev(), requires_grad=True) if scale is not None else None
    kw = dict(logit_scale=s) if s is not None else dict(tau=TAU)
    out = region.region_step(t["pred"], t["emb"], t["comb"], inp["masks"], gather=False, bg_mode=bg_mode, memory=memory, **kw)
    out.loss.backward(torch.tensor(seed, device=dev()))
    torch.cuda.synchronize()
    monkeypatch.setattr(ops, "_call", real)
    parts = {k: getattr(out, k).detach().clone() for k in ("loss", "seg", "fg", "bg", "nce")}
    parts["regions"] = out.regions.detach().clone()
    grads = {k: t[k].grad for k in t}
    grads["logit_scale"] = s.grad if s is not None else None
    return parts, grads, calls


@pytest.mark.parametrize("path", [dict(tail=True), dict(tail=False, bg_mode=1)], ids=["tail", "chain_bg1"])
def test_empty_memory_is_bit_equal_on_the_step(path, monkeypatch):
    from cor_b200 import region
    inp = _bench_inputs()
    m = region.RegionMemory(8192, 256, dev())
    for scale in (None, 1.0 / TAU):
        a = _step(inp, monkeypatch, None, scale=scale, **path)
        b = _step(inp, monkeypatch, m, scale=scale, **path)
        for k in a[0]:
            assert torch.equal(a[0][k], b[0][k]), k
        for k in a[1]:
            assert (a[1][k] is None and b[1][k] is None) or torch.equal(a[1][k], b[1][k]), k
        if path["tail"]:
            assert any(c.startswith("cor_step_tail_fwd") for c in b[2])


def _step_oracle(parts, comb, mem, s, g):
    """nce, d(g nce)/d comb and d(g nce)/d regions by the fp64 oracle on the step's own pooled rows."""
    B, M, C = parts["regions"].shape
    R = parts["regions"].reshape(B * M, C)
    return oracle_nce(R, comb.reshape(B, C), torch.arange(B, device=dev()) * M, mem, s, g)


def test_region_step_with_a_full_memory(monkeypatch):
    inp = _bench_inputs()
    m = _filled(8192, 256, 8192 + 1000)
    a = _step(inp, monkeypatch, None)
    b = _step(inp, monkeypatch, m)
    assert "cor_step_tail_fwd_mem" in b[2] and "cor_step_tail_bwd" in b[2] and "cor_memory_scan" in b[2]
    for k in ("seg", "fg", "bg", "regions"):
        assert torch.equal(a[0][k], b[0][k]), k
    assert torch.equal(a[1]["pred"], b[1]["pred"])
    nce, gq, gr, _ = _step_oracle(b[0], inp["comb"], m.rows(), 1.0 / TAU, 0.7)
    assert abs(float(b[0]["nce"]) - nce) <= 1e-3 * abs(nce)
    assert float(b[0]["nce"]) > float(a[0]["nce"])          # more negatives, higher loss
    # g_comb = the InfoNCE part (oracle) + the fg / bg part, which the memory does not change (the step without it)
    _, gq0, _, _ = _step_oracle(a[0], inp["comb"], m.rows()[:0], 1.0 / TAU, 0.7)
    want = a[1]["comb"].reshape(16, 256).double().cpu() - gq0 + gq
    assert rel(b[1]["comb"].reshape(16, 256), want) < 4e-3
    # g_emb: the memory changes it only through the current rows' coefficients; against the chain's emb gradient with
    # the same memory (an independent kernel path) and for a visible change from the step without a memory
    c = _step(inp, monkeypatch, m, tail=False)
    assert rel(b[1]["emb"].float(), c[1]["emb"].float()) < 1e-3
    assert rel(b[1]["emb"].float(), a[1]["emb"].float()) > 1e-4


def test_backward_after_enqueue_raises(monkeypatch):
    from cor_b200 import CorError, ops
    inp = _bench_inputs()
    m = _filled(1024, 256, 600)
    t = {k: inp[k].clone().requires_grad_(True) for k in ("pred", "emb", "comb")}
    from cor_b200 import region
    out = region.region_step(t["pred"], t["emb"], t["comb"], inp["masks"], gather=False, memory=m)
    m.enqueue(out.regions)
    with pytest.raises(CorError, match="enqueue after backward"):
        out.loss.backward()
    g = torch.Generator(device=dev()).manual_seed(2)
    R, Q = _unit(64, 256, g).requires_grad_(True), _unit(4, 256, g).requires_grad_(True)
    loss = ops.infonce_loss(R, Q, torch.arange(4, device=dev()), memory=m)
    m.reset()
    with pytest.raises(CorError, match="enqueue after backward"):
        loss.backward()


def test_graph_replay_matches_eager_steps():
    from cor_b200 import region
    import bench
    cfg = bench.CFG
    inp = _bench_inputs()
    mk = lambda: region.StepBuffers(cfg["B"], cfg["M"], cfg["C"], cfg["h"], cfg["w"], cfg["H"], cfg["W"], cfg["hp"], cfg["wp"],
                                    device=dev(), emb_dtype=torch.bfloat16)
    m_graph, m_eager = _filled(8192, 256, 7000, seed=4), _filled(8192, 256, 7000, seed=4)
    bufs = mk()
    bufs.load(inp)
    bufs.capture(tau=TAU, gather=False, memory=m_graph)
    torch.cuda.synchronize()
    assert torch.equal(m_graph.state, m_eager.state) and torch.equal(m_graph.bank, m_eager.bank), "capture moved the memory"
    eager = mk()
    eager.load(inp)
    for i in range(5):                                     # the memory fills at step 2 and wraps from then on
        bufs.replay()
        torch.cuda.synchronize()
        loss_e, grads_e = eager._step(True, True, dict(tau=TAU, gather=False, memory=m_eager))
        torch.cuda.synchronize()
        assert torch.equal(bufs.loss.reshape(()), loss_e.reshape(())), i
        for k in ("pred", "comb", "emb"):
            assert torch.equal(bufs.grads[k], grads_e[k]), (i, k)
    assert m_graph.state[:2].tolist() == m_eager.state[:2].tolist() == [(7000 + 5 * 1024) % 8192, 8192]
    assert torch.equal(m_graph.bank, m_eager.bank)


def test_two_runs_are_bit_identical(monkeypatch):
    inp = _bench_inputs()
    runs = [_step(inp, monkeypatch, _filled(65536, 256, 70000), scale=1.0 / TAU) for _ in range(2)]
    for k in runs[0][0]:
        assert torch.equal(runs[0][0][k], runs[1][0][k]), k
    for k in runs[0][1]:
        assert torch.equal(runs[0][1][k], runs[1][1][k]), k


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_multi_rank_memory_is_rank_local():
    n = min(torch.cuda.device_count(), 8)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "_memory_worker.py")]
    r = subprocess.run(cmd, cwd=ROOT, env=dict(os.environ, NCCL_DEBUG="WARN"), capture_output=True, text=True, timeout=240)
    assert r.returncode == 0 and "MEMORY_OK" in r.stdout, r.stdout[-3000:] + "\n" + r.stderr[-3000:]
