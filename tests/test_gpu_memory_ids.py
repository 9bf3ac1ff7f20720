"""Region memory with row ids (``RegionMemory.enqueue(ids=)``, ``query_ids=``): a memory row whose id equals a query's id
is left out of that query's negatives and gradients, inside the scan and dQ kernels.

* The ring: ids land at the slots of their rows, one per row or one per image on its row 0, across a wrap; an enqueue
  without ids writes -1 over the old ones.
* Nothing matches: loss and every gradient are bit-equal to the same call without ``query_ids`` (``ops.infonce_loss`` on
  both engines, ``region_step`` on the one-launch tail and on the kernel chain).
* Everything matches: bit-equal to the call without the memory, also when the first 32-row chunk is excluded and later
  rows are not (the scan's running max starts at -inf).
* An fp64 oracle over the non-excluded rows at several fills, a wrapped ring among them; a memory of bf16 copies of the
  targets' own rows, tagged with the query ids, has the loss of a memory without those copies.
* A captured graph with an ids buffer replays eager steps bit for bit; two runs are bit-identical.
* On >= 2 GPUs each rank's memory and query ids are its own (worker script)."""
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


def _ids(n, lo, hi, g):
    return torch.randint(lo, hi, (n,), device=dev(), generator=g, dtype=torch.int64)


def _filled(K, D, n_rows, id_range=(-1, 20), seed=3):
    """A memory of capacity K after pushing n_rows unit rows in batches of at most K // 2 + 1 (wraps when n_rows > K), with
    random ids in id_range (-1: no id) on every other batch and no ids on the rest."""
    from cor_b200 import region
    m = region.RegionMemory(K, D, dev())
    g = torch.Generator(device=dev()).manual_seed(seed)
    left, i = n_rows, 0
    while left > 0:
        n = min(left, max(1, K // 2 + 1))
        m.enqueue(_unit(n, D, g), ids=_ids(n, *id_range, g) if i % 2 == 0 else None)
        left -= n
        i += 1
    return m


def oracle_nce_x(R, Q, T, mem, mem_ids, qids, s, g=1.0):
    """fp64 InfoNCE over R and the memory rows whose id is not the query's (or is negative); operands rounded to bf16 as
    the kernels see them, memory rows constant: (loss, d/d queries, d/d regions, d/d s)."""
    R64 = R.bfloat16().double().cpu().requires_grad_(True)
    Q64 = Q.bfloat16().double().cpu().requires_grad_(True)
    M64 = mem.double().cpu()
    st = torch.tensor(float(s), dtype=torch.float64, requires_grad=True)
    logits = st * (Q64 @ torch.cat([R64, M64]).t())
    mi, qi = mem_ids.cpu(), qids.cpu()
    excl = (mi[None, :] >= 0) & (mi[None, :] == qi[:, None])
    keep = torch.cat([torch.ones(Q.shape[0], R.shape[0], dtype=torch.bool), ~excl], 1)
    logits = logits.masked_fill(~keep, float("-inf"))
    loss = (torch.logsumexp(logits, 1) - logits[torch.arange(Q.shape[0]), T.cpu()]).mean()
    (g * loss).backward()
    return float(loss), Q64.grad, R64.grad, float(st.grad)


def rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).norm() / b.norm())


def _nce(R, Q, T, memory=None, scale=None, g=1.0, engine="auto", query_ids=None):
    from cor_b200 import ops
    r, q = R.clone().requires_grad_(True), Q.clone().requires_grad_(True)
    s = torch.tensor(scale, dtype=torch.float32, device=dev(), requires_grad=True) if scale is not None else None
    kw = dict(logit_scale=s) if s is not None else dict(tau=TAU)
    loss = ops.infonce_loss(r, q, T, engine=engine, memory=memory, query_ids=query_ids, **kw)
    loss.backward(torch.tensor(g, device=dev()))
    torch.cuda.synchronize()
    return loss.detach(), r.grad, q.grad, (s.grad if s is not None else None)


def _same(a, b):
    for x, y in zip(a, b):
        assert (x is None and y is None) or torch.equal(x, y)


def test_ring_ids_slots_groups_and_wrap():
    from cor_b200 import region
    K, C, B, M = 1000, 128, 6, 64
    m = region.RegionMemory(K, C, dev())
    assert m.ids.shape == (K,) and bool((m.ids == -1).all())
    g = torch.Generator(device=dev()).manual_seed(1)
    ref = torch.full((K,), -1, dtype=torch.int64, device=dev())
    head = 0
    for step in range(7):                                  # 384 rows a step: the third, fifth and seventh wrap mid-batch
        rows = torch.randn(B, M, C, device=dev(), generator=g)
        kind = step % 3
        if kind == 0:                                      # one id per row
            ids = _ids(B * M, -3, 50, g).view(B, M)
            want = ids.reshape(-1)
        elif kind == 1:                                    # one id per image, on its row 0
            ids = _ids(B, 0, 50, g)
            want = torch.full((B, M), -1, dtype=torch.int64, device=dev())
            want[:, 0] = ids
            want = want.reshape(-1)
        else:                                              # no ids: -1 over whatever the slots held
            ids, want = None, torch.full((B * M,), -1, dtype=torch.int64, device=dev())
        m.enqueue(rows, ids=ids)
        ref[(head + torch.arange(B * M, device=dev())) % K] = want
        head = (head + B * M) % K
        torch.cuda.synchronize()
        assert torch.equal(m.ids, ref), step
        assert m.state[:2].tolist() == [head, min((step + 1) * B * M, K)]
    assert torch.equal(m.row_ids(), torch.cat([ref[head:], ref[:head]]))
    m2 = region.RegionMemory(K, C, dev())
    m2.enqueue(torch.randn(5, C, device=dev()), ids=torch.arange(5, device=dev()))
    assert m2.row_ids().tolist() == [0, 1, 2, 3, 4]


@pytest.mark.parametrize("Nq,Nr,engine", [(16, 4096, "stream"), (256, 8192, "umma")])
def test_nothing_matches_is_bit_equal_on_infonce_loss(Nq, Nr, engine):
    g = torch.Generator(device=dev()).manual_seed(5)
    R, Q = _unit(Nr, 256, g), _unit(Nq, 256, g)
    T = torch.randint(0, Nr, (Nq,), device=dev(), generator=g)
    m = _filled(8192, 256, 8192 + 3000)
    qids = _ids(Nq, 100, 200, g)                          # none among the memory's ids
    qids[0] = -1                                           # a negative id matches nothing, -1 rows included
    for scale in (None, 1.0 / TAU):
        _same(_nce(R, Q, T, m, scale, engine=engine), _nce(R, Q, T, m, scale, engine=engine, query_ids=qids))


def _step(inp, monkeypatch, memory=None, tail=True, bg_mode=0, scale=None, seed=0.7, query_ids=None):
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
    out = region.region_step(t["pred"], t["emb"], t["comb"], inp["masks"], gather=False, bg_mode=bg_mode, memory=memory,
                             query_ids=query_ids, **kw)
    out.loss.backward(torch.tensor(seed, device=dev()))
    torch.cuda.synchronize()
    monkeypatch.setattr(ops, "_call", real)
    parts = {k: getattr(out, k).detach().clone() for k in ("loss", "seg", "fg", "bg", "nce")}
    parts["regions"] = out.regions.detach().clone()
    grads = {k: t[k].grad for k in t}
    grads["logit_scale"] = s.grad if s is not None else None
    return parts, grads, calls


def _same_step(a, b):
    for k in a[0]:
        assert torch.equal(a[0][k], b[0][k]), k
    for k in a[1]:
        assert (a[1][k] is None and b[1][k] is None) or torch.equal(a[1][k], b[1][k]), k


PATHS = [dict(tail=True), dict(tail=False, bg_mode=1)]


@pytest.mark.parametrize("path", PATHS, ids=["tail", "chain_bg1"])
def test_nothing_matches_is_bit_equal_on_the_step(path, monkeypatch):
    inp = _bench_inputs()
    m = _filled(8192, 256, 8192 + 1000)
    qids = torch.arange(16, device=dev()) + 1000
    for scale in (None, 1.0 / TAU):
        a = _step(inp, monkeypatch, m, scale=scale, **path)
        b = _step(inp, monkeypatch, m, scale=scale, query_ids=qids, **path)
        _same_step(a, b)
        assert "cor_memory_exclude" in b[2] and "cor_memory_scan_x" in b[2] and "cor_memory_dq_x" in b[2]
        assert "cor_memory_exclude" not in a[2] and "cor_memory_scan" in a[2] and "cor_memory_dq" in a[2]
        if path["tail"]:
            assert "cor_step_tail_fwd_mem" in b[2]


@pytest.mark.parametrize("Nq,Nr,engine", [(16, 4096, "stream"), (256, 8192, "umma")])
def test_everything_matches_is_bit_equal_to_no_memory(Nq, Nr, engine):
    from cor_b200 import region
    g = torch.Generator(device=dev()).manual_seed(6)
    R, Q = _unit(Nr, 256, g), _unit(Nq, 256, g)
    T = torch.randint(0, Nr, (Nq,), device=dev(), generator=g)
    qids = torch.full((Nq,), 7, dtype=torch.int64, device=dev())
    for K, n in ((1, 1), (300, 300), (8192, 8192 + 500)):
        m = region.RegionMemory(K, 256, dev())
        left = n
        while left:
            k = min(left, K)
            m.enqueue(_unit(k, 256, g), ids=torch.full((k,), 7, dtype=torch.int64, device=dev()))
            left -= k
        for scale in (None, 1.0 / TAU):
            _same(_nce(R, Q, T, None, scale, engine=engine), _nce(R, Q, T, m, scale, engine=engine, query_ids=qids))


@pytest.mark.parametrize("path", PATHS, ids=["tail", "chain_bg1"])
def test_everything_matches_is_bit_equal_on_the_step(path, monkeypatch):
    inp = _bench_inputs()
    from cor_b200 import region
    m = region.RegionMemory(4096, 256, dev())
    g = torch.Generator(device=dev()).manual_seed(8)
    m.enqueue(_unit(3000, 256, g), ids=torch.arange(3000, device=dev()) % 16)
    a = _step(inp, monkeypatch, None, scale=1.0 / TAU, **path)
    b = _step(inp, monkeypatch, m, scale=1.0 / TAU, query_ids=torch.arange(16, device=dev()), **path)
    # each triplet b excludes its rows (ids == b) only: the loss rises; a memory where every row is every query's
    m2 = region.RegionMemory(4096, 256, dev())
    m2.enqueue(_unit(3000, 256, g), ids=torch.full((3000,), 5, dtype=torch.int64, device=dev()))
    c = _step(inp, monkeypatch, m2, scale=1.0 / TAU, query_ids=torch.full((16,), 5, dtype=torch.int64, device=dev()), **path)
    _same_step(a, c)
    assert float(b[0]["nce"]) > float(a[0]["nce"])


def test_first_chunk_excluded_later_rows_not():
    """Rows 0..31 (the first mask word of every query's scan) carry query 0's id, the rest carry none: query 0's running
    max starts at -inf and must come out finite; against the oracle over the rows it keeps."""
    from cor_b200 import region
    g = torch.Generator(device=dev()).manual_seed(9)
    Nq, Nr, D = 16, 1024, 256
    R, Q = _unit(Nr, D, g), _unit(Nq, D, g)
    T = torch.randint(0, Nr, (Nq,), device=dev(), generator=g)
    qids = torch.arange(Nq, device=dev()) + 10
    for K, n_first in ((200, 32), (8192, 128), (8192, 8192)):
        m = region.RegionMemory(K, D, dev())
        m.enqueue(_unit(n_first, D, g), ids=torch.full((n_first,), 10, dtype=torch.int64, device=dev()))
        if K > n_first:
            m.enqueue(_unit(K - n_first, D, g))
        got = _nce(R, Q, T, m, scale=1.0 / TAU, g=0.7, query_ids=qids)
        loss, gq, gr, gs = oracle_nce_x(R, Q, T, m.rows(), m.row_ids(), qids, 1.0 / TAU, g=0.7)
        assert torch.isfinite(got[0]) and abs(float(got[0]) - loss) <= 1e-3 * abs(loss), (K, n_first)
        assert rel(got[2], gq) < 4e-3 and rel(got[1], gr) < 4e-3
        assert abs(float(got[3]) - gs) <= 1e-3 * abs(gs)


# (Nq, K, rows pushed): partly full, full, and full after a wrap
FILL = [(16, 127, 60), (16, 8192, 5000), (1, 127, 200), (16, 8192, 8192 + 3000), (64, 65536, 70000), (256, 8192, 8192)]


@pytest.mark.parametrize("Nq,K,n_rows", FILL)
def test_against_the_oracle(Nq, K, n_rows):
    D, Nr = 256, 1024
    g = torch.Generator(device=dev()).manual_seed(11)
    R, Q = _unit(Nr, D, g), _unit(Nq, D, g)
    T = torch.randint(0, Nr, (Nq,), device=dev(), generator=g)
    m = _filled(K, D, n_rows, id_range=(-1, 12))
    qids = _ids(Nq, 0, 12, g)
    got = _nce(R, Q, T, m, scale=1.0 / TAU, g=0.7, query_ids=qids)
    loss, gq, gr, gs = oracle_nce_x(R, Q, T, m.rows(), m.row_ids(), qids, 1.0 / TAU, g=0.7)
    assert abs(float(got[0]) - loss) <= 1e-3 * abs(loss)
    assert rel(got[2], gq) < 4e-3 and rel(got[1], gr) < 4e-3
    assert abs(float(got[3]) - gs) <= 1e-3 * abs(gs)


@pytest.mark.parametrize("Nq,Nr,engine", [(16, 4096, "stream"), (256, 8192, "umma")])
def test_copies_of_the_targets_are_left_out(Nq, Nr, engine):
    """Triplets that share their target object: every query looks for region t0, and the memory holds five bf16 copies of
    it (earlier epochs' pooled rows) tagged with its id among unrelated rows.  With query_ids the loss and gradients are
    those of the memory without the copies; without them the loss sits on the duplicates' floor, log 6 higher at most."""
    from cor_b200 import region
    g = torch.Generator(device=dev()).manual_seed(12)
    D, K = 256, 8192
    R, Q = _unit(Nr, D, g), _unit(Nq, D, g)
    T = torch.full((Nq,), 17, dtype=torch.int64, device=dev())
    Q = torch.nn.functional.normalize(Q + 2.0 * R[17], dim=-1)         # queries close to their target: a confident model
    qids = torch.full((Nq,), 4242, dtype=torch.int64, device=dev())
    others = _unit(6000, D, g)
    with_copies, without = region.RegionMemory(K, D, dev()), region.RegionMemory(K, D, dev())
    with_copies.enqueue(others[:3000])
    with_copies.enqueue(R[17].expand(5, D).bfloat16(), ids=qids[:5])
    with_copies.enqueue(others[3000:])
    without.enqueue(others)
    got = _nce(R, Q, T, with_copies, scale=1.0 / TAU, g=0.7, engine=engine, query_ids=qids)
    ref = _nce(R, Q, T, without, scale=1.0 / TAU, g=0.7, engine=engine)
    raw = _nce(R, Q, T, with_copies, scale=1.0 / TAU, g=0.7, engine=engine)
    assert abs(float(got[0]) - float(ref[0])) <= 1e-4 * abs(float(ref[0])) + 1e-6      # the same terms, summed in another order
    assert rel(got[2], ref[2]) < 1e-3 and rel(got[1], ref[1]) < 1e-3
    assert abs(float(got[3]) - float(ref[3])) <= 1e-3 * abs(float(ref[3]))
    assert float(raw[0]) > float(ref[0]) + 1.0                         # five duplicates of the target: a floor near log 6
    loss, gq, gr, gs = oracle_nce_x(R, Q, T, with_copies.rows(), with_copies.row_ids(), qids, 1.0 / TAU, g=0.7)
    assert abs(float(got[0]) - loss) <= 1e-3 * abs(loss) and rel(got[2], gq) < 4e-3 and rel(got[1], gr) < 4e-3


@pytest.mark.parametrize("Nq,Nr,engine", [(16, 4096, "stream"), (256, 8192, "umma")])
def test_own_target_copies_against_the_oracle(Nq, Nr, engine):
    """Distinct targets: each query's own target row is in the memory, tagged with its id, beside the other queries'
    copies, which stay negatives for it."""
    from cor_b200 import region
    g = torch.Generator(device=dev()).manual_seed(13)
    D, K = 256, 8192
    R, Q = _unit(Nr, D, g), _unit(Nq, D, g)
    T = torch.randperm(Nr, device=dev(), generator=g)[:Nq]
    Q = torch.nn.functional.normalize(Q + 2.0 * R[T], dim=-1)
    qids = torch.randperm(10 * Nq, device=dev(), generator=g)[:Nq]
    m = region.RegionMemory(K, D, dev())
    m.enqueue(_unit(3000, D, g))
    m.enqueue(R[T].bfloat16(), ids=qids)
    m.enqueue(_unit(3000, D, g))
    got = _nce(R, Q, T, m, scale=1.0 / TAU, g=0.7, engine=engine, query_ids=qids)
    raw = _nce(R, Q, T, m, scale=1.0 / TAU, g=0.7, engine=engine)
    loss, gq, gr, gs = oracle_nce_x(R, Q, T, m.rows(), m.row_ids(), qids, 1.0 / TAU, g=0.7)
    assert abs(float(got[0]) - loss) <= 1e-3 * abs(loss)
    assert rel(got[2], gq) < 4e-3 and rel(got[1], gr) < 4e-3
    assert abs(float(got[3]) - gs) <= 1e-3 * abs(gs) + 1e-5
    assert float(raw[0]) > float(got[0]) + 0.5                         # its own copy as a negative: near log 2 per query


@pytest.mark.parametrize("path", PATHS, ids=["tail", "chain_bg1"])
def test_step_with_its_own_rows_in_memory_against_the_oracle(path, monkeypatch):
    """A step's pooled rows pushed with the triplets' ids on each image's row 0 ([B] form), then the same step with those
    ids: each triplet leaves its own ground-truth row out and scores the other 63 rows of every image."""
    from cor_b200 import region
    inp = _bench_inputs()
    g = torch.Generator(device=dev()).manual_seed(14)
    qids = torch.arange(16, device=dev()) * 3 + 1
    m = region.RegionMemory(8192, 256, dev())
    m.enqueue(_unit(2000, 256, g), ids=_ids(2000, 0, 60, g))
    first = _step(inp, monkeypatch, None, **path)
    m.enqueue(first[0]["regions"], ids=qids)
    b = _step(inp, monkeypatch, m, scale=1.0 / TAU, query_ids=qids, **path)
    assert "cor_memory_dq_x" in b[2]
    B, M, C = b[0]["regions"].shape
    nce, gq, _, gs = oracle_nce_x(b[0]["regions"].reshape(B * M, C), inp["comb"].reshape(B, C), torch.arange(B, device=dev()) * M,
                                  m.rows(), m.row_ids(), qids, 1.0 / TAU, g=0.7)
    assert abs(float(b[0]["nce"]) - nce) <= 1e-3 * abs(nce)
    assert abs(float(b[1]["logit_scale"]) - gs) <= 2e-3 * abs(gs) + 1e-4   # g_scale: the InfoNCE term only
    # g_comb = the InfoNCE part (oracle) + the fg / bg part, which the memory does not change (the step without it)
    _, gq0, _, _ = oracle_nce_x(b[0]["regions"].reshape(B * M, C), inp["comb"].reshape(B, C), torch.arange(B, device=dev()) * M,
                                m.rows()[:0], m.row_ids()[:0], qids, 1.0 / TAU, g=0.7)
    want = first[1]["comb"].reshape(B, C).double().cpu() - gq0 + gq
    assert rel(b[1]["comb"].reshape(B, C), want) < 4e-3
    a = _step(inp, monkeypatch, m, scale=1.0 / TAU, **path)                # the same memory, no ids: every copy a negative
    assert float(a[0]["nce"]) > float(b[0]["nce"])


def _bufs(ids):
    from cor_b200 import region
    import bench
    cfg = bench.CFG
    return region.StepBuffers(cfg["B"], cfg["M"], cfg["C"], cfg["h"], cfg["w"], cfg["H"], cfg["W"], cfg["hp"], cfg["wp"], device=dev(),
                              emb_dtype=torch.bfloat16, ids=ids)


def test_graph_replay_with_ids_matches_eager_steps():
    inp = _bench_inputs()
    inp["ids"] = torch.arange(16, device=dev()) % 5         # repeated ids: triplets that share a target
    plain = _bufs(False)
    assert "ids" not in plain.d
    bufs = _bufs(True)
    assert bufs.h2d_bytes == plain.h2d_bytes + 16 * 8
    m_graph, m_eager = _filled(8192, 256, 7000, id_range=(-1, 5), seed=4), _filled(8192, 256, 7000, id_range=(-1, 5), seed=4)
    bufs.load(inp)
    bufs.capture(tau=TAU, gather=False, memory=m_graph)
    torch.cuda.synchronize()
    assert torch.equal(m_graph.state, m_eager.state) and torch.equal(m_graph.bank, m_eager.bank)
    assert torch.equal(m_graph.ids, m_eager.ids), "capture moved the memory's ids"
    eager = _bufs(True)
    eager.load(inp)
    for i in range(5):
        bufs.replay()
        torch.cuda.synchronize()
        loss_e, grads_e = eager._step(True, True, dict(tau=TAU, gather=False, memory=m_eager))
        torch.cuda.synchronize()
        assert torch.equal(bufs.loss.reshape(()), loss_e.reshape(())), i
        for k in ("pred", "comb", "emb"):
            assert torch.equal(bufs.grads[k], grads_e[k]), (i, k)
    assert torch.equal(m_graph.bank, m_eager.bank) and torch.equal(m_graph.ids, m_eager.ids)
    rid = m_graph.row_ids()[-16 * 64:].view(16, 64)          # the last step's rows: its ids on row 0 of each image
    assert torch.equal(rid[:, 0], inp["ids"]) and bool((rid[:, 1:] == -1).all())


def test_two_runs_are_bit_identical(monkeypatch):
    inp = _bench_inputs()
    qids = torch.arange(16, device=dev()) % 7
    runs = [_step(inp, monkeypatch, _filled(65536, 256, 70000, id_range=(-1, 7)), scale=1.0 / TAU, query_ids=qids) for _ in range(2)]
    _same_step(runs[0], runs[1])


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_multi_rank_query_ids_are_rank_local():
    n = min(torch.cuda.device_count(), 8)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "_memory_ids_worker.py")]
    r = subprocess.run(cmd, cwd=ROOT, env=dict(os.environ, NCCL_DEBUG="WARN"), capture_output=True, text=True, timeout=240)
    assert r.returncode == 0 and "MEMORY_IDS_OK" in r.stdout, r.stdout[-3000:] + "\n" + r.stderr[-3000:]
