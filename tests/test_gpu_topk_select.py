"""Top-k without S (cor_topk_select): the selecting epilogue of the tensor-core similarity kernel plus one select /
re-score / sort CTA per query.  Results must equal the oracle's total order (score desc, index asc) exactly, including
ties at the cut and galleries that make every tile compact.  On large galleries, where the oracle is too slow, they must
equal the route that writes S on the same rows.  Run with ``-m gpu`` on a B200."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def dev():
    return torch.device("cuda:0")


def cu(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(dev())


def s_route(r16, q16, k):
    """The route that writes S on the tensor cores (cor_sim_umma_fwd) and selects from it (cor_topk)."""
    from cor_b200 import ops
    Nr, D = r16.shape
    Nq = q16.shape[0]
    S, _ = ops._sim_forward(r16, q16, 1.0, True, False, "umma")
    idx = torch.empty((Nq, k), dtype=torch.int64, device=dev())
    score = torch.empty((Nq, k), dtype=torch.float32, device=dev())
    ops._call("cor_topk", dev(), ops.ptr(S), ops.ptr(r16), ops.ptr(q16), Nr, Nq, D, k, ops.ptr(idx), ops.ptr(score))
    return idx, score


def fused(r16, q16, k):
    from cor_b200 import ops
    return ops._topk_select(r16, q16, k)


def assert_oracle(regions, queries, k):
    from cor_b200 import ops
    from oracle import np_oracle as no
    idx, sc = fused(ops._to_bf16_rows(cu(regions)), ops._to_bf16_rows(cu(queries)), k)
    ridx, rsc = no.topk_retrieve(regions, queries, k)
    np.testing.assert_array_equal(idx.cpu().numpy(), ridx)
    np.testing.assert_array_equal(sc.cpu().numpy(), rsc)


def device_rows(seed, n, D):
    g = torch.Generator(device=dev()).manual_seed(seed)
    x = torch.randn(n, D, device=dev(), generator=g)
    return torch.nn.functional.normalize(x, dim=-1).bfloat16()


# every Nr, Nq, D and k of the coverage list at least once: Nr not a multiple of 128, one and several query tiles, k = Nr
@pytest.mark.parametrize("Nr,Nq,D,k", [
    (200, 1, 64, 1), (200, 16, 192, 200), (200, 300, 256, 50), (1000, 256, 256, 10), (1000, 300, 64, 256), (1000, 1, 192, 256),
    (4096, 300, 192, 50), (4096, 16, 256, 256), (4096, 256, 64, 1), (100000, 256, 256, 10), (100000, 16, 64, 50),
    (100000, 300, 192, 1), (100000, 1, 256, 256)])
def test_topk_select_equals_oracle(Nr, Nq, D, k):
    from cor_b200 import synth
    g = synth.make_gallery(300 + Nq + k, Nr, Nq, D=D, duplicate=True)
    assert_oracle(g["regions"], g["queries"], k)


@pytest.mark.parametrize("k", [10, 256])
def test_more_duplicates_of_the_best_row_than_a_list_holds(k):
    """2 000 exact copies of the best row, spread over every CTA: more than any list's capacity (ncand + 128), so the
    smallest indices must win inside each list and again in the union."""
    from cor_b200 import synth
    g = synth.make_gallery(71, 60000, 16, D=256)
    r, q = g["regions"], g["queries"]
    copies = np.arange(5, 60000, 30)[:2000]
    r[copies] = q[0]
    assert_oracle(r, q, k)


@pytest.mark.parametrize("k", [1, 50, 256])
def test_zero_query_every_score_ties(k):
    from cor_b200 import synth
    g = synth.make_gallery(73, 30000, 20, D=192)
    q = g["queries"].copy()
    q[7] = 0.0
    assert_oracle(g["regions"], q, k)


@pytest.mark.parametrize("k", [10, 256])
def test_scores_rising_with_the_index_compact_every_tile(k):
    """The gallery sorted by query 0's score: its every tile beats the threshold, so every tile compacts."""
    from cor_b200 import synth
    from oracle import np_oracle as no
    g = synth.make_gallery(79, 50000, 64, D=128)
    s0 = no.region_query_similarity(g["regions"], g["queries"][:1])[0]
    r = g["regions"][np.argsort(s0, kind="stable")]
    assert_oracle(r, g["queries"], k)


@pytest.mark.parametrize("k", [10, 256])
def test_256_queries_2m_regions_equal_the_s_route(k):
    r16, q16 = device_rows(81, 2_000_000, 256), device_rows(82, 256, 256)
    idx, sc = fused(r16, q16, k)
    ridx, rsc = s_route(r16, q16, k)
    assert torch.equal(idx, ridx) and torch.equal(sc, rsc)


def test_8192_queries_6m_regions_where_s_would_not_fit():
    """S would be 8 192 x 6 M x 4 B = 196 GB.  A seeded sample of 64 queries is checked against the S route on those
    queries only, and the call's peak memory stays within its inputs, outputs and reported work bytes."""
    from cor_b200 import _lib, ops
    Nr, Nq, D, k = 6_000_000, 8192, 256, 10
    r16, q16 = device_rows(83, Nr, D), device_rows(84, Nq, D)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    assert ops._topk_fused(Nq, Nr, D, k, "auto")          # the public op takes the fused path here
    idx, sc = ops.topk_retrieve(r16, q16, k)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    work = _lib.load().cor_topk_select_work_bytes(Nq, Nr, D, k)
    outputs = Nq * k * (8 + 4)
    # the work buffer as the test harness hands it out (a 4 KB canary behind it), plus the allocator's rounding
    assert peak <= outputs + work + 4096 + 3 * 512, (peak, outputs, work)
    sample = torch.from_numpy(np.random.default_rng(85).choice(Nq, 64, replace=False)).to(dev())
    ridx, rsc = s_route(r16, q16[sample].contiguous(), k)
    assert torch.equal(idx[sample], ridx) and torch.equal(sc[sample], rsc)


def test_deterministic_and_graph_capturable():
    r16, q16 = device_rows(87, 300_000, 192), device_rows(88, 300, 192)
    a = fused(r16, q16, 50)
    b = fused(r16, q16, 50)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fused(r16, q16, 50)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = fused(r16, q16, 50)
    out[0].zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out[0], a[0]) and torch.equal(out[1], a[1])
