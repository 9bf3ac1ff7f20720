"""CPU checks of top-k without S: cor_topk_select refuses bad arguments with COR_EINVAL before any device query, its work
size depends on Nq and k but not on Nr, ops.topk_retrieve raises CorError for a width mismatch, k outside
1..min(Nr, 256) and CPU tensors, and it takes the fused path only on the shapes where it measured faster or S is too
large."""
import ctypes
import os

import pytest
import torch

from cor_b200 import _lib, build

EINVAL = -1


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        build.build()
    return _lib.load()


def test_topk_select_refuses_bad_arguments(lib):
    null, one = ctypes.c_void_p(None), ctypes.c_void_p(16)
    cases = [
        (null, one, 100, 4, 256, 10, one, one, one),      # null regions
        (one, null, 100, 4, 256, 10, one, one, one),      # null queries
        (one, one, 100, 4, 256, 10, null, one, one),      # null idx
        (one, one, 100, 4, 256, 10, one, null, one),      # null score
        (one, one, 100, 4, 256, 10, one, one, null),      # null work
        (one, one, 100, 4, 256, 0, one, one, one),        # k < 1
        (one, one, 100, 4, 256, 101, one, one, one),      # k > Nr
        (one, one, 1000, 4, 256, 257, one, one, one),     # k > 256
        (one, one, 0, 4, 256, 1, one, one, one),          # Nr < 1
        (one, one, 100, 0, 256, 10, one, one, one),       # Nq < 1
        (one, one, 100, 4, 96, 10, one, one, one),        # D not a tensor-core width
        (one, one, 100, 4, 320, 10, one, one, one),       # D > 256
    ]
    for args in cases:
        assert lib.cor_topk_select(*args, null) == EINVAL, args
        assert lib.cor_last_error()
    for bad in ((0, 100, 256, 10), (4, 0, 256, 10), (4, 100, 256, 0), (4, 1000, 256, 257)):
        assert lib.cor_topk_select_work_bytes(*bad) == 0, bad


def test_python_layer_refuses_bad_arguments():
    from cor_b200 import ops, region
    r, q = torch.zeros(100, 256), torch.zeros(4, 256)
    for args, msg in (((r, torch.zeros(4, 128), 5), "differ in width"), ((r, q, 0), "1 <= k"), ((r, q, 101), "Nr=100"),
                      ((torch.zeros(1000, 256), q, 257), "min\\(Nr, 256\\)"), ((r, q, 5), "CUDA")):
        with pytest.raises(_lib.CorError, match=msg):
            ops.topk_retrieve(*args)
    with pytest.raises(_lib.CorError, match="CUDA"):
        region.topk_regions(r, q, 5)
    assert ops._KERNELS_PER_CALL["cor_topk_select"] == 2
    assert ops._topk_fused(256, 1 << 20, 256, 10, "auto") and ops._topk_fused(8192, 6_000_000, 64, 256, "umma")
    assert not ops._topk_fused(256, 4096, 256, 10, "auto") and not ops._topk_fused(256, 1 << 20, 256, 256, "auto")
    assert not ops._topk_fused(256, 1 << 20, 256, 10, "stream") and not ops._topk_fused(8192, 6_000_000, 96, 10, "auto")
