"""Argument checks of the fused linear layer and its GEMM (cor_b200/linear.py, csrc/gemm_umma.cu) that need no device:
the combinations ``linear()`` refuses, and the bad ``gemm()`` / ``cor_gemm_bf16`` arguments that come back as errors
before anything is launched."""
import ctypes
import os

import pytest
import torch

from cor_b200 import _lib, build
from cor_b200._lib import CorError
from cor_b200.linear import gemm, linear


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        build.build()
    return _lib.load()


@pytest.mark.parametrize("act,with_res,with_mask,words", [
    ("relu", True, False, ("relu", "residual")),
    ("sigmoid", True, False, ("sigmoid", "residual")),
    ("sigmoid", False, True, ("sigmoid", "drop_mask")),
    ("sigmoid", True, True, ("sigmoid", "residual")),
])
def test_linear_refuses_activation_backward_through_a_changed_output(act, with_res, with_mask, words):
    """relu and sigmoid differentiate through the layer's stored output; a residual (or, for sigmoid, a dropout mask) changes
    that output, so the backward would be wrong.  The refusal comes before any device check: CPU tensors reach it."""
    x, w = torch.ones(4, 8), torch.ones(16, 8)
    res = torch.zeros(4, 16) if with_res else None
    mask = torch.ones(4, 16) if with_mask else None
    with pytest.raises(CorError) as e:
        linear(x, w, None, act, mask, residual=res)
    msg = str(e.value)
    assert all(wd in msg for wd in words), msg
    assert "CUDA" not in msg


@pytest.mark.parametrize("act,with_res,with_mask", [(None, True, False), ("gelu", True, True), ("relu", False, True)])
def test_linear_accepts_the_combinations_its_backward_handles(act, with_res, with_mask):
    """The accepted combinations get as far as the device check (and no further on CPU tensors: there is no CPU path)."""
    x, w = torch.ones(4, 8), torch.ones(16, 8)
    res = torch.zeros(4, 16) if with_res else None
    mask = torch.ones(4, 16) if with_mask else None
    with pytest.raises(CorError, match="CUDA tensors"):
        linear(x, w, None, act, mask, residual=res)


@pytest.mark.parametrize("a,b", [
    (torch.ones(8, 64), torch.ones(8, 64, dtype=torch.bfloat16)),                         # fp32 operand
    (torch.ones(8, 64, dtype=torch.bfloat16), torch.ones(8, 64, dtype=torch.float16)),    # fp16 operand
    (torch.ones(2, 8, 64, dtype=torch.bfloat16), torch.ones(8, 64, dtype=torch.bfloat16)),  # 3-D operand
])
def test_gemm_refuses_operands_that_are_not_2d_bf16(a, b):
    with pytest.raises(CorError, match="2-D bf16"):
        gemm(a, b, 8, 8, 64)


def test_gemm_refuses_cpu_operands():
    a = torch.ones(8, 64, dtype=torch.bfloat16)
    with pytest.raises(CorError, match="CUDA tensors"):
        gemm(a, a, 8, 8, 64)


def test_gemm_entry_rejects_bad_arguments_before_any_launch(lib):
    """cor_gemm_bf16's checks that precede the tensor maps: COR_EINVAL with a message, no device touched."""
    null = ctypes.c_void_p(None)
    one = ctypes.c_void_p(16)

    def args(A=one, B=one, C=one, M=8, N=8, K=64, batch=1, act=0, residual=null, res_dtype=0, c_dtype=0):
        return (A, 0, 8, 0, B, 0, 8, 0, M, N, K, batch, 1.0, null, act, null, null, residual, res_dtype, 8, C, c_dtype, 8, null, 0,
                null, null)

    cases = {
        "null A": args(A=null), "null B": args(B=null), "null C": args(C=null),
        "M = 0": args(M=0), "N = 0": args(N=0), "batch = 0": args(batch=0), "negative K": args(K=-64),
        "u8 output": args(c_dtype=2), "u8 residual": args(residual=one, res_dtype=2),
        "act -1": args(act=-1), "act 4": args(act=4),
    }
    for what, a in cases.items():
        assert lib.cor_gemm_bf16(*a) == -1, what
        assert lib.cor_last_error(), what
