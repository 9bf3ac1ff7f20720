"""Linear layers on the tcgen05 GEMM of ``csrc/gemm_umma.cu`` (bf16 operands, fp32 accumulate), forward and backward.

``linear(x, weight, bias, act, drop_mask)`` is ``drop_mask * act(x @ weight.T + bias)`` as ONE kernel (the bias,
activation and dropout mask live in the GEMM epilogue); its backward is one element-wise kernel (``cor_act_bwd``: the
epilogue's derivative, bf16 ``dZ`` and the bias gradient) and two more GEMMs that read the SAME buffers in the other
orientation -- ``dX = dZ W`` takes ``W [out, in]`` as an MN-major operand, ``dW = dZ^T X`` takes both ``dZ`` and ``X``
MN-major -- so nothing is ever transposed in memory.  Under bf16 autocast the reference's ``nn.Linear`` computes the
same way (bf16 operands, fp32 accumulate, lib/support_branch.py:47-54 inside utils/trainer_v3_g.py:51).
"""
from __future__ import annotations

from typing import Optional

import torch

from . import _lib as L
from . import ops
from ._lib import ACT_GELU, ACT_NONE, ACT_RELU, ACT_SIGMOID, CorError

__all__ = ["gemm", "linear", "ln_rows", "ln_channels_first", "dwconv7_rows", "cast_bf16", "ACT_NONE", "ACT_RELU", "ACT_GELU", "ACT_SIGMOID"]

_ACTS = {None: ACT_NONE, "none": ACT_NONE, "relu": ACT_RELU, "gelu": ACT_GELU, "sigmoid": ACT_SIGMOID}


def cast_bf16(a: torch.Tensor, b: Optional[torch.Tensor] = None) -> torch.Tensor:
    """bf16 copy of ``a`` ([rows, c0] f32), or of ``cat(a, b, dim=-1)`` -- one kernel."""
    dev = L.require_cuda(a, b)
    a = a.float().contiguous()
    rows, c0 = a.shape
    c1 = 0
    if b is not None:
        b = b.float().contiguous()
        if b.shape[0] != rows:
            raise CorError(f"cast_bf16: row counts differ ({rows} vs {b.shape[0]})")
        c1 = b.shape[1]
    out = torch.empty((rows, c0 + c1), dtype=torch.bfloat16, device=dev)
    ops._call("cor_cast_cat_bf16", dev, ops.ptr(a), c0, ops.ptr(b), c1, ops._ll(rows), ops.ptr(out))
    return out


def gemm(a: torch.Tensor, b: torch.Tensor, M: int, N: int, K: int, *, a_mn: bool = False, b_mn: bool = False, batch: int = 1,
         a_batch_rows: int = 0, b_batch_rows: int = 0, alpha: float = 1.0, bias: Optional[torch.Tensor] = None, act: int = ACT_NONE,
         emul: Optional[torch.Tensor] = None, colscale: Optional[torch.Tensor] = None, residual: Optional[torch.Tensor] = None,
         out_dtype: torch.dtype = torch.float32, want_pre: bool = False, ksplit: int = 0):
    """C[b][m][n] = epilogue(alpha * sum_k A[b](m,k) B[b](n,k)); see include/cor_b200.h (cor_gemm_bf16).  ``a`` / ``b`` are
    2-D bf16 tensors; ``x_mn`` says the operand is stored [K, rows] instead of [rows, K].  Returns C [batch*M, N] (and the
    bf16 pre-activation when ``want_pre``)."""
    if a.dtype != torch.bfloat16 or b.dtype != torch.bfloat16 or a.dim() != 2 or b.dim() != 2:
        raise CorError("gemm: operands must be 2-D bf16 tensors")
    dev = L.require_cuda(a, b, bias, emul, colscale, residual)
    a, b = a.contiguous(), b.contiguous()
    lib = L.load()
    C = torch.empty((batch * M, N), dtype=out_dtype, device=dev)
    pre = torch.empty((batch * M, N), dtype=torch.bfloat16, device=dev) if want_pre else None
    work = ops._work(lib.cor_gemm_bf16_work_bytes(M, N, K, batch, ksplit), dev)
    res = residual.contiguous() if residual is not None else None
    ops._call("cor_gemm_bf16", dev, ops.ptr(a), int(a_mn), ops._ll(a.shape[0]), ops._ll(a_batch_rows), ops.ptr(b), int(b_mn),
              ops._ll(b.shape[0]), ops._ll(b_batch_rows), M, N, K, batch, ops._f(alpha), ops.ptr(bias), int(act), ops.ptr(emul),
              ops.ptr(colscale), ops.ptr(res), (L.dtype_code(res) if res is not None else L.F32), ops._ll(N), ops.ptr(C), L.dtype_code(C),
              ops._ll(N), ops.ptr(pre), int(ksplit), ops.ptr(work))
    return (C, pre) if want_pre else C


_w16_cache = {}


def _weight_bf16(w: torch.Tensor) -> torch.Tensor:
    """bf16 copy of a weight.  Cached only for parameters (or views of parameters, e.g. ``conv.weight.view(out, in)``):
    keyed on the parameter object (weak reference) and its ``_version``, which an optimizer's in-place update bumps.
    Computed weights (e.g. a product of two parameters) are cast on every call."""
    import weakref
    base = w._base if w._base is not None else w
    if not isinstance(base, torch.nn.Parameter):
        return cast_bf16(w.detach().reshape(w.shape[0], -1))
    key = (id(base), tuple(w.shape), w.storage_offset())
    hit = _w16_cache.get(key)
    if hit is not None and hit[0]() is base and hit[1] == base._version:
        return hit[2]
    w16 = cast_bf16(w.detach().reshape(w.shape[0], -1))
    _w16_cache[key] = (weakref.ref(base), base._version, w16)
    return w16


class _LinearFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, act, drop_mask, x2, colscale, residual, out_bf16):
        dev = L.require_cuda(x, weight, bias, drop_mask, x2, colscale, residual)
        rows = x.shape[0]
        x16 = cast_bf16(x, x2) if x.dtype != torch.bfloat16 or x2 is not None else x.contiguous()   # torch.cat((x, x2), -1) fused with the cast
        w16 = _weight_bf16(weight)
        N, K = w16.shape
        if x16.shape[1] != K:
            raise CorError(f"linear: input width {x16.shape[1]} != weight in_features {K}")
        if colscale is not None and act != ACT_NONE:
            raise CorError("linear: a column scale goes with no activation (ConvNeXt's gamma * pwconv2(.))")
        b32 = bias.float().contiguous() if bias is not None else None
        m32 = drop_mask.float().contiguous() if drop_mask is not None else None
        cs = colscale.float().contiguous() if colscale is not None else None
        want_pre = act == ACT_GELU or (cs is not None and colscale.requires_grad)
        out = gemm(x16, w16, rows, N, K, bias=b32, act=act, emul=m32, colscale=cs, residual=residual, want_pre=want_pre,
                   out_dtype=torch.bfloat16 if out_bf16 else torch.float32)
        y, pre = out if want_pre else (out, None)
        # relu / sigmoid differentiate through the stored OUTPUT (linear() refuses a residual with either, and a mask with sigmoid)
        ctx.save_for_backward(x16, w16, (y.float() if y.dtype != torch.float32 else y) if act in (ACT_RELU, ACT_SIGMOID) else None, pre, m32, cs)
        ctx.cfg = (act, x.shape[1], x.requires_grad, x2 is not None and x2.requires_grad, weight.requires_grad,
                   bias is not None and bias.requires_grad, colscale is not None and colscale.requires_grad,
                   residual is not None and residual.requires_grad, x.dtype, weight.dtype, tuple(weight.shape), rows, N)
        return y

    @staticmethod
    def backward(ctx, gy):
        x16, w16, y, pre, m32, cs = ctx.saved_tensors
        act, c0, need_x, need_x2, need_w, need_b, need_cs, need_res, xdt, wdt, wshape, rows, N = ctx.cfg
        dev = x16.device
        K = x16.shape[1]
        gy = (gy if gy.dtype in (torch.float32, torch.bfloat16) else gy.float()).contiguous()
        dz = torch.empty((rows, N), dtype=torch.bfloat16, device=dev)
        db = torch.empty((N,), dtype=torch.float32, device=dev) if need_b else None
        dcs = torch.empty((N,), dtype=torch.float32, device=dev) if need_cs else None
        work = ops._work(L.load().cor_act_bwd_work_bytes(rows, N), dev) if (need_b or need_cs) else None
        ops._call("cor_act_bwd", dev, ops.ptr(gy), L.dtype_code(gy), ops.ptr(y), ops.ptr(pre), ops.ptr(m32), ops.ptr(cs), int(act), ops._ll(rows), N,
                  ops.ptr(dz), ops.ptr(db), ops.ptr(dcs), ops.ptr(work))
        gx = gx2 = gw = None
        if need_x or need_x2:
            # dX = dZ W : W [N, K] read as the MN-major B (k = out features); a bf16 input gets its gradient in bf16 straight
            # from the epilogue
            g_in = gemm(dz, w16, rows, K, N, b_mn=True, out_dtype=torch.bfloat16 if (xdt == torch.bfloat16 and c0 == K) else torch.float32)
            gx = (g_in[:, :c0] if c0 != K else g_in).to(xdt) if need_x else None
            gx2 = g_in[:, c0:].to(xdt) if need_x2 else None
        if need_w:
            gw = gemm(dz, x16, N, K, rows, a_mn=True, b_mn=True).view(wshape).to(wdt)   # dW = dZ^T X : both operands MN-major (k = rows)
        return gx, gw, db, None, None, gx2, dcs, ((gy if gy.dtype == torch.float32 else gy.float()) if need_res else None), None


def linear(x: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor] = None, act: Optional[str] = None,
           drop_mask: Optional[torch.Tensor] = None, x2: Optional[torch.Tensor] = None, colscale: Optional[torch.Tensor] = None,
           residual: Optional[torch.Tensor] = None, out_bf16: bool = False) -> torch.Tensor:
    """``residual + colscale * drop_mask * act(cat(x, x2) @ weight.T + bias)`` -> f32 [rows, out_features]; x [rows, in] f32
    or bf16 (any leading shape is flattened by the caller).  ``drop_mask`` holds 0 or 1/(1-p) per element (what
    ``F.dropout`` multiplies by); ``colscale`` [out] and ``residual`` [rows, out] are ConvNeXt's layer scale and skip
    connection (mask_adapter.py:215-221), fused into the same GEMM epilogue.  ``out_bf16`` writes the result in bf16 (the next
    GEMM's A operand: no fp32 round trip of a wide hidden activation)."""
    # relu and sigmoid differentiate through the stored output, which a residual or (for sigmoid) a mask has changed
    if act in ("relu", "sigmoid") and residual is not None:
        raise CorError(f"linear: act={act!r} with a residual is not supported (its backward would read relu/sigmoid through the residual)")
    if act == "sigmoid" and drop_mask is not None:
        raise CorError("linear: act='sigmoid' with a drop_mask is not supported (its backward would read the sigmoid through the mask)")
    return _LinearFn.apply(x, weight, bias, _ACTS[act], drop_mask, x2, colscale, residual, bool(out_bf16))


class _LnRowsFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, eps, act, out_bf16):
        dev = L.require_cuda(x, weight, bias)
        x = x.float().contiguous()
        rows, Cc = x.shape
        w, b = weight.float().contiguous(), bias.float().contiguous()
        y = torch.empty((rows, Cc), dtype=torch.bfloat16 if out_bf16 else torch.float32, device=dev)
        stats = torch.empty((rows, 2), dtype=torch.float32, device=dev)
        ops._call("cor_ln_rows_fwd", dev, ops.ptr(x), ops.ptr(w), ops.ptr(b), ops._ll(rows), Cc, ops._f(eps), int(act), ops.ptr(y),
                  L.dtype_code(y), ops.ptr(stats))
        ctx.save_for_backward(x, w, b, stats)
        ctx.cfg = (int(act), weight.dtype)
        return y

    @staticmethod
    def backward(ctx, gy):
        x, w, b, stats = ctx.saved_tensors
        act, wdt = ctx.cfg
        dev = x.device
        rows, Cc = x.shape
        gy = (gy if gy.dtype in (torch.float32, torch.bfloat16) else gy.float()).contiguous()
        dx = torch.empty_like(x)
        dw = torch.empty((Cc,), dtype=torch.float32, device=dev)
        db = torch.empty((Cc,), dtype=torch.float32, device=dev)
        work = ops._work(L.load().cor_ln_rows_work_bytes(rows, Cc), dev)
        ops._call("cor_ln_rows_bwd", dev, ops.ptr(gy), L.dtype_code(gy), ops.ptr(x), ops.ptr(w), ops.ptr(b), ops.ptr(stats), ops._ll(rows), Cc, act, ops.ptr(dx),
                  ops.ptr(dw), ops.ptr(db), ops.ptr(work))
        return dx, dw.to(wdt), db.to(wdt), None, None, None


def ln_rows(x: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor, eps: float = 1e-6, act: Optional[str] = None,
            out_bf16: bool = False) -> torch.Tensor:
    """Row-wise LayerNorm over the last axis of x [rows, C] (+ optional GELU), biased variance -- both data formats of the
    reference's LayerNorm (mask_adapter.py:226-251) once the tensor is laid out channels-last.  ``out_bf16`` writes the next
    GEMM's A operand directly."""
    return _LnRowsFn.apply(x, weight, bias, float(eps), _ACTS[act], bool(out_bf16))


class _LnCfFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, eps, act):
        dev = L.require_cuda(x, weight, bias)
        xc = x.float().contiguous()
        N, Cc = xc.shape[0], xc.shape[1]
        P = xc[0, 0].numel()
        w, b = weight.detach().float().contiguous(), bias.detach().float().contiguous()
        y = torch.empty_like(xc)
        ops._call("cor_ln_cf_fwd", dev, ops.ptr(xc), ops.ptr(w), ops.ptr(b), ops._ll(N), Cc, ops._ll(P), ops._f(eps), int(act), ops.ptr(y))
        ctx.save_for_backward(xc, w, b)
        ctx.cfg = (float(eps), int(act), weight.dtype, x.dtype)
        return y

    @staticmethod
    def backward(ctx, gy):
        xc, w, b = ctx.saved_tensors
        eps, act, wdt, xdt = ctx.cfg
        dev = xc.device
        N, Cc = xc.shape[0], xc.shape[1]
        P = xc[0, 0].numel()
        gy = gy.float().contiguous()
        dx = torch.empty_like(xc)
        dw = torch.empty((Cc,), dtype=torch.float32, device=dev)
        db = torch.empty((Cc,), dtype=torch.float32, device=dev)
        work = ops._work(L.load().cor_ln_cf_work_bytes(N, Cc, P), dev)
        ops._call("cor_ln_cf_bwd", dev, ops.ptr(gy), ops.ptr(xc), ops.ptr(w), ops.ptr(b), ops._ll(N), Cc, ops._ll(P), ops._f(eps), act,
                  ops.ptr(dx), ops.ptr(dw), ops.ptr(db), ops.ptr(work))
        return dx.to(xdt), dw.to(wdt), db.to(wdt), None, None


def ln_channels_first(x: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor, eps: float = 1e-6, act: Optional[str] = None) -> torch.Tensor:
    """LayerNorm over dim 1 of x [N, C, *spatial] (C <= 32) + optional GELU in one launch -- the reference's
    LayerNorm(data_format="channels_first") (mask_adapter.py:240-251) as used inside mask_downscaling (:128-142)."""
    return _LnCfFn.apply(x, weight, bias, float(eps), _ACTS[act])


class _DwConv7Fn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x_rows, weight, bias, n, h, w):
        dev = L.require_cuda(x_rows, weight, bias)
        x = x_rows.float().contiguous()
        Cc = x.shape[1]
        wt = weight.float().reshape(Cc, 49).contiguous()
        b = bias.float().contiguous() if bias is not None else None
        out = torch.empty_like(x)
        ops._call("cor_dwconv7_cl", dev, ops.ptr(x), ops.ptr(wt), ops.ptr(b), ops.ptr(out), n, h, w, Cc, 0)
        ctx.save_for_backward(x, wt)
        ctx.cfg = (n, h, w, weight.dtype, tuple(weight.shape), bias is not None, x_rows.requires_grad, weight.requires_grad)
        return out

    @staticmethod
    def backward(ctx, gy):
        x, wt = ctx.saved_tensors
        n, h, w, wdt, wshape, has_b, need_x, need_w = ctx.cfg
        dev = x.device
        Cc = x.shape[1]
        gy = gy.float().contiguous()
        gx = gw = gb = None
        if need_x:
            gx = torch.empty_like(x)
            ops._call("cor_dwconv7_cl", dev, ops.ptr(gy), ops.ptr(wt), None, ops.ptr(gx), n, h, w, Cc, 1)       # flipped kernel
        if need_w or has_b:
            gw32 = torch.empty((Cc, 49), dtype=torch.float32, device=dev)
            gb32 = torch.empty((Cc,), dtype=torch.float32, device=dev) if has_b else None
            work = ops._work(L.load().cor_dwconv7_work_bytes(n, h, w, Cc), dev)
            ops._call("cor_dwconv7_cl_wgrad", dev, ops.ptr(x), ops.ptr(gy), ops.ptr(gw32), ops.ptr(gb32), n, h, w, Cc, ops.ptr(work))
            gw = gw32.view(wshape).to(wdt)
            gb = gb32.to(wdt) if has_b else None
        return gx, gw, gb, None, None, None


def dwconv7_rows(x_rows: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor], n: int, h: int, w: int) -> torch.Tensor:
    """Depth-wise 7x7 convolution (padding 3) of n maps given as channels-last rows [n*h*w, C] -> rows of the same shape:
    ``nn.Conv2d(C, C, 7, padding=3, groups=C)`` (mask_adapter.py:196-199) without leaving the rows layout."""
    return _DwConv7Fn.apply(x_rows, weight, bias, int(n), int(h), int(w))


def dwconv7_ok(Cc: int, h: int, w: int) -> bool:
    return Cc % 32 == 0 and (w + 6) * 7 * 32 * 4 * 2 <= 200 * 1024
