"""torch-facing operators over libcor_b200.so: thin autograd wrappers, no arithmetic of their own.

PyTorch here is plumbing (device memory, streams, autograd tape); every number is produced by the
CUDA kernels behind the C ABI in include/cor_b200.h.  All ops raise on non-CUDA tensors.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import Optional

import torch

from . import _lib as L
from ._lib import BF16, F32, U8, W_CLAMP, W_PLAIN, W_SIGMOID, CorError, check, dtype_code, ptr, require_cuda, stream_ptr

__all__ = [
    "mask_prep", "region_pool", "fgbg_losses", "seg_loss", "l2_normalize", "similarity", "infonce_loss",
    "topk_retrieve", "val_postprocess", "RegionPool", "W_PLAIN", "W_CLAMP", "W_SIGMOID", "seg_coef", "clear_caches",
]

_f = C.c_float
_i = C.c_int
_ll = C.c_longlong

# launch counter: bench.py reports how many of OUR kernels ran inside the timed region
LAUNCHES = {"count": 0}
_KERNELS_PER_CALL = {
    "cor_mask_prep": 2, "cor_pool_stream_fwd": 1, "cor_pool_umma_fwd": 1, "cor_rows_finalize": 1,
    "cor_rows_finalize_bwd": 1, "cor_pool_bwd_feat": 1, "cor_pool_bwd_umma": 1, "cor_pool_bwd_maps": 1, "cor_fgbg_loss_fwd": 2,
    "cor_fgbg_loss_bwd": 1, "cor_seg_loss_fwd": 2, "cor_seg_loss_bwd": 1, "cor_sim_stream_fwd": 2,
    "cor_sim_umma_fwd": 2, "cor_infonce_bwd_umma": 3, "cor_gemm_bf16": 1, "cor_cast_cat_bf16": 1, "cor_act_bwd": 2, "cor_ln_rows_fwd": 1, "cor_ln_rows_bwd": 2, "cor_dwconv7_cl": 1, "cor_dwconv7_cl_wgrad": 2,
    "cor_hyper_logits_fwd": 1, "cor_hyper_logits_bwd": 2, "cor_sim_lse_parts": 1, "cor_infonce_tail": 1, "cor_infonce_fwd": 1, "cor_infonce_bwd": 2, "cor_topk": 1, "cor_l2_normalize": 1,
    "cor_val_post": 3, "cor_soft_metrics": 2, "cor_step_tail_fwd": 1, "cor_step_tail_bwd": 1,
    # device-resident logit scale: the same kernels; the tensor-core backward adds one fold launch when the scale's
    # gradient is wanted
    "cor_sim_stream_fwd_ls": 2, "cor_sim_umma_fwd_ls": 2, "cor_sim_lse_parts_ls": 1, "cor_infonce_tail_ls": 1, "cor_infonce_fwd_ls": 1,
    "cor_infonce_bwd_ls": 2, "cor_infonce_bwd_umma_ls": 4, "cor_step_tail_fwd_ls": 1, "cor_step_tail_bwd_ls": 1,
    "cor_peer_gather_sim_ls": 1,
    # cross-batch region memory: cor_memory_dq is 2 launches, 3 with the logit scale's gradient (its caller passes the count)
    "cor_memory_reset": 1, "cor_memory_enqueue": 1, "cor_memory_scan": 1, "cor_infonce_tail_mem": 1, "cor_step_tail_fwd_mem": 1,
    "cor_memory_dq": 2,
    # top-k without S: the selecting similarity kernel, then select / re-score / sort
    "cor_topk_select": 2,
}


# optional per-call CUDA-event timing (bench.py's roofline leg): {"name": [(start, end), ...]}
TIMING = {"events": None}


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _call(name: str, dev, *args, launches: Optional[int] = None):
    """One C-ABI call on ``dev``'s current stream.  Host cost matters for the launch-bound small shapes (a few dozen calls
    per module forward): the device guard is taken only when ``dev`` is not already current and the stream handle comes
    from the raw accessor (no Stream object).  ``launches`` overrides the table's kernel count for entries whose count
    depends on their arguments."""
    lib = L.load()
    ev = TIMING["events"]
    idx = dev.index
    if ev is None and idx is not None and _raw_stream is not None and torch.cuda.current_device() == idx:
        rc = getattr(lib, name)(*args, L.C.c_void_p(_raw_stream(idx)))
    else:
        with torch.cuda.device(dev):
            if ev is not None:
                st = torch.cuda.current_stream()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(st)
                rc = getattr(lib, name)(*args, stream_ptr())
                b.record(st)
                ev.setdefault(name, []).append((a, b))
            else:
                rc = getattr(lib, name)(*args, stream_ptr())
    LAUNCHES["count"] += _KERNELS_PER_CALL.get(name, 1) if launches is None else launches
    check(rc, name)


def _work(nbytes: int, dev) -> torch.Tensor:
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=dev)


def _as_supported_float(t: torch.Tensor) -> torch.Tensor:
    if t.dtype not in (torch.float32, torch.bfloat16):
        t = t.float()
    return t.contiguous()


def _mask_scale(masks: torch.Tensor, mask_scale: Optional[float]) -> float:
    if mask_scale is not None:
        return float(mask_scale)
    return 1.0 / 255.0 if masks.dtype == torch.uint8 else 1.0


# --------------------------------------------------------------------------------------------------
# mask resample + sums
# --------------------------------------------------------------------------------------------------
def mask_prep(masks: torch.Tensor, hw, transform: int = W_PLAIN, want_f32: bool = True, bf16_out: Optional[torch.Tensor] = None,
              group: int = 0, group_stride: int = 0, mask_scale: Optional[float] = None):
    """masks [N,Hm,Wm] (f32/bf16/u8) -> (w_f32 [N,h*w] or None, stats [N,4]).  If ``bf16_out`` is
    given (a [*, ldw=h*w]-rowed bf16 buffer) transform(r) is also written there, row of mask n at
    (n // group) * group_stride + (n % group) * h*w elements."""
    dev = require_cuda(masks, bf16_out)
    if masks.dtype not in (torch.float32, torch.bfloat16, torch.uint8):
        masks = masks.float()
    masks = masks.contiguous()
    N, Hm, Wm = masks.shape
    h, w = int(hw[0]), int(hw[1])
    P = h * w
    lib = L.load()
    w32 = torch.empty((N, P), dtype=torch.float32, device=dev) if want_f32 else None
    stats = torch.empty((N, 4), dtype=torch.float32, device=dev)
    work = _work(lib.cor_mask_prep_work_bytes(N, Hm, Wm, h, w), dev)
    _call("cor_mask_prep", dev, ptr(masks), dtype_code(masks), _f(_mask_scale(masks, mask_scale)), N, Hm, Wm, h, w,
          int(transform), ptr(w32), ptr(bf16_out), _ll(P), int(group), _ll(group_stride), ptr(stats), ptr(work))
    return w32, stats


# --------------------------------------------------------------------------------------------------
# region pooling
# --------------------------------------------------------------------------------------------------
@dataclass
class RegionPool:
    """Result of :func:`region_pool`."""
    fg: torch.Tensor                      # [B, R/G, C] f32 (unit rows when normalize)
    bg: Optional[torch.Tensor]            # [B, R/G, C] f32 or None
    stats: torch.Tensor                   # [B*R, 4] {sum m, sum 1-m, den, den_bf16}
    fg_bf16: Optional[torch.Tensor] = None
    engine: str = "stream"


_umma_w_cache = {}


def _umma_weight_buffer(dev, B, Rp, R, P, ones_row=True):
    """Cached bf16 weight operand [B, Rp, P] of the tensor-core pooling GEMM: rows < R are rewritten by
    mask_prep every call, padding rows stay zero, and (with ``ones_row``) row R is all ones so that its
    pooled sum is sum_p F -- the background by subtraction."""
    key = (dev.index, B, Rp, R, P, bool(ones_row))
    buf = _umma_w_cache.get(key)
    if buf is None:
        # never evicted: a captured CUDA graph (StepBuffers.capture) holds the raw pointer.  One buffer per shape, so
        # calls of the same shape must stay on one stream at a time; clear_caches() frees them explicitly.
        buf = torch.zeros((B, Rp, P), dtype=torch.bfloat16, device=dev)
        if ones_row:
            buf[:, R, :] = 1.0
        _umma_w_cache[key] = buf
    buf._cor_epoch = getattr(buf, "_cor_epoch", 0) + 1       # every hand-out precedes a rewrite by mask_prep: a backward that
    return buf                                                # wants these weights checks that no later forward replaced them


def clear_caches():
    """Free the cached operand buffers.  Only when no captured graph that used them will be replayed again."""
    _umma_w_cache.clear()


def umma_pool_eligible(feat: torch.Tensor, R: int, P: int, transform: int, group: int, pair: bool = True) -> bool:
    """Shapes the tcgen05 pooling GEMM serves: bf16 features, 16 <= R, R (+1 ones row when the background
    is wanted) <= 256 (UMMA N), whole 64-pixel K blocks and 128-channel M tiles."""
    C = feat.shape[1]
    return (feat.dtype == torch.bfloat16 and R >= 16 and R + (1 if pair else 0) <= 256 and P % 64 == 0 and C % 128 == 0
            and transform in (W_PLAIN, W_CLAMP) and group == 1)


class _RegionPoolFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feat, masks, transform, normalize, pair, group, eps, mask_scale, engine, want_bf16):
        dev = require_cuda(feat, masks)
        feat_c = _as_supported_float(feat)
        B, Cc, h, w = feat_c.shape
        P = h * w
        if masks.dim() != 4 or masks.shape[0] != B:
            raise CorError(f"region_pool: masks must be [B,R,H,W] with B={B}, got {tuple(masks.shape)}")
        R = masks.shape[1]
        if R % group:
            raise CorError(f"region_pool: R={R} not divisible by group={group}")
        flat = masks.reshape(B * R, masks.shape[2], masks.shape[3])
        need_w32 = True
        use_umma = engine == "umma" or (engine == "auto" and umma_pool_eligible(feat_c, R, P, transform, group, pair))
        if use_umma and not umma_pool_eligible(feat_c, R, P, transform, group, pair):
            raise CorError("region_pool: engine='umma' needs bf16 features, 16 <= R <= 256 (255 with background rows), P % 64 == 0, C % 128 == 0")
        rows_out = B * R // group
        fg = torch.empty((rows_out, Cc), dtype=torch.float32, device=dev)
        bg = torch.empty((rows_out, Cc), dtype=torch.float32, device=dev) if pair else None
        fg16 = torch.empty((rows_out, Cc), dtype=torch.bfloat16, device=dev) if want_bf16 else None
        inv_fg = torch.empty((rows_out,), dtype=torch.float32, device=dev)
        inv_bg = torch.empty((rows_out,), dtype=torch.float32, device=dev) if pair else None
        lib = L.load()
        if use_umma:
            Rp = (R + (1 if pair else 0) + 15) // 16 * 16
            w16 = _umma_weight_buffer(dev, B, Rp, R, P, ones_row=pair)
            need_w32 = feat.requires_grad      # backward runs on the fp32 weights
            w32, stats = mask_prep(flat, (h, w), transform, want_f32=need_w32, bf16_out=w16, group=R, group_stride=Rp * P,
                                   mask_scale=mask_scale)
            ks = lib.cor_pool_umma_ksplit(B, Cc, P)
            part = torch.empty((ks, B, Rp, Cc), dtype=torch.float32, device=dev)   # split-K partials; row R = sum_p F
            _call("cor_pool_umma_fwd", dev, ptr(feat_c), ptr(w16), B, Cc, P, Rp, ptr(part))
            den_col = 3
            fg_sum = None
            split = B * Rp * Cc
            _call("cor_rows_finalize", dev, ptr(part), R, _ll(Rp * Cc), ks, _ll(split), ptr(stats[:, den_col:]), 4, _f(eps), B * R, Cc,
                  1, int(normalize), None, _f(0.0), ptr(fg), ptr(fg16), ptr(inv_fg))
            if pair:
                all_sum = part[0, :, R, :]        # view: image b at b * Rp * C floats, split k at k * split
                _call("cor_rows_finalize", dev, ptr(part), R, _ll(Rp * Cc), ks, _ll(split), ptr(stats[:, den_col:]), 4, _f(eps), B * R,
                      Cc, 1, int(normalize), ptr(all_sum), _f(float(P)), ptr(bg), None, ptr(inv_bg))
            bg_sum = None
        else:
            den_col = 2
            w32, stats = mask_prep(flat, (h, w), transform, want_f32=True, mask_scale=mask_scale)
            fg_sum = torch.empty((B, R, Cc), dtype=torch.float32, device=dev)
            bg_sum = torch.empty((B, R, Cc), dtype=torch.float32, device=dev) if pair else None
            _call("cor_pool_stream_fwd", dev, ptr(feat_c), dtype_code(feat_c), ptr(w32), _ll(P), B, Cc, P, R, int(transform),
                  ptr(fg_sum), ptr(bg_sum))
            _call("cor_rows_finalize", dev, ptr(fg_sum), 0, _ll(0), 1, _ll(0), ptr(stats[:, den_col:]), 4, _f(eps), B * R, Cc, int(group),
                  int(normalize), None, _f(0.0), ptr(fg), ptr(fg16), ptr(inv_fg))
            if pair:
                # background denominators: P - den  (sum_p (1 - w))
                den_bg = (float(P) - stats[:, den_col]).contiguous()
                ctx.den_bg = den_bg
                _call("cor_rows_finalize", dev, ptr(bg_sum), 0, _ll(0), 1, _ll(0), ptr(den_bg), 1, _f(eps), B * R, Cc, int(group),
                      int(normalize), None, _f(0.0), ptr(bg), None, ptr(inv_bg))
        ctx.cfg = (B, Cc, h, w, R, int(transform), bool(normalize), bool(pair), int(group), float(eps), den_col, use_umma,
                   feat_c.dtype, feat.dtype, tuple(masks.shape))
        ctx.feat_needs = feat.requires_grad
        ctx.engine = engine
        ctx.maps_need = masks.requires_grad
        saved_feat = feat_c if masks.requires_grad else None
        ctx.save_for_backward(w32 if need_w32 else None, stats, fg, bg, inv_fg, inv_bg, saved_feat,
                              fg_sum if masks.requires_grad else None)
        ctx.mark_non_differentiable(stats)
        ctx.set_materialize_grads(False)
        outs = (fg.view(B, R // group, Cc), bg.view(B, R // group, Cc) if pair else None, stats, fg16)
        if fg16 is not None:
            ctx.mark_non_differentiable(fg16)
        return outs

    @staticmethod
    def backward(ctx, g_fg, g_bg, _g_stats, _g16):
        w32, stats, fg, bg, inv_fg, inv_bg, feat_c, fg_sum = ctx.saved_tensors
        (B, Cc, h, w, R, transform, normalize, pair, group, eps, den_col, use_umma, feat_dtype, feat_in_dtype,
         mask_shape) = ctx.cfg
        dev = fg.device
        P = h * w
        g_feat = g_maps = None
        if not (ctx.feat_needs or ctx.maps_need) or (g_fg is None and g_bg is None):
            return (None,) * 10
        if w32 is None:
            raise CorError("region_pool backward: fp32 weights were not saved")
        zeros = None
        if g_fg is None:
            zeros = torch.zeros_like(fg)
        gs_fg = torch.empty((B * R, Cc), dtype=torch.float32, device=dev)
        _call("cor_rows_finalize_bwd", dev, ptr((g_fg.reshape(-1, Cc).float().contiguous() if g_fg is not None else zeros)),
              ptr(fg), ptr(inv_fg), ptr(stats[:, den_col:]), 4, _f(eps), B * R, Cc, group, int(normalize), 0, _f(0.0), ptr(gs_fg))
        gs_bg = None
        if pair and g_bg is not None:
            gs_bg = torch.empty((B * R, Cc), dtype=torch.float32, device=dev)
            if use_umma:
                _call("cor_rows_finalize_bwd", dev, ptr(g_bg.reshape(-1, Cc).float().contiguous()), ptr(bg), ptr(inv_bg),
                      ptr(stats[:, den_col:]), 4, _f(eps), B * R, Cc, group, int(normalize), 1, _f(float(P)), ptr(gs_bg))
            else:
                _call("cor_rows_finalize_bwd", dev, ptr(g_bg.reshape(-1, Cc).float().contiguous()), ptr(bg), ptr(inv_bg),
                      ptr(ctx.den_bg), 1, _f(eps), B * R, Cc, group, int(normalize), 0, _f(0.0), ptr(gs_bg))
        if ctx.feat_needs:
            g_feat_c = torch.empty((B, Cc, h, w), dtype=feat_dtype, device=dev)
            tc = ctx.engine != "stream" and L.load().cor_pool_bwd_umma_ok(B, Cc, P, R, int(gs_bg is not None))
            _call("cor_pool_bwd_umma" if tc else "cor_pool_bwd_feat", dev, ptr(gs_fg), ptr(gs_bg), ptr(w32), _ll(P), B, Cc, P, R,
                  transform, ptr(g_feat_c), L._DTYPES[feat_dtype])
            g_feat = g_feat_c if feat_in_dtype == feat_dtype else g_feat_c.to(feat_in_dtype)
        if ctx.maps_need:
            if transform != W_SIGMOID:
                raise CorError("region_pool backward: only sigmoid maps (MaskAdapter tail) are differentiable; masks carry no grad")
            if tuple(mask_shape[2:]) != (h, w):
                raise CorError("region_pool backward: maps must already be at the feature resolution")
            den = stats[:, den_col].contiguous()
            pooled = fg_sum.reshape(B * R, Cc) / den[:, None]
            g_pooled = gs_fg * den[:, None]
            g_maps = torch.empty((B * R, P), dtype=torch.float32, device=dev)
            _call("cor_pool_bwd_maps", dev, ptr(feat_c), L._DTYPES[feat_c.dtype], ptr(w32), _ll(P), ptr(g_pooled), ptr(pooled),
                  ptr(den), B, Cc, P, R, ptr(g_maps))
            g_maps = g_maps.view(mask_shape)
        return g_feat, g_maps, None, None, None, None, None, None, None, None


def region_pool(feat: torch.Tensor, masks: torch.Tensor, *, transform: int = W_CLAMP, normalize: bool = True, pair: bool = False,
                group: int = 1, eps: float = 1e-8, mask_scale: Optional[float] = None, engine: str = "auto",
                want_bf16: bool = False) -> RegionPool:
    """Mask-guided region pooling: feat [B,C,h,w] x masks [B,R,H,W] -> [B,R/group,C].

    row(b,r) = sum_p w F / (sum_p w + eps) with w = transform(bilinear(mask)); optional mean over
    groups of ``group`` rows, optional L2-normalise, optional background rows (w -> 1-w).
    engine: "stream" (CUDA-core, exact fp32), "umma" (tcgen05 tensor cores, bf16 operands) or "auto".
    """
    fg, bg, stats, fg16 = _RegionPoolFn.apply(feat, masks, int(transform), bool(normalize), bool(pair), int(group), float(eps),
                                              mask_scale, engine, bool(want_bf16))
    return RegionPool(fg=fg, bg=bg, stats=stats, fg_bf16=fg16)


# --------------------------------------------------------------------------------------------------
# fg / bg cosine losses
# --------------------------------------------------------------------------------------------------
def _rows2d(t: torch.Tensor):
    """[n,C] f32 view with unit inner stride (row stride may exceed C: no copy for strided slices)."""
    if t.dtype != torch.float32:
        t = t.float()
    if t.dim() != 2 or t.stride(1) != 1:
        t = t.reshape(t.shape[0], -1).contiguous()
    return t


class _FgBgFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, fg_rows, bg_rows, comb, stats, bg_mode):
        dev = require_cuda(fg_rows, bg_rows, comb, stats)
        n, Cc = fg_rows.shape
        if comb.numel() != n * Cc or (bg_rows is not None and tuple(bg_rows.shape) != (n, Cc)):
            raise CorError(f"fgbg_losses: pooled rows are [{n},{Cc}] but comb has {tuple(comb.shape)}"
                           + (f" and bg rows {tuple(bg_rows.shape)}" if bg_rows is not None else "")
                           + " (the composed query must have the feature map's channel count)")
        fg_c = _rows2d(fg_rows)
        bg_c = _rows2d(bg_rows) if bg_rows is not None else None
        comb_c = _rows2d(comb)
        stats_c = _rows2d(stats)
        lib = L.load()
        out4 = torch.empty(4, dtype=torch.float32, device=dev)
        aux = torch.empty(lib.cor_fgbg_aux_floats(n, Cc), dtype=torch.float32, device=dev)
        _call("cor_fgbg_loss_fwd", dev, ptr(fg_c), _ll(fg_c.stride(0)), ptr(bg_c), _ll(bg_c.stride(0) if bg_c is not None else 0),
              ptr(comb_c), _ll(comb_c.stride(0)), ptr(stats_c), _ll(stats_c.stride(0)), n, Cc, int(bg_mode), ptr(out4), ptr(aux))
        ctx.save_for_backward(fg_c, bg_c, comb_c, out4, aux)
        ctx.bg_mode = int(bg_mode)
        ctx.comb_dtype = comb.dtype
        ctx.comb_shape = tuple(comb.shape)
        return out4[:2].clone(), out4[2:].clone()

    @staticmethod
    def backward(ctx, g2, _gcount):
        fg_c, bg_c, comb_c, out4, aux = ctx.saved_tensors
        dev = fg_c.device
        n, Cc = fg_c.shape
        g2 = g2.float().contiguous()
        g_fg = torch.empty((n, Cc), dtype=torch.float32, device=dev)
        g_bg = torch.empty((n, Cc), dtype=torch.float32, device=dev) if bg_c is not None else None
        g_comb = torch.empty((n, Cc), dtype=torch.float32, device=dev)
        _call("cor_fgbg_loss_bwd", dev, ptr(fg_c), _ll(fg_c.stride(0)), ptr(bg_c), _ll(bg_c.stride(0) if bg_c is not None else 0),
              ptr(comb_c), _ll(comb_c.stride(0)), n, Cc, ctx.bg_mode, ptr(out4), ptr(aux), ptr(g2), _ll(1), _f(1.0), _f(1.0), ptr(g_fg), _ll(Cc), 0, ptr(g_bg),
              _ll(Cc), ptr(g_comb), _ll(Cc), 0)
        return g_fg, g_bg, g_comb.view(ctx.comb_shape).to(ctx.comb_dtype), None, None


def fgbg_losses(fg_rows: torch.Tensor, bg_rows: Optional[torch.Tensor], comb: torch.Tensor, stats: torch.Tensor,
                bg_mode: int = 0):
    """(losses[2] = {fg, bg}, counts[2] = {#valid fg, #valid bg}) from pooled unit rows [n,C], the
    composed queries [n,C] and the mask_prep stats [n,4].  bg_mode 0 = reference broadcast form."""
    return _FgBgFn.apply(fg_rows, bg_rows, comb, stats, bg_mode)


# --------------------------------------------------------------------------------------------------
# segmentation loss
# --------------------------------------------------------------------------------------------------
def seg_coef(**terms) -> tuple:
    """Coefficient vector of the segmentation loss: seg_coef(wbce=1, wiou=1) is loss_func.py:31."""
    names = ("wbce", "wiou", "dice", "bce", "iou", "wdice", "focal")
    bad = set(terms) - set(names)
    if bad:
        raise CorError(f"seg_coef: unknown terms {sorted(bad)} (known: {names})")
    return tuple(float(terms.get(n, 0.0)) for n in names)


def _coef_array(coef):
    return (C.c_float * L.SEG_NTERMS)(*coef)


class _SegLossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred, mask, coef, mask_scale, focal_alpha, focal_gamma, dice_smooth):
        dev = require_cuda(pred, mask)
        pred_c = _as_supported_float(pred)
        if mask.dtype not in (torch.float32, torch.bfloat16, torch.uint8):
            mask = mask.float()
        if pred_c.dim() != 4 or mask.dim() != 4 or pred_c.shape[:2] != mask.shape[:2]:
            raise CorError(f"seg_loss: pred {tuple(pred.shape)} and mask {tuple(mask.shape)} must be [N,C,H,W] with equal N,C")
        Hm, Wm = mask.shape[2:]
        # a [N,1,H,W] slice of a larger [N,M,H,W] tensor is read in place through its sample stride (no copy)
        if mask.shape[1] == 1 and mask.stride(3) == 1 and mask.stride(2) == Wm and mask.stride(0) >= Hm * Wm:
            mask_c, nstride = mask, mask.stride(0)
        else:
            mask_c, nstride = mask.contiguous(), Hm * Wm
        N = pred_c.shape[0] * pred_c.shape[1]
        H, W = pred_c.shape[2:]
        lib = L.load()
        out8 = torch.empty(8, dtype=torch.float32, device=dev)
        per = torch.empty((N, lib.cor_seg_loss_npartials()), dtype=torch.float32, device=dev)
        need = pred.requires_grad
        t_save = torch.empty((N, H, W), dtype=torch.float32, device=dev) if need else None
        w_save = torch.empty((N, H, W), dtype=torch.float32, device=dev) if need else None
        work = _work(lib.cor_seg_loss_work_bytes(N, H, W), dev)
        _call("cor_seg_loss_fwd", dev, ptr(pred_c), dtype_code(pred_c), ptr(mask_c), dtype_code(mask_c),
              _f(_mask_scale(mask_c, mask_scale)), N, H, W, Hm, Wm, _ll(nstride), _coef_array(coef), _f(focal_alpha), _f(focal_gamma),
              _f(dice_smooth), ptr(out8), ptr(per), ptr(t_save), ptr(w_save), ptr(work))
        ctx.save_for_backward(pred_c, t_save, w_save, per)
        ctx.cfg = (N, H, W, tuple(coef), float(dice_smooth), float(focal_alpha), float(focal_gamma), pred.dtype)
        return out8[0].clone(), out8.clone()

    @staticmethod
    def backward(ctx, g_loss, _g_extra):
        pred_c, t_save, w_save, per = ctx.saved_tensors
        N, H, W, coef, dice_smooth, focal_alpha, focal_gamma, in_dtype = ctx.cfg
        dev = pred_c.device
        g = g_loss.reshape(1).float().contiguous()
        g_pred = torch.empty_like(pred_c)
        _call("cor_seg_loss_bwd", dev, ptr(pred_c), dtype_code(pred_c), ptr(t_save), ptr(w_save), ptr(per), N, H, W, _coef_array(coef),
              _f(dice_smooth), _f(focal_alpha), _f(focal_gamma), ptr(g), ptr(g_pred), dtype_code(g_pred))
        return g_pred.to(in_dtype), None, None, None, None, None, None


def seg_loss(pred: torch.Tensor, mask: torch.Tensor, w1: float = 1.0, w2: float = 1.0, mask_scale: Optional[float] = None,
             focal_alpha: float = 0.25, focal_gamma: float = 2.0, dice_smooth: float = 1.0, return_extras: bool = False,
             coef: Optional[tuple] = None):
    """Weighted BCE + weighted IoU (loss_func.py:5-32); ``mask`` may be at any resolution -- it is
    bilinearly resampled to the logit grid inside the kernel (trainer_v3_g.py:67).  ``coef``
    (:func:`seg_coef`) selects another combination of the seven per-sample terms the kernel produces
    (dice / plain bce / iou / weighted dice / focal are Class N); all of them are differentiable.
    With ``return_extras`` also returns the 8-vector {loss, dice, focal, wbce, wiou, bce, iou, wdice}."""
    if coef is None:
        coef = seg_coef(wbce=w1, wiou=w2)
    want_focal = return_extras or coef[L.SEG_FOCAL] != 0.0       # the focal term is a powf per pixel: only on request
    loss, extra = _SegLossFn.apply(pred, mask, tuple(coef), mask_scale, float(focal_alpha),
                                   float(focal_gamma) if want_focal else -1.0, float(dice_smooth))
    return (loss, extra) if return_extras else loss


# --------------------------------------------------------------------------------------------------
# L2 normalise, similarity, InfoNCE, top-k
# --------------------------------------------------------------------------------------------------
class _L2NormFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, want_bf16):
        dev = require_cuda(x)
        xc = _as_supported_float(x)
        D = xc.shape[-1]
        n = xc.numel() // D
        y = torch.empty((n, D), dtype=torch.float32, device=dev)
        y16 = torch.empty((n, D), dtype=torch.bfloat16, device=dev) if want_bf16 else None
        inv = torch.empty((n,), dtype=torch.float32, device=dev)
        _call("cor_l2_normalize", dev, ptr(xc), dtype_code(xc), n, D, ptr(y), ptr(y16), ptr(inv))
        ctx.save_for_backward(y, inv)
        ctx.shape = tuple(x.shape)
        ctx.in_dtype = x.dtype
        if y16 is not None:
            ctx.mark_non_differentiable(y16)
        return y.view(x.shape), (y16.view(x.shape) if y16 is not None else None)

    @staticmethod
    def backward(ctx, g, _g16):
        y, inv = ctx.saved_tensors
        dev = y.device
        n, D = y.shape
        gc = g.reshape(n, D).float().contiguous()
        ones = torch.ones((n,), dtype=torch.float32, device=dev)
        gx = torch.empty((n, D), dtype=torch.float32, device=dev)
        _call("cor_rows_finalize_bwd", dev, ptr(gc), ptr(y), ptr(inv), ptr(ones), 1, _f(0.0), n, D, 1, 1, 0, _f(0.0), ptr(gx))
        return gx.view(ctx.shape).to(ctx.in_dtype), None


def l2_normalize(x: torch.Tensor, want_bf16: bool = False):
    """x / max(||x||_2, 1e-12) along the last dim (support_branch.py:85).  Returns f32 (and bf16)."""
    y, y16 = _L2NormFn.apply(x, want_bf16)
    return (y, y16) if want_bf16 else y


def _sim_engine(Nq: int, Nr: int, D: int, engine: str) -> str:
    if engine != "auto":
        return engine
    # tensor-core kernel: whenever the tile shape fits and either there are enough queries to fill an MMA or the
    # region stream is long (measured at 16 x 102 400 x 256: 31.7 us against 144 us for the streaming kernel)
    if D % 64 == 0 and 64 <= D <= 256 and (Nq >= 32 or Nr >= 8192):
        return "umma"
    return "stream"


def check_logit_scale(logit_scale: Optional[torch.Tensor], tau: Optional[float], who: str) -> None:
    """A logit scale replaces ``tau``: a 0-dim fp32 CUDA tensor, never passed together with ``tau``."""
    if logit_scale is None:
        return
    if tau is not None:
        raise CorError(f"{who}: pass either tau or logit_scale, not both")
    if not isinstance(logit_scale, torch.Tensor) or logit_scale.dim() != 0 or logit_scale.dtype != torch.float32:
        raise CorError(f"{who}: logit_scale must be a 0-dim float32 tensor, got "
                       + (f"shape {tuple(logit_scale.shape)} {logit_scale.dtype}" if isinstance(logit_scale, torch.Tensor) else repr(logit_scale)))
    if not logit_scale.is_cuda:
        raise CorError(f"{who}: logit_scale must be a CUDA tensor (the kernels read it from device memory)")


def _tau_arg(name: str, inv_tau: float, scale: Optional[torch.Tensor]):
    """(entry name, argument) of an InfoNCE entry: the float inv_tau, or the ``_ls`` twin that reads the device scale."""
    return (name, _f(inv_tau)) if scale is None else (name + "_ls", ptr(scale))


def _tail_entry(name: str, inv_tau: float, scale: Optional[torch.Tensor], mem_args: Optional[tuple]):
    """(entry name, tau-position arguments) of an InfoNCE tail entry: the choice of ``_tau_arg``, or with a region memory's
    ``mem_args`` = (mem_part, mem_nparts, mem_state) the ``_mem`` twin, which takes inv_tau and the scale (NULL: inv_tau)."""
    if mem_args is None:
        name, ta = _tau_arg(name, inv_tau, scale)
        return name, (ta,)
    return name + "_mem", (_f(inv_tau), ptr(scale), *mem_args)


def _sim_forward(r16, q16, inv_tau, want_S, want_lse, engine, scale=None):
    dev = r16.device
    Nr, D = r16.shape
    Nq = q16.shape[0]
    lib = L.load()
    S = torch.empty((Nq, Nr), dtype=torch.float32, device=dev) if want_S else None
    lse = torch.empty((Nq,), dtype=torch.float32, device=dev) if want_lse else None
    work = _work(lib.cor_sim_work_bytes(Nq, Nr, D), dev)
    name, ta = _tau_arg("cor_sim_umma_fwd" if _sim_engine(Nq, Nr, D, engine) == "umma" else "cor_sim_stream_fwd", inv_tau, scale)
    _call(name, dev, ptr(r16), ptr(q16), Nr, Nq, D, ta, ptr(S), ptr(lse), ptr(work))
    return S, lse


def _sim_lse_parts(r16, q16, inv_tau, engine, scale=None):
    """Similarity producer that leaves its log-sum-exp partials in a work buffer: (work, nparts, qt) for cor_infonce_tail."""
    import ctypes as C
    dev = r16.device
    Nr, D = r16.shape
    Nq = q16.shape[0]
    lib = L.load()
    work = _work(lib.cor_sim_work_bytes(Nq, Nr, D), dev)
    nparts, qt = C.c_int(0), C.c_int(0)
    eng = 1 if _sim_engine(Nq, Nr, D, engine) == "umma" else 0
    name, ta = _tau_arg("cor_sim_lse_parts", inv_tau, scale)
    _call(name, dev, eng, ptr(r16), ptr(q16), Nr, Nq, D, ta, ptr(work), C.byref(nparts), C.byref(qt))
    return work, nparts.value, qt.value


def check_memory(memory, D: int, dev, who: str) -> None:
    """A region memory (``region.RegionMemory``) serves queries of its own width on its own device."""
    if memory is None:
        return
    if not all(hasattr(memory, a) for a in ("bank", "state", "K", "C", "enqueues")):
        raise CorError(f"{who}: memory must be a RegionMemory, got {type(memory).__name__}")
    if memory.C != D:
        raise CorError(f"{who}: the memory holds rows of width C={memory.C}, the queries have D={D}")
    if dev is not None and memory.bank.device != dev:
        raise CorError(f"{who}: the memory is on {memory.bank.device}, the call on {dev}")


def _memory_scan_work(memory, Nq: int, D: int, dev) -> torch.Tensor:
    return _work(L.load().cor_memory_scan_work_bytes(Nq, memory.K, D), dev)


def _memory_scan(memory, q16, inv_tau, scale=None, work=None):
    """Log-sum-exp partials of the queries against the memory's valid rows (tensor cores): (work, nparts) for the
    ``_mem`` tail entries.  ``work``: a buffer from _memory_scan_work allocated on the stream that consumes the partials."""
    dev = q16.device
    Nq, D = q16.shape
    if work is None:
        work = _memory_scan_work(memory, Nq, D, dev)
    nparts = C.c_int(0)
    _call("cor_memory_scan", dev, ptr(memory.bank), memory.K, ptr(memory.state), ptr(q16), Nq, D, _f(inv_tau), ptr(scale), ptr(work),
          C.byref(nparts))
    return work, nparts.value


def _memory_dq(memory, q16, lse, inv_tau, scale, g_loss, g_mul, g_queries, g_scale):
    """ADD the memory rows' share of the InfoNCE gradient into g_queries [Nq, D] and g_scale (either may be None)."""
    if g_queries is None and g_scale is None:
        return
    dev = q16.device
    Nq, D = q16.shape
    work = _work(L.load().cor_memory_dq_work_bytes(Nq, memory.K, D), dev)
    _call("cor_memory_dq", dev, ptr(memory.bank), memory.K, ptr(memory.state), ptr(q16), Nq, D, _f(inv_tau), ptr(scale), ptr(lse),
          ptr(g_loss), _f(g_mul), ptr(g_queries), ptr(g_scale), ptr(work), launches=1 + (g_queries is not None) + (g_scale is not None))


def check_memory_unchanged(mem_rec, who: str) -> None:
    """A backward over memory rows needs the rows its forward scored: refuse it after an enqueue in between."""
    if mem_rec is not None and mem_rec[0].enqueues != mem_rec[1]:
        raise CorError(f"{who}: the region memory was enqueued between forward and backward, so the rows the forward scored "
                       "may have been overwritten; enqueue after backward()")


def _to_bf16_rows(x: torch.Tensor) -> torch.Tensor:
    """[.., D] -> bf16 [rows, D] on our own cast kernel (fp32 input) -- not an ATen copy."""
    x2 = x.reshape(-1, x.shape[-1])
    if x2.dtype == torch.bfloat16:
        return x2.contiguous()
    x2 = x2.float().contiguous()
    out = torch.empty(x2.shape, dtype=torch.bfloat16, device=x2.device)
    _call("cor_cast_cat_bf16", x2.device, ptr(x2), x2.shape[1], None, 0, _ll(x2.shape[0]), ptr(out))
    return out


def similarity(regions: torch.Tensor, queries: torch.Tensor, engine: str = "auto") -> torch.Tensor:
    """S[q, r] = <queries[q], regions[r]> with bf16 operands and fp32 accumulation: [Nq, Nr] f32."""
    require_cuda(regions, queries)
    S, _ = _sim_forward(_to_bf16_rows(regions), _to_bf16_rows(queries), 1.0, True, False, engine)
    return S


def _infonce_bwd_dense(Nq: int, Nr: int, D: int, engine: str) -> bool:
    """Dense (GEMM) InfoNCE backward for the many-query regime; the streaming kernel keeps the few-query one (a rank's
    own queries against gathered regions) and everything the tensor-core similarity kernel does not take."""
    if engine == "stream":
        return False
    return Nq >= 128 and D in (64, 128, 192, 256) and Nq * Nr >= (1 << 19)


class _InfoNCEFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, regions, queries, targets, tau, engine, regions_bf16, logit_scale, memory):
        dev = require_cuda(regions, queries, targets, logit_scale)
        check_memory(memory, queries.shape[-1], dev, "infonce_loss")
        r16 = regions_bf16.reshape(-1, regions_bf16.shape[-1]).contiguous() if regions_bf16 is not None else _to_bf16_rows(regions)
        q16 = _to_bf16_rows(queries)
        Nr, D = r16.shape
        Nq = q16.shape[0]
        tg = targets.to(torch.int64).contiguous()
        inv_tau = 1.0 / float(tau) if logit_scale is None else 0.0
        _, lse = _sim_forward(r16, q16, inv_tau, False, True, engine, logit_scale)
        loss = torch.empty(1, dtype=torch.float32, device=dev)
        tgt = torch.empty((Nq,), dtype=torch.float32, device=dev)
        if memory is None:
            name, ta = _tau_arg("cor_infonce_fwd", inv_tau, logit_scale)
            _call(name, dev, ptr(r16), ptr(q16), ptr(tg), ptr(lse), Nr, Nq, D, ta, ptr(loss), ptr(tgt))
        else:
            # the tail entry in its lse-in form: it merges the memory's partials into the current rows' lse (in place) and
            # forms the loss as cor_infonce_fwd does, so an empty memory changes no bit
            mwork, mparts = _memory_scan(memory, q16, inv_tau, logit_scale)
            name, tas = _tail_entry("cor_infonce_tail", inv_tau, logit_scale, (ptr(mwork), mparts, ptr(memory.state)))
            _call(name, dev, None, 0, 0, ptr(r16), ptr(q16), ptr(tg), Nr, Nq, D, *tas, ptr(lse), ptr(loss), ptr(tgt), None, None,
                  _f(0.0), _f(0.0), _f(0.0), None)
        ctx.mem = None if memory is None else (memory, memory.enqueues)
        # the scale is saved as an input: an in-place write to it before backward trips autograd's version check
        ctx.save_for_backward(r16, q16, tg, lse, logit_scale)
        ctx.engine = engine
        ctx.cfg = (inv_tau, regions.dtype, queries.dtype, tuple(regions.shape), tuple(queries.shape),
                   regions.requires_grad, queries.requires_grad)
        return loss[0].clone()

    @staticmethod
    def backward(ctx, g):
        check_memory_unchanged(ctx.mem, "infonce_loss backward")
        r16, q16, tg, lse, sc = ctx.saved_tensors
        inv_tau, rdt, qdt, rshape, qshape, r_need, q_need = ctx.cfg
        s_need = sc is not None and ctx.needs_input_grad[6]
        dev = r16.device
        Nr, D = r16.shape
        Nq = q16.shape[0]
        lib = L.load()
        gl = g.reshape(1).float().contiguous()
        gs = torch.empty((), dtype=torch.float32, device=dev) if s_need else None
        gs_arg = () if sc is None else (ptr(gs),)
        if _infonce_bwd_dense(Nq, Nr, D, ctx.engine):
            # hundreds of queries: both products on our tensor-core kernel (csrc/nce_bwd_umma.cu) -- the S tile is
            # recomputed, turned into bf16 coefficients in registers and fed straight back as an MMA operand; no S, no P,
            # no library GEMM.  The scale's gradient comes out of the dQ launch, which therefore runs whenever it is wanted.
            gq = torch.empty((Nq, D), dtype=torch.float32, device=dev) if q_need else None
            gr = torch.empty((Nr, D), dtype=torch.float32, device=dev) if r_need else None
            work = _work(lib.cor_infonce_bwd_umma_work_bytes(Nq, Nr, D), dev)
            name, ta = _tau_arg("cor_infonce_bwd_umma", inv_tau, sc)
            _call(name, dev, ptr(r16), ptr(q16), Nr, Nq, D, ta, ptr(lse), ptr(tg), ptr(gl), _f(1.0), ptr(gr), ptr(gq), *gs_arg, ptr(work))
        else:
            gr = torch.empty((Nr, D), dtype=torch.float32, device=dev)
            gq = torch.empty((Nq, D), dtype=torch.float32, device=dev)
            work = _work(lib.cor_sim_work_bytes(Nq, Nr, D), dev)
            name, ta = _tau_arg("cor_infonce_bwd", inv_tau, sc)
            _call(name, dev, ptr(r16), ptr(q16), ptr(tg), ptr(lse), Nr, Nq, D, ta, ptr(gl), _f(1.0), ptr(gr), ptr(gq), *gs_arg, ptr(work))
        if ctx.mem is not None:          # the memory rows' share, added into what the current rows' backward wrote
            _memory_dq(ctx.mem[0], q16, lse, inv_tau, sc, gl, 1.0, gq if q_need else None, gs)
        return ((gr.view(rshape).to(rdt) if r_need else None), (gq.view(qshape).to(qdt) if q_need else None), None, None, None, None, gs,
                None)


def infonce_loss(regions: torch.Tensor, queries: torch.Tensor, targets: torch.Tensor, tau: Optional[float] = None, engine: str = "auto",
                 regions_bf16: Optional[torch.Tensor] = None, logit_scale: Optional[torch.Tensor] = None, memory=None) -> torch.Tensor:
    """mean_q CE(s * S[q,:], targets[q]) with S = queries @ regions^T (bf16 operands, fp32 accumulate) and s = 1/tau
    (tau defaults to 0.07).  Gradients flow straight through the bf16 rounding to ``regions`` and ``queries``.

    ``logit_scale``: a learnable temperature -- a 0-dim float32 CUDA tensor s > 0 used in place of 1/tau (pass one or
    the other).  The kernels read it from device memory, and when it requires grad d loss / d s reaches it through
    autograd, e.g. ``logit_scale = log_s.exp()`` with a parameter ``log_s`` as in CLIP.

    ``memory``: a ``region.RegionMemory`` whose valid rows join the negatives of every query (never a target, no gradient
    of their own); the queries and the scale get the memory terms of their gradient.  Enqueue into it after backward()."""
    check_logit_scale(logit_scale, tau, "infonce_loss")
    check_memory(memory, queries.shape[-1], None, "infonce_loss")
    return _InfoNCEFn.apply(regions, queries, targets, 0.07 if tau is None else float(tau), engine, regions_bf16, logit_scale, memory)


# Measured on one B200 at 1000 W (profiles/r06_topk_bench.log), D = 256: at k = 10 the fused path takes 2.65 against
# 12.5 ms at 256 x 1 M and 24.7 against 75.1 ms at 4 096 x 1 M, but 0.195 against 0.040 ms at 256 x 4 096 (S in L2);
# at k = 256 the S route wins at every size measured, up to S = 16 GB (4 096 x 1 M).  Beyond 16 GB of S the fused path is
# taken whatever k: its memory does not grow with the gallery.  Sizes between the measured points are not measured.
_TOPK_FUSED_MAX_K = 10
_TOPK_FUSED_MIN_ROWS = 1 << 20
_TOPK_S_MAX_BYTES = 16 << 30


def _topk_fused(Nq: int, Nr: int, D: int, k: int, engine: str) -> bool:
    """Top-k that selects inside the tensor-core similarity kernel (cor_topk_select) instead of writing S."""
    if engine not in ("auto", "umma") or D not in (64, 128, 192, 256):
        return False
    return (k <= _TOPK_FUSED_MAX_K and Nr >= _TOPK_FUSED_MIN_ROWS) or Nq * Nr * 4 > _TOPK_S_MAX_BYTES


def _topk_select(r16: torch.Tensor, q16: torch.Tensor, k: int):
    """cor_topk_select on bf16 rows: (idx, score) without writing S."""
    dev = r16.device
    Nr, D = r16.shape
    Nq = q16.shape[0]
    idx = torch.empty((Nq, k), dtype=torch.int64, device=dev)
    score = torch.empty((Nq, k), dtype=torch.float32, device=dev)
    work = _work(L.load().cor_topk_select_work_bytes(Nq, Nr, D, int(k)), dev)
    _call("cor_topk_select", dev, ptr(r16), ptr(q16), Nr, Nq, D, int(k), ptr(idx), ptr(score), ptr(work))
    return idx, score


def topk_retrieve(regions: torch.Tensor, queries: torch.Tensor, k: int, engine: str = "auto"):
    """Per query the k best regions under (score desc, index asc): (idx [Nq,k] int64, score [Nq,k] f32), 1 <= k <=
    min(Nr, 256).  Prefilter on tensor-core / streaming scores, exact fp64 re-score of the top k+slack candidates.

    With ``engine`` "auto" or "umma", D in {64, 128, 192, 256} and either k <= 10 on a gallery of at least 2^20 rows or
    a score matrix S of more than 16 GB, the tensor-core similarity kernel keeps each query's candidates while it
    scores, so S [Nq, Nr] is never written: the call's memory is the gallery, the queries, the outputs and
    ``cor_topk_select_work_bytes`` of scratch, which does not grow with Nr.  Other shapes write S (on the tensor cores,
    or on the CUDA cores with ``engine="stream"`` and other widths) and select from it, which measured faster there.
    A gallery of bf16 rows is read in place; fp32 rows are first cast to a bf16 copy."""
    if regions.shape[-1] != queries.shape[-1]:
        raise CorError(f"topk_retrieve: regions {tuple(regions.shape)} and queries {tuple(queries.shape)} differ in width")
    Nr = regions.numel() // max(regions.shape[-1], 1)
    if not 1 <= int(k) <= min(Nr, 256):
        raise CorError(f"topk_retrieve: need 1 <= k <= min(Nr, 256), got k={k} with Nr={Nr}")
    dev = require_cuda(regions, queries)
    r16, q16 = _to_bf16_rows(regions), _to_bf16_rows(queries)
    Nr, D = r16.shape
    Nq = q16.shape[0]
    if _topk_fused(Nq, Nr, D, int(k), engine):
        return _topk_select(r16, q16, int(k))
    idx = torch.empty((Nq, k), dtype=torch.int64, device=dev)
    score = torch.empty((Nq, k), dtype=torch.float32, device=dev)
    S, _ = _sim_forward(r16, q16, 1.0, True, False, engine)
    _call("cor_topk", dev, ptr(S), ptr(r16), ptr(q16), Nr, Nq, D, int(k), ptr(idx), ptr(score))
    return idx, score


# --------------------------------------------------------------------------------------------------
# validation post-process
# --------------------------------------------------------------------------------------------------
def val_postprocess(pred: torch.Tensor, size=None, gt: Optional[torch.Tensor] = None, want_post: bool = True,
                    want_hard: bool = False, gt_scale: Optional[float] = None, post_first: bool = False):
    """sigmoid + per-sample min-max of (optionally upsampled) logits; returns dict with ``post``
    [N,1,Ho,Wo] f32, ``hard`` uint8 (0/255), ``metrics`` [N,5] {dice,mae,iou,mdice,miou} if gt given.
    ``post_first=False`` is the in-training validation order (resize logits, then sigmoid + min-max,
    trainer_v3_g.py:226-231); ``post_first=True`` is the offline evaluator's (sigmoid + min-max at the logit
    size, then bilinear resize of the map to the ground-truth size and > 0.5, vailder.py:427-430,466,473)."""
    dev = require_cuda(pred, gt)
    pc = _as_supported_float(pred)
    if pc.dim() != 4 or pc.shape[1] != 1:
        raise CorError(f"val_postprocess: pred must be [N,1,H,W], got {tuple(pred.shape)}")
    N, _, H, W = pc.shape
    Ho, Wo = (H, W) if size is None else (int(size[0]), int(size[1]))
    lib = L.load()
    post = torch.empty((N, 1, Ho, Wo), dtype=torch.float32, device=dev) if want_post else None
    hard = torch.empty((N, 1, Ho, Wo), dtype=torch.uint8, device=dev) if want_hard else None
    metrics = None
    gc = None
    if gt is not None:
        gc = gt if gt.dtype in (torch.float32, torch.uint8) else gt.float()
        gc = gc.contiguous()
        if gc.numel() != N * Ho * Wo:
            raise CorError("val_postprocess: gt must have the output resolution")
        metrics = torch.empty((N, 5), dtype=torch.float32, device=dev)
    work = _work(lib.cor_val_post_work_bytes(N, Ho, Wo), dev)
    _call("cor_val_post", dev, ptr(pc), dtype_code(pc), N, H, W, Ho, Wo, int(post_first), ptr(post), ptr(hard), ptr(gc),
          (dtype_code(gc) if gc is not None else F32), _f(_mask_scale(gc, gt_scale) if gc is not None else 1.0), ptr(metrics), ptr(work))
    return {"post": post, "hard": hard, "metrics": metrics}


def soft_metrics(pred: torch.Tensor, gt: torch.Tensor, smooth: float = 1e-5, gt_scale: Optional[float] = None) -> torch.Tensor:
    """[N,5] = {dice, mae, iou, mdice, miou} of utils/trainer_v3_g.py:381-443 in one pass over (pred, gt)."""
    dev = require_cuda(pred, gt)
    if pred.shape != gt.shape:
        raise CorError(f"Shape mismatch: pred {tuple(pred.shape)} vs gt {tuple(gt.shape)}")
    N = pred.shape[0]
    pc = pred.reshape(N, -1).float().contiguous()
    gc = gt.reshape(N, -1)
    gc = (gc if gc.dtype in (torch.float32, torch.uint8) else gc.float()).contiguous()
    lib = L.load()
    out = torch.empty((N, 5), dtype=torch.float32, device=dev)
    work = _work(lib.cor_val_post_work_bytes(N, 1, 1), dev)
    _call("cor_soft_metrics", dev, ptr(pc), ptr(gc), dtype_code(gc), _f(_mask_scale(gc, gt_scale)), N, _ll(pc.shape[1]), _f(smooth),
          ptr(out), ptr(work))
    return out
