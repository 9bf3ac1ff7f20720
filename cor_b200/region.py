"""Region-level retrieval and scoring (north-star extensions, "Class N" in SURVEY.md section 0):
multi-mask region pooling, the full region x query similarity matrix, InfoNCE over (all-gathered)
negatives, top-k retrieval, and the fused training step the benchmark times.

None of these has a reference implementation; where they overlap the reference they reduce to it:
row (b,m) of ``pool_regions`` equals ``loss_func.mask_pooling(emb[b], masks[b,m])`` and the target
column of the similarity matrix equals the cosine inside ``fg_feat_similarity_loss``.
"""
from __future__ import annotations

import os
from dataclasses import dataclass
from typing import Optional

import torch

from . import dist as cdist
from . import ops
from . import peer
from ._lib import CorError

__all__ = ["pool_regions", "region_query_similarity", "region_infonce_loss", "topk_regions", "region_step", "RegionStepOut",
           "StepBuffers"]


def pool_regions(emb: torch.Tensor, masks: torch.Tensor, background: bool = False, engine: str = "auto", want_bf16: bool = True):
    """emb [B,C,h,w] x candidate masks [B,M,H,W] -> ops.RegionPool with unit rows fg [B,M,C]
    (and bg when ``background``), plus per-mask stats (validity, denominators)."""
    return ops.region_pool(emb, masks, transform=ops.W_CLAMP, normalize=True, pair=background, engine=engine, want_bf16=want_bf16)


def region_query_similarity(regions: torch.Tensor, queries: torch.Tensor, engine: str = "auto") -> torch.Tensor:
    """[Nr,D] unit region rows x [Nq,D] unit queries -> cosine matrix S [Nq,Nr] (bf16 operands, fp32 accumulate)."""
    return ops.similarity(regions, queries, engine)


def region_infonce_loss(regions: torch.Tensor, queries: torch.Tensor, targets: torch.Tensor, tau: Optional[float] = None,
                        gather: bool = True, engine: str = "auto", regions_bf16: Optional[torch.Tensor] = None,
                        logit_scale: Optional[torch.Tensor] = None) -> torch.Tensor:
    """InfoNCE of each local query against ALL regions.  With ``gather`` (and an initialised process
    group) the region rows are all-gathered across ranks first and ``targets`` -- indices into the
    LOCAL region rows -- are offset by rank * n_local.  tau (default 0.07) is a build choice (the reference defines
    none); ``logit_scale`` replaces 1/tau with a device tensor that can be learned (see ``ops.infonce_loss``).  Each
    rank's loss is the mean over its own queries, so the scale's gradient is rank-local, like the queries'."""
    ops.check_logit_scale(logit_scale, tau, "region_infonce_loss")
    regions = regions.reshape(-1, regions.shape[-1])
    rank, ws = cdist.world()
    if gather and ws > 1:
        n_local = regions.shape[0]
        regions = cdist.all_gather_rows(regions)
        targets = targets + rank * n_local
        regions_bf16 = None
    return ops.infonce_loss(regions, queries.reshape(-1, queries.shape[-1]), targets, tau, engine, regions_bf16, logit_scale)


def topk_regions(regions: torch.Tensor, queries: torch.Tensor, k: int, sharded: bool = False, engine: str = "auto"):
    """Top-k regions per query, total order (score desc, index asc).  With ``sharded`` each rank holds
    a contiguous, equal shard of the gallery: local top-k, all-gather of k*(score,idx), k-way merge.
    Takes no temperature or logit scale: a positive scale does not change the ranking."""
    idx, score = ops.topk_retrieve(regions, queries, min(k, regions.shape[0]), engine)
    rank, ws = cdist.world()
    if sharded and ws > 1:
        return cdist.merge_topk(idx, score, rank * regions.shape[0], k)
    return idx, score


@dataclass
class RegionStepOut:
    loss: torch.Tensor
    seg: torch.Tensor
    fg: torch.Tensor
    bg: torch.Tensor
    nce: torch.Tensor
    regions: torch.Tensor          # [B, M, C] unit rows (detached view for retrieval)


_target_cache = {}


def _target_rows(dev, B, M, offset):
    """Row index of every triplet's ground-truth region (b * M + offset), cached per shape."""
    key = (dev.index, B, M, offset)
    t = _target_cache.get(key)
    if t is None:
        # never evicted (a few bytes each): captured graphs hold the raw pointer
        t = torch.arange(B, device=dev, dtype=torch.int64) * M + offset
        _target_cache[key] = t
    return t


_side_streams = {}


def _side_stream(dev):
    """One extra stream per device for the branch of the step that does not depend on the pooled rows."""
    st = _side_streams.get(dev.index)
    if st is None:
        st = torch.cuda.Stream(device=dev)
        _side_streams[dev.index] = st
    return st


def _overlap_enabled():
    return os.environ.get("COR_STEP_OVERLAP", "1") != "0"


def _step_tail_ok(B: int, M: int, C: int, multi_rank: bool, bg_mode: int, sim_engine: str) -> bool:
    """Whether the fused step runs its region tail as one forward and one backward launch (csrc/step_tail.cu): one rank's
    rows only, bg_mode 0 and a streaming-similarity shape (<= 16 queries, C % 8 == 0, C <= 256).  ``COR_STEP_TAIL=0`` keeps
    the kernel chain it replaces (A/B)."""
    return (os.environ.get("COR_STEP_TAIL", "1") != "0" and not multi_rank and bg_mode == 0 and B <= 16 and C % 8 == 0 and C <= 256
            and ops._sim_engine(B, B * M, C, sim_engine) == "stream")


_tail_counters = {}


def _tail_counter(dev, B, M, C):
    """Zero-initialised arrival counters of the step-tail kernels, cached per shape: every launch leaves them zero again."""
    key = (dev.index, B, M, C)
    t = _tail_counters.get(key)
    if t is None:
        # never evicted (128 bytes each): captured graphs hold the raw pointer
        from . import _lib as L
        t = torch.zeros(L.load().cor_step_tail_counter_words(), dtype=torch.int32, device=dev)
        _tail_counters[key] = t
    return t


def _peer_fused_ok(n_queries: int, C: int, n_regions: int = 0, sim_engine: str = "auto") -> bool:
    """Shapes the fused gather + similarity kernel serves (a rank's <= 16 queries, one 16-byte vector per lane) and for which
    it wins: whenever the separate path would score on the streaming kernel.  Once the gathered gallery is large enough for
    the tensor-core similarity kernel (8 GPUs x 1024 regions) the pull kernel + that kernel measure 3 us faster per step
    (0.848 vs 0.851 ms at 8 GPUs; at 2 GPUs the fused kernel wins 0.8136 vs 0.8161 ms).  ``COR_PEER_FUSED=0`` / ``=2``
    force the separate / the fused kernels (A/B)."""
    knob = os.environ.get("COR_PEER_FUSED", "1")
    if knob == "0" or n_queries > 16 or C % 8 or C > 256:
        return False
    if knob == "2":
        return True
    return ops._sim_engine(n_queries, n_regions, C, sim_engine) != "umma"


class _FusedStepFn(torch.autograd.Function):
    """The whole region path as ONE autograd node: every kernel of the forward is launched back to
    back on the current stream, the backward is written out by hand, and no tensor glue (slices,
    zeros + scatter, tiny adds) sits between them.  Used by :func:`region_step` when the tensor-core
    pooling engine applies; the modular ops remain the general path."""

    @staticmethod
    def forward(ctx, pred, emb, comb, masks, tau, nce_weight, gather, sim_engine, bg_mode, w_fg, w_bg, logit_scale):
        from . import _lib as L
        ptr, _f, _ll, call = ops.ptr, ops._f, ops._ll, ops._call
        dev = L.require_cuda(pred, emb, comb, masks, logit_scale)
        sc = logit_scale                       # device logit scale (replaces 1/tau in every InfoNCE launch) or None
        tau_arg = lambda name, inv_tau: ops._tau_arg(name, inv_tau, sc)
        lib = L.load()
        B, M = masks.shape[:2]
        Cc, h, w = emb.shape[1:]
        P = h * w
        if masks.dtype not in (torch.float32, torch.bfloat16, torch.uint8):
            masks = masks.float()            # bool / fp16 / fp64 masks: one conversion serves mask_prep and the seg loss
        emb_c = emb.contiguous()
        pred_c = ops._as_supported_float(pred)
        comb_c = comb.reshape(B, -1).float().contiguous()
        f32 = dict(dtype=torch.float32, device=dev)
        need_emb = emb.requires_grad
        # 5. segmentation loss against the GT mask, resample fused.  It depends on neither the resampled weights nor the
        #    pooled rows, so it is issued FIRST, on a side stream (a parallel branch once the step is captured in a CUDA
        #    graph): its instruction-bound tiles run underneath the HBM-bound mask resample.
        gt = masks[:, 0]                       # [B,Hm,Wm] view; read in place through its sample stride
        Hm, Wm = gt.shape[1:]
        if not (gt.stride(2) == 1 and gt.stride(1) == Wm):
            gt = gt.contiguous()
        N = B
        H, W = pred_c.shape[2:]
        out8 = torch.empty(8, **f32)
        per = torch.empty((N, lib.cor_seg_loss_npartials()), **f32)
        need_pred = pred.requires_grad
        t_save = torch.empty((N, H, W), **f32) if need_pred else None
        w_save = torch.empty((N, H, W), **f32) if need_pred else None
        seg_work = ops._work(lib.cor_seg_loss_work_bytes(N, H, W), dev)
        cur = torch.cuda.current_stream(dev)
        side = _side_stream(dev) if _overlap_enabled() else None
        if side is not None:
            side.wait_stream(cur)
        # multi-GPU: the bf16 rows land directly in this rank's peer-mapped buffer (cor_b200/peer.py), else in a local one.
        # "Have my peers finished reading what I published last step?" is asked HERE, on the side stream at the very
        # start of the step (one 32-thread CTA polling local flags): by the time the row epilogue needs the answer the
        # 0.7 ms mask resample has gone by, so the wait never sits on the critical path.
        rank, ws = cdist.world()
        px = peer.get_exchange(B * M, Cc, dev) if (gather and ws > 1) else None
        ev_px = None
        if px is not None:
            with torch.cuda.stream(side if side is not None else cur):
                px.before_produce(0)
                if side is not None:
                    ev_px = torch.cuda.Event()
                    ev_px.record(side)
        q16 = torch.empty((B, comb_c.shape[1]), dtype=torch.bfloat16, device=dev)
        ev_q = None
        with torch.cuda.stream(side if side is not None else cur):
            call("cor_cast_cat_bf16", dev, ptr(comb_c), comb_c.shape[1], None, 0, _ll(B), ptr(q16))   # bf16 queries, off the main chain
            if side is not None:
                ev_q = torch.cuda.Event()
                ev_q.record(side)
            call("cor_seg_loss_fwd", dev, ptr(pred_c), L.dtype_code(pred_c), ptr(gt), L.dtype_code(gt), _f(ops._mask_scale(gt, None)), N, H, W,
                 Hm, Wm, _ll(gt.stride(0)), None, _f(0.25), _f(-1.0), _f(1.0), ptr(out8), ptr(per), ptr(t_save), ptr(w_save),
                 ptr(seg_work))
        # 1. masks -> bf16 weights (+ raw fp32 weights for the backward) + full-resolution stats
        Rp = (M + 1 + 15) // 16 * 16
        w16 = ops._umma_weight_buffer(dev, B, Rp, M, P)
        w32, stats = ops.mask_prep(masks.reshape(B * M, *masks.shape[2:]), (h, w), ops.W_CLAMP, want_f32=need_emb, bf16_out=w16,
                                   group=M, group_stride=Rp * P)
        # 2. pooling GEMM (split-K partials), 3. row epilogues: all fg rows, bg rows of the GT masks only
        ks = lib.cor_pool_umma_ksplit(B, Cc, P)
        part = torch.empty((ks, B, Rp, Cc), **f32)
        call("cor_pool_umma_fwd", dev, ptr(emb_c), ptr(w16), B, Cc, P, Rp, ptr(part))
        tail = _step_tail_ok(B, M, Cc, gather and ws > 1, int(bg_mode), sim_engine)
        ctx.tail = _tail_counter(dev, B, M, Cc) if tail else None
        if tail:
            # 3.-6. in ONE launch: unit rows (+ bf16 copy), their scores against the queries, the bg rows and fg / bg cosine
            # statistics of the GT masks, and in its last CTA the log-sum-exp merge, the InfoNCE, fg / bg losses and the total
            fg = torch.empty((B * M, Cc), **f32)
            fg16 = torch.empty((B * M, Cc), dtype=torch.bfloat16, device=dev)
            inv_fg = torch.empty((B * M,), **f32)
            bg = torch.empty((B, Cc), **f32)
            inv_bg = torch.empty((B,), **f32)
            out4 = torch.empty(4, **f32)
            aux = torch.empty(lib.cor_fgbg_aux_floats(B, Cc), **f32)
            r16, offset, ws, n_local = fg16, 0, 1, B * M
            targets = _target_rows(dev, B, M, 0)
            lse = torch.empty((B,), **f32)
            nce = torch.empty(1, **f32)
            tgt = torch.empty((B,), **f32)
            loss = torch.empty(1, **f32)
            inv_tau = 1.0 / float(tau)
            work = ops._work(lib.cor_step_tail_work_bytes(B, M, Cc), dev)
            if side is not None:
                cur.wait_stream(side)        # join: the total needs the segmentation loss, the scores the bf16 queries
            name, ta = tau_arg("cor_step_tail_fwd", inv_tau)
            call(name, dev, ptr(part), ks, _ll(B * Rp * Cc), Rp, B, M, Cc, _f(float(P)), ptr(stats), ptr(q16), ptr(comb_c),
                 ptr(targets), ta, ptr(out8), _f(w_fg), _f(w_bg), _f(nce_weight), ptr(fg), ptr(fg16), ptr(inv_fg), ptr(bg),
                 ptr(inv_bg), ptr(out4), ptr(aux), ptr(lse), ptr(nce), ptr(tgt), ptr(loss), ptr(work), ptr(ctx.tail))
        else:
            fg = torch.empty((B * M, Cc), **f32)
            fg16 = px.pub if px is not None else torch.empty((B * M, Cc), dtype=torch.bfloat16, device=dev)
            if ev_px is not None:
                cur.wait_event(ev_px)
            inv_fg = torch.empty((B * M,), **f32)
            split = B * Rp * Cc
            call("cor_rows_finalize", dev, ptr(part), M, _ll(Rp * Cc), ks, _ll(split), ptr(stats[:, 3:]), 4, _f(1e-8), B * M, Cc, 1, 1,
                 None, _f(0.0), ptr(fg), ptr(fg16), ptr(inv_fg))
            if px is not None:
                px.signal(0)                     # the bg rows, fg/bg loss and segmentation loss below hide the rank skew
            # 4. background rows + fg / bg cosine losses on the GT rows (row b*M of fg, row b of bg): a second branch off the
            #    fg rows, on the side stream, parallel to the similarity / InfoNCE chain below
            bg = torch.empty((B, Cc), **f32)
            inv_bg = torch.empty((B,), **f32)
            out4 = torch.empty(4, **f32)
            aux = torch.empty(lib.cor_fgbg_aux_floats(B, Cc), **f32)
            if side is not None:
                side.wait_stream(cur)
            with torch.cuda.stream(side if side is not None else cur):
                call("cor_rows_finalize", dev, ptr(part), 1, _ll(Rp * Cc), ks, _ll(split), ptr(stats[:, 3:]), 4 * M, _f(1e-8), B, Cc, 1, 1,
                     ptr(part[0, :, M, :]), _f(float(P)), ptr(bg), None, ptr(inv_bg))
                call("cor_fgbg_loss_fwd", dev, ptr(fg), _ll(M * Cc), ptr(bg), _ll(Cc), ptr(comb_c), _ll(Cc), ptr(stats), _ll(4 * M), B, Cc,
                     int(bg_mode), ptr(out4), ptr(aux))
            # 6. InfoNCE of every composed query against all (gathered) regions
            if ev_q is not None:
                cur.wait_event(ev_q)
            n_local = B * M
            inv_tau = 1.0 / float(tau)
            fused_parts = None
            if gather and ws > 1:
                r16 = torch.empty((ws * n_local, Cc), dtype=torch.bfloat16, device=dev)
                if px is not None and _peer_fused_ok(B, Cc, ws * n_local, sim_engine):
                    # ONE kernel: pull the peers' rows over NVLink, keep a local copy for the backward, and score every row
                    # against this rank's queries while it is in registers (all-gather fused with its consumer)
                    fused_parts = px.gather_sim(r16, q16, inv_tau, sc)
                elif px is not None:
                    px.gather(r16)               # our own pull-over-NVLink kernel: no NCCL on the data path
                else:
                    torch.distributed.all_gather_into_tensor(r16, fg16)
                offset = rank * n_local
            else:
                r16, offset, ws = fg16, 0, 1
            targets = _target_rows(dev, B, M, offset)
            nce = torch.empty(1, **f32)
            tgt = torch.empty((B,), **f32)
            loss = torch.empty(1, **f32)
            # similarity with its log-sum-exp partials left in the work buffer, then ONE tail kernel: partial merge -> lse,
            # target logits, InfoNCE mean and the step's total loss
            sim_work, nparts, qt = fused_parts if fused_parts is not None else ops._sim_lse_parts(r16, q16, inv_tau, sim_engine, sc)
            lse = torch.empty((B,), **f32)
            if side is not None:
                cur.wait_stream(side)        # join: the total needs the segmentation and fg/bg losses
            name, ta = tau_arg("cor_infonce_tail", inv_tau)
            call(name, dev, ptr(sim_work), nparts, qt, ptr(r16), ptr(q16), ptr(targets), r16.shape[0], B, Cc, ta,
                 ptr(lse), ptr(nce), ptr(tgt), ptr(out8), ptr(out4), _f(w_fg), _f(w_bg), _f(nce_weight), ptr(loss))
        # the scale is saved as an input: an in-place write to it before backward trips autograd's version check
        ctx.save_for_backward(pred_c, t_save, w_save, per, fg, bg, inv_fg, inv_bg, comb_c, stats, out4, aux, r16, q16, targets, lse, w32, sc)
        ctx.cfg = (B, M, Cc, h, w, float(inv_tau), float(nce_weight), int(bg_mode), float(w_fg), float(w_bg), ws, offset, n_local,
                   pred.dtype, emb.dtype, comb.dtype, tuple(comb.shape), need_pred, need_emb, comb.requires_grad)
        ctx.px = px
        ctx.w16 = (w16, getattr(w16, "_cor_epoch", -1))      # not a saved tensor: a cached operand buffer, validated by its epoch
        ctx.mark_non_differentiable(fg, out8, out4, nce)
        ctx.set_materialize_grads(False)     # no zero-filled gradients for the auxiliary outputs
        return loss[0], out8, out4, nce, fg

    @staticmethod
    def backward(ctx, g_loss, *_unused):
        from . import _lib as L
        ptr, _f, _ll, call = ops.ptr, ops._f, ops._ll, ops._call
        (pred_c, t_save, w_save, per, fg, bg, inv_fg, inv_bg, comb_c, stats, out4, aux, r16, q16, targets, lse, w32, sc) = ctx.saved_tensors
        (B, M, Cc, h, w, inv_tau, nce_weight, bg_mode, w_fg, w_bg, ws, offset, n_local, pred_dt, emb_dt, comb_dt, comb_shape,
         need_pred, need_emb, need_comb) = ctx.cfg
        dev = fg.device
        lib = L.load()
        P = h * w
        f32 = dict(dtype=torch.float32, device=dev)
        if g_loss is None:
            return (None,) * 12
        g = g_loss.reshape(1).float().contiguous()
        g_pred = g_emb = g_comb = None
        need_scale = sc is not None and ctx.needs_input_grad[11]
        # d loss / d scale: written by the InfoNCE backward over THIS rank's queries (the launch that writes g_queries)
        g_scale = torch.empty((), **f32) if need_scale else None
        tau_arg = lambda name: ops._tau_arg(name, inv_tau, sc)
        gs_arg = () if sc is None else (ptr(g_scale),)          # the _ls backward entries take the gradient pointer
        cur = torch.cuda.current_stream(dev)
        side = _side_stream(dev) if (_overlap_enabled() and need_pred) else None

        def seg_bwd():
            if not need_pred:
                return None
            N, H, W = t_save.shape
            gp = torch.empty_like(pred_c)
            if side is not None:
                side.wait_stream(cur)
            with torch.cuda.stream(side if side is not None else cur):
                call("cor_seg_loss_bwd", dev, ptr(pred_c), L.dtype_code(pred_c), ptr(t_save), ptr(w_save), ptr(per), N, H, W, None, _f(1.0),
                     _f(0.25), _f(-1.0), ptr(g), ptr(gp), L.dtype_code(gp))
            return gp

        px = ctx.px
        ev_px = None
        if px is not None and ws > 1:
            # same idea as in the forward: ask early, on the side stream, whether the peers are done with last step's `gall`
            if side is not None:
                side.wait_stream(cur)
                with torch.cuda.stream(side):
                    px.before_produce(1)
                    ev_px = torch.cuda.Event()
                    ev_px.record(side)
            else:
                px.before_produce(1)
        if px is None or side is not None:
            g_pred = seg_bwd()               # side stream: runs underneath the InfoNCE / pooling backward
        w16, w16_epoch = ctx.w16
        gemm_ok = bg_mode != 1 and w16 is not None and getattr(w16, "_cor_epoch", -1) == w16_epoch and Cc % 8 == 0 and P % 8 == 0
        if ctx.tail is not None and (gemm_ok or not need_emb):
            # ONE launch: InfoNCE + fg-loss gradient of every row, through the row epilogue, cast to bf16 into the K-padded
            # operand of the pooling-backward GEMM; and the query gradient (+ fg / bg terms) in extra CTAs, one set per query
            Kp = (M + 63) // 64 * 64
            a16 = torch.empty((B * Kp, Cc), dtype=torch.bfloat16, device=dev) if need_emb else None
            g_q = torch.empty((B, Cc), **f32) if need_comb else None
            work = ops._work(lib.cor_step_tail_work_bytes(B, M, Cc), dev)
            name, ta = tau_arg("cor_step_tail_bwd")
            call(name, dev, ptr(r16), ptr(q16), ptr(targets), ptr(lse), B, M, Cc, ta, ptr(g), _f(nce_weight),
                 ptr(fg), ptr(inv_fg), ptr(stats), ptr(comb_c), ptr(out4), ptr(aux), _f(w_fg), _f(w_bg), ptr(a16), Kp, ptr(g_q),
                 *gs_arg, ptr(work), ptr(ctx.tail))
            if need_comb:
                g_comb = g_q.view(comb_shape).to(comb_dt)
            if need_emb:
                from .linear import gemm
                Rp = w16.shape[1]
                out_dt = emb_dt if emb_dt in (torch.float32, torch.bfloat16) else torch.float32
                g_emb = gemm(a16, w16.view(B * Rp, P), Cc, P, Kp, a_mn=True, b_mn=True, batch=B, a_batch_rows=Kp, b_batch_rows=Rp,
                             out_dtype=out_dt).view(B, Cc, h, w).to(emb_dt)
        else:
            # InfoNCE backward first: it WRITES g_regions (this rank's rows) and g_queries ...
            Nr = r16.shape[0]
            g_regions = torch.empty((n_local, Cc), **f32)
            g_q = torch.empty((B, Cc), **f32)
            work = ops._work(lib.cor_sim_work_bytes(B, Nr, Cc), dev)
            if ws > 1:
                # gradient of every gathered row, then a reduce-scatter back to the owning rank: measured faster than a
                # collective-free backward that all-gathers the queries instead (profiles/README.md)
                if ev_px is not None:
                    cur.wait_event(ev_px)
                g_all = px.gall if px is not None else torch.empty((Nr, Cc), **f32)
                name, ta = tau_arg("cor_infonce_bwd")
                call(name, dev, ptr(r16), ptr(q16), ptr(targets), ptr(lse), Nr, B, Cc, ta, ptr(g), _f(nce_weight),
                     ptr(g_all), ptr(g_q), *gs_arg, ptr(work))
                if px is not None:
                    px.signal(1)
                    if side is None:
                        g_pred = seg_bwd()       # independent work between the signal and the pull hides the rank skew
                    px.reduce(g_regions)         # fixed rank order: bit-identical from run to run
                else:
                    torch.distributed.reduce_scatter_tensor(g_regions, g_all, op=torch.distributed.ReduceOp.SUM)
            else:
                name, ta = tau_arg("cor_infonce_bwd")
                call(name, dev, ptr(r16), ptr(q16), ptr(targets), ptr(lse), Nr, B, Cc, ta, ptr(g), _f(nce_weight),
                     ptr(g_regions), ptr(g_q), *gs_arg, ptr(work))
            # ... then the fg/bg backward ADDS its GT-row gradients into g_regions (row b*M) and g_queries
            g_bg = torch.empty((B, Cc), **f32) if bg_mode == 1 else None
            call("cor_fgbg_loss_bwd", dev, ptr(fg), _ll(M * Cc), ptr(bg), _ll(Cc), ptr(comb_c), _ll(Cc), B, Cc, bg_mode, ptr(out4), ptr(aux),
                 ptr(g), _ll(0), _f(w_fg), _f(w_bg), ptr(g_regions), _ll(M * Cc), 1, ptr(g_bg), _ll(Cc), ptr(g_q), _ll(Cc), 1)
            if need_comb:
                g_comb = g_q.view(comb_shape).to(comb_dt)
            if need_emb:
                gs_fg = torch.empty((B * M, Cc), **f32)
                call("cor_rows_finalize_bwd", dev, ptr(g_regions), ptr(fg), ptr(inv_fg), ptr(stats[:, 3:]), 4, _f(1e-8), B * M, Cc, 1, 1, 0,
                     _f(0.0), ptr(gs_fg))
                gs_bg_full = None
                if g_bg is not None:          # paired bg mode: background gradient lives on the GT rows only
                    gs_bg = torch.empty((B, Cc), **f32)
                    call("cor_rows_finalize_bwd", dev, ptr(g_bg), ptr(bg), ptr(inv_bg), ptr(stats[:, 3:]), 4 * M, _f(1e-8), B, Cc, 1, 1, 1,
                         _f(float(P)), ptr(gs_bg))
                    gs_bg_full = torch.zeros((B, M, Cc), **f32)
                    gs_bg_full[:, 0, :] = gs_bg
                g_emb_c = torch.empty((B, Cc, h, w), dtype=emb_dt if emb_dt in (torch.float32, torch.bfloat16) else torch.float32, device=dev)
                if gs_bg_full is None and gemm_ok:
                    # d emb[b] (C x P) = gs[b]^T (C x M) w[b] (M x P): one batched tcgen05 GEMM on the bf16 weights the forward's
                    # pooling GEMM used (still in their buffer: no later forward of this shape has rewritten them), both operands
                    # MN-major as they lie; the gradient rows are cast to bf16 and zero-padded to a whole 64-row K block, which makes
                    # the other operand's rows beyond M (the ones row, the next image) irrelevant.  Persistent tiles with coalesced
                    # stores: 2-3x faster than the one-shot pool_bwd_umma kernel, which rebuilds both operands from fp32.
                    from .linear import gemm
                    Kp = (M + 63) // 64 * 64
                    a16 = torch.empty((B * Kp, Cc), dtype=torch.bfloat16, device=dev)
                    call("cor_cast_pad_rows_bf16", dev, ptr(gs_fg), B, M, Kp, Cc, ptr(a16))
                    Rp = w16.shape[1]
                    g_emb_c = gemm(a16, w16.view(B * Rp, P), Cc, P, Kp, a_mn=True, b_mn=True, batch=B, a_batch_rows=Kp, b_batch_rows=Rp,
                                   out_dtype=g_emb_c.dtype).view(B, Cc, h, w)
                else:
                    name = "cor_pool_bwd_umma" if lib.cor_pool_bwd_umma_ok(B, Cc, P, M, int(gs_bg_full is not None)) else "cor_pool_bwd_feat"
                    call(name, dev, ptr(gs_fg), ptr(gs_bg_full), ptr(w32), _ll(P), B, Cc, P, M, ops.W_CLAMP, ptr(g_emb_c), L._DTYPES[g_emb_c.dtype])
                g_emb = g_emb_c.to(emb_dt)
        if side is not None:
            cur.wait_stream(side)
        if g_pred is not None:
            g_pred = g_pred.to(pred_dt)
        return g_pred, g_emb, g_comb, None, None, None, None, None, None, None, None, g_scale


def _fused_ok(emb, masks, pool_engine):
    B, M = masks.shape[:2]
    P = emb.shape[2] * emb.shape[3]
    return pool_engine in ("auto", "umma") and ops.umma_pool_eligible(emb, M, P, ops.W_CLAMP, 1, True) and emb.shape[1] % 8 == 0


def region_step(pred: torch.Tensor, emb: torch.Tensor, comb: torch.Tensor, masks: torch.Tensor, *, tau: Optional[float] = None,
                nce_weight: float = 1.0, gather: bool = True, pool_engine: str = "auto", sim_engine: str = "auto",
                bg_mode: int = 0, fused: bool = True, logit_scale: Optional[torch.Tensor] = None) -> RegionStepOut:
    """One forward of the whole region path for a batch of triplets with M candidate masks each
    (mask 0 of every image is the ground-truth ``query_mask``):

        seg  = wbce_with_wiou_loss(pred, resample(masks[:,0]))                 trainer_v3_g.py:67-68
        fg,bg = fg/bg_feat_similarity_loss(emb, comb, masks[:,0])              trainer_v3_g.py:69-71
        nce  = InfoNCE(comb_b vs all B*M (x world) pooled regions, target = region (b,0))   [Class N]
        loss = seg + 5 fg + 5 bg + nce_weight * nce

    The InfoNCE logits are S / tau (tau defaults to 0.07), or ``logit_scale * S`` for a learnable temperature:
    ``logit_scale`` is a 0-dim float32 tensor s > 0 on the step's device, passed instead of ``tau``.  The kernels read
    it from device memory, and d loss / d s reaches it through autograd when it requires grad.

    ONE pass over the masks and ONE pass over the feature map serve fg, bg and all M regions.  With bf16
    features and >= 16 masks the step runs as a single fused autograd node (tensor-core pooling, hand
    written backward); other shapes compose the modular ops.
    """
    ops.check_logit_scale(logit_scale, tau, "region_step")
    if logit_scale is not None and logit_scale.device != emb.device:
        raise CorError(f"region_step: logit_scale is on {logit_scale.device}, the step on {emb.device}")
    B, M = masks.shape[:2]
    if comb.shape[0] != B or emb.shape[0] != B or pred.shape[0] != B:
        raise CorError("region_step: batch sizes differ")
    if comb.numel() != B * emb.shape[1]:
        raise CorError(f"region_step: comb {tuple(comb.shape)} must hold one row of C={emb.shape[1]} channels per triplet "
                       "(the kernels read the queries with the feature map's row width)")
    if fused and _fused_ok(emb, masks, pool_engine) and pred.dim() == 4 and pred.shape[1] == 1:
        loss, out8, out4, nce, fg = _FusedStepFn.apply(pred, emb, comb, masks, 0.07 if tau is None else float(tau), float(nce_weight),
                                                       bool(gather), sim_engine, int(bg_mode), 5.0, 5.0, logit_scale)
        return RegionStepOut(loss=loss, seg=out8[0], fg=out4[0], bg=out4[1], nce=nce[0], regions=fg.view(B, M, -1))
    pool = ops.region_pool(emb, masks, transform=ops.W_CLAMP, normalize=True, pair=True, engine=pool_engine, want_bf16=True)
    Cc = pool.fg.shape[-1]
    q = comb.reshape(B, -1)
    gt_rows = torch.arange(B, device=emb.device) * M
    losses, _ = ops.fgbg_losses(pool.fg[:, 0, :], pool.bg[:, 0, :], q, pool.stats.view(B, M, 4)[:, 0, :], bg_mode)
    seg = ops.seg_loss(pred, masks[:, 0:1])
    nce = region_infonce_loss(pool.fg.reshape(B * M, Cc), q, gt_rows, tau, gather, sim_engine,
                              regions_bf16=pool.fg_bf16, logit_scale=logit_scale)
    loss = seg + 5 * losses[0] + 5 * losses[1] + nce_weight * nce
    return RegionStepOut(loss=loss, seg=seg, fg=losses[0], bg=losses[1], nce=nce, regions=pool.fg.detach())


class StepBuffers:
    """Static device buffers (+ a pinned loss slot) for the end-to-end call: the public entry a trainer
    uses when its batch arrives from a DataLoader on the host.  ``run`` copies this step's inputs
    host->device on the current stream, runs :func:`region_step` (+ backward) and returns the loss on
    the host, so the timed region of ``bench.py``'s e2e leg contains the copies.

    ``capture()`` records forward + backward of the step ONCE into a CUDA graph over these static
    buffers (launch-bound inner loop: ~30 small kernels); afterwards ``run`` / ``replay`` re-issue
    the whole step with a single graph launch.  Gradients land in ``self.grads``.

    ``capture(logit_scale=s)`` (s a 0-dim float32 tensor on the device) learns the temperature: the graph reads ``s``
    from device memory at every replay, so a value written into it (``s.copy_(log_s.exp())``) takes effect without a
    recapture, and d loss / d s lands in ``self.grads["logit_scale"]``, overwritten by every replay."""

    def __init__(self, B, M, C=256, h=64, w=64, H=1024, W=1024, hp=256, wp=256, D=None, device="cuda",
                 emb_dtype=torch.bfloat16, mask_dtype=torch.float32):
        if D is not None and D != C:
            raise CorError(f"StepBuffers: the composed query width D={D} must equal the feature channels C={C}")
        D = C
        self.device = torch.device(device)
        mk = lambda shape, dt: torch.empty(shape, dtype=dt, device=self.device)
        self.d = {"pred": mk((B, 1, hp, wp), emb_dtype), "emb": mk((B, C, h, w), emb_dtype), "comb": mk((B, 1, D), torch.float32),
                  "masks": mk((B, M, H, W), mask_dtype)}
        self.loss_host = torch.empty((), dtype=torch.float32).pin_memory()
        self._seed = torch.ones((), dtype=torch.float32, device=self.device)
        self.graph = None
        self.loss = None
        self.grads = {}
        self.launches_per_step = 0

    @property
    def h2d_bytes(self):
        return sum(t.numel() * t.element_size() for t in self.d.values())

    def load(self, src: dict):
        """Copy one batch (host pinned or device tensors) into the static buffers on the current stream."""
        for k, t in self.d.items():
            t.copy_(src[k], non_blocking=True)

    def _step(self, backward, emb_grad, kw):
        pred = self.d["pred"].detach().requires_grad_(backward)
        comb = self.d["comb"].detach().requires_grad_(backward)
        emb = self.d["emb"].detach().requires_grad_(backward and emb_grad)
        kw = dict(kw)
        scale = kw.pop("logit_scale", None)
        if scale is not None:
            scale = scale.detach().requires_grad_(backward)      # a leaf over the caller's storage: read in place
        out = region_step(pred, emb, comb, self.d["masks"], logit_scale=scale, **kw)
        if backward:
            out.loss.backward(gradient=self._seed)      # a resident 1.0: no per-step fill kernel from autograd
        grads = {"pred": pred.grad, "comb": comb.grad, "emb": emb.grad}
        if scale is not None:
            grads["logit_scale"] = scale.grad
        return out.loss.detach(), grads

    def capture(self, backward: bool = True, emb_grad: bool = True, warmup: int = 3, **kw):
        """Warm up on a side stream, then capture fwd+bwd of the step into a CUDA graph."""
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):
            for _ in range(warmup):
                self._step(backward, emb_grad, kw)
        torch.cuda.current_stream(self.device).wait_stream(side)
        torch.cuda.synchronize(self.device)
        n0 = ops.LAUNCHES["count"]
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self.loss, self.grads = self._step(backward, emb_grad, kw)
        self.launches_per_step = ops.LAUNCHES["count"] - n0
        self.graph = g
        return self

    def replay(self):
        self.graph.replay()
        ops.LAUNCHES["count"] += self.launches_per_step
        return self.loss

    def run(self, host: dict, backward: bool = True, emb_grad: bool = True, **kw) -> float:
        self.load(host)
        if self.graph is not None:
            loss = self.replay()
        else:
            loss, self.grads = self._step(backward, emb_grad, kw)
        self.loss_host.copy_(loss, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        if peer._CACHE:
            peer.check_all()             # a peer wait that expired (COR_PEER_TIMEOUT_S) invalidates the step: raise
        return float(self.loss_host)
