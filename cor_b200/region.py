"""Region-level retrieval and scoring (north-star extensions, "Class N" in SURVEY.md section 0):
multi-mask region pooling, the full region x query similarity matrix, InfoNCE over (all-gathered)
negatives, top-k retrieval, and the fused training step the benchmark times.

None of these has a reference implementation; where they overlap the reference they reduce to it:
row (b,m) of ``pool_regions`` equals ``loss_func.mask_pooling(emb[b], masks[b,m])`` and the target
column of the similarity matrix equals the cosine inside ``fg_feat_similarity_loss``.
"""
from __future__ import annotations

import functools
import os
from collections import namedtuple
from dataclasses import dataclass
from typing import Optional

import torch

from . import _lib as L
from . import dist as cdist
from . import ops
from . import peer
from ._lib import CorError
from .linear import gemm
from .ops import _f, _ll, ptr

__all__ = ["pool_regions", "region_query_similarity", "region_infonce_loss", "topk_regions", "region_step", "RegionStepOut",
           "StepBuffers", "RegionMemory"]


class RegionMemory:
    """Cross-batch memory of region embeddings (as XBM, "Cross-Batch Memory for Embedding Learning"): a ring of at most
    ``capacity`` bf16 unit rows of width ``C`` whose valid rows serve the InfoNCE of ``region_step``,
    ``region_infonce_loss`` and ``ops.infonce_loss`` (``memory=``) as extra negatives.  Memory rows are never targets and
    get no gradient; the queries and the logit scale get the memory terms of theirs.

    The head and fill count live in device memory ({head, count} in ``state``), so a captured CUDA graph that enqueues
    advances them at every replay.  Enqueue AFTER backward(): a backward whose forward scored the memory raises
    ``CorError`` if the memory was enqueued in between (``enqueues`` counts the calls on the host).  Each rank of a
    data-parallel job owns its memory and scores it against its own queries only.  C must be 64, 128, 192 or 256.

    Every slot also carries an int64 row id (``ids``, -1 = none), set by ``enqueue(rows, ids=...)``.  A call given
    ``query_ids`` leaves each query's same-id rows out of its negatives and its gradients: with the target object's id on
    the rows pushed from a step, a later step that looks for the same object does not score it as a negative (XBM keeps
    a label with every memory row for this reason)."""

    def __init__(self, capacity: int, C: int, device="cuda"):
        if int(capacity) < 1:
            raise CorError(f"RegionMemory: capacity must be >= 1, got {capacity}")
        if int(C) not in (64, 128, 192, 256):
            raise CorError(f"RegionMemory: C={C} must be 64, 128, 192 or 256 (the widths the tensor-core kernels take)")
        device = torch.device(device)
        if device.type != "cuda":
            raise CorError(f"RegionMemory: the memory lives on a CUDA device, got {device}")
        self.K, self.C = int(capacity), int(C)
        # zero rows: the last partly filled tile of a scan reads rows past the fill, which must be finite
        self.bank = torch.zeros((self.K, self.C), dtype=torch.bfloat16, device=device)
        self.state = torch.zeros(L.load().cor_memory_state_words(), dtype=torch.int32, device=device)
        self.ids = torch.full((self.K,), -1, dtype=torch.int64, device=device)
        self.enqueues = 0

    @property
    def device(self):
        return self.bank.device

    def enqueue(self, rows: torch.Tensor, ids: Optional[torch.Tensor] = None) -> None:
        """Push ``rows`` (fp32 or bf16 [..., C], e.g. ``RegionStepOut.regions``; 1 <= n <= capacity rows) as bf16 at the
        head, overwriting the oldest rows once full.  One kernel on the current stream, no host synchronisation.

        ``ids``: int64 row ids on the memory's device, shaped ``rows.shape[:-1]`` (one per row) or, for rows [B, M, C],
        [B]: the id of each image's row 0 (the ground-truth region of ``region_step``), its other rows getting -1.  Without
        ``ids`` every pushed row gets -1."""
        if rows.dtype not in (torch.float32, torch.bfloat16):
            raise CorError(f"RegionMemory.enqueue: rows must be float32 or bfloat16, got {rows.dtype}")
        if rows.dim() < 1 or rows.shape[-1] != self.C:
            raise CorError(f"RegionMemory.enqueue: rows {tuple(rows.shape)} must be [..., C={self.C}]")
        n = rows.numel() // self.C
        if not 1 <= n <= self.K:
            raise CorError(f"RegionMemory.enqueue: {n} rows, the memory takes 1 to {self.K} at once")
        dev = L.require_cuda(rows)
        if dev != self.device:
            raise CorError(f"RegionMemory.enqueue: rows on {dev}, the memory on {self.device}")
        group = 1
        if ids is not None:
            lead = tuple(rows.shape[:-1])
            if not isinstance(ids, torch.Tensor) or ids.dtype != torch.int64:
                raise CorError("RegionMemory.enqueue: ids must be an int64 tensor, got "
                               + (str(ids.dtype) if isinstance(ids, torch.Tensor) else type(ids).__name__))
            if rows.dim() == 3 and tuple(ids.shape) == lead[:1]:
                group = rows.shape[1]
            elif tuple(ids.shape) != lead:
                raise CorError(f"RegionMemory.enqueue: ids {tuple(ids.shape)} must be {lead} (one per row)"
                               + (f" or {lead[:1]} (one per image, on its row 0)" if rows.dim() == 3 else ""))
            if ids.device != self.device:
                raise CorError(f"RegionMemory.enqueue: ids on {ids.device}, the memory on {self.device}")
            ids = ids.contiguous()
        rc = rows.detach().reshape(n, self.C).contiguous()
        ops._call("cor_memory_enqueue_ids", dev, ops.ptr(rc), L.dtype_code(rc), n, self.C, ops.ptr(self.bank), self.K, ops.ptr(self.state),
                  ops.ptr(self.ids), ops.ptr(ids), group)
        self.enqueues += 1

    def reset(self) -> None:
        """Empty the memory (one memset of the state on the current stream)."""
        ops._call("cor_memory_reset", self.device, ops.ptr(self.state))
        self.enqueues += 1

    def count(self) -> int:
        """Valid rows (synchronises with the device)."""
        return int(self.state[1].item())

    def rows(self) -> torch.Tensor:
        """The valid rows, oldest first, as bf16 [count, C] (synchronises with the device)."""
        head, count = (int(v) for v in self.state[:2].tolist())
        if count < self.K:
            return self.bank[:count].clone()
        return torch.cat([self.bank[head:], self.bank[:head]])

    def row_ids(self) -> torch.Tensor:
        """The ids of the valid rows, oldest first, as int64 [count], in the order of ``rows()`` (synchronises)."""
        head, count = (int(v) for v in self.state[:2].tolist())
        if count < self.K:
            return self.ids[:count].clone()
        return torch.cat([self.ids[head:], self.ids[:head]])


def pool_regions(emb: torch.Tensor, masks: torch.Tensor, background: bool = False, engine: str = "auto", want_bf16: bool = True):
    """emb [B,C,h,w] x candidate masks [B,M,H,W] -> ops.RegionPool with unit rows fg [B,M,C]
    (and bg when ``background``), plus per-mask stats (validity, denominators)."""
    return ops.region_pool(emb, masks, transform=ops.W_CLAMP, normalize=True, pair=background, engine=engine, want_bf16=want_bf16)


def region_query_similarity(regions: torch.Tensor, queries: torch.Tensor, engine: str = "auto") -> torch.Tensor:
    """[Nr,D] unit region rows x [Nq,D] unit queries -> cosine matrix S [Nq,Nr] (bf16 operands, fp32 accumulate)."""
    return ops.similarity(regions, queries, engine)


def region_infonce_loss(regions: torch.Tensor, queries: torch.Tensor, targets: torch.Tensor, tau: Optional[float] = None,
                        gather: bool = True, engine: str = "auto", regions_bf16: Optional[torch.Tensor] = None,
                        logit_scale: Optional[torch.Tensor] = None, memory: Optional[RegionMemory] = None,
                        query_ids: Optional[torch.Tensor] = None) -> torch.Tensor:
    """InfoNCE of each local query against ALL regions.  With ``gather`` (and an initialised process
    group) the region rows are all-gathered across ranks first and ``targets`` -- indices into the
    LOCAL region rows -- are offset by rank * n_local.  tau (default 0.07) is a build choice (the reference defines
    none); ``logit_scale`` replaces 1/tau with a device tensor that can be learned (see ``ops.infonce_loss``).  Each
    rank's loss is the mean over its own queries, so the scale's gradient is rank-local, like the queries'.  ``memory``
    (a :class:`RegionMemory`) adds its valid rows to every query's negatives; each rank scores its own memory.
    ``query_ids`` (int64, one per local query, with ``memory``): leave each query's same-id memory rows out (see
    ``ops.infonce_loss``); each rank's ids are those of its own queries and memory."""
    ops.check_logit_scale(logit_scale, tau, "region_infonce_loss")
    regions = regions.reshape(-1, regions.shape[-1])
    rank, ws = cdist.world()
    if gather and ws > 1:
        n_local = regions.shape[0]
        regions = cdist.all_gather_rows(regions)
        targets = targets + rank * n_local
        regions_bf16 = None
    return ops.infonce_loss(regions, queries.reshape(-1, queries.shape[-1]), targets, tau, engine, regions_bf16, logit_scale, memory,
                            query_ids)


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


@functools.cache
def _target_rows(dev, B, M, offset):
    """Row index of every triplet's ground-truth region (b * M + offset), cached per shape and never evicted (a few bytes
    each): captured graphs hold the raw pointer."""
    return torch.arange(B, device=dev, dtype=torch.int64) * M + offset


@functools.cache
def _side_stream(dev):
    """One extra stream per device for the branch of the step that does not depend on the pooled rows."""
    return torch.cuda.Stream(device=dev)


def _overlap_enabled():
    return os.environ.get("COR_STEP_OVERLAP", "1") != "0"


def _step_tail_ok(B: int, M: int, C: int, multi_rank: bool, bg_mode: int, sim_engine: str) -> bool:
    """Whether the fused step runs its region tail as one forward and one backward launch (csrc/step_tail.cu): one rank's
    rows only, bg_mode 0 and a streaming-similarity shape (<= 16 queries, C % 8 == 0, C <= 256).  ``COR_STEP_TAIL=0`` keeps
    the kernel chain it replaces (A/B)."""
    return (os.environ.get("COR_STEP_TAIL", "1") != "0" and not multi_rank and bg_mode == 0 and B <= 16 and C % 8 == 0 and C <= 256
            and ops._sim_engine(B, B * M, C, sim_engine) == "stream")


@functools.cache
def _tail_counter(dev, B, M, C):
    """Zero-initialised arrival counters of the step-tail kernels, cached per shape: every launch leaves them zero again.
    Never evicted (128 bytes each): captured graphs hold the raw pointer."""
    return torch.zeros(L.load().cor_step_tail_counter_words(), dtype=torch.int32, device=dev)


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


# the fused step's shape and scalars, fixed before its first launch and read again by its backward.  ws: the ranks whose
# rows the InfoNCE scores (1 unless the rows are gathered); offset: this rank's first row among them
_StepCfg = namedtuple("_StepCfg", "B M Cc h w inv_tau nce_weight bg_mode w_fg w_bg ws offset pred_dt emb_dt comb_dt comb_shape "
                                  "need_pred need_emb need_comb")
# the tensors the step's backward reads, kept through save_for_backward
_Saved = namedtuple("_Saved", "pred_c t_save w_save per fg bg inv_fg inv_bg comb_c stats out4 aux r16 q16 targets lse w32 scale")
_Side = namedtuple("_Side", "q16 ev_q ev_px mem_args excl out8 t_save w_save per scratch")
_Rows = namedtuple("_Rows", "fg inv_fg bg inv_bg out4 aux lse nce tgt loss")


def _side_branch(cfg, dev, cur, side, px, pred_c, masks, comb_c, memory, sc, query_ids) -> _Side:
    """What needs neither the resampled weights nor the pooled rows, issued FIRST on the side stream (a parallel branch once
    captured in a CUDA graph), else on the current one: the peer-exit wait, the bf16 queries, the memory scan and the
    segmentation loss, whose instruction-bound tiles run underneath the HBM-bound mask resample.  ``scratch``: the work
    buffers the side stream writes, to keep alive until the tail joins it.  ``excl``: with ``query_ids``, the memory's
    exclusion mask, built just before the scan and kept for the backward's memory dQ."""
    lib = L.load()
    f32 = dict(dtype=torch.float32, device=dev)
    gt = masks[:, 0]                       # [B,Hm,Wm] view; read in place through its sample stride
    Hm, Wm = gt.shape[1:]
    if not (gt.stride(2) == 1 and gt.stride(1) == Wm):
        gt = gt.contiguous()
    N, D = comb_c.shape
    H, W = pred_c.shape[2:]
    out8 = torch.empty(8, **f32)
    per = torch.empty((N, lib.cor_seg_loss_npartials()), **f32)
    t_save = torch.empty((N, H, W), **f32) if cfg.need_pred else None
    w_save = torch.empty((N, H, W), **f32) if cfg.need_pred else None
    seg_work = ops._work(lib.cor_seg_loss_work_bytes(N, H, W), dev)
    stream = side if side is not None else cur
    if side is not None:
        side.wait_stream(cur)
    # "Have my peers finished reading the rows I published last step?" is asked HERE, at the very start of the step (one
    # 32-thread CTA polling local flags): by the time the row epilogue needs the answer the 0.7 ms mask resample has gone
    # by, so the wait never sits on the critical path.
    ev_px = mem_args = None
    if px is not None:
        with torch.cuda.stream(stream):
            px.before_produce(0)
        ev_px = side.record_event() if side is not None else None
    q16 = torch.empty((N, D), dtype=torch.bfloat16, device=dev)
    # allocated on the consuming stream: its block is reused only after the tail that reads it
    mwork = ops._memory_scan_work(memory, N, D, dev) if memory is not None else None
    # its last reader is the memory dQ of the backward, on the current stream
    excl = ops._memory_exclude_work(memory, N, dev) if query_ids is not None else None
    with torch.cuda.stream(stream):
        ops._call("cor_cast_cat_bf16", dev, ptr(comb_c), D, None, 0, _ll(N), ptr(q16))
        ev_q = side.record_event() if side is not None else None
        if memory is not None:
            if excl is not None:
                ops._memory_exclude(memory, query_ids, excl)
            mwork, mparts = ops._memory_scan(memory, q16, cfg.inv_tau, sc, mwork, excl)
            mem_args = (ptr(mwork), mparts, ptr(memory.state))
        ops._call("cor_seg_loss_fwd", dev, ptr(pred_c), L.dtype_code(pred_c), ptr(gt), L.dtype_code(gt), _f(ops._mask_scale(gt, None)),
                  N, H, W, Hm, Wm, _ll(gt.stride(0)), None, _f(0.25), _f(-1.0), _f(1.0), ptr(out8), ptr(per), ptr(t_save),
                  ptr(w_save), ptr(seg_work))
    return _Side(q16, ev_q, ev_px, mem_args, excl, out8, t_save, w_save, per, (seg_work, mwork))


def _pool(cfg, dev, emb_c, masks):
    """masks -> bf16 weights in the cached GEMM operand (+ raw fp32 weights for the backward) + full-resolution stats, then
    the pooling GEMM: (w16, w32, stats, split-K partials [ksplit, B, Rp, C]), row M = the all-ones weight row's sum."""
    B, M, Cc, P = cfg.B, cfg.M, cfg.Cc, cfg.h * cfg.w
    Rp = (M + 1 + 15) // 16 * 16
    w16 = ops._umma_weight_buffer(dev, B, Rp, M, P)
    w32, stats = ops.mask_prep(masks.reshape(B * M, *masks.shape[2:]), (cfg.h, cfg.w), ops.W_CLAMP, want_f32=cfg.need_emb,
                               bf16_out=w16, group=M, group_stride=Rp * P)
    part = torch.empty((L.load().cor_pool_umma_ksplit(B, Cc, P), B, Rp, Cc), dtype=torch.float32, device=dev)
    ops._call("cor_pool_umma_fwd", dev, ptr(emb_c), ptr(w16), B, Cc, P, Rp, ptr(part))
    return w16, w32, stats, part


def _row_outputs(dev, B, M, Cc) -> _Rows:
    """What either tail writes: unit rows + inverse norms, the GT masks' bg rows + inverse norms, the fg / bg losses + their
    auxiliaries, and the InfoNCE's log-sum-exp, mean and target logits with the step's total loss."""
    e = lambda *shape: torch.empty(shape, dtype=torch.float32, device=dev)
    return _Rows(fg=e(B * M, Cc), inv_fg=e(B * M), bg=e(B, Cc), inv_bg=e(B), out4=e(4), aux=e(L.load().cor_fgbg_aux_floats(B, Cc)),
                 lse=e(B), nce=e(1), tgt=e(B), loss=e(1))


def _tail_forward(cfg, dev, cur, side, part, stats, comb_c, sc, sd, counter):
    """The region tail in ONE launch (csrc/step_tail.cu): unit rows (+ bf16 copy), their scores against the queries, the bg
    rows and fg / bg cosine statistics of the GT masks, and in its last CTA the log-sum-exp merge (with the memory's
    partials), the InfoNCE, fg / bg losses and the total.  Returns (_Rows, the scored bf16 rows, their targets)."""
    B, M, Cc, Rp = cfg.B, cfg.M, cfg.Cc, part.shape[2]
    o = _row_outputs(dev, B, M, Cc)
    fg16 = torch.empty((B * M, Cc), dtype=torch.bfloat16, device=dev)
    targets = _target_rows(dev, B, M, 0)
    work = ops._work(L.load().cor_step_tail_work_bytes(B, M, Cc), dev)
    if side is not None:
        cur.wait_stream(side)            # join: the total needs the segmentation loss, the scores the bf16 queries
    name, tas = ops._tail_entry("cor_step_tail_fwd", cfg.inv_tau, sc, sd.mem_args)
    ops._call(name, dev, ptr(part), part.shape[0], _ll(B * Rp * Cc), Rp, B, M, Cc, _f(float(cfg.h * cfg.w)), ptr(stats), ptr(sd.q16),
              ptr(comb_c), ptr(targets), *tas, ptr(sd.out8), _f(cfg.w_fg), _f(cfg.w_bg), _f(cfg.nce_weight), ptr(o.fg), ptr(fg16),
              ptr(o.inv_fg), ptr(o.bg), ptr(o.inv_bg), ptr(o.out4), ptr(o.aux), ptr(o.lse), ptr(o.nce), ptr(o.tgt), ptr(o.loss), ptr(work),
              ptr(counter))
    return o, fg16, targets


def _chain_forward(cfg, dev, cur, side, part, stats, comb_c, sc, sd, px, sim_engine):
    """The region tail as a kernel chain where the one-launch tail does not serve: the row epilogue, the bg rows and fg / bg
    losses on the side stream, the gather (or fused gather + similarity) and cor_infonce_tail.  Returns as _tail_forward."""
    B, M, Cc = cfg.B, cfg.M, cfg.Cc
    ks, Rp = part.shape[0], part.shape[2]
    n_local, split = B * M, B * Rp * Cc
    o = _row_outputs(dev, B, M, Cc)
    # multi-GPU: the bf16 rows land directly in this rank's peer-mapped buffer (cor_b200/peer.py), else in a local one
    fg16 = px.pub if px is not None else torch.empty((n_local, Cc), dtype=torch.bfloat16, device=dev)
    if sd.ev_px is not None:
        cur.wait_event(sd.ev_px)
    ops._call("cor_rows_finalize", dev, ptr(part), M, _ll(Rp * Cc), ks, _ll(split), ptr(stats[:, 3:]), 4, _f(1e-8), n_local, Cc, 1, 1,
              None, _f(0.0), ptr(o.fg), ptr(fg16), ptr(o.inv_fg))
    if px is not None:
        px.signal(0)                     # the bg rows, fg/bg loss and segmentation loss below hide the rank skew
    # background rows + fg / bg cosine losses on the GT rows (row b*M of fg, row b of bg): a second branch off the fg rows,
    # on the side stream, parallel to the similarity / InfoNCE chain below
    if side is not None:
        side.wait_stream(cur)
    with torch.cuda.stream(side if side is not None else cur):
        ops._call("cor_rows_finalize", dev, ptr(part), 1, _ll(Rp * Cc), ks, _ll(split), ptr(stats[:, 3:]), 4 * M, _f(1e-8), B, Cc, 1, 1,
                  ptr(part[0, :, M, :]), _f(float(cfg.h * cfg.w)), ptr(o.bg), None, ptr(o.inv_bg))
        ops._call("cor_fgbg_loss_fwd", dev, ptr(o.fg), _ll(M * Cc), ptr(o.bg), _ll(Cc), ptr(comb_c), _ll(Cc), ptr(stats), _ll(4 * M), B,
                  Cc, cfg.bg_mode, ptr(o.out4), ptr(o.aux))
    # InfoNCE of every composed query against all (gathered) regions
    if sd.ev_q is not None:
        cur.wait_event(sd.ev_q)
    r16, fused_parts = fg16, None
    if cfg.ws > 1:
        r16 = torch.empty((cfg.ws * n_local, Cc), dtype=torch.bfloat16, device=dev)
        if px is not None and _peer_fused_ok(B, Cc, cfg.ws * n_local, sim_engine):
            # ONE kernel: pull the peers' rows over NVLink, keep a local copy for the backward, and score every row against
            # this rank's queries while it is in registers (all-gather fused with its consumer)
            fused_parts = px.gather_sim(r16, sd.q16, cfg.inv_tau, sc)
        elif px is not None:
            px.gather(r16)               # our own pull-over-NVLink kernel: no NCCL on the data path
        else:
            torch.distributed.all_gather_into_tensor(r16, fg16)
    targets = _target_rows(dev, B, M, cfg.offset)
    # similarity with its log-sum-exp partials left in the work buffer, then ONE tail kernel: partial merge (with this rank's
    # memory, scored against its own queries) -> lse, target logits, InfoNCE mean and the step's total loss
    sim_work, nparts, qt = fused_parts if fused_parts is not None else ops._sim_lse_parts(r16, sd.q16, cfg.inv_tau, sim_engine, sc)
    if side is not None:
        cur.wait_stream(side)            # join: the total needs the segmentation and fg/bg losses
    name, tas = ops._tail_entry("cor_infonce_tail", cfg.inv_tau, sc, sd.mem_args)
    ops._call(name, dev, ptr(sim_work), nparts, qt, ptr(r16), ptr(sd.q16), ptr(targets), r16.shape[0], B, Cc, *tas, ptr(o.lse),
              ptr(o.nce), ptr(o.tgt), ptr(sd.out8), ptr(o.out4), _f(cfg.w_fg), _f(cfg.w_bg), _f(cfg.nce_weight), ptr(o.loss))
    return o, r16, targets


def _seg_backward(cfg, s, g, cur, side):
    """Gradient of the segmentation loss wrt pred (None when pred needs none), on the side stream when there is one."""
    if not cfg.need_pred:
        return None
    N, H, W = s.t_save.shape
    gp = torch.empty_like(s.pred_c)
    if side is not None:
        side.wait_stream(cur)
    with torch.cuda.stream(side if side is not None else cur):
        ops._call("cor_seg_loss_bwd", gp.device, ptr(s.pred_c), L.dtype_code(s.pred_c), ptr(s.t_save), ptr(s.w_save), ptr(s.per), N, H,
                  W, None, _f(1.0), _f(0.25), _f(-1.0), ptr(g), ptr(gp), L.dtype_code(gp))
    return gp


def _pool_bwd_gemm(a16, w16, B, Cc, P, Kp, out_dtype):
    """d emb[b] (C x P) = gs[b]^T (C x M) w[b] (M x P) -> [B*C, P]: one batched tcgen05 GEMM on the bf16 weights the forward's
    pooling GEMM used (the caller checked that no later forward of this shape has rewritten them), both operands MN-major
    as they lie.  ``a16`` holds the gradient rows in bf16, zero-padded to whole 64-row K blocks (Kp), which makes the
    weight rows beyond M (the ones row, the next image) irrelevant.  Persistent tiles with coalesced stores: 2-3x faster
    than the one-shot pool_bwd_umma kernel, which rebuilds both operands from fp32."""
    Rp = w16.shape[1]
    return gemm(a16, w16.view(B * Rp, P), Cc, P, Kp, a_mn=True, b_mn=True, batch=B, a_batch_rows=Kp, b_batch_rows=Rp, out_dtype=out_dtype)


def _tail_backward(ctx, s, g, g_scale):
    """(g_emb, g_comb) from ONE launch: InfoNCE + fg-loss gradient of every row, through the row epilogue, cast to bf16 into
    the K-padded operand of the pooling-backward GEMM; and the query gradient (+ fg / bg terms) in extra CTAs, one set per
    query.  Then the memory's share of the query gradient, and the GEMM."""
    cfg = ctx.cfg
    B, M, Cc = cfg.B, cfg.M, cfg.Cc
    dev = s.fg.device
    Kp = (M + 63) // 64 * 64
    a16 = torch.empty((B * Kp, Cc), dtype=torch.bfloat16, device=dev) if cfg.need_emb else None
    g_q = torch.empty((B, Cc), dtype=torch.float32, device=dev) if cfg.need_comb else None
    work = ops._work(L.load().cor_step_tail_work_bytes(B, M, Cc), dev)
    name, ta = ops._tau_arg("cor_step_tail_bwd", cfg.inv_tau, s.scale)
    gs_arg = () if s.scale is None else (ptr(g_scale),)          # the _ls backward entries take the gradient pointer
    ops._call(name, dev, ptr(s.r16), ptr(s.q16), ptr(s.targets), ptr(s.lse), B, M, Cc, ta, ptr(g), _f(cfg.nce_weight), ptr(s.fg),
              ptr(s.inv_fg), ptr(s.stats), ptr(s.comb_c), ptr(s.out4), ptr(s.aux), _f(cfg.w_fg), _f(cfg.w_bg), ptr(a16), Kp, ptr(g_q),
              *gs_arg, ptr(work), ptr(ctx.tail))
    if ctx.mem is not None:
        ops._memory_dq(ctx.mem[0], s.q16, s.lse, cfg.inv_tau, s.scale, g, cfg.nce_weight, g_q, g_scale, ctx.mem[2])
    g_comb = g_q.view(cfg.comb_shape).to(cfg.comb_dt) if cfg.need_comb else None
    if not cfg.need_emb:
        return None, g_comb
    out_dt = cfg.emb_dt if cfg.emb_dt in (torch.float32, torch.bfloat16) else torch.float32
    return _pool_bwd_gemm(a16, ctx.w16[0], B, Cc, cfg.h * cfg.w, Kp, out_dt).view(B, Cc, cfg.h, cfg.w).to(cfg.emb_dt), g_comb


def _chain_backward(ctx, s, g, g_scale, g_pred, gemm_ok, cur, side, ev_px):
    """Backward of the kernel chain, and of a one-launch tail whose bf16 weights were rewritten since: (g_emb, g_comb, g_pred),
    the last computed here, between the signal and the pull, when there is a peer exchange and no side stream."""
    cfg, px = ctx.cfg, ctx.px
    B, M, Cc, P = cfg.B, cfg.M, cfg.Cc, cfg.h * cfg.w
    dev = s.fg.device
    lib = L.load()
    f32 = dict(dtype=torch.float32, device=dev)
    # InfoNCE backward first: it WRITES g_regions (this rank's rows) and g_queries ...
    Nr = s.r16.shape[0]
    g_regions = torch.empty((B * M, Cc), **f32)
    g_q = torch.empty((B, Cc), **f32)
    work = ops._work(lib.cor_sim_work_bytes(B, Nr, Cc), dev)
    if ev_px is not None:
        cur.wait_event(ev_px)
    # several ranks: gradient of every gathered row, then a reduce-scatter back to the owning rank: measured faster than a
    # collective-free backward that all-gathers the queries instead (profiles/README.md)
    g_rows = g_regions if cfg.ws == 1 else px.gall if px is not None else torch.empty((Nr, Cc), **f32)
    name, ta = ops._tau_arg("cor_infonce_bwd", cfg.inv_tau, s.scale)
    gs_arg = () if s.scale is None else (ptr(g_scale),)
    ops._call(name, dev, ptr(s.r16), ptr(s.q16), ptr(s.targets), ptr(s.lse), Nr, B, Cc, ta, ptr(g), _f(cfg.nce_weight), ptr(g_rows),
              ptr(g_q), *gs_arg, ptr(work))
    if px is not None:
        px.signal(1)
        if side is None:
            g_pred = _seg_backward(cfg, s, g, cur, None)   # independent work between the signal and the pull hides the rank skew
        px.reduce(g_regions)             # fixed rank order: bit-identical from run to run
    elif cfg.ws > 1:
        torch.distributed.reduce_scatter_tensor(g_regions, g_rows, op=torch.distributed.ReduceOp.SUM)
    # ... then the fg/bg backward ADDS its GT-row gradients into g_regions (row b*M) and g_queries
    g_bg = torch.empty((B, Cc), **f32) if cfg.bg_mode == 1 else None
    ops._call("cor_fgbg_loss_bwd", dev, ptr(s.fg), _ll(M * Cc), ptr(s.bg), _ll(Cc), ptr(s.comb_c), _ll(Cc), B, Cc, cfg.bg_mode, ptr(s.out4),
              ptr(s.aux), ptr(g), _ll(0), _f(cfg.w_fg), _f(cfg.w_bg), ptr(g_regions), _ll(M * Cc), 1, ptr(g_bg), _ll(Cc), ptr(g_q), _ll(Cc), 1)
    if ctx.mem is not None:              # this rank's memory, against this rank's queries
        ops._memory_dq(ctx.mem[0], s.q16, s.lse, cfg.inv_tau, s.scale, g, cfg.nce_weight, g_q if cfg.need_comb else None, g_scale,
                       ctx.mem[2])
    g_comb = g_q.view(cfg.comb_shape).to(cfg.comb_dt) if cfg.need_comb else None
    if not cfg.need_emb:
        return None, g_comb, g_pred
    gs_fg = torch.empty((B * M, Cc), **f32)
    ops._call("cor_rows_finalize_bwd", dev, ptr(g_regions), ptr(s.fg), ptr(s.inv_fg), ptr(s.stats[:, 3:]), 4, _f(1e-8), B * M, Cc, 1, 1,
              0, _f(0.0), ptr(gs_fg))
    out_dt = cfg.emb_dt if cfg.emb_dt in (torch.float32, torch.bfloat16) else torch.float32
    if gemm_ok:                          # implies bg_mode 0: no background gradient
        Kp = (M + 63) // 64 * 64
        a16 = torch.empty((B * Kp, Cc), dtype=torch.bfloat16, device=dev)
        ops._call("cor_cast_pad_rows_bf16", dev, ptr(gs_fg), B, M, Kp, Cc, ptr(a16))
        return _pool_bwd_gemm(a16, ctx.w16[0], B, Cc, P, Kp, out_dt).view(B, Cc, cfg.h, cfg.w).to(cfg.emb_dt), g_comb, g_pred
    gs_bg_full = None
    if g_bg is not None:                 # paired bg mode: background gradient lives on the GT rows only
        gs_bg = torch.empty((B, Cc), **f32)
        ops._call("cor_rows_finalize_bwd", dev, ptr(g_bg), ptr(s.bg), ptr(s.inv_bg), ptr(s.stats[:, 3:]), 4 * M, _f(1e-8), B, Cc, 1, 1, 1,
                  _f(float(P)), ptr(gs_bg))
        gs_bg_full = torch.zeros((B, M, Cc), **f32)
        gs_bg_full[:, 0, :] = gs_bg
    g_emb = torch.empty((B, Cc, cfg.h, cfg.w), dtype=out_dt, device=dev)
    name = "cor_pool_bwd_umma" if lib.cor_pool_bwd_umma_ok(B, Cc, P, M, int(gs_bg_full is not None)) else "cor_pool_bwd_feat"
    ops._call(name, dev, ptr(gs_fg), ptr(gs_bg_full), ptr(s.w32), _ll(P), B, Cc, P, M, ops.W_CLAMP, ptr(g_emb), L._DTYPES[g_emb.dtype])
    return g_emb.to(cfg.emb_dt), g_comb, g_pred


class _FusedStepFn(torch.autograd.Function):
    """The whole region path as ONE autograd node, hand-written backward, no tensor glue (slices, zeros + scatter, tiny adds)
    between its kernels: the side branch, the pooling, then the one-launch tail where it applies, else the kernel chain.
    Used by :func:`region_step` when the tensor-core pooling engine applies; the modular ops remain the general path."""

    @staticmethod
    def forward(ctx, pred, emb, comb, masks, tau, nce_weight, gather, sim_engine, bg_mode, w_fg, w_bg, logit_scale, memory, query_ids):
        dev = L.require_cuda(pred, emb, comb, masks, logit_scale)
        sc = logit_scale                       # device logit scale (replaces 1/tau in every InfoNCE launch) or None
        B, M = masks.shape[:2]
        Cc, h, w = emb.shape[1:]
        if masks.dtype not in (torch.float32, torch.bfloat16, torch.uint8):
            masks = masks.float()            # bool / fp16 / fp64 masks: one conversion serves mask_prep and the seg loss
        emb_c = emb.contiguous()
        pred_c = ops._as_supported_float(pred)
        comb_c = comb.reshape(B, -1).float().contiguous()
        rank, ws = cdist.world()
        multi_rank = gather and ws > 1
        cfg = _StepCfg(B, M, Cc, h, w, 1.0 / float(tau), float(nce_weight), int(bg_mode), float(w_fg), float(w_bg), ws if multi_rank else 1,
                       rank * B * M if multi_rank else 0, pred.dtype, emb.dtype, comb.dtype, tuple(comb.shape), pred.requires_grad,
                       emb.requires_grad, comb.requires_grad)
        cur = torch.cuda.current_stream(dev)
        side = _side_stream(dev) if _overlap_enabled() else None
        px = peer.get_exchange(B * M, Cc, dev) if multi_rank else None
        sd = _side_branch(cfg, dev, cur, side, px, pred_c, masks, comb_c, memory, sc, query_ids)
        w16, w32, stats, part = _pool(cfg, dev, emb_c, masks)
        ctx.tail = _tail_counter(dev, B, M, Cc) if _step_tail_ok(B, M, Cc, multi_rank, cfg.bg_mode, sim_engine) else None
        if ctx.tail is not None:
            o, r16, targets = _tail_forward(cfg, dev, cur, side, part, stats, comb_c, sc, sd, ctx.tail)
        else:
            o, r16, targets = _chain_forward(cfg, dev, cur, side, part, stats, comb_c, sc, sd, px, sim_engine)
        # the scale is saved as an input: an in-place write to it before backward trips autograd's version check
        ctx.save_for_backward(*_Saved(pred_c=pred_c, t_save=sd.t_save, w_save=sd.w_save, per=sd.per, fg=o.fg, bg=o.bg, inv_fg=o.inv_fg,
                                      inv_bg=o.inv_bg, comb_c=comb_c, stats=stats, out4=o.out4, aux=o.aux, r16=r16, q16=sd.q16,
                                      targets=targets, lse=o.lse, w32=w32, scale=sc))
        ctx.cfg, ctx.px = cfg, px
        ctx.mem = None if memory is None else (memory, memory.enqueues, sd.excl)
        ctx.w16 = (w16, getattr(w16, "_cor_epoch", -1))      # not a saved tensor: a cached operand buffer, validated by its epoch
        ctx.mark_non_differentiable(o.fg, sd.out8, o.out4, o.nce)
        ctx.set_materialize_grads(False)     # no zero-filled gradients for the auxiliary outputs
        return o.loss[0], sd.out8, o.out4, o.nce, o.fg

    @staticmethod
    def backward(ctx, g_loss, *_unused):
        if g_loss is None:
            return (None,) * 14
        ops.check_memory_unchanged(ctx.mem, "region_step backward")
        cfg, s, px = ctx.cfg, _Saved(*ctx.saved_tensors), ctx.px
        dev = s.fg.device
        g = g_loss.reshape(1).float().contiguous()
        # d loss / d scale: written by the InfoNCE backward over THIS rank's queries (the launch that writes g_queries)
        g_scale = torch.empty((), dtype=torch.float32, device=dev) if s.scale is not None and ctx.needs_input_grad[11] else None
        cur = torch.cuda.current_stream(dev)
        side = _side_stream(dev) if (_overlap_enabled() and cfg.need_pred) else None
        ev_px = None
        if px is not None and cfg.ws > 1:
            # as in the forward: ask early, on the side stream, whether the peers are done with last step's `gall`
            if side is not None:
                side.wait_stream(cur)
            with torch.cuda.stream(side if side is not None else cur):
                px.before_produce(1)
            ev_px = side.record_event() if side is not None else None
        # on the side stream it runs underneath the InfoNCE / pooling backward
        g_pred = _seg_backward(cfg, s, g, cur, side) if px is None or side is not None else None
        w16, w16_epoch = ctx.w16
        gemm_ok = (cfg.bg_mode != 1 and w16 is not None and getattr(w16, "_cor_epoch", -1) == w16_epoch and cfg.Cc % 8 == 0
                   and (cfg.h * cfg.w) % 8 == 0)
        # a tail forward whose bf16 weights a later forward of this shape rewrote takes the chain's fp32 pooling backward
        use_tail = ctx.tail is not None and (gemm_ok or not cfg.need_emb)
        if use_tail:
            g_emb, g_comb = _tail_backward(ctx, s, g, g_scale)
        else:
            g_emb, g_comb, g_pred = _chain_backward(ctx, s, g, g_scale, g_pred, gemm_ok, cur, side, ev_px)
        if side is not None:
            cur.wait_stream(side)
        if g_pred is not None:
            g_pred = g_pred.to(cfg.pred_dt)
        return g_pred, g_emb, g_comb, None, None, None, None, None, None, None, None, g_scale, None, None


def _fused_ok(emb, masks, pool_engine):
    B, M = masks.shape[:2]
    P = emb.shape[2] * emb.shape[3]
    return pool_engine in ("auto", "umma") and ops.umma_pool_eligible(emb, M, P, ops.W_CLAMP, 1, True) and emb.shape[1] % 8 == 0


def region_step(pred: torch.Tensor, emb: torch.Tensor, comb: torch.Tensor, masks: torch.Tensor, *, tau: Optional[float] = None,
                nce_weight: float = 1.0, gather: bool = True, pool_engine: str = "auto", sim_engine: str = "auto",
                bg_mode: int = 0, fused: bool = True, logit_scale: Optional[torch.Tensor] = None,
                memory: Optional[RegionMemory] = None, query_ids: Optional[torch.Tensor] = None) -> RegionStepOut:
    """One forward of the whole region path for a batch of triplets with M candidate masks each
    (mask 0 of every image is the ground-truth ``query_mask``):

        seg  = wbce_with_wiou_loss(pred, resample(masks[:,0]))                 trainer_v3_g.py:67-68
        fg,bg = fg/bg_feat_similarity_loss(emb, comb, masks[:,0])              trainer_v3_g.py:69-71
        nce  = InfoNCE(comb_b vs all B*M (x world) pooled regions, target = region (b,0))   [Class N]
        loss = seg + 5 fg + 5 bg + nce_weight * nce

    The InfoNCE logits are S / tau (tau defaults to 0.07), or ``logit_scale * S`` for a learnable temperature:
    ``logit_scale`` is a 0-dim float32 tensor s > 0 on the step's device, passed instead of ``tau``.  The kernels read
    it from device memory, and d loss / d s reaches it through autograd when it requires grad.

    ``memory`` (a :class:`RegionMemory` of width C on the step's device) adds its valid rows to every query's InfoNCE
    negatives: nce = mean_b (logsumexp over the current rows and the memory - target logit).  The step stays on its fused
    kernels; the memory is scanned on tensor cores beside the mask resample.  Push the batch with
    ``memory.enqueue(out.regions)`` after backward() (``StepBuffers.capture(memory=...)`` does it inside the graph).

    ``query_ids`` (int64 [B] on the step's device, with ``memory``): an id per triplet, e.g. its target object's.  Memory
    rows with the same id (pushed by ``memory.enqueue(out.regions, ids=query_ids)``) are left out of that triplet's
    negatives and gradients, so an earlier pooled row of the object it looks for is not scored against it.

    ONE pass over the masks and ONE pass over the feature map serve fg, bg and all M regions.  With bf16
    features and >= 16 masks the step runs as a single fused autograd node (tensor-core pooling, hand
    written backward); other shapes compose the modular ops.
    """
    ops.check_logit_scale(logit_scale, tau, "region_step")
    if logit_scale is not None and logit_scale.device != emb.device:
        raise CorError(f"region_step: logit_scale is on {logit_scale.device}, the step on {emb.device}")
    ops.check_memory(memory, emb.shape[1], emb.device if emb.is_cuda else None, "region_step")
    B, M = masks.shape[:2]
    ops.check_query_ids(query_ids, memory, B, emb.device if emb.is_cuda else None, "region_step")
    if comb.shape[0] != B or emb.shape[0] != B or pred.shape[0] != B:
        raise CorError("region_step: batch sizes differ")
    if comb.numel() != B * emb.shape[1]:
        raise CorError(f"region_step: comb {tuple(comb.shape)} must hold one row of C={emb.shape[1]} channels per triplet "
                       "(the kernels read the queries with the feature map's row width)")
    if fused and _fused_ok(emb, masks, pool_engine) and pred.dim() == 4 and pred.shape[1] == 1:
        loss, out8, out4, nce, fg = _FusedStepFn.apply(pred, emb, comb, masks, 0.07 if tau is None else float(tau), float(nce_weight),
                                                       bool(gather), sim_engine, int(bg_mode), 5.0, 5.0, logit_scale, memory, query_ids)
        return RegionStepOut(loss=loss, seg=out8[0], fg=out4[0], bg=out4[1], nce=nce[0], regions=fg.view(B, M, -1))
    pool = ops.region_pool(emb, masks, transform=ops.W_CLAMP, normalize=True, pair=True, engine=pool_engine, want_bf16=True)
    Cc = pool.fg.shape[-1]
    q = comb.reshape(B, -1)
    gt_rows = torch.arange(B, device=emb.device) * M
    losses, _ = ops.fgbg_losses(pool.fg[:, 0, :], pool.bg[:, 0, :], q, pool.stats.view(B, M, 4)[:, 0, :], bg_mode)
    seg = ops.seg_loss(pred, masks[:, 0:1])
    nce = region_infonce_loss(pool.fg.reshape(B * M, Cc), q, gt_rows, tau, gather, sim_engine,
                              regions_bf16=pool.fg_bf16, logit_scale=logit_scale, memory=memory, query_ids=query_ids)
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
    recapture, and d loss / d s lands in ``self.grads["logit_scale"]``, overwritten by every replay.

    ``capture(memory=m)`` / ``run(..., memory=m)`` (m a :class:`RegionMemory`): every step scores against the memory, then
    after the backward pushes its regions with ``m.enqueue``, inside the graph, so each replay advances the memory.
    ``capture`` leaves the memory as it found it (its warm-up steps are undone).

    ``ids=True`` adds a static int64 buffer ``d["ids"]`` [B], one id per triplet (e.g. its target object's), that
    ``load`` fills like the others.  With a memory every step then scores with ``query_ids=d["ids"]`` and pushes its
    regions with ``ids=d["ids"]`` (on each image's ground-truth row), so a replay never scores a triplet against earlier
    pooled rows of its own target."""

    def __init__(self, B, M, C=256, h=64, w=64, H=1024, W=1024, hp=256, wp=256, D=None, device="cuda",
                 emb_dtype=torch.bfloat16, mask_dtype=torch.float32, ids: bool = False):
        if D is not None and D != C:
            raise CorError(f"StepBuffers: the composed query width D={D} must equal the feature channels C={C}")
        D = C
        self.device = torch.device(device)
        mk = lambda shape, dt: torch.empty(shape, dtype=dt, device=self.device)
        self.d = {"pred": mk((B, 1, hp, wp), emb_dtype), "emb": mk((B, C, h, w), emb_dtype), "comb": mk((B, 1, D), torch.float32),
                  "masks": mk((B, M, H, W), mask_dtype)}
        if ids:
            self.d["ids"] = mk((B,), torch.int64)
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
        memory = kw.pop("memory", None)
        if scale is not None:
            scale = scale.detach().requires_grad_(backward)      # a leaf over the caller's storage: read in place
        ids = self.d.get("ids") if memory is not None else None
        out = region_step(pred, emb, comb, self.d["masks"], logit_scale=scale, memory=memory, query_ids=ids, **kw)
        if backward:
            out.loss.backward(gradient=self._seed)      # a resident 1.0: no per-step fill kernel from autograd
        if memory is not None:
            memory.enqueue(out.regions, ids=ids)         # after the backward, which needs the rows the forward scored
        grads = {"pred": pred.grad, "comb": comb.grad, "emb": emb.grad}
        if scale is not None:
            grads["logit_scale"] = scale.grad
        return out.loss.detach(), grads

    def capture(self, backward: bool = True, emb_grad: bool = True, warmup: int = 3, **kw):
        """Warm up on a side stream, then capture fwd+bwd of the step into a CUDA graph."""
        memory = kw.get("memory")
        saved = (memory.bank.clone(), memory.state.clone(), memory.ids.clone()) if memory is not None else None
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):
            for _ in range(warmup):
                self._step(backward, emb_grad, kw)
        torch.cuda.current_stream(self.device).wait_stream(side)
        torch.cuda.synchronize(self.device)
        if saved is not None:                            # undo the warm-up's enqueues
            memory.bank.copy_(saved[0])
            memory.state.copy_(saved[1])
            memory.ids.copy_(saved[2])
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
