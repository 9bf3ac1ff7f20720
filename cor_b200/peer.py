"""NVLink peer-memory exchange of the region rows (SURVEY.md §8e): the B200-native replacement of the NCCL
all-gather / reduce-scatter pair around the similarity stage of ``region_step``.

One process per GPU on one node.  Every rank cudaMallocs one region (``cor_peer_alloc``), exports it with CUDA IPC,
the 64-byte handles travel once through ``torch.distributed`` (the plumbing), and every rank maps its peers'
regions.  After that the exchange is two of our own kernels per step (``cor_peer_gather_rows`` forward,
``cor_peer_reduce_rows`` backward) that pull over NVLink and synchronise through flags in peer memory - no NCCL call
on the data path, capturable in a CUDA graph.  Layout of a rank's region::

    [ flags | pub: n_local x C bf16 | gall: world*n_local x C f32 ]      (each part 256-byte aligned)

``pub`` is written in place by ``cor_rows_finalize`` and ``gall`` by ``cor_infonce_bwd``, so the exchange adds no
staging copy.  Setting ``COR_PEER=0`` (or a failed IPC mapping on any rank) keeps the NCCL collectives.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch
import torch.distributed as dist

from . import _lib as L

__all__ = ["PeerExchange", "get_exchange", "enabled"]

_CACHE: dict = {}


class _Raw:
    """A __cuda_array_interface__ view of raw device memory (the owner keeps it alive)."""

    def __init__(self, ptr: int, nbytes: int):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}


def _align(n: int, a: int = 256) -> int:
    return (n + a - 1) // a * a


def enabled() -> bool:
    return os.environ.get("COR_PEER", "1") != "0"


class PeerExchange:
    """Symmetric buffers + mapped peer pointers for one (n_local, C) shape.  Collective constructor: every rank of
    ``group`` must call it; ``ok`` is the same on all ranks."""

    def __init__(self, n_local: int, Cc: int, device: torch.device, group=None):
        lib = L.load()
        self.lib = lib
        self.group = group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.n_local, self.C = n_local, Cc
        self.device = torch.device(device)
        self.dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.ok = False
        self._last = None                  # channel of the last exchange launched
        self.base = None
        self.mapped: list = []
        flag_b = _align(lib.cor_peer_flag_bytes())
        pub_b = _align(n_local * Cc * 2)
        gall_b = _align(self.world * n_local * Cc * 4)
        self.off_pub, self.off_gall = flag_b, flag_b + pub_b
        self.nbytes = flag_b + pub_b + gall_b
        good = self.world <= lib.cor_peer_max_world()
        handle = b""
        if good:
            base = C.c_void_p()
            if lib.cor_peer_alloc(self.dev_index, self.nbytes, C.byref(base)) == 0:
                self.base = base.value
                buf = C.create_string_buffer(64)
                good = lib.cor_peer_export(C.c_void_p(self.base), buf) == 0
                handle = buf.raw
            else:
                good = False
        handles = [None] * self.world
        dist.all_gather_object(handles, (good, handle), group=group)
        good = all(h[0] for h in handles)
        ptrs = []
        if good:
            for r, (_, h) in enumerate(handles):
                if r == self.rank:
                    ptrs.append(self.base)
                    continue
                p = C.c_void_p()
                if lib.cor_peer_open(self.dev_index, h, C.byref(p)) != 0:
                    good = False
                    break
                self.mapped.append(p.value)
                ptrs.append(p.value)
        votes = [None] * self.world          # object collective: works over NCCL and over gloo (one-GPU emulation in the tests)
        dist.all_gather_object(votes, bool(good), group=group)
        if not all(votes):
            self.close()
            return
        i64 = dict(dtype=torch.int64, device=self.device)
        self.flag_ptrs = torch.tensor(ptrs, **i64)
        self.pub_ptrs = torch.tensor([p + self.off_pub for p in ptrs], **i64)
        self.gall_ptrs = torch.tensor([p + self.off_gall for p in ptrs], **i64)
        self.state = torch.zeros(max(lib.cor_peer_state_bytes() // 4, 12), dtype=torch.int32, device=self.device)
        self._err_word = lib.cor_peer_error_word()
        self._raw = _Raw(self.base, self.nbytes)
        whole = torch.as_tensor(self._raw, device=self.device)
        self.pub = whole[self.off_pub:self.off_pub + n_local * Cc * 2].view(torch.bfloat16).view(n_local, Cc)
        self.gall = whole[self.off_gall:self.off_gall + self.world * n_local * Cc * 4].view(torch.float32).view(self.world * n_local, Cc)
        torch.cuda.synchronize(self.device)
        dist.barrier(group=group)
        self.ok = True

    # -- protocol (csrc/peer.cu) --------------------------------------------------------------------------------------
    def _ctl(self, name, channel):
        from . import ops
        ops._call(name, self.device, ops.ptr(self.flag_ptrs), ops.ptr(self.state), self.rank, self.world, channel)

    def before_produce(self, channel: int):
        """Call before the kernel that overwrites ``pub`` (channel 0) / ``gall`` (channel 1).  The peers have provably
        finished reading the previous contents once an exchange on the OTHER channel ran in between (its enter barrier
        orders them); only when the same channel is used twice in a row is a wait kernel needed.  That shortcut rests
        on host-side history, which a CUDA graph would freeze: a captured step ALWAYS carries the wait (one 32-thread
        CTA polling local flags), so that eager forward-only calls between replays cannot tear the rows."""
        if self._last == channel or torch.cuda.is_current_stream_capturing():
            self._ctl("cor_peer_wait_exit", channel)

    def check(self):
        """Raise CorError if any wait of this exchange expired (COR_PEER_TIMEOUT_S).  Synchronises the device: call it
        where the step already syncs (``StepBuffers.run`` does), not inside a captured region."""
        word = int(self.state[self._err_word].item()) & 0xFFFFFFFF
        if word:
            raise L.CorError(f"peer exchange: rank {self.rank} gave up waiting for a peer at epoch {word & 0x7FFFFFFF} "
                             "(COR_PEER_TIMEOUT_S); results since then are invalid")

    def signal(self, channel: int):
        """Call right after the producer kernel: tells the peers this rank's buffer is ready for the next exchange."""
        self._ctl("cor_peer_signal", channel)

    def gather(self, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """[world*n_local, C] bf16 = every rank's ``pub`` (rank-major).  ``signal(0)`` must have been issued."""
        from . import ops
        if out is None:
            out = torch.empty((self.world * self.n_local, self.C), dtype=torch.bfloat16, device=self.device)
        ops._call("cor_peer_gather_rows", self.device, ops.ptr(self.pub_ptrs), ops.ptr(out), ops._ll(self.n_local * self.C * 2),
                  ops.ptr(self.flag_ptrs), ops.ptr(self.state), self.rank, self.world, 0)
        self._last = 0
        return out

    def gather_sim(self, out: torch.Tensor, q16: torch.Tensor, inv_tau: float, logit_scale: Optional[torch.Tensor] = None):
        """Fused all-gather + similarity (csrc/peer.cu, peer_gather_sim_kernel): fills ``out`` [world*n_local, C] bf16 like
        :meth:`gather` AND scores every row against this rank's queries ``q16`` [Nq <= 16, C] bf16 while it is in registers.
        ``logit_scale`` (0-dim f32 on the device) replaces ``inv_tau`` when given.
        Returns ``(work, nparts, qt)`` -- the log-sum-exp partials for ``cor_infonce_tail``."""
        import ctypes as C_
        from . import ops
        work = ops._work(self.lib.cor_peer_gather_sim_work_bytes(), self.device)
        nparts = C_.c_int(0)
        name, ta = ops._tau_arg("cor_peer_gather_sim", inv_tau, logit_scale)
        ops._call(name, self.device, ops.ptr(self.pub_ptrs), ops.ptr(out), ops._ll(self.n_local), self.C, ops.ptr(q16),
                  int(q16.shape[0]), ta, ops.ptr(work), C_.byref(nparts), ops.ptr(self.flag_ptrs), ops.ptr(self.state),
                  self.rank, self.world, 0)
        self._last = 0
        return work, nparts.value, 16

    def reduce(self, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """[n_local, C] f32 = sum over ranks (ascending) of their ``gall`` slice for this rank.  ``signal(1)`` first."""
        from . import ops
        if out is None:
            out = torch.empty((self.n_local, self.C), dtype=torch.float32, device=self.device)
        ops._call("cor_peer_reduce_rows", self.device, ops.ptr(self.gall_ptrs), ops.ptr(out), ops._ll(self.n_local * self.C),
                  ops.ptr(self.flag_ptrs), ops.ptr(self.state), self.rank, self.world, 1)
        self._last = 1
        return out

    def close(self):
        lib = self.lib
        for p in self.mapped:
            lib.cor_peer_close(C.c_void_p(p))
        self.mapped = []
        if self.base is not None:
            lib.cor_peer_free(C.c_void_p(self.base))
            self.base = None
        self.ok = False


def get_exchange(n_local: int, Cc: int, device, group=None) -> Optional[PeerExchange]:
    """The cached exchange for this shape, or None when peer memory is off / unavailable (-> NCCL).  Collective on
    first use per shape."""
    if not enabled() or not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return None
    if dist.get_backend(group) != "nccl":
        return None
    key = (n_local, Cc, torch.device(device).index, id(group))
    px = _CACHE.get(key)
    if px is None:
        px = PeerExchange(n_local, Cc, torch.device(device), group)
        _CACHE[key] = px
    return px if px.ok else None


def check_all():
    """``PeerExchange.check`` on every live exchange."""
    for px in _CACHE.values():
        if px.ok:
            px.check()


def release_all():
    """Unmap and free every cached exchange (call before tearing the process group down)."""
    for px in _CACHE.values():
        px.close()
    _CACHE.clear()
