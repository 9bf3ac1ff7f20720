"""ctypes binding of libcor_b200.so (include/cor_b200.h).  No fallback: if the library is missing
or a call fails, this raises -- the product path never routes around the CUDA kernels."""
from __future__ import annotations

import ctypes as C
import os
import re
import threading

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libcor_b200.so")
HEADER = os.path.join(os.path.dirname(HERE), "include", "cor_b200.h")

F32, BF16, U8 = 0, 1, 2
ABI_VERSION = 3
# terms of the segmentation loss (include/cor_b200.h COR_SEG_*)
ACT_NONE, ACT_RELU, ACT_GELU, ACT_SIGMOID = range(4)
SEG_WBCE, SEG_WIOU, SEG_DICE, SEG_BCE, SEG_IOU, SEG_WDICE, SEG_FOCAL, SEG_NTERMS = range(8)
W_PLAIN, W_CLAMP, W_SIGMOID = 0, 1, 2

_DTYPES = {torch.float32: F32, torch.bfloat16: BF16, torch.uint8: U8}

_lib = None
_lock = threading.Lock()


class CorError(RuntimeError):
    """A libcor_b200 call returned a non-zero status."""


def declared_symbols(header: str = HEADER):
    """Names of every function include/cor_b200.h declares (used by the CPU export test)."""
    text = re.sub(r"/\*.*?\*/", "", open(header).read(), flags=re.S)
    return sorted(set(re.findall(r"\b(cor_[a-z0-9_]+)\s*\(", text)))


def _sig(lib, name, restype, *argtypes):
    fn = getattr(lib, name)
    fn.restype = restype
    fn.argtypes = list(argtypes)
    return fn


def load(path: str = LIB_PATH):
    """dlopen the library (works without a GPU: cudart is linked statically) and type every entry.
    ``COR_B200_LIB`` points at another build of the same ABI (A/B runs of two kernel versions on one box)."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = os.environ.get("COR_B200_LIB", path)
        if not os.path.exists(path):
            raise CorError(
                f"{path} not found: build it with `python -m cor_b200.build` (nvcc, sm_100a). "
                "cor_b200 has no CPU or PyTorch fallback by design.")
        lib = C.CDLL(path)
        p, i, f, ll, sz = C.c_void_p, C.c_int, C.c_float, C.c_longlong, C.c_size_t
        _sig(lib, "cor_abi_version", i)
        _sig(lib, "cor_last_error", C.c_char_p)
        _sig(lib, "cor_device_info", i, C.POINTER(i), C.POINTER(i), C.POINTER(i))
        _sig(lib, "cor_mask_prep_work_bytes", sz, i, i, i, i, i)
        _sig(lib, "cor_mask_prep", i, p, i, f, i, i, i, i, i, i, p, p, ll, i, ll, p, p, p)
        _sig(lib, "cor_pool_stream_fwd", i, p, i, p, ll, i, i, i, i, i, p, p, p)
        _sig(lib, "cor_pool_umma_work_bytes", sz, i, i, i, i)
        _sig(lib, "cor_pool_umma_ksplit", i, i, i, i)
        _sig(lib, "cor_pool_umma_fwd", i, p, p, i, i, i, i, p, p)
        _sig(lib, "cor_rows_finalize", i, p, i, ll, i, ll, p, i, f, i, i, i, i, p, f, p, p, p, p)
        _sig(lib, "cor_rows_finalize_bwd", i, p, p, p, p, i, f, i, i, i, i, i, f, p, p)
        _sig(lib, "cor_pool_bwd_feat", i, p, p, p, ll, i, i, i, i, i, p, i, p)
        _sig(lib, "cor_pool_bwd_umma_ok", i, i, i, i, i, i)
        _sig(lib, "cor_pool_bwd_umma", i, p, p, p, ll, i, i, i, i, i, p, i, p)
        _sig(lib, "cor_pool_bwd_maps", i, p, i, p, ll, p, p, p, i, i, i, i, p, p)
        _sig(lib, "cor_fgbg_aux_floats", sz, i, i)
        _sig(lib, "cor_fgbg_loss_fwd", i, p, ll, p, ll, p, ll, p, ll, i, i, i, p, p, p)
        _sig(lib, "cor_fgbg_loss_bwd", i, p, ll, p, ll, p, ll, i, i, i, p, p, p, ll, f, f, p, ll, i, p, ll, p, ll, i, p)
        _sig(lib, "cor_step_tail_counter_words", i)
        _sig(lib, "cor_step_tail_work_bytes", sz, i, i, i)
        _sig(lib, "cor_step_tail_fwd", i, p, i, ll, i, i, i, i, f, p, p, p, p, f, p, f, f, f, p, p, p, p, p, p, p, p, p, p, p, p, p, p)
        _sig(lib, "cor_step_tail_bwd", i, p, p, p, p, i, i, i, f, p, f, p, p, p, p, p, p, f, f, p, i, p, p, p, p)
        _sig(lib, "cor_step_tail_fwd_ls", i, p, i, ll, i, i, i, i, f, p, p, p, p, p, p, f, f, f, p, p, p, p, p, p, p, p, p, p, p, p, p, p)
        _sig(lib, "cor_step_tail_bwd_ls", i, p, p, p, p, i, i, i, p, p, f, p, p, p, p, p, p, f, f, p, i, p, p, p, p, p)
        _sig(lib, "cor_seg_loss_work_bytes", sz, i, i, i)
        _sig(lib, "cor_seg_loss_npartials", i)
        fp = C.POINTER(C.c_float)
        _sig(lib, "cor_seg_loss_fwd", i, p, i, p, i, f, i, i, i, i, i, ll, fp, f, f, f, p, p, p, p, p, p)
        _sig(lib, "cor_seg_loss_bwd", i, p, i, p, p, p, i, i, i, fp, f, f, f, p, p, i, p)
        _sig(lib, "cor_sim_work_bytes", sz, i, i, i)
        _sig(lib, "cor_sim_stream_fwd", i, p, p, i, i, i, f, p, p, p, p)
        _sig(lib, "cor_sim_umma_fwd", i, p, p, i, i, i, f, p, p, p, p)
        _sig(lib, "cor_infonce_fwd", i, p, p, p, p, i, i, i, f, p, p, p)
        _sig(lib, "cor_sim_lse_parts", i, i, p, p, i, i, i, f, p, C.POINTER(i), C.POINTER(i), p)
        _sig(lib, "cor_infonce_tail", i, p, i, i, p, p, p, i, i, i, f, p, p, p, p, p, f, f, f, p, p)
        _sig(lib, "cor_infonce_bwd", i, p, p, p, p, i, i, i, f, p, f, p, p, p, p)
        _sig(lib, "cor_infonce_bwd_umma_work_bytes", sz, i, i, i)
        _sig(lib, "cor_infonce_bwd_umma", i, p, p, i, i, i, f, p, p, p, f, p, p, p, p)
        # the same entries with the logit scale read from device memory (and its gradient written there)
        _sig(lib, "cor_sim_stream_fwd_ls", i, p, p, i, i, i, p, p, p, p, p)
        _sig(lib, "cor_sim_umma_fwd_ls", i, p, p, i, i, i, p, p, p, p, p)
        _sig(lib, "cor_sim_lse_parts_ls", i, i, p, p, i, i, i, p, p, C.POINTER(i), C.POINTER(i), p)
        _sig(lib, "cor_infonce_tail_ls", i, p, i, i, p, p, p, i, i, i, p, p, p, p, p, p, f, f, f, p, p)
        _sig(lib, "cor_infonce_fwd_ls", i, p, p, p, p, i, i, i, p, p, p, p)
        _sig(lib, "cor_infonce_bwd_ls", i, p, p, p, p, i, i, i, p, p, f, p, p, p, p, p)
        _sig(lib, "cor_infonce_bwd_umma_ls", i, p, p, i, i, i, p, p, p, p, f, p, p, p, p, p)
        _sig(lib, "cor_topk", i, p, p, p, i, i, i, i, p, p, p)
        _sig(lib, "cor_l2_normalize", i, p, i, i, i, p, p, p, p)
        _sig(lib, "cor_gemm_bf16_work_bytes", sz, i, i, i, i, i)
        _sig(lib, "cor_gemm_bf16", i, p, i, ll, ll, p, i, ll, ll, i, i, i, i, f, p, i, p, p, p, i, ll, p, i, ll, p, i, p, p)
        _sig(lib, "cor_cast_cat_bf16", i, p, i, p, i, ll, p, p)
        _sig(lib, "cor_cast_pad_rows_bf16", i, p, i, i, i, i, p, p)
        _sig(lib, "cor_act_bwd_work_bytes", sz, ll, i)
        _sig(lib, "cor_act_bwd", i, p, i, p, p, p, p, i, ll, i, p, p, p, p, p)
        _sig(lib, "cor_dwconv7_work_bytes", sz, i, i, i, i)
        _sig(lib, "cor_dwconv7_cl", i, p, p, p, p, i, i, i, i, i, p)
        _sig(lib, "cor_dwconv7_cl_wgrad", i, p, p, p, p, i, i, i, i, p, p)
        _sig(lib, "cor_ln_rows_work_bytes", sz, ll, i)
        _sig(lib, "cor_ln_rows_fwd", i, p, p, p, ll, i, f, i, p, i, p, p)
        _sig(lib, "cor_ln_rows_bwd", i, p, i, p, p, p, p, ll, i, i, p, p, p, p, p)
        _sig(lib, "cor_ln_cf_work_bytes", sz, ll, i, ll)
        _sig(lib, "cor_ln_cf_fwd", i, p, p, p, ll, i, ll, f, i, p, p)
        _sig(lib, "cor_ln_cf_bwd", i, p, p, p, p, ll, i, ll, f, i, p, p, p, p, p)
        _sig(lib, "cor_adapter_tail_weights", i, p, i, i, i, i, i, p, p, p)
        _sig(lib, "cor_adapter_tail_bwd", i, p, p, p, i, i, i, i, p, p)
        _sig(lib, "cor_hyper_logits_work_bytes", sz, i, i, i, ll)
        _sig(lib, "cor_hyper_logits_fwd", i, p, p, i, p, i, i, i, i, i, i, ll, p)
        _sig(lib, "cor_hyper_logits_bwd", i, p, p, i, p, i, p, p, i, i, i, i, i, ll, p, p)
        _sig(lib, "cor_val_post_work_bytes", sz, i, i, i)
        _sig(lib, "cor_val_post", i, p, i, i, i, i, i, i, i, p, p, p, i, f, p, p, p)
        _sig(lib, "cor_soft_metrics", i, p, p, i, f, i, ll, f, p, p, p)
        pp = C.POINTER(C.c_void_p)
        _sig(lib, "cor_peer_max_world", i)
        _sig(lib, "cor_peer_flag_bytes", sz)
        _sig(lib, "cor_peer_state_bytes", sz)
        _sig(lib, "cor_peer_error_word", i)
        _sig(lib, "cor_peer_alloc", i, i, sz, pp)
        _sig(lib, "cor_peer_free", i, p)
        _sig(lib, "cor_peer_export", i, p, C.c_char_p)
        _sig(lib, "cor_peer_open", i, i, C.c_char_p, pp)
        _sig(lib, "cor_peer_close", i, p)
        _sig(lib, "cor_peer_signal", i, p, p, i, i, i, p)
        _sig(lib, "cor_peer_wait_exit", i, p, p, i, i, i, p)
        _sig(lib, "cor_peer_gather_rows", i, p, p, ll, p, p, i, i, i, p)
        _sig(lib, "cor_peer_reduce_rows", i, p, p, ll, p, p, i, i, i, p)
        _sig(lib, "cor_peer_gather_sim_work_bytes", sz)
        _sig(lib, "cor_peer_gather_sim", i, p, p, ll, i, p, i, f, p, p, p, p, i, i, i, p)
        _sig(lib, "cor_peer_gather_sim_ls", i, p, p, ll, i, p, i, p, p, p, p, p, i, i, i, p)
        if lib.cor_abi_version() != ABI_VERSION:
            raise CorError(f"ABI version mismatch: library {lib.cor_abi_version()}, binding {ABI_VERSION}; rebuild with `python -m cor_b200.build`")
        _lib = lib
        return lib


def check(rc: int, what: str):
    if rc != 0:
        msg = load().cor_last_error().decode(errors="replace")
        raise CorError(f"{what} failed (status {rc}): {msg}")


_device_ok = set()


def require_cuda(*tensors):
    """Every tensor must live on one sm_100 CUDA device.  Raises otherwise (no CPU fallback)."""
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise CorError("cor_b200 kernels need CUDA tensors (sm_100a); got a %s tensor. "
                           "There is no CPU fallback by design." % t.device)
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise CorError(f"tensors on different devices: {dev} vs {t.device}")
    if dev is not None and dev.index not in _device_ok:
        with torch.cuda.device(dev):
            check(load().cor_device_info(None, None, None), "cor_device_info")
        _device_ok.add(dev.index)
    return dev


def dtype_code(t: torch.Tensor) -> int:
    try:
        return _DTYPES[t.dtype]
    except KeyError:
        raise CorError(f"unsupported dtype {t.dtype} (supported: float32, bfloat16, uint8)") from None


def ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
