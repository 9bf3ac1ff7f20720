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


# C types of the header -> ctypes.  Every pointer is a c_void_p; a type outside this table is an error, not a guess.
_SCALARS = {"int": C.c_int, "float": C.c_float, "long long": C.c_longlong, "size_t": C.c_size_t, "cor_stream_t": C.c_void_p}
_DECL = re.compile(r"^[ \t]*([A-Za-z_][\w \t*]*?)\s*\b(cor_\w+)\s*\(([^;]*?)\)\s*;", re.M)


def _ctype(fn: str, t: str, returned: bool = False):
    t = " ".join(t.replace("*", " * ").split())
    if returned and t == "const char *":
        return C.c_char_p                     # cor_last_error(): check() decodes it
    if "*" in t and re.fullmatch(r"[\w *]+", t):
        return C.c_void_p
    if t in _SCALARS:
        return _SCALARS[t]
    raise CorError(f"{fn}: no ctypes mapping for the type `{t}` declared in the header")


def declarations(header: str = HEADER):
    """{name: (restype, argtypes)} of every function the header declares, typed from the header itself."""
    if not os.path.exists(header):
        raise CorError(f"{header} not found: the C ABI header types every entry of libcor_b200.so")
    text = re.sub(r"/\*.*?\*/|//[^\n]*", "", open(header).read(), flags=re.S)
    decls = {}
    for ret, name, params in _DECL.findall(text):
        params = [] if params.strip() in ("", "void") else params.split(",")
        decls[name] = (_ctype(name, ret, returned=True), [_ctype(name, re.sub(r"\b\w+\s*$", "", p)) for p in params])
    return decls


def declared_symbols(header: str = HEADER):
    """Names of every function include/cor_b200.h declares (used by the CPU export test)."""
    return sorted(declarations(header))


def load(path: str = LIB_PATH):
    """dlopen the library (works without a GPU: cudart is linked statically) and type every entry from the header.
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
        decls = declarations()
        lib = C.CDLL(path)
        for name, (restype, argtypes) in decls.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = restype, argtypes
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
