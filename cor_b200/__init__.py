"""cor_b200 -- B200 (sm_100a) kernels for CORE's region pooling, scoring and loss path.

Public surface (mirrors the reference, wangtong627/COR):
  cor_b200.loss_func      drop-in for utils/loss_func.py
  cor_b200.mask_adapter   drop-in for the pooling modules of lib/support_model/mask_adapter.py
  cor_b200.hooks.install  rebinds those names inside an unmodified reference checkout
  cor_b200.region         multi-mask pooling, similarity matrix, InfoNCE, top-k, fused step
  cor_b200.ops            the operator layer over the C ABI (include/cor_b200.h)
All compute is in cor_b200/libcor_b200.so (build: ``python -m cor_b200.build``); there is no CPU
or PyTorch fallback.  ``cor_b200.synth`` (numpy only) generates the benchmark inputs.
"""
__version__ = "0.1.0"

from ._lib import CorError  # noqa: E402,F401


def __getattr__(name):
    # cor_b200.RegionMemory without importing the region layer (and torch.distributed) at package import
    if name == "RegionMemory":
        from .region import RegionMemory
        return RegionMemory
    raise AttributeError(f"module {__name__!r} has no attribute {name!r}")
