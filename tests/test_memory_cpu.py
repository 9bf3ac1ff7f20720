"""CPU checks of the cross-batch region memory: every new C entry refuses bad arguments with COR_EINVAL before any device
query, and the Python layer raises CorError for a wrong device, a width that differs from the rows, capacity < 1, more
rows than the capacity and an unsupported dtype."""
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


def test_new_entries_refuse_bad_arguments(lib):
    null, one = ctypes.c_void_p(None), ctypes.c_void_p(16)
    nparts = ctypes.byref(ctypes.c_int())
    cases = [
        ("cor_memory_reset", (null, null)),                                               # null state
        ("cor_memory_enqueue", (one, 0, 4, 256, one, 8, null, null)),                     # null state
        ("cor_memory_enqueue", (one, 0, 4, 256, null, 8, one, null)),                     # null bank
        ("cor_memory_enqueue", (one, 0, 1, 256, one, 0, one, null)),                      # K < 1
        ("cor_memory_enqueue", (one, 0, 0, 256, one, 8, one, null)),                      # n <= 0
        ("cor_memory_enqueue", (one, 0, 9, 256, one, 8, one, null)),                      # n > K
        ("cor_memory_enqueue", (one, 0, 4, 96, one, 8, one, null)),                       # unsupported width
        ("cor_memory_enqueue", (one, 2, 4, 256, one, 8, one, null)),                      # uint8 rows
        ("cor_memory_scan", (one, 8, null, one, 4, 256, 14.0, null, one, nparts, null)),  # null state
        ("cor_memory_scan", (null, 8, one, one, 4, 256, 14.0, null, one, nparts, null)),  # null bank
        ("cor_memory_scan", (one, 0, one, one, 4, 256, 14.0, null, one, nparts, null)),   # K < 1
        ("cor_memory_scan", (one, 8, one, one, 4, 100, 14.0, null, one, nparts, null)),   # unsupported width
        ("cor_memory_dq", (one, 8, null, one, 4, 256, 14.0, null, one, one, 1.0, one, null, one, null)),   # null state
        ("cor_memory_dq", (null, 8, one, one, 4, 256, 14.0, null, one, one, 1.0, one, null, one, null)),   # null bank
        ("cor_memory_dq", (one, 0, one, one, 4, 256, 14.0, null, one, one, 1.0, one, null, one, null)),    # K < 1
        ("cor_memory_dq", (one, 8, one, one, 4, 320, 14.0, null, one, one, 1.0, one, null, one, null)),    # unsupported width
        ("cor_memory_dq", (one, 8, one, one, 4, 256, 14.0, null, one, one, 1.0, one, one, one, null)),     # scale grad, no scale
        ("cor_infonce_tail_mem", (one, 4, 16, one, one, one, 8, 4, 64, 14.0, null, one, 4, null, one, one, one, null, null,
                                  0.0, 0.0, 0.0, null, null)),                            # memory partials without the state
        ("cor_step_tail_fwd_mem", (one, 1, 0, 17, 4, 16, 64, 1.0, one, one, one, one, 14.0, null, one, 0, one, one, 5.0, 5.0, 1.0,
                                   *([one] * 13), null)),                                 # memory partials, nparts = 0
    ]
    for name, args in cases:
        assert getattr(lib, name)(*args) == EINVAL, name
        assert lib.cor_last_error(), name
    assert lib.cor_memory_state_words() >= 3
    assert lib.cor_memory_scan_work_bytes(0, 8, 256) == 0 and lib.cor_memory_dq_work_bytes(4, 0, 256) == 0


def test_python_layer_refuses_bad_arguments():
    import cor_b200
    from cor_b200 import ops, region
    for args, msg in (((0, 256), "capacity"), ((8, 100), "C=100"), ((8, 256, "cpu"), "CUDA device")):
        with pytest.raises(_lib.CorError, match=msg):
            region.RegionMemory(*args)
    assert cor_b200.RegionMemory is region.RegionMemory
    # a memory's host-side argument checks, on CPU storage (they run before any device is touched)
    m = region.RegionMemory.__new__(region.RegionMemory)
    m.K, m.C, m.enqueues = 8, 128, 0
    m.bank, m.state = torch.zeros(8, 128, dtype=torch.bfloat16), torch.zeros(4, dtype=torch.int32)
    for rows, msg in ((torch.zeros(4, 128, dtype=torch.float16), "float32 or bfloat16"), (torch.zeros(4, 64), "C=128"),
                      (torch.zeros(9, 128), "1 to 8"), (torch.zeros(0, 128), "1 to 8"), (torch.zeros(4, 128), "CUDA")):
        with pytest.raises(_lib.CorError, match=msg):
            m.enqueue(rows)
    assert m.enqueues == 0
    x = torch.zeros(4, 256)
    with pytest.raises(_lib.CorError, match="width C=128"):
        ops.infonce_loss(x, x, torch.zeros(4, dtype=torch.int64), memory=m)
    with pytest.raises(_lib.CorError, match="must be a RegionMemory"):
        ops.infonce_loss(x, x, torch.zeros(4, dtype=torch.int64), memory=object())
    with pytest.raises(_lib.CorError, match="width C=128"):
        region.region_step(x, torch.zeros(1, 256, 4, 4), x, torch.zeros(1, 16, 8, 8), memory=m)
