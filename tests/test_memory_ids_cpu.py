"""CPU checks of the region memory's row ids: the new C entries refuse bad arguments with COR_EINVAL before any launch,
and the Python layer raises CorError for query ids without a memory, of the wrong dtype, shape or device, and for
enqueue ids of the wrong dtype, shape or device -- after the checks enqueue made before ids existed."""
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
        ("cor_memory_enqueue_ids", (one, 0, 4, 256, one, 8, one, null, one, 1, null)),       # null id ring
        ("cor_memory_enqueue_ids", (one, 0, 4, 256, one, 8, null, one, one, 1, null)),       # null state
        ("cor_memory_enqueue_ids", (one, 0, 4, 256, null, 8, one, one, one, 1, null)),       # null bank
        ("cor_memory_enqueue_ids", (one, 0, 4, 256, one, 8, one, one, one, 0, null)),        # group < 1
        ("cor_memory_enqueue_ids", (one, 0, 4, 256, one, 8, one, one, one, 3, null)),        # group does not divide n
        ("cor_memory_enqueue_ids", (one, 0, 9, 256, one, 8, one, one, one, 1, null)),        # n > K
        ("cor_memory_enqueue_ids", (one, 0, 1, 256, one, 0, one, one, one, 1, null)),        # K < 1
        ("cor_memory_enqueue_ids", (one, 0, 4, 96, one, 8, one, one, one, 1, null)),         # unsupported width
        ("cor_memory_enqueue_ids", (one, 2, 4, 256, one, 8, one, one, one, 1, null)),        # uint8 rows
        ("cor_memory_exclude", (null, 8, one, one, 4, one, null)),                           # null id ring
        ("cor_memory_exclude", (one, 8, null, one, 4, one, null)),                           # null state
        ("cor_memory_exclude", (one, 8, one, null, 4, one, null)),                           # null query ids
        ("cor_memory_exclude", (one, 8, one, one, 4, null, null)),                           # null mask
        ("cor_memory_exclude", (one, 0, one, one, 4, one, null)),                            # K < 1
        ("cor_memory_exclude", (one, 8, one, one, 0, one, null)),                            # Nq < 1
        ("cor_memory_scan_x", (one, 8, one, one, 4, 256, 14.0, null, null, one, nparts, null)),   # null mask
        ("cor_memory_scan_x", (one, 8, null, one, 4, 256, 14.0, null, one, one, nparts, null)),   # null state
        ("cor_memory_scan_x", (one, 0, one, one, 4, 256, 14.0, null, one, one, nparts, null)),    # K < 1
        ("cor_memory_scan_x", (one, 8, one, one, 0, 256, 14.0, null, one, one, nparts, null)),    # Nq < 1
        ("cor_memory_scan_x", (one, 8, one, one, 4, 100, 14.0, null, one, one, nparts, null)),    # unsupported width
        ("cor_memory_dq_x", (one, 8, one, one, 4, 256, 14.0, null, null, one, one, 1.0, one, null, one, null)),   # null mask
        ("cor_memory_dq_x", (one, 8, null, one, 4, 256, 14.0, null, one, one, one, 1.0, one, null, one, null)),   # null state
        ("cor_memory_dq_x", (one, 0, one, one, 4, 256, 14.0, null, one, one, one, 1.0, one, null, one, null)),    # K < 1
        ("cor_memory_dq_x", (one, 8, one, one, 4, 320, 14.0, null, one, one, one, 1.0, one, null, one, null)),    # unsupported width
        ("cor_memory_dq_x", (one, 8, one, one, 4, 256, 14.0, null, one, one, one, 1.0, null, null, one, null)),   # nothing to compute
        ("cor_memory_dq_x", (one, 8, one, one, 4, 256, 14.0, null, one, one, one, 1.0, one, one, one, null)),     # scale grad, no scale
    ]
    for name, args in cases:
        assert getattr(lib, name)(*args) == EINVAL, name
        assert lib.cor_last_error(), name
    assert lib.cor_memory_exclude_bytes(0, 8) == 0 and lib.cor_memory_exclude_bytes(4, 0) == 0
    assert lib.cor_memory_exclude_bytes(16, 65536) == 16 * 2048 * 4 and lib.cor_memory_exclude_bytes(3, 33) == 3 * 2 * 4


def _cpu_memory(K=8, C=256):
    """A RegionMemory's host-side state on CPU storage: its argument checks run before any device is touched."""
    from cor_b200 import region
    m = region.RegionMemory.__new__(region.RegionMemory)
    m.K, m.C, m.enqueues = K, C, 0
    m.bank, m.state = torch.zeros(K, C, dtype=torch.bfloat16), torch.zeros(4, dtype=torch.int32)
    m.ids = torch.full((K,), -1, dtype=torch.int64)
    return m


def test_query_ids_are_checked():
    from cor_b200 import ops, region
    x, t = torch.zeros(4, 256), torch.zeros(4, dtype=torch.int64)
    q4 = torch.zeros(4, dtype=torch.int64)
    with pytest.raises(_lib.CorError, match="together with memory="):
        ops.infonce_loss(x, x, t, query_ids=q4)
    with pytest.raises(_lib.CorError, match="together with memory="):
        region.region_infonce_loss(x, x, t, gather=False, query_ids=q4)
    with pytest.raises(_lib.CorError, match="together with memory="):
        region.region_step(x[:1], torch.zeros(1, 256, 4, 4), x[:1], torch.zeros(1, 16, 8, 8), query_ids=q4[:1])
    m = _cpu_memory()
    for q, msg in ((q4.int(), "int64"), ([0, 1, 2, 3], "int64"), (torch.zeros(3, dtype=torch.int64), r"must be \[4\]"),
                   (torch.zeros(4, 1, dtype=torch.int64), r"must be \[4\]"), (q4, "query_ids are on cpu")):
        with pytest.raises(_lib.CorError, match=msg):
            ops.infonce_loss(x, x, t, memory=m, query_ids=q)
    with pytest.raises(_lib.CorError, match=r"must be \[1\]"):
        region.region_step(x[:1], torch.zeros(1, 256, 4, 4), x[:1], torch.zeros(1, 16, 8, 8), memory=m, query_ids=q4)
    with pytest.raises(_lib.CorError, match="query_ids are on cpu"):
        region.region_step(x[:1], torch.zeros(1, 256, 4, 4), x[:1], torch.zeros(1, 16, 8, 8), memory=m, query_ids=q4[:1])
    # a memory object without an id ring (built before ids existed) takes no query ids
    del m.ids
    with pytest.raises(_lib.CorError, match="keeps row ids"):
        ops.infonce_loss(x, x, t, memory=m, query_ids=q4)


def test_enqueue_ids_are_checked_after_the_rows(monkeypatch):
    m = _cpu_memory(8, 128)
    # the rows' own errors come first, whatever the ids
    bad = torch.zeros(3, dtype=torch.int32)
    for rows, msg in ((torch.zeros(4, 128, dtype=torch.float16), "float32 or bfloat16"), (torch.zeros(4, 64), "C=128"),
                      (torch.zeros(9, 128), "1 to 8"), (torch.zeros(4, 128), "CUDA")):
        with pytest.raises(_lib.CorError, match=msg):
            m.enqueue(rows, ids=bad)
    # past the device checks (the memory and the rows on one device, here the host), the ids' own
    monkeypatch.setattr(_lib, "require_cuda", lambda *t: torch.device("cpu"))
    rows2, rows3 = torch.zeros(4, 128), torch.zeros(2, 4, 128)
    for rows, ids, msg in ((rows2, torch.zeros(4, dtype=torch.int32), "int64"), (rows2, [0, 1, 2, 3], "int64"),
                           (rows2, torch.zeros(3, dtype=torch.int64), r"must be \(4,\)"),
                           (rows2, torch.zeros(4, 1, dtype=torch.int64), r"must be \(4,\)"),
                           (rows3, torch.zeros(4, dtype=torch.int64), r"must be \(2, 4\) .* or \(2,\)"),
                           (rows3, torch.zeros(2, 4, 1, dtype=torch.int64), r"must be \(2, 4\)")):
        with pytest.raises(_lib.CorError, match=msg):
            m.enqueue(rows, ids=ids)
    assert m.enqueues == 0
