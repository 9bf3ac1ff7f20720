"""CPU checks of the learnable logit scale: every new C entry rejects a NULL scale before touching a device, and the
Python entries reject tau together with logit_scale, and a scale that is not a 0-dim float32 CUDA tensor."""
import ctypes
import os

import pytest
import torch

from cor_b200 import _lib, build


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        build.build()
    return _lib.load()


def test_new_entries_reject_a_null_scale(lib):
    null, one = ctypes.c_void_p(None), ctypes.c_void_p(16)
    cases = {
        "cor_sim_stream_fwd_ls": (one, one, 8, 4, 64, null, one, one, one, null),
        "cor_sim_umma_fwd_ls": (one, one, 8, 4, 64, null, one, one, one, null),
        "cor_sim_lse_parts_ls": (0, one, one, 8, 4, 64, null, one, ctypes.byref(ctypes.c_int()), ctypes.byref(ctypes.c_int()), null),
        "cor_infonce_tail_ls": (one, 4, 16, one, one, one, 8, 4, 64, null, one, one, one, null, null, 0.0, 0.0, 0.0, null, null),
        "cor_infonce_fwd_ls": (one, one, one, one, 8, 4, 64, null, one, one, null),
        "cor_infonce_bwd_ls": (one, one, one, one, 8, 4, 64, null, one, 1.0, one, one, one, one, null),
        "cor_infonce_bwd_umma_ls": (one, one, 64, 64, 64, null, one, one, one, 1.0, one, one, one, one, null),
        "cor_step_tail_fwd_ls": (one, 1, 0, 17, 4, 16, 64, 1.0, one, one, one, one, null, one, 5.0, 5.0, 1.0,
                                 *([one] * 13), null),
        "cor_step_tail_bwd_ls": (one, one, one, one, 4, 16, 64, null, one, 1.0, one, one, one, one, one, one, 5.0, 5.0, one, 64, one, one,
                                 one, one, null),
        "cor_peer_gather_sim_ls": (one, one, 64, 64, one, 4, null, one, one, one, one, 0, 2, 0, null),
    }
    assert set(cases) == {n for n in _lib.declared_symbols() if n.endswith("_ls")}
    for name, args in cases.items():
        assert getattr(lib, name)(*args) == -1, name
        assert b"logit_scale" in lib.cor_last_error(), name


def test_region_step_validates_the_scale():
    from cor_b200 import ops, region
    x = torch.zeros(1)
    bad = [(dict(tau=0.07, logit_scale=torch.tensor(14.0)), "either tau or logit_scale"),
           (dict(logit_scale=torch.ones(2)), "0-dim float32"),
           (dict(logit_scale=torch.tensor(14.0, dtype=torch.float64)), "0-dim float32"),
           (dict(logit_scale=torch.tensor(14.0)), "CUDA tensor")]
    for kw, msg in bad:
        with pytest.raises(_lib.CorError, match=msg):
            region.region_step(x, x, x, x, **kw)
        with pytest.raises(_lib.CorError, match=msg):
            ops.infonce_loss(x, x, x, **kw)
        with pytest.raises(_lib.CorError, match=msg):
            region.region_infonce_loss(x, x, x, **kw)
