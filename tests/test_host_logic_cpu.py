"""Host-side decisions added in round 2 that need no GPU: which exchange / pooling-tail / mask-branch path a shape takes."""
import os

import torch
import torch.nn as nn


def test_fused_gather_similarity_is_chosen_where_the_streaming_kernel_would_score(monkeypatch):
    from cor_b200 import region
    monkeypatch.delenv("COR_PEER_FUSED", raising=False)
    assert region._peer_fused_ok(16, 256, 2 * 1024)            # 2 GPUs x 1024 regions: streaming similarity -> fused
    assert region._peer_fused_ok(16, 256, 4 * 1024)
    assert not region._peer_fused_ok(16, 256, 8 * 1024)        # 8 192 regions: the tensor-core similarity kernel takes over
    assert not region._peer_fused_ok(17, 256, 2048)            # more than one query tile
    assert not region._peer_fused_ok(16, 260, 2048)            # one 16-byte vector per lane: C <= 256, C % 8 == 0
    assert not region._peer_fused_ok(16, 252, 2048)
    assert region._peer_fused_ok(16, 256, 8 * 1024, "stream")  # an explicit streaming engine keeps the fusion
    monkeypatch.setenv("COR_PEER_FUSED", "0")
    assert not region._peer_fused_ok(16, 256, 2048)
    monkeypatch.setenv("COR_PEER_FUSED", "2")
    assert region._peer_fused_ok(16, 256, 8 * 1024)
    assert not region._peer_fused_ok(32, 256, 8 * 1024)        # the kernel's own limits still hold when forced


def test_pooling_tail_and_mask_branch_eligibility():
    from cor_b200 import mask_adapter as ma
    maps, feat = torch.zeros(2, 16, 24, 24), torch.zeros(2, 768, 24, 24)
    assert not ma._tail_gemm_ok(maps, feat, 8)                 # CPU tensors never take a CUDA path
    m = ma.MaskAdapterPooling(x_in_channel=768, mask_adatpet_network_in_channel=512, mask_downscaling_mid_channel=16,
                              mask_adatpet_network_mid_channel=256, num_output_maps=8)
    md = m.get_mask_map.mask_downscaling
    assert ma._md_fusable(md)                                  # the reference's own layout: conv, LN2d, GELU, conv, LN2d, GELU, conv
    other = nn.Sequential(*list(md.children())[:6], nn.Identity())
    other[2] = nn.ReLU()
    assert not ma._md_fusable(other)
    tanh = nn.Sequential(*list(md.children()))
    tanh[5] = nn.GELU(approximate="tanh")
    assert not ma._md_fusable(tanh)


def test_seg_coefficients_and_act_codes_are_stable():
    from cor_b200 import _lib as L
    assert (L.ACT_NONE, L.ACT_RELU, L.ACT_GELU, L.ACT_SIGMOID) == (0, 1, 2, 3)
    assert L.ABI_VERSION == 3
