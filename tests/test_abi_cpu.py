"""CPU checks of the drop-in boundary: the C-ABI library loads without a GPU and exports every
symbol include/cor_b200.h declares; the product path refuses CPU tensors instead of falling back."""
import ctypes
import inspect
import os

import pytest
import torch

from cor_b200 import _lib, build
from oracle.build_ref import REFERENCE


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        build.build()
    return _lib.load()


def test_library_exports_every_declared_symbol(lib):
    names = _lib.declared_symbols()
    assert len(names) >= 25
    raw = ctypes.CDLL(_lib.LIB_PATH)
    missing = [n for n in names if not hasattr(raw, n)]
    assert not missing, f"declared in include/cor_b200.h but not exported: {missing}"
    assert lib.cor_abi_version() == _lib.ABI_VERSION == 3


def test_no_torch_types_in_the_header():
    """The boundary is a plain C ABI: extern "C", pointers and sizes only."""
    text = open(_lib.HEADER).read()
    code = "\n".join(l for l in text.splitlines() if not l.lstrip().startswith(("*", "/*", "//")))
    assert 'extern "C"' in text
    for banned in ("at::", "torch::", "c10::", "std::", "class ", "template"):
        assert banned not in code, banned


def test_size_queries_need_no_gpu(lib):
    # max(64x64 tiles = 16, strips of >= 16 rows = 16) records of cor_seg_loss_npartials() doubles per sample
    assert lib.cor_seg_loss_npartials() == 10
    assert lib.cor_seg_loss_work_bytes(16, 256, 256) == 16 * 16 * 10 * 8
    assert lib.cor_fgbg_aux_floats(16, 256) == 16 * 8 + 3 * 256
    assert lib.cor_mask_prep_work_bytes(4, 64, 64, 16, 16) > 0


def test_cpu_tensors_are_refused_not_served():
    from cor_b200 import loss_func, mask_adapter, ops
    x = torch.randn(2, 1, 32, 32)
    with pytest.raises(_lib.CorError, match="no CPU fallback"):
        loss_func.wbce_with_wiou_loss(x, torch.rand(2, 1, 32, 32))
    with pytest.raises(_lib.CorError, match="no CPU fallback"):
        mask_adapter.MaskedPooling()(torch.randn(2, 8, 4, 4), torch.rand(2, 1, 16, 16))
    with pytest.raises(_lib.CorError, match="no CPU fallback"):
        ops.similarity(torch.randn(8, 16), torch.randn(2, 16))


def test_product_never_imports_the_oracle():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for dirpath, _, files in os.walk(os.path.join(root, "cor_b200")):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f"{f} imports the oracle"


def test_dropin_signatures_match_the_reference():
    """Argument names of the reference entry points (utils/loss_func.py:5,35,59,88;
    lib/support_model/mask_adapter.py:13,31-37,52)."""
    from cor_b200 import loss_func as lf
    from cor_b200 import mask_adapter as ma
    sig = lambda f: list(inspect.signature(f).parameters)
    assert sig(lf.wbce_with_wiou_loss) == ["pred", "mask", "w1", "w2"]
    assert sig(lf.mask_pooling) == ["embeddings", "mask"]
    assert sig(lf.fg_feat_similarity_loss) == ["query_image_embeddings", "comb_support_feat", "query_mask"]
    assert sig(lf.bg_feat_similarity_loss) == ["query_image_embeddings", "comb_support_feat", "query_mask"]
    from cor_b200 import metrics as mt
    assert sig(mt.compute_dice) == ["pred", "gt", "smooth"] and sig(mt.compute_mae) == ["pred", "gt"]
    assert sig(mt.compute_miou) == ["pred", "gt", "smooth"]
    assert sig(ma.MaskedPooling.forward) == ["self", "clip_feature", "mask"]
    assert sig(ma.MaskAdapterPooling.forward) == ["self", "clip_feature", "mask"]
    assert sig(ma.MaskAdapterPooling.__init__) == ["self", "x_in_channel", "mask_adatpet_network_in_channel",
                                                   "mask_downscaling_mid_channel", "mask_adatpet_network_mid_channel",
                                                   "num_output_maps"]


def test_mask_adapter_parameter_names_match_reference_checkpoints():
    """strict checkpoint loading (my_test.py:145) needs identical state_dict keys; the expected key
    list was captured from the reference module (SupportBranch config, support_branch.py:30-36)."""
    from cor_b200.mask_adapter import MaskAdapterPooling
    m = MaskAdapterPooling(x_in_channel=64, mask_adatpet_network_in_channel=32, mask_downscaling_mid_channel=16,
                           mask_adatpet_network_mid_channel=32, num_output_maps=8)
    keys = set(m.state_dict().keys())
    expect = {"channel_clip_to_maskadapter.conv.weight", "channel_clip_to_maskadapter.norm.weight", "get_mask_map.fuse.weight",
              "get_mask_map.cnext1.gamma", "get_mask_map.cnext1.dwconv.weight", "get_mask_map.cnext2.pwconv1.weight",
              "get_mask_map.cnext3.pwconv2.bias", "get_mask_map.cnext3.norm.weight", "get_mask_map.norm.bias",
              "get_mask_map.final.weight", "get_mask_map.mask_downscaling.0.weight", "get_mask_map.mask_downscaling.1.weight",
              "get_mask_map.mask_downscaling.3.weight", "get_mask_map.mask_downscaling.4.bias",
              "get_mask_map.mask_downscaling.6.weight"}
    assert expect <= keys
    if os.path.isdir(REFERENCE):   # with a reference checkout: compare against the real module
        import sys
        sys.path.insert(0, REFERENCE)
        from lib.support_model.mask_adapter import MaskAdapterPooling as Ref
        r = Ref(x_in_channel=64, mask_adatpet_network_in_channel=32, mask_downscaling_mid_channel=16,
                mask_adatpet_network_mid_channel=32, num_output_maps=8)
        assert {k: tuple(v.shape) for k, v in r.state_dict().items()} == {k: tuple(v.shape) for k, v in m.state_dict().items()}
        m.load_state_dict(r.state_dict(), strict=True)


@pytest.mark.skipif(not os.path.isdir(REFERENCE), reason="needs a checkout of the reference named by COR_REFERENCE")
def test_hooks_install_into_the_real_reference():
    """hooks.install() rebinds the reference's own names; SupportBranch (support_branch.py:29-40) then
    builds with the patched pooling classes, parameters and error behaviour untouched."""
    import sys
    import types
    sys.path.insert(0, REFERENCE)
    for name in ("open_clip", "accelerate"):
        if name not in sys.modules:
            m = types.ModuleType(name)
            m.Accelerator = object
            m.DistributedType = types.SimpleNamespace(MULTI_GPU="MULTI_GPU", DEEPSPEED="DEEPSPEED")
            sys.modules[name] = m
    from cor_b200 import hooks, loss_func, mask_adapter
    import utils.loss_func as ref_lf
    import lib.support_model.mask_adapter as ref_ma
    import lib.support_model.siglip_openclip as ref_sig
    orig = ref_lf.wbce_with_wiou_loss
    done = hooks.install()
    try:
        assert "utils.loss_func" in done and "lib.support_model.mask_adapter" in done
        assert ref_lf.wbce_with_wiou_loss is loss_func.wbce_with_wiou_loss
        assert ref_lf.fg_feat_similarity_loss is loss_func.fg_feat_similarity_loss
        ref_sig.SigLIP = lambda *a, **k: torch.nn.Identity()
        import lib.support_branch as sb
        sb.SigLIP = ref_sig.SigLIP
        branch = sb.SupportBranch("ViT-B-16-SigLIP-384", "unused", mask_pooling="MaskAdapterPooling")
        assert any(k.startswith("mask_pooling.get_mask_map.") for k in branch.state_dict())
        with pytest.raises(_lib.CorError, match="no CPU fallback"):      # the patched forward is the CUDA path
            branch.mask_pooling(torch.randn(1, 768, 24, 24), torch.rand(1, 1, 24, 24))
        with pytest.raises(ValueError):
            sb.SupportBranch("ViT-B-16-SigLIP-384", "unused", mask_pooling="nope")
        assert type(sb.SupportBranch("ViT-B-16-SigLIP-384", "unused", mask_pooling="MaskedPooling").mask_pooling).forward \
            is hooks._masked_forward
        # the composed-query head and the decoder's hypernetwork product are rebound on the reference's own classes too
        from cor_b200 import mask_decoder as md, support_head as sh
        import lib.sam_model.mask_decoder as ref_md
        assert sb.SupportBranch.forward is sh.support_branch_forward
        assert ref_md.MaskDecoder.predict_masks is md.predict_masks
        assert "lib.support_branch" in done and "lib.sam_model.mask_decoder" in done
    finally:
        hooks.uninstall()
    assert ref_lf.wbce_with_wiou_loss is orig
    assert ref_ma.MaskedPooling.forward is not hooks._masked_forward


def test_argument_validation_fails_before_any_launch(lib):
    """Bad arguments come back as COR_EINVAL (-1) with a message, before the library touches a device: the error
    behaviour a binding in another host language would rely on (INTEGRATION.md contract)."""
    EINVAL = -1
    null = ctypes.c_void_p(None)
    one = ctypes.c_void_p(16)          # any non-null value: validation must reject the call before dereferencing it
    cases = [
        ("cor_peer_gather_rows", (null, one, 1024, one, one, 0, 2, 0, null)),            # null source table
        ("cor_peer_gather_rows", (one, one, 1000, one, one, 0, 2, 0, null)),             # bytes not a multiple of 16
        ("cor_peer_gather_rows", (one, one, 1024, one, one, 3, 2, 0, null)),             # rank outside the world
        ("cor_peer_reduce_rows", (one, one, 1024, one, one, 0, 64, 1, null)),            # world beyond cor_peer_max_world()
        ("cor_peer_gather_sim", (one, one, 64, 256, one, 17, 14.0, one, one, one, one, 0, 2, 0, null)),   # more queries than a tile
        ("cor_peer_signal", (one, one, 0, 2, 5, null)),                                  # channel out of range
        ("cor_infonce_tail", (null, 4, 16, one, one, one, 8, 4, 64, 1.0, one, one, one, null, null, 0.0, 0.0, 0.0, null, null)),
        ("cor_infonce_tail", (one, 4, 16, one, one, one, 8, 4, 64, 1.0, one, one, one, null, null, 0.0, 0.0, 0.0, one, null)),  # total without seg/fgbg
        ("cor_sim_umma_fwd", (one, one, 8, 4, 64, 1.0, one, one, one, null)),             # S and lse in one call
        ("cor_sim_lse_parts", (0, one, one, 8, 4, 64, 1.0, one, None, None, null)),      # nowhere to report the layout
        ("cor_topk", (one, one, one, 8, 4, 64, 9, one, one, null)),                      # k > Nr
        ("cor_gemm_bf16", (one, 0, 8, 0, one, 0, 8, 0, 8, 8, 0, 1, 1.0, null, 0, null, null, null, 0, 8, one, 0, 8, null, 0, null, null)),  # K = 0
        ("cor_gemm_bf16", (one, 0, 8, 0, one, 0, 8, 0, 8, 8, 64, 1, 1.0, null, 9, null, null, null, 0, 8, one, 0, 8, null, 0, null, null)), # unknown activation
        ("cor_hyper_logits_fwd", (one, one, 0, one, 0, 2, 4, 0, 5, 32, 64, null)),       # more tokens than exist
        ("cor_ln_cf_fwd", (one, one, one, 4, 33, 64, 1e-6, 0, one, null)),               # more channels than the kernel holds
        ("cor_adapter_tail_weights", (one, 2, 12, 64, 8, 64, one, one, null)),           # R not a multiple of the group
        ("cor_adapter_tail_bwd", (one, one, null, 2, 16, 64, 8, one, null)),             # null gradient
        ("cor_infonce_bwd_umma", (one, one, 64, 64, 100, 1.0, one, one, one, 1.0, one, one, one, null)),   # D not a multiple of 64
        ("cor_act_bwd", (one, 0, null, null, null, null, 1, 4, 4, one, null, null, null, null)),   # relu without the activation output
        ("cor_ln_rows_fwd", (one, one, one, 8, 2048, 1e-6, 0, one, 0, null, null)),      # more channels than a warp holds
    ]
    for name, args in cases:
        rc = getattr(lib, name)(*args)
        assert rc == EINVAL, (name, rc)
        assert lib.cor_last_error(), name
    assert lib.cor_peer_max_world() >= 8 and lib.cor_peer_flag_bytes() >= 4 * 2 * 2 * 8 and lib.cor_peer_state_bytes() >= 16


def test_header_is_plain_c_and_a_c_host_can_bind_it(lib, tmp_path):
    """include/cor_b200.h compiles as C99 (not only as C++) and a C program linked against the library can call it."""
    import shutil
    import subprocess
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no gcc")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    libdir = os.path.dirname(_lib.LIB_PATH)
    exe = str(tmp_path / "c_abi_probe")
    cmd = [gcc, "-std=c99", "-Wall", "-Werror", "-pedantic", "-I", os.path.join(root, "include"), os.path.join(root, "examples", "c_abi_probe.c"),
           "-L", libdir, "-l:libcor_b200.so", f"-Wl,-rpath,{libdir}", "-o", exe]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0, (r.returncode, r.stdout, r.stderr)
    assert "ABI v3" in r.stdout and "-> -1" in r.stdout
