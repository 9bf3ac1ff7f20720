"""Generate tests/golden/*.npz by running the UNMODIFIED reference (wangtong627/COR) here.

Needs a checkout of the reference, named by COR_REFERENCE (the same variable oracle/build_ref.py reads):

    COR_REFERENCE=/path/to/COR python oracle/gen_golden.py

Every fixture stores the inputs (compressed) and the reference's outputs and autograd
gradients, all float32, computed on CPU in fp32 by importing the reference's own modules
(`utils.loss_func`, `lib.support_model.mask_adapter`, and the metric functions of
`utils.trainer_v3_g`, which is loaded with a stub `accelerate`).  Nothing from the reference is
copied into this repo; only the numeric vectors are.
"""
from __future__ import annotations

import os
import sys
import types

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, ROOT)

from cor_b200 import synth  # noqa: E402
from oracle.build_ref import REFERENCE as REF  # noqa: E402

sys.path.insert(0, REF)


def _stub(name, **attrs):
    m = types.ModuleType(name)
    for k, v in attrs.items():
        setattr(m, k, v)
    sys.modules[name] = m
    return m


def load_reference():
    _stub("accelerate", Accelerator=object, DistributedType=types.SimpleNamespace(MULTI_GPU="MULTI_GPU", DEEPSPEED="DEEPSPEED"))
    _stub("accelerate.utils", DistributedType=types.SimpleNamespace(MULTI_GPU="MULTI_GPU", DEEPSPEED="DEEPSPEED"))
    from utils import loss_func
    from lib.support_model import mask_adapter
    try:
        from utils import trainer_v3_g as trainer
    except Exception as e:  # pragma: no cover - diagnostics only
        print("trainer import failed, metrics fixtures use loss_func only:", e)
        trainer = None
    return loss_func, mask_adapter, trainer


def t(x, grad=False):
    return torch.from_numpy(np.ascontiguousarray(x)).clone().requires_grad_(grad)


def save(name, **arrays):
    os.makedirs(OUT, exist_ok=True)
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **{k: np.asarray(v) for k, v in arrays.items()})
    print(f"{name}: {os.path.getsize(path) / 1024:.1f} KiB  keys={sorted(arrays)}")


def main():
    if not os.path.isdir(REF):
        raise SystemExit("set COR_REFERENCE to a checkout of the reference (wangtong627/COR)")
    torch.manual_seed(0)
    torch.set_num_threads(4)
    lf, ma, trainer = load_reference()
    rng = np.random.default_rng(20260118)

    # ---- a1 MaskedPooling (mask_adapter.py:13-25): integer and non-integer resample ----
    for tag, (C, hw, HW, soft) in {"int16": (48, 24, 384, False), "so400m": (40, 27, 384, True), "same": (24, 12, 12, True)}.items():
        feat = rng.standard_normal((2, C, hw, hw)).astype(np.float32)
        mask = synth.make_masks(rng, 2, 1, HW, HW, soft=soft, degenerate=False)
        f = t(feat, True)
        out = ma.MaskedPooling()(f, t(mask))
        g = rng.standard_normal(out.shape).astype(np.float32)
        out.backward(t(g))
        save(f"masked_pooling_{tag}", feat=feat, mask=mask, out=out.detach().numpy(), gout=g, gfeat=f.grad.numpy())

    # ---- a2 MaskAdapterPooling tail (mask_adapter.py:62-80) through the real module ----
    torch.manual_seed(1)
    mod = ma.MaskAdapterPooling(x_in_channel=40, mask_adatpet_network_in_channel=32, mask_downscaling_mid_channel=16,
                                mask_adatpet_network_mid_channel=32, num_output_maps=8).eval()
    grabbed = {}
    mod.get_mask_map.register_forward_hook(lambda m, i, o: grabbed.__setitem__("maps", o))
    feat = rng.standard_normal((2, 40, 24, 24)).astype(np.float32)
    mask = synth.make_masks(rng, 2, 3, 96, 96, degenerate=False)
    f = t(feat, True)
    out = mod(f, t(mask))                                  # [2,3,40]
    maps = grabbed["maps"]
    maps.retain_grad()
    g = rng.standard_normal(out.shape).astype(np.float32)
    # gradient of the TAIL only: d out / d maps and d out / d feat with maps held fixed
    maps_leaf = maps.detach().clone().requires_grad_(True)
    f2 = t(feat, True)
    B, C = 2, 40
    N = maps_leaf.size(1)
    w = F.softmax(F.logsigmoid(F.interpolate(maps_leaf, size=(24, 24), mode="bilinear", align_corners=False)).view(B, N, -1), dim=-1)
    tail = torch.bmm(w, f2.view(B, C, -1).permute(0, 2, 1)).reshape(B, N // 8, 8, -1).mean(dim=-2)
    assert torch.allclose(tail, out.detach(), atol=1e-6), "tail replay must equal the module output"
    tail.backward(t(g))
    save("mask_adapter_tail", feat=feat, maps=maps.detach().numpy(), out=out.detach().numpy(), gout=g,
         gfeat=f2.grad.numpy(), gmaps=maps_leaf.grad.numpy(), num_output_maps=np.int64(8))

    # ---- a4 mask_pooling (loss_func.py:35-56) ----
    emb = rng.standard_normal((3, 32, 16, 16)).astype(np.float32)
    mask = synth.make_masks(rng, 3, 1, 256, 256, soft=True, degenerate=False)
    mask[2] = mask[2] * 1.5 - 0.2                          # out of [0,1]: exercises the clamp
    e = t(emb, True)
    out = lf.mask_pooling(e, t(mask))
    g = rng.standard_normal(out.shape).astype(np.float32)
    out.backward(t(g))
    save("mask_pooling", emb=emb, mask=mask, out=out.detach().numpy(), gout=g, gemb=e.grad.numpy())

    # ---- a5/a6 fg / bg losses (loss_func.py:59-126), incl. empty and full masks ----
    for tag, B in {"b5": 5, "b1": 1}.items():
        emb = rng.standard_normal((B, 32, 16, 16)).astype(np.float32)
        comb = synth.unit_rows(rng, B, 1, 32)
        mask = synth.make_masks(rng, B, 1, 256, 256, degenerate=False)
        if B > 1:
            mask[1] = 0.0                                  # fg-invalid
            mask[3] = 1.0                                  # bg-invalid
        res = {}
        for name, fn in (("fg", lf.fg_feat_similarity_loss), ("bg", lf.bg_feat_similarity_loss)):
            e, c = t(emb, True), t(comb, True)
            v = fn(e, c, t(mask))
            v.backward()
            res[name] = v.detach().numpy()
            res["gemb_" + name] = e.grad.numpy()
            res["gcomb_" + name] = c.grad.numpy()
        save(f"fgbg_{tag}", emb=emb, comb=comb, mask=mask, **res)
    # all-invalid -> grad-less zeros
    emb = rng.standard_normal((2, 8, 8, 8)).astype(np.float32)
    comb = synth.unit_rows(rng, 2, 1, 8)
    z = np.zeros((2, 1, 64, 64), np.float32)
    fgv = lf.fg_feat_similarity_loss(t(emb, True), t(comb, True), t(z))
    bgv = lf.bg_feat_similarity_loss(t(emb, True), t(comb, True), t(z + 1))
    save("fgbg_allinvalid", emb=emb, comb=comb, fg=fgv.numpy(), bg=bgv.numpy(),
         fg_requires_grad=np.bool_(fgv.requires_grad), bg_requires_grad=np.bool_(bgv.requires_grad))

    # ---- a7 wbce_with_wiou_loss (loss_func.py:5-32) ----
    for tag, (B, Cc, H, W) in {"sq64": (2, 1, 64, 64), "rect": (2, 2, 48, 80), "tiny": (1, 1, 20, 20)}.items():
        pred = np.concatenate([synth.make_logits(rng, B, H, W) for _ in range(Cc)], 1)
        mask = synth.make_masks(rng, B, Cc, H, W, soft=True, degenerate=False)
        p = t(pred, True)
        v = lf.wbce_with_wiou_loss(p, t(mask))
        v.backward()
        save(f"wbce_wiou_{tag}", pred=pred, mask=mask, loss=v.detach().numpy(), gpred=p.grad.numpy())
    # weights w1/w2
    p = t(pred, True)
    v = lf.wbce_with_wiou_loss(p, t(mask), w1=0.3, w2=1.7)
    save("wbce_wiou_weights", pred=pred, mask=mask, loss=v.detach().numpy(), w1=np.float32(0.3), w2=np.float32(1.7))

    # ---- a8 trainer composition (trainer_v3_g.py:67-73) ----
    d = synth.make_triplets(7, B=4, M=1, C=32, h=16, w=16, H=256, W=256, hp=64, wp=64, degenerate=False)
    d["masks"][2] = 0.0
    p, e, c, qm = t(d["pred"], True), t(d["emb"], True), t(d["comb"], True), t(d["masks"])
    target = F.interpolate(qm, size=p.shape[2:], mode="bilinear", align_corners=False)
    seg = lf.wbce_with_wiou_loss(p, target)
    feat = 5 * lf.fg_feat_similarity_loss(e, c, qm) + 5 * lf.bg_feat_similarity_loss(e, c, qm)
    total = seg + feat
    total.backward()
    save("trainer_step", **d, seg=seg.detach().numpy(), total=total.detach().numpy(), target=target.numpy(),
         gpred=p.grad.numpy(), gemb=e.grad.numpy(), gcomb=c.grad.numpy())

    # ---- a10 validation post-process (trainer_v3_g.py:226-231; vailder.py:427-430,473) ----
    pred = synth.make_logits(rng, 2, 32, 32)
    up = F.interpolate(t(pred), size=(128, 128), mode="bilinear", align_corners=False)
    pr = torch.sigmoid(up)
    mn, mx = torch.amin(pr, dim=(1, 2, 3), keepdim=True), torch.amax(pr, dim=(1, 2, 3), keepdim=True)
    post = (pr - mn) / (mx - mn + 1e-8)
    pr0 = torch.sigmoid(t(pred))
    post0 = (pr0 - torch.amin(pr0, dim=(1, 2, 3), keepdim=True)) / (torch.amax(pr0, dim=(1, 2, 3), keepdim=True) - torch.amin(pr0, dim=(1, 2, 3), keepdim=True) + 1e-8)
    gt = synth.make_masks(rng, 2, 1, 128, 128, degenerate=False)
    extra = {}
    if trainer is not None:
        for k in ("dice", "mae", "iou", "mdice", "miou"):
            extra[k] = getattr(trainer, "compute_" + k)(post, t(gt)).numpy()
    # offline evaluator (vailder.py:427-430,459-473): normalise at 32x32, cv2.resize to the GT size, binarise
    import cv2
    gt_hw = (75, 100)
    resized = np.stack([cv2.resize(post0.numpy()[i, 0], (gt_hw[1], gt_hw[0]), interpolation=cv2.INTER_LINEAR) for i in range(2)])[:, None]
    save("vailder_hard", pred=pred, resized=resized.astype(np.float32), hard=((resized > 0.5).astype(np.uint8) * 255),
         gt_hw=np.asarray(gt_hw))
    save("val_post", pred=pred, post_up=post.numpy(), post_same=post0.numpy(), gt=gt,
         hard_up=((post.numpy() > 0.5).astype(np.uint8) * 255), **extra)


if __name__ == "__main__":
    main()
