"""Recipe for ``oracle/_ref/``: the reference's OWN hot-path modules, placed where the tests and the bench can import them.

TEST / BASELINE INFRASTRUCTURE ONLY (see oracle/np_oracle.py header).  The reference is Python: there is nothing to
compile, so "building" the real reference for this path means copying the two importable modules that hold it --

    utils/loss_func.py                    (wbce_with_wiou_loss, mask_pooling, fg/bg_feat_similarity_loss)
    lib/support_model/mask_adapter.py     (MaskedPooling, MaskAdapterPooling and its ConvNeXt head)
    lib/support_model/cir_feature_fuse.py (CirFuseModule: the composed-query head's fusion)

-- byte for byte into ``oracle/_ref/`` (git-ignored: reference sources never enter this repository's history; a copy of
the working tree carries the directory along like a built .so).  ``MANIFEST.json`` records the
sha256 of every file so a consumer can tell the copy is unmodified.  Run by ``__graft_entry__.build()`` whenever
``COR_REFERENCE`` names a checkout of the reference (wangtong627/COR); without one nothing is copied and the tests that
run the reference's own modules skip.

    python oracle/build_ref.py [--reference DIR]
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import shutil

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_ref")
FILES = ("utils/loss_func.py", "lib/support_model/mask_adapter.py", "lib/support_model/cir_feature_fuse.py")
REFERENCE = os.environ.get("COR_REFERENCE", "")


def build(reference: str = REFERENCE) -> str | None:
    if not reference or not os.path.isdir(reference):
        return None
    manifest = {}
    for rel in FILES:
        src, dst = os.path.join(reference, rel), os.path.join(OUT, rel)
        os.makedirs(os.path.dirname(dst), exist_ok=True)
        shutil.copyfile(src, dst)
        manifest[rel] = hashlib.sha256(open(dst, "rb").read()).hexdigest()
    # package markers so that `import utils.loss_func` / `import lib.support_model.mask_adapter` resolve under _ref/
    for d in ("utils", "lib", "lib/support_model"):
        init = os.path.join(OUT, d, "__init__.py")
        if not os.path.exists(init):
            open(init, "w").close()
    with open(os.path.join(OUT, "MANIFEST.json"), "w") as f:
        json.dump({"source": reference, "files": manifest}, f, indent=1)
    return OUT


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", default=REFERENCE)
    print(build(ap.parse_args().reference))
