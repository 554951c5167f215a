"""Golden values for the tests that compare against the UNMODIFIED reference directly (tests/test_eval_postprocess.py,
tests/test_png_tail.py, tests/test_oracle.py): the reference's outputs on exactly the inputs those tests build
-> tests/golden/reference_checks.json.  Needs the reference tree (oracle/ref_import.py) and OpenCV:

    python -m oracle.gen_golden_reference_checks
"""
from __future__ import annotations

import hashlib
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import ref_import  # noqa: E402
from oracle.gen_golden import synth_images  # noqa: E402

PATH = os.path.join(ROOT, "tests", "golden", "reference_checks.json")
PNG_SEED, PNG_SHAPES = 11, ((1, 1), (5, 7), (120, 33), (64, 64))


def png_masks():
    rng = np.random.default_rng(PNG_SEED)
    return [(shape, rng.random(shape) > 0.6) for shape in PNG_SHAPES]


def tensor_sha256(t: torch.Tensor) -> str:
    return hashlib.sha256(t.detach().cpu().contiguous().numpy().tobytes()).hexdigest()


def eval_postprocess_case():
    from focoos.models.fai_detr.config import DETRConfig as RC
    from focoos.models.fai_detr.ports import DETRModelOutput as RO
    from focoos.models.fai_detr.processor import DETRProcessor as RP
    from focoos.nn.backbone.resnet import ResnetConfig as RB
    from tests.test_eval_postprocess import _case

    class Entry:  # DatasetEntry duck type
        def __init__(self, d):
            self.height, self.width = d["height"], d["width"]

    logits, boxes, entries = _case()
    ref = RP(RC(backbone_config=RB(), num_classes=20), image_size=640).eval_postprocess(RO(boxes=boxes, logits=logits, loss=None), [Entry(e) for e in entries], top_k=100)
    return [{"scores": r["instances"].scores.tolist(), "classes": r["instances"].classes.tolist(), "boxes": r["instances"].boxes.tensor.tolist(),
             "image_size": list(r["instances"].image_size)} for r in ref]


def oracle_case():
    from tests.parity_utils import seeded_sd

    fm = ref_import.get_reference_model("fai-detr-l-obj365")
    fm.model.load_state_dict(seeded_sd(0), strict=True)
    imgs = synth_images(7, [(480, 640)])
    with torch.no_grad():
        x, _ = fm.processor.preprocess(imgs, device=torch.device("cpu"), dtype=torch.float32)
        out = fm.model(x)
    return {"input_shape": list(x.shape), "input_sha256": tensor_sha256(x),
            "sorted_max_logits": np.sort(out.logits.numpy().max(-1), axis=1).tolist()}


def main():
    ref_import.install()
    import cv2  # the real OpenCV (ref_import stubs it only when it is absent)
    assert not type(cv2).__name__.startswith("_Dummy"), "OpenCV is needed to generate the goldens"
    from focoos.utils.vision import binary_mask_to_base64

    g = {"_meta": {"cv2": cv2.__version__, "torch": torch.__version__, "source": "unmodified reference (focoos), CPU, fp32"},
         "png_b64": {"x".join(map(str, s)): binary_mask_to_base64(m) for s, m in png_masks()},
         "eval_postprocess": eval_postprocess_case(),
         "oracle_vs_reference": oracle_case()}
    with open(PATH, "w") as f:
        json.dump(g, f, indent=1)
    print("wrote", PATH, os.path.getsize(PATH), "bytes")


if __name__ == "__main__":
    main()
