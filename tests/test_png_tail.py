"""The PNG / base64 tail of the segmentation post-process (SURVEY §8 a17 / f2; reference utils/vision.py:264-293, pinned in the reference by
tests/utils/test_vision.py:154-160): byte-identical strings to the unmodified reference function (goldens from oracle/gen_golden_png.py and
oracle/gen_golden_reference_checks.py), and the decoded image is the mask."""
import json
import os

import numpy as np
import pytest

from focoos_b200.processor import base64_to_binary_mask, binary_mask_to_base64
from oracle.gen_golden_reference_checks import png_masks

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "png_masks.json")
REFERENCE_CHECKS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_checks.json")


def _cases():
    with open(GOLDEN) as f:
        g = json.load(f)
    for k, v in g.items():
        if k != "_meta":
            n = int(np.prod(v["shape"]))
            yield k, np.unpackbits(np.array(v["bits"], dtype=np.uint8))[:n].reshape(v["shape"]).astype(bool), v["b64"]


@pytest.mark.parametrize("name,mask,b64", list(_cases()))
def test_base64_png_equals_the_reference_string(name, mask, b64):
    pytest.importorskip("cv2")
    assert binary_mask_to_base64(mask) == b64
    assert np.array_equal(base64_to_binary_mask(b64), mask), "decodes back to the mask"


def test_reference_fixture_mask():
    """tests/utils/conftest.py:11-26 of the reference: [[1,0],[0,1]] -> the OpenCV PNG string"""
    m = np.array([[1, 0], [0, 1]], dtype=bool)
    s = binary_mask_to_base64(m)
    assert isinstance(s, str) and np.array_equal(base64_to_binary_mask(s), m)


def test_against_the_live_reference_function():
    """seeded random masks of several shapes -> the strings the reference function returned for them"""
    pytest.importorskip("cv2")
    with open(REFERENCE_CHECKS) as f:
        ref = json.load(f)["png_b64"]
    masks = png_masks()
    assert len(masks) == len(ref)
    for shape, m in masks:
        assert binary_mask_to_base64(m) == ref["x".join(map(str, shape))]
