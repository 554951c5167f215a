"""DETRProcessor.eval_postprocess (SURVEY §8 f3): host logic on the CPU reference backend against what the UNMODIFIED reference's
`DETRProcessor.eval_postprocess` returns for the same case (tests/golden/reference_checks.json, oracle/gen_golden_reference_checks.py),
and the CUDA kernel against the CPU reference operator (-m gpu)."""
import json
import os

import numpy as np
import pytest
import torch

from focoos_b200 import DETRConfig, DETRProcessor, ops
from focoos_b200.ports import DETRModelOutput
from oracle.ops_ref import RefBackend

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_checks.json")


def _case(B=3, Q=300, C=20, seed=0):
    g = torch.Generator().manual_seed(seed)
    logits = torch.rand((B, Q, C), generator=g)
    c = torch.rand((B, Q, 2), generator=g)
    wh = torch.rand((B, Q, 2), generator=g) * 0.6
    boxes = torch.cat([c - wh / 2, c + wh / 2], -1)           # some reach outside [0,1] -> clipped
    boxes[:, ::17, 2] = boxes[:, ::17, 0]                      # some are empty after scaling -> dropped
    boxes[:, 5::23] = 1.5                                      # fully outside -> clipped to zero area -> dropped
    entries = [{"height": 480, "width": 640}, {"height": 333, "width": 500}, {"height": None, "width": None}][:B]
    return logits, boxes, entries


@pytest.fixture()
def ref_backend():
    ops._backend = RefBackend()
    yield
    ops._backend = None


def _check_against(res, ref_scores, ref_labels, ref_boxes):
    assert len(res) == len(ref_scores)
    for r, s, l, b in zip(res, ref_scores, ref_labels, ref_boxes):
        inst = r["instances"]
        assert len(inst) == len(s)
        assert np.array_equal(inst.classes.cpu().numpy(), l)
        assert np.allclose(inst.scores.cpu().numpy(), s, atol=0)
        assert np.abs(inst.boxes.tensor.cpu().numpy() - b).max() <= 1e-4 if len(s) else True


def test_eval_postprocess_matches_the_reference(ref_backend):
    with open(GOLDEN) as f:
        ref = json.load(f)["eval_postprocess"]
    logits, boxes, entries = _case()
    ours = DETRProcessor(DETRConfig(num_classes=20), image_size=640).eval_postprocess(DETRModelOutput(boxes=boxes, logits=logits), entries, top_k=100)
    _check_against(ours, [np.array(r["scores"], dtype=np.float32) for r in ref], [np.array(r["classes"], dtype=np.int64) for r in ref],
                   [np.array(r["boxes"], dtype=np.float32).reshape(-1, 4) for r in ref])
    assert [o["instances"].image_size for o in ours] == [tuple(r["image_size"]) for r in ref]


@pytest.mark.gpu
def test_eval_postprocess_kernel_matches_the_cpu_reference_operator():
    logits, boxes, entries = _case(seed=3)
    proc = DETRProcessor(DETRConfig(num_classes=20), image_size=640)
    ops._backend = RefBackend()
    try:
        ref = proc.eval_postprocess(DETRModelOutput(boxes=boxes, logits=logits), entries, top_k=300)
    finally:
        ops._backend = None
    got = proc.eval_postprocess(DETRModelOutput(boxes=boxes.cuda(), logits=logits.cuda()), entries, top_k=300)
    _check_against(got, [r["instances"].scores.numpy() for r in ref], [r["instances"].classes.numpy() for r in ref], [r["instances"].boxes.tensor.numpy() for r in ref])
    assert all(g["instances"].scores.is_cuda for g in got)
