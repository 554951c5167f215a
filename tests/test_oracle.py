"""Pins the CPU oracle (oracle/detr_oracle.py) to the committed golden fixtures produced by the
UNMODIFIED reference (oracle/gen_golden.py, oracle/gen_golden_reference_checks.py)."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import detr_oracle as O
from oracle.gen_golden import state_dict_digest, synth_images
from oracle.gen_golden_reference_checks import tensor_sha256
from tests.parity_utils import compare_queries, golden_meta, load_golden, seeded_sd


@pytest.fixture(scope="module")
def sd():
    return seeded_sd(0)


def test_seeded_weights_reproduce(sd):
    assert state_dict_digest(sd) == golden_meta()["weights_sha256"]


def test_anchor_validity():
    # SURVEY Appendix A.13: outermost ring of the 80x80 level is invalid, logit-space anchors there are 0
    a, v = O.generate_anchors([(20, 20), (40, 40), (80, 80)])
    assert a.shape == (1, 8400, 4) and int((~v).sum()) == 80 * 4 - 4
    assert float(a[0, ~v[0, :, 0]].abs().max()) == 0.0


def test_oracle_vs_golden_case_a(sd):
    g = load_golden("detr_l_obj365_b2_640")
    imgs = synth_images(1, [(640, 640)] * 2)
    taps = {}
    with torch.no_grad():
        x = O.detr_preprocess(imgs, (640, 640))
        s, b = O.detr_forward(sd, x, O.DetrOracleConfig(), taps)
    assert np.abs(x[:, :, 100:108, 200:208].numpy() - g["pre_image_patch"]).max() == 0
    for t in ("res2", "res3", "res4", "res5"):
        v = taps[t]
        sl = v[:, :: max(1, v.shape[1] // 8)][:, :8, :: max(1, v.shape[2] // 20), :: max(1, v.shape[3] // 20)].numpy()
        assert np.abs(sl - g["tap_" + t]).max() <= 1e-4 * g["tapstat_" + t][2]
    ds, db = compare_queries(g["scores"], g["boxes"], g["enc_topk_ind"], s.numpy(), b.numpy(), taps["topk_ind"].numpy())
    assert ds < 1e-4 and db < 1e-4, (ds, db)
    dets = O.detr_postprocess(s, b, [(640, 640)] * 2, threshold=0.5)
    for i, d in enumerate(dets):
        n = int(g["det_count"][i])
        assert len(d.scores) == n
        assert sorted(d.labels) == sorted(g["det_labels"][i, :n].tolist())
        assert sorted(map(tuple, d.boxes)) == sorted(map(tuple, g["det_boxes"][i, :n].tolist()))
        assert np.abs(np.array(d.scores) - g["det_scores"][i, :n]).max() < 1e-5


def test_oracle_vs_golden_ragged(sd):
    g = load_golden("detr_l_obj365_b3_ragged")
    sizes = [tuple(s) for s in g["image_sizes"].tolist()]
    imgs = synth_images(2, sizes)
    taps = {}
    with torch.no_grad():
        x = O.detr_preprocess(imgs, (640, 640))
        s, b = O.detr_forward(sd, x, O.DetrOracleConfig(), taps)
    assert np.abs(x[:, :, 100:108, 200:208].numpy() - g["pre_image_patch"]).max() < 1e-4
    ds, db = compare_queries(g["scores"], g["boxes"], g["enc_topk_ind"], s.numpy(), b.numpy(), taps["topk_ind"].numpy())
    assert ds < 1e-4 and db < 1e-4, (ds, db)
    dets = O.detr_postprocess(s, b, sizes, threshold=float(g["threshold"]))
    for i, d in enumerate(dets):
        n = int(g["det_count"][i])
        assert len(d.scores) == n
        assert sorted(d.labels) == sorted(g["det_labels"][i, :n].tolist())
        gb = np.array(sorted(map(tuple, g["det_boxes"][i, :n].tolist())))
        ob = np.array(sorted(map(tuple, d.boxes)))
        assert np.abs(gb - ob).max() <= 1  # round() of a coordinate that sits within 1e-4 px of .5


def test_oracle_vs_live_reference(sd):
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_checks.json")) as f:
        ref = json.load(f)["oracle_vs_reference"]
    imgs = synth_images(7, [(480, 640)])
    with torch.no_grad():
        xo = O.detr_preprocess(imgs, (640, 640))
        taps = {}
        s, b = O.detr_forward(sd, xo, O.DetrOracleConfig(), taps)
    # bit-identical pre-processed input
    assert list(xo.shape) == ref["input_shape"] and tensor_sha256(xo) == ref["input_sha256"]
    # same SET of queries, per-query values equal up to fp32 reassociation
    assert np.abs(np.array(ref["sorted_max_logits"], dtype=np.float32) - np.sort(s.numpy().max(-1), axis=1)).max() < 1e-4
