"""CPU: pins the numpy forward restatement and the generated prototxt against cv2.dnn executing the
reference's own model files, and against the committed golden head blobs."""
import os
import re
import tempfile

import numpy as np
import pytest

from conftest import GOLDEN, WEIGHTS, caffemodel
from oracle import topology
from oracle.inputs import letterbox_bgr_u8
from oracle.mnet_numpy import MnetOracle, preprocess_bgr_u8


def test_macs_match_survey():
    m = topology.conv_macs(448, 448)
    assert m == {"full3x3": 297593856, "pw": 165781504, "dw": 17385984, "deconv": 1003520, "total": 481764864}
    assert topology.conv_macs(896, 1280)["total"] == 2752942080


@pytest.mark.parametrize("model", ["mnet-deconv-0517", "mnet25"])
def test_numpy_forward_vs_golden_heads(model, golden_image):
    inp = letterbox_bgr_u8(golden_image, 448, 448)
    out = MnetOracle(caffemodel(model)).forward(preprocess_bgr_u8(inp))
    gold = np.load(os.path.join(GOLDEN, f"heads_{model}_448.npz"))
    for name in topology.OUTPUT_BLOBS:
        assert out[name][0].shape == gold[name].shape
        assert np.abs(out[name][0] - gold[name]).max() < 2e-5, name


def test_generated_prototxt_runs_in_cv2_and_matches_numpy():
    import cv2
    rng = np.random.default_rng(3)
    img = rng.integers(0, 256, (64, 96, 3), dtype=np.uint8)
    x = preprocess_bgr_u8(img)
    with tempfile.TemporaryDirectory() as d:
        p = os.path.join(d, "gen.prototxt")
        open(p, "w").write(topology.to_prototxt(64, 96))
        net = cv2.dnn.readNetFromCaffe(p, caffemodel("mnet25"))
        net.setInput(x)
        outs = net.forward(topology.OUTPUT_BLOBS)
    mine = MnetOracle(caffemodel("mnet25")).forward(x)
    for name, o in zip(topology.OUTPUT_BLOBS, outs):
        assert np.abs(o - mine[name]).max() < 2e-5, name


def test_generated_prototxt_equals_reference_prototxt():
    """cv2.dnn runs the reference's own prototxt (committed byte-identical under tests/golden/weights) and the generated one
    on the same caffemodel: identical head blobs."""
    import cv2
    rng = np.random.default_rng(4)
    x = preprocess_bgr_u8(rng.integers(0, 256, (96, 64, 3), dtype=np.uint8))
    for model in ("mnet-deconv-0517", "mnet25"):
        txt = open(os.path.join(WEIGHTS, f"{model}.prototxt")).read()
        txt, n = re.subn(r"shape: \{ dim: 1 dim: 3 dim: \d+ dim: \d+ \}", "shape: { dim: 1 dim: 3 dim: 96 dim: 64 }", txt)
        assert n == 1
        with tempfile.TemporaryDirectory() as d:
            pr, pg = os.path.join(d, "r.prototxt"), os.path.join(d, "g.prototxt")
            open(pr, "w").write(txt)
            open(pg, "w").write(topology.to_prototxt(96, 64))
            a = cv2.dnn.readNetFromCaffe(pr, caffemodel(model))
            b = cv2.dnn.readNetFromCaffe(pg, caffemodel(model))
            a.setInput(x)
            b.setInput(x)
            for u, v in zip(a.forward(topology.OUTPUT_BLOBS), b.forward(topology.OUTPUT_BLOBS)):
                assert np.array_equal(u, v)


def test_committed_fixtures_are_the_reference_files():
    """Every committed copy of a reference data file has the SHA-256 that file has in the reference
    (tests/golden/reference_sha256.json, written by tests/golden/make_golden.py)."""
    import hashlib
    import json
    digests = json.load(open(os.path.join(GOLDEN, "reference_sha256.json")))
    files = {"data/img.jpg": os.path.join(GOLDEN, "data", "img.jpg")}
    for f in ("mnet25.caffemodel", "mnet-deconv-0517.caffemodel", "mnet25.prototxt", "mnet-deconv-0517.prototxt",
              "mnet-deconv-0517.table.int8"):
        files[f"model/{f}"] = os.path.join(WEIGHTS, f)
    assert sorted(digests) == sorted(files)
    for name, path in files.items():
        assert hashlib.sha256(open(path, "rb").read()).hexdigest() == digests[name], name


def test_int8_oracle_within_calibration_tolerance_of_fp32(golden_image):
    """The integer scheme (oracle/mnet_int8.py: table scales + per-channel weight scales) against the FP32
    oracle on the golden photo: per-tensor RMS error of a few LSB, same 5 faces, boxes within 2 px."""
    from conftest import WEIGHTS
    from oracle.mnet_int8 import Int8Oracle, read_table
    from oracle.postproc import PostprocOracle
    table = os.path.join(WEIGHTS, "mnet-deconv-0517.table.int8")
    t = read_table(table)
    assert len(t) == 210 and abs(t["data"] - 2.00836) < 1e-4          # SURVEY.md Appendix C
    inp = letterbox_bgr_u8(golden_image, 448, 448)
    o8 = Int8Oracle(caffemodel("mnet-deconv-0517"), table)
    blobs, tens = o8.forward(inp[None], want_tensors=True)
    ref = MnetOracle(caffemodel("mnet-deconv-0517")).forward(preprocess_bgr_u8(inp), want=list(tens.keys()))
    for name, (q, s) in tens.items():
        rms = np.sqrt(np.mean((q.astype(np.float32) * np.float32(s) - ref[name]) ** 2)) / s
        assert rms < 4.0, (name, rms)
    po = PostprocOracle()
    r8 = po.postprocess([b[0] for b in blobs], 448, 448, 0.9, 0.4)["faces"]
    gold = np.load(os.path.join(GOLDEN, "dets_mnet-deconv-0517_448x448.npz"))["faces_thr0.9"]
    assert len(r8) == len(gold) == 5
    for g in gold:
        c = r8[np.argmin(np.abs(r8[:, 1:3] - g[1:3]).sum(1))]
        assert np.abs(c[1:5] - g[1:5]).max() < 2.0 and abs(c[0] - g[0]) < 0.03
