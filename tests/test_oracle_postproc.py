"""CPU: pins the plain-C post-process restatement (oracle/postproc.c) against the reference's own
compiled code (oracle/_ref: the reference's RetinaFace.cpp built unmodified behind a fake engine), as
recorded on the same seeded inputs in tests/golden/postproc_reference.npz (tests/golden/make_golden.py),
and against the committed golden detections."""
import hashlib
import os

import numpy as np
import pytest

from conftest import GOLDEN
from oracle.postproc import STRIDES, PostprocOracle, synth_heads

REF = np.load(os.path.join(GOLDEN, "postproc_reference.npz"))


def _sha256(arrays) -> bytes:
    return hashlib.sha256(b"".join(np.ascontiguousarray(a, dtype=np.float32).tobytes() for a in arrays)).digest()


def assert_reference_output(mine: np.ndarray, key: str) -> None:
    """`mine` is, byte for byte, the array oracle/_ref computed for `key`: same shape, same first rows, same SHA-256."""
    shape, rows = tuple(REF[key + "__shape"]), REF[key + "__rows"]
    assert mine.shape == shape, (key, mine.shape, shape)
    assert np.array_equal(mine[:len(rows)], rows), (key, mine[:len(rows)], rows)
    assert _sha256([mine]) == REF[key + "__sha256"].tobytes(), key


@pytest.fixture(scope="module")
def oracle():
    return PostprocOracle()


def test_base_anchors_values(oracle):
    # SURVEY.md 8a2: values printed by the reference's own generate_anchors_fpn
    exp = {32: [[-248, -248, 263, 263], [-120, -120, 135, 135]], 16: [[-56, -56, 71, 71], [-24, -24, 39, 39]],
           8: [[-8, -8, 23, 23], [0, 0, 15, 15]]}
    for s in STRIDES:
        assert oracle.base_anchors(s).tolist() == exp[s]


@pytest.mark.parametrize("hw", [(448, 448), (896, 1280), (320, 320)])
def test_anchors_match_reference(oracle, hw):
    for s in STRIDES:
        base = oracle.base_anchors(s)
        assert np.array_equal(base, REF[f"base_{hw[0]}x{hw[1]}_s{s}"])
        # anchors_plane: index k*H*W + ih*W + iw
        h, w = hw[0] // s, hw[1] // s
        ys, xs = np.mgrid[0:h, 0:w]
        mine = [np.stack([base[k, 0] + xs * s, base[k, 1] + ys * s, base[k, 2] + xs * s, base[k, 3] + ys * s], -1).reshape(-1, 4)
                for k in range(2)]
        assert_reference_output(np.concatenate(mine).astype(np.float32), f"plane_{hw[0]}x{hw[1]}_s{s}")


@pytest.mark.parametrize("hw", [(448, 448), (896, 1280)])
@pytest.mark.parametrize("ncand", [0, 1, 7, 64, 1024, 4000])
def test_postprocess_bit_exact_vs_reference(oracle, hw, ncand):
    key = f"{hw[0]}x{hw[1]}_n{ncand}"
    heads = synth_heads(hw[0], hw[1], ncand, seed=ncand + 11)
    assert _sha256(heads) == REF[f"pp_{key}__heads_sha256"].tobytes(), "synthetic heads differ from those the reference ran on"
    for thr in (0.9, 0.5):
        mine = oracle.postprocess(heads, hw[0], hw[1], thr, 0.4)   # reference postProcess hard-codes NMS 0.4
        assert_reference_output(mine["faces"], f"pp_{key}_thr{thr}")
        if thr == 0.9:
            assert len(mine["cand"]) == ncand
    # RetinaFace::nms with other thresholds, on the same candidates
    cands = oracle.postprocess(heads, hw[0], hw[1], 0.9, 0.4)["cand"]
    assert _sha256([cands]) == REF[f"nms_{key}__cands_sha256"].tobytes()
    for nt in (0.0, 0.3, 0.7, 1.0):
        a, _ = oracle.nms(cands, nt)
        assert_reference_output(a, f"nms_{key}_nt{nt}")


def test_edge_cases(oracle):
    h = w = 64
    heads = synth_heads(h, w, 0)
    r = oracle.postprocess(heads, h, w, 0.9, 0.4)
    assert len(r["faces"]) == 0 and len(r["cand"]) == 0
    # every anchor is a candidate
    heads = synth_heads(h, w, 10_000)
    r = oracle.postprocess(heads, h, w, 0.9, 0.4)
    assert len(r["cand"]) == 2 * (2 * 2 + 4 * 4 + 8 * 8)
    # strict threshold: conf == thr is dropped (RetinaFace.cpp:693 `conf <= threshold`)
    heads = synth_heads(h, w, 0)
    heads[0][2, 0, 0] = np.float32(0.9)
    assert len(oracle.postprocess(heads, h, w, np.float32(0.9), 0.4)["cand"]) == 0
    heads[0][2, 0, 0] = np.nextafter(np.float32(0.9), np.float32(1))
    assert len(oracle.postprocess(heads, h, w, np.float32(0.9), 0.4)["cand"]) == 1
    # ties: equal scores keep emission order
    heads = synth_heads(h, w, 0)
    heads[6][2, 0, 0] = 0.95   # stride 8, anchor 0, j 0
    heads[0][2, 1, 1] = 0.95   # stride 32, anchor 0, j 3 -> emitted first
    r = oracle.postprocess(heads, h, w, 0.9, 1.0)
    assert r["idx"].tolist() == sorted(r["idx"].tolist()) and len(r["idx"]) == 2


@pytest.mark.parametrize("model", ["mnet-deconv-0517", "mnet25"])
def test_golden_detections_from_golden_heads(oracle, model):
    """heads frozen from cv2.dnn(reference prototxt+caffemodel) -> oracle == detections frozen from oracle/_ref."""
    heads_npz = np.load(os.path.join(GOLDEN, f"heads_{model}_448.npz"))
    from oracle.topology import OUTPUT_BLOBS
    heads = [heads_npz[n] for n in OUTPUT_BLOBS]
    dets = np.load(os.path.join(GOLDEN, f"dets_{model}_448x448.npz"))
    for thr in (0.9, 0.5, 0.02):
        r = oracle.postprocess(heads, 448, 448, thr, 0.4)
        assert np.array_equal(r["faces"], dets[f"faces_thr{thr}"])
    assert dets["faces_thr0.9"].shape == (5, 15)   # SURVEY.md 8c: 27 candidates -> 5 faces
