#!/usr/bin/env python
"""Generates the committed golden fixtures FROM THE REFERENCE ITSELF.

Needs a checkout of the reference project:   python tests/golden/make_golden.py <reference-dir> [files] [dets] [postproc]
(no group named = all three).  The tests read only what this writes; none of them needs the reference.

What it freezes (the reference has no tests / golden vectors of its own, SURVEY.md section 4):
  files     data/img.jpg, weights/*.caffemodel, weights/*.prototxt, weights/*.table.int8 -- the reference's DATA artefacts
            (its only image fixture, the trained weights, the network descriptions and the INT8 calibration cache the hot
            path consumes).  Byte-identical copies; no reference source code is copied.  reference_sha256.json records
            the SHA-256 of each file as it lies in the reference.
  dets      heads_<model>_448.npz -- the 9 head blobs for data/img.jpg letterboxed to 448x448, from cv2.dnn executing the
            reference's OWN prototxt (input-dim line rewritten) + caffemodel.
            dets_<model>_<HxW>.npz -- detections from the reference's OWN compiled post-process (oracle/_ref:
            RetinaFace::postProcess, thr 0.9 / NMS 0.4 as in main.cpp:43) on those heads, plus head checksums.
  postproc  postproc_reference.npz -- what oracle/_ref computes on the seeded synthetic heads of
            tests/test_oracle_postproc.py and tests/test_gpu_parity.py: base anchors, anchor planes, post-process and
            NMS outputs.  Arrays too large to store whole are kept as <key>__shape, <key>__sha256 (of the float32
            bytes) and their first rows (<key>__rows); <key>__heads_sha256 / <key>__cands_sha256 pin the synthetic input.
"""
import hashlib
import json
import os
import re
import shutil
import subprocess
import sys
import tempfile

import cv2
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import topology  # noqa: E402
from oracle.inputs import letterbox_bgr_u8  # noqa: E402
from oracle.mnet_numpy import preprocess_bgr_u8  # noqa: E402
from oracle.postproc import STRIDES, PostprocOracle, ReferencePostproc, build, synth_heads  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
MODELS = ("mnet-deconv-0517", "mnet25")
MODEL_FILES = ("mnet25.caffemodel", "mnet-deconv-0517.caffemodel", "mnet25.prototxt", "mnet-deconv-0517.prototxt",
               "mnet-deconv-0517.table.int8")
SAMPLE_ROWS = 4


def sha256(a) -> np.ndarray:
    data = a if isinstance(a, bytes) else np.ascontiguousarray(a, dtype=np.float32).tobytes()
    return np.frombuffer(hashlib.sha256(data).digest(), dtype=np.uint8)


def heads_sha256(heads) -> np.ndarray:
    return sha256(b"".join(np.ascontiguousarray(h, dtype=np.float32).tobytes() for h in heads))


def digest(out: dict, key: str, a: np.ndarray) -> None:
    """Shape, SHA-256 and the first rows of `a`, under `key`."""
    out[key + "__shape"] = np.array(a.shape, dtype=np.int64)
    out[key + "__sha256"] = sha256(a)
    out[key + "__rows"] = a[:SAMPLE_ROWS]


def ref_net(ref_dir: str, model: str, h: int, w: int):
    txt = open(f"{ref_dir}/model/{model}.prototxt").read()
    txt, n = re.subn(r"shape: \{ dim: 1 dim: 3 dim: \d+ dim: \d+ \}", f"shape: {{ dim: 1 dim: 3 dim: {h} dim: {w} }}", txt)
    assert n == 1
    d = tempfile.mkdtemp()
    p = os.path.join(d, "ref.prototxt")
    open(p, "w").write(txt)
    return cv2.dnn.readNetFromCaffe(p, f"{ref_dir}/model/{model}.caffemodel")


def make_files(ref_dir: str) -> None:
    os.makedirs(f"{OUT}/data", exist_ok=True)
    os.makedirs(f"{OUT}/weights", exist_ok=True)
    shutil.copyfile(f"{ref_dir}/data/img.jpg", f"{OUT}/data/img.jpg")
    digests = {"data/img.jpg": hashlib.sha256(open(f"{ref_dir}/data/img.jpg", "rb").read()).hexdigest()}
    for f in MODEL_FILES:
        shutil.copyfile(f"{ref_dir}/model/{f}", f"{OUT}/weights/{f}")
        digests[f"model/{f}"] = hashlib.sha256(open(f"{ref_dir}/model/{f}", "rb").read()).hexdigest()
    with open(f"{OUT}/reference_sha256.json", "w") as fh:
        json.dump(digests, fh, indent=1, sort_keys=True)
        fh.write("\n")


def make_dets(ref_dir: str) -> None:
    img = cv2.imread(f"{OUT}/data/img.jpg")
    assert img.shape == (886, 1280, 3)
    for model in MODELS:
        for (h, w) in ((448, 448), (896, 1280)):
            inp = letterbox_bgr_u8(img, h, w)
            net = ref_net(ref_dir, model, h, w)
            net.setInput(preprocess_bgr_u8(inp))
            heads = [np.ascontiguousarray(b[0]) for b in net.forward(topology.OUTPUT_BLOBS)]
            ref = ReferencePostproc(h, w)
            out = {"input_sha256": np.frombuffer(hashlib.sha256(inp.tobytes()).digest(), dtype=np.uint8)}
            for thr in (0.9, 0.5, 0.02):
                out[f"faces_thr{thr}"] = ref.postprocess(heads, thr)
            ref.close()
            out["head_sums"] = np.array([b.astype(np.float64).sum() for b in heads])
            out["head_abs_sums"] = np.array([np.abs(b.astype(np.float64)).sum() for b in heads])
            np.savez_compressed(f"{OUT}/dets_{model}_{h}x{w}.npz", **out)
            if (h, w) == (448, 448):
                np.savez_compressed(f"{OUT}/heads_{model}_448.npz", **{n: b for n, b in zip(topology.OUTPUT_BLOBS, heads)})
            print(model, h, w, {k: v.shape for k, v in out.items() if k.startswith("faces")})
            print("  top face thr0.9:", out["faces_thr0.9"][0][:5])


def make_postproc() -> None:
    """The cases of test_oracle_postproc.py (anchors, post-process, NMS) and of test_gpu_parity.py
    (test_postprocess_matches_reference_compiled_code), run through oracle/_ref."""
    oracle = PostprocOracle()
    out = {}
    for hw in ((448, 448), (896, 1280), (320, 320)):
        ref = ReferencePostproc(*hw)
        for s in STRIDES:
            out[f"base_{hw[0]}x{hw[1]}_s{s}"] = ref.base_anchors(s)
            digest(out, f"plane_{hw[0]}x{hw[1]}_s{s}", ref.anchor_plane(s))
        ref.close()
    for hw in ((448, 448), (896, 1280)):
        ref = ReferencePostproc(*hw)
        for ncand in (0, 1, 7, 64, 1024, 4000):
            key = f"{hw[0]}x{hw[1]}_n{ncand}"
            heads = synth_heads(hw[0], hw[1], ncand, seed=ncand + 11)
            out[f"pp_{key}__heads_sha256"] = heads_sha256(heads)
            for thr in (0.9, 0.5):
                digest(out, f"pp_{key}_thr{thr}", ref.postprocess(heads, thr))
            cands = oracle.postprocess(heads, hw[0], hw[1], 0.9, 0.4)["cand"]
            out[f"nms_{key}__cands_sha256"] = sha256(cands)
            for nt in (0.0, 0.3, 0.7, 1.0):
                digest(out, f"nms_{key}_nt{nt}", ref.nms(cands, nt))
        ref.close()
    ref = ReferencePostproc(448, 448)
    for ncand in (5, 300, 2000):
        heads = synth_heads(448, 448, ncand, seed=7 + ncand)
        out[f"gpu_448x448_n{ncand}__heads_sha256"] = heads_sha256(heads)
        out[f"gpu_448x448_n{ncand}"] = ref.postprocess(heads, 0.9)
    ref.close()
    np.savez_compressed(f"{OUT}/postproc_reference.npz", **out)
    print("postproc_reference.npz:", len(out), "arrays")


def main(argv) -> None:
    if len(argv) < 2 or not os.path.isfile(os.path.join(argv[1], "retinaface", "RetinaFace.cpp")):
        raise SystemExit(__doc__)
    ref_dir = os.path.abspath(argv[1])
    groups = argv[2:] or ["files", "dets", "postproc"]
    build(force=True)
    subprocess.check_call([os.path.join(ROOT, "oracle", "build_ref.sh")], env=dict(os.environ, RF_REFERENCE_ROOT=ref_dir))
    if "files" in groups:
        make_files(ref_dir)
    if "dets" in groups:
        make_dets(ref_dir)
    if "postproc" in groups:
        make_postproc()


if __name__ == "__main__":
    main(sys.argv)
