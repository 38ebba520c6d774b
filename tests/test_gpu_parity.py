"""GPU (-m gpu): parity of the CUDA path, called through the C ABI, against the oracle and the
committed golden fixtures.  Tolerances are written next to each assertion.

Nothing here reads /root/reference (absent on the GPU box): golden fixtures + the oracle only.
"""
import os

import numpy as np
import pytest

from conftest import GOLDEN, caffemodel
from oracle import topology
from oracle.inputs import letterbox_bgr_u8, s_noise_batch, s_real_batch
from oracle.mnet_numpy import MnetOracle, preprocess_bgr_u8
from oracle.postproc import PostprocOracle, synth_heads

pytestmark = pytest.mark.gpu

# FP32 mode: same math as the oracle up to summation order -> observed ~1e-5; gate at 2e-4 abs.
TOL_FP32 = 2e-4


def _engine(model, h, w, prec, **kw):
    from retinaface_b200 import Engine
    return Engine(caffemodel(model), h, w, precision=prec, **kw)


def _compare_dets(mine, mine_idx, ref, label="", max_faces=None):
    """Selection (anchor emission indices, order) bit-exact; scores + landmarks bit-exact; box corners
    within 4e-6 relative (the exp() rounding noted in postproc.cu)."""
    ridx, rfaces = ref["idx"], ref["faces"]
    if max_faces is not None and len(ridx) > max_faces:   # output capacity clamp keeps the top-scoring prefix
        ridx, rfaces = ridx[:max_faces], rfaces[:max_faces]
    assert mine_idx.tolist() == ridx.tolist(), label
    a, b = mine, rfaces
    assert a.shape == b.shape, label
    if len(a) == 0:
        return
    assert np.array_equal(a[:, 0], b[:, 0]), label            # scores
    assert np.array_equal(a[:, 5:], b[:, 5:]), label          # landmarks
    assert np.allclose(a[:, 1:5], b[:, 1:5], rtol=4e-6, atol=1e-4), label


@pytest.fixture(scope="module")
def post_oracle():
    return PostprocOracle()


@pytest.mark.parametrize("hw", [(448, 448), (896, 1280)])
def test_postprocess_kernels_vs_oracle(post_oracle, hw):
    """rf_postprocess (decode + threshold + sort + NMS kernels) on synthetic S-nms head tensors."""
    from retinaface_b200 import RF_PREC_FP32
    h, w = hw
    eng = _engine("mnet25", h, w, RF_PREC_FP32, max_batch=4, max_faces=8192)
    try:
        for ncand in (0, 1, 37, 64, 1024, 4000, 8192):
            batch = [synth_heads(h, w, ncand, seed=100 + ncand + i) for i in range(3)]
            heads = [np.stack([b[k] for b in batch]) for k in range(9)]
            for thr, nms in ((0.9, 0.4), (0.5, 0.4), (0.9, 0.0), (0.9, 1.0)):
                if ncand > 1024 and (thr, nms) != (0.9, 0.4):
                    continue
                faces, idx, ncands = eng.postprocess(heads, thr, nms)
                for i in range(3):
                    ref = post_oracle.postprocess(batch[i], h, w, thr, nms)
                    assert ncands[i] == len(ref["cand"]), (ncand, thr, nms, i)
                    _compare_dets(faces[i], idx[i], ref, f"ncand={ncand} thr={thr} nms={nms} img={i}", max_faces=8192)
    finally:
        eng.close()


def test_postprocess_matches_reference_compiled_code():
    """Same, against what oracle/_ref (the reference's own RetinaFace::postProcess) computed on the same synthetic heads
    (tests/golden/postproc_reference.npz, written by tests/golden/make_golden.py)."""
    import hashlib
    from retinaface_b200 import RF_PREC_FP32
    h = w = 448
    gold = np.load(os.path.join(GOLDEN, "postproc_reference.npz"))
    eng = _engine("mnet25", h, w, RF_PREC_FP32, max_batch=1, max_faces=4096)
    try:
        for ncand in (5, 300, 2000):
            heads = synth_heads(h, w, ncand, seed=7 + ncand)
            digest = hashlib.sha256(b"".join(np.ascontiguousarray(x, dtype=np.float32).tobytes() for x in heads)).digest()
            assert digest == gold[f"gpu_448x448_n{ncand}__heads_sha256"].tobytes(), "synthetic heads differ from those the reference ran on"
            faces, idx, _ = eng.postprocess([x[None] for x in heads], 0.9, 0.4)
            theirs = gold[f"gpu_448x448_n{ncand}"]
            assert faces[0].shape == theirs.shape
            assert np.array_equal(faces[0][:, 0], theirs[:, 0])
            assert np.array_equal(faces[0][:, 5:], theirs[:, 5:])
            assert np.allclose(faces[0][:, 1:5], theirs[:, 1:5], rtol=4e-6, atol=1e-4)
    finally:
        eng.close()


def test_postprocess_edge_cases(post_oracle):
    from retinaface_b200 import RF_PREC_FP32
    h = w = 64
    eng = _engine("mnet25", h, w, RF_PREC_FP32, max_batch=2, max_faces=512)
    try:
        # every anchor a candidate (168 of them), strict threshold, ties broken by emission order
        heads = synth_heads(h, w, 10_000)
        faces, idx, nc = eng.postprocess([x[None] for x in heads], 0.9, 0.4)
        ref = post_oracle.postprocess(heads, h, w, 0.9, 0.4)
        assert nc[0] == 168
        _compare_dets(faces[0], idx[0], ref)
        z = synth_heads(h, w, 0)
        z[0][2, 0, 0] = np.float32(0.9)
        assert eng.postprocess([x[None] for x in z], 0.9, 0.4)[2][0] == 0          # conf == thr dropped
        z[6][2, 0, 0] = 0.95
        z[0][2, 1, 1] = 0.95
        faces, idx, nc = eng.postprocess([x[None] for x in z], 0.9, 1.0)
        assert nc[0] == 2 and idx[0].tolist() == sorted(idx[0].tolist())
        # max_faces clamp keeps the top-scoring ones
        small = _engine("mnet25", h, w, RF_PREC_FP32, max_batch=1, max_faces=4)
        f2, i2, _ = small.postprocess([x[None] for x in heads], 0.9, 0.4)
        assert len(f2[0]) == 4 and np.array_equal(f2[0], faces_all(eng, heads)[:4])
        small.close()
    finally:
        eng.close()


def faces_all(eng, heads):
    return eng.postprocess([x[None] for x in heads], 0.9, 0.4)[0][0]


@pytest.mark.parametrize("model", ["mnet-deconv-0517", "mnet25"])
def test_fp32_forward_heads_vs_golden_and_oracle(model, golden_image):
    """FP32 CUDA forward vs (a) golden head blobs frozen from cv2.dnn on the reference's own model
    files, (b) the numpy oracle on seeded noise; plus every intermediate activation."""
    from retinaface_b200 import RF_PREC_FP32
    eng = _engine(model, 448, 448, RF_PREC_FP32, max_batch=2)
    try:
        eng.debug_keep_all()
        inp = letterbox_bgr_u8(golden_image, 448, 448)
        noise = s_noise_batch(1, 448, 448, seed=0)[0]
        batch = np.stack([inp, noise])
        heads = eng.forward_heads(batch)
        gold = np.load(os.path.join(GOLDEN, f"heads_{model}_448.npz"))
        for k, name in enumerate(topology.OUTPUT_BLOBS):
            err = np.abs(heads[k][0] - gold[name]).max()
            assert err < TOL_FP32, (name, err)
        orc = MnetOracle(caffemodel(model))
        inter = ["mobilenet0_relu0_fwd", "mobilenet0_relu1_fwd", "mobilenet0_relu2_fwd", "mobilenet0_relu10_fwd",
                 "mobilenet0_relu22_fwd", "mobilenet0_relu26_fwd", "rf_c3_lateral_relu", "_plus0", "rf_c2_aggr_relu",
                 "_plus1", "rf_c1_aggr_relu", "rf_c3_det_concat_relu", "rf_c2_det_concat_relu", "rf_c1_det_concat_relu"]
        x = np.concatenate([preprocess_bgr_u8(inp), preprocess_bgr_u8(noise)])
        ref = orc.forward(x, want=list(topology.OUTPUT_BLOBS) + inter)
        for name in inter:
            got = eng.debug_tensor(name, 2)
            scale = max(1.0, float(np.abs(ref[name]).max()))
            err = np.abs(got - ref[name]).max() / scale
            assert err < TOL_FP32, (name, err)
        for k, name in enumerate(topology.OUTPUT_BLOBS):
            err = np.abs(heads[k] - ref[name]).max()
            assert err < TOL_FP32, (name, err)
    finally:
        eng.close()


@pytest.mark.parametrize("hw", [(448, 448), (896, 1280)])
def test_fp32_detect_matches_golden_detections(hw, golden_image, post_oracle):
    """End to end through rf_detect_batch (host images in, faces out) against the detections frozen
    from the reference's own post-process on cv2.dnn heads: same faces, same order; coordinates within
    2e-3 px (FP32 conv summation order), scores within 1e-5."""
    from retinaface_b200 import RF_PREC_FP32
    h, w = hw
    for model in ("mnet-deconv-0517", "mnet25"):
        eng = _engine(model, h, w, RF_PREC_FP32, max_batch=2, max_image=(1024, 1536))
        try:
            dets = np.load(os.path.join(GOLDEN, f"dets_{model}_{h}x{w}.npz"))
            inp = letterbox_bgr_u8(golden_image, h, w)
            for thr in (0.9, 0.5):
                faces, idx = eng.detect_batch([inp, inp], thr, 0.4, want_index=True)
                g = dets[f"faces_thr{thr}"]
                for f in faces:
                    assert f.shape == g.shape, (model, hw, thr, f.shape, g.shape)
                    assert np.abs(f[:, 0] - g[:, 0]).max() < 1e-5
                    assert np.abs(f[:, 1:] - g[:, 1:]).max() < 2e-3
                assert np.array_equal(faces[0], faces[1])
            # consistency: rf_forward_heads -> oracle post-process == rf_detect_batch, selection bit-exact
            heads = eng.forward_heads(inp[None])
            ref = post_oracle.postprocess([x[0] for x in heads], h, w, 0.5, 0.4)
            faces, idx = eng.detect_batch([inp], 0.5, 0.4, want_index=True)
            _compare_dets(faces[0], idx[0], ref, f"{model} {hw}")
            if hw == (448, 448):
                # the un-letterboxed 1280x886 photo through the GPU letterbox kernel: same result
                f2 = eng.detect_batch([golden_image], 0.5, 0.4)
                assert np.array_equal(f2[0], faces[0])
        finally:
            eng.close()


def test_preprocess_letterbox_bit_exact(golden_image):
    """rf_preprocess (GPU letterbox kernel) vs the oracle's cv2.resize-based letterbox: identical bytes."""
    from retinaface_b200 import RF_PREC_FP32
    rng = np.random.default_rng(5)
    eng = _engine("mnet25", 448, 448, RF_PREC_FP32, max_batch=1, max_image=(2048, 2048))
    try:
        cases = [golden_image, rng.integers(0, 256, (333, 517, 3), dtype=np.uint8), rng.integers(0, 256, (900, 700, 3), dtype=np.uint8),
                 rng.integers(0, 256, (896, 896, 3), dtype=np.uint8), rng.integers(0, 256, (100, 448, 3), dtype=np.uint8),
                 rng.integers(0, 256, (448, 448, 3), dtype=np.uint8), rng.integers(0, 256, (2000, 31, 3), dtype=np.uint8),
                 rng.integers(0, 256, (1, 1, 3), dtype=np.uint8)]
        for img in cases:
            assert np.array_equal(eng.preprocess(img), letterbox_bgr_u8(img, 448, 448)), img.shape
    finally:
        eng.close()


@pytest.mark.parametrize("model", ["mnet25", "mnet-deconv-0517"])
def test_fp16_forward_and_detect(model, golden_image, post_oracle):
    """FP16 path (configs[1]): head tensors vs golden FP32 heads within FP16 tolerance
    (cls_prob abs 5e-3, deltas abs 2e-2 over ALL anchors; observed 3e-3 / 1e-2), detections on the golden image:
    same faces as the FP32 golden ones, scores within 1e-3 (north_star's FP16 tolerance; observed 1.2e-4) and
    boxes / landmarks within 0.1 px (observed 0.02 px); and internal consistency
    (its own heads -> oracle post-process == its own detect) bit-exact in selection."""
    from retinaface_b200 import RF_PREC_FP16
    eng = _engine(model, 448, 448, RF_PREC_FP16, max_batch=8)
    try:
        inp = letterbox_bgr_u8(golden_image, 448, 448)
        batch = s_real_batch(inp, 8)
        heads = eng.forward_heads(batch)
        gold = np.load(os.path.join(GOLDEN, f"heads_{model}_448.npz"))
        for k, name in enumerate(topology.OUTPUT_BLOBS):
            err = np.abs(heads[k][0] - gold[name]).max()
            assert err < (5e-3 if "cls_prob" in name else 2e-2), (name, err)
        dets = np.load(os.path.join(GOLDEN, f"dets_{model}_448x448.npz"))["faces_thr0.9"]
        faces, idx = eng.detect_batch(list(batch), 0.9, 0.4, want_index=True)
        assert faces[0].shape == dets.shape
        assert np.abs(faces[0][:, 0] - dets[:, 0]).max() < 1e-3
        assert np.abs(faces[0][:, 1:] - dets[:, 1:]).max() < 0.1
        for i in range(8):
            ref = post_oracle.postprocess([x[i] for x in heads], 448, 448, 0.9, 0.4)
            _compare_dets(faces[i], idx[i], ref, f"fp16 img {i}")
            assert len(faces[i]) >= 4
    finally:
        eng.close()


def test_fp16_tensor_core_layers_vs_oracle(golden_image):
    """tcgen05 path, layer by layer: every materialised activation of the FP16 engine against the FP32
    numpy oracle (relative to the tensor's max: 2e-2, FP16 storage through up to 30 layers), and against the
    FP16 SIMT kernels (RF_FLAG_NO_TENSORCORE, which also selects the CUDA-core stem) that share the storage
    rounding but not the FP16 operand rounding of the stem's pointwise GEMM (2e-2 as well)."""
    from retinaface_b200 import RF_PREC_FP16
    from retinaface_b200.capi import RF_FLAG_NO_TENSORCORE
    inp = letterbox_bgr_u8(golden_image, 448, 448)
    noise = s_noise_batch(1, 448, 448, seed=1)[0]
    batch = np.stack([inp, noise, np.roll(inp, 40, axis=1)])
    tc = _engine("mnet25", 448, 448, RF_PREC_FP16, max_batch=3)
    simt = _engine("mnet25", 448, 448, RF_PREC_FP16, max_batch=3, flags=RF_FLAG_NO_TENSORCORE)
    try:
        tc.debug_keep_all()
        simt.debug_keep_all()
        h_tc = tc.forward_heads(batch)
        h_simt = simt.forward_heads(batch)
        names = ["mobilenet0_relu2_fwd", "mobilenet0_relu4_fwd", "mobilenet0_relu6_fwd",
                 "mobilenet0_relu8_fwd", "mobilenet0_relu10_fwd", "mobilenet0_relu12_fwd", "mobilenet0_relu22_fwd",
                 "mobilenet0_relu24_fwd", "mobilenet0_relu26_fwd", "rf_c3_lateral_relu", "rf_c3_det_context_conv1_relu",
                 "rf_c3_det_concat_relu", "rf_c2_lateral_relu", "rf_c2_aggr_relu", "rf_c2_det_concat_relu",
                 "rf_c1_red_conv_relu", "rf_c1_aggr_relu", "rf_c1_det_context_conv1_relu",
                 "rf_c1_det_context_conv3_1_relu", "rf_c1_det_concat_relu"]
        x = np.concatenate([preprocess_bgr_u8(b) for b in batch])
        ref = MnetOracle(caffemodel("mnet25")).forward(x, want=names)
        for name in names:
            a, b = tc.debug_tensor(name, 3), simt.debug_tensor(name, 3)
            scale = float(np.abs(ref[name]).max())
            e_ref = np.abs(a - ref[name]).max() / scale
            e_simt = np.abs(a - b).max() / scale
            assert e_ref < 2e-2, (name, "vs oracle", e_ref)
            assert e_simt < 2e-2, (name, "vs simt fp16", e_simt)
        for k in range(9):
            assert np.abs(h_tc[k] - h_simt[k]).max() < 2e-2, k
    finally:
        tc.close()
        simt.close()


@pytest.mark.parametrize("hw", [(448, 448), (96, 160), (416, 288)])
def test_fp16_tensor_core_stem_vs_oracle(hw, golden_image):
    """stem_tc.cuh (conv0 and conv2 as tcgen05 GEMMs, conv0 weights rounded to FP16) against the FP32 numpy
    oracle and against the CUDA-core stem (RF_FLAG_SIMT_STEM, FP32 weights): mobilenet0_relu2_fwd within 2e-3 of
    the tensor's max (FP16 storage of the output alone is 5e-4), including sizes whose 16x16 tiles are partial."""
    from retinaface_b200 import RF_PREC_FP16
    from retinaface_b200.capi import RF_FLAG_SIMT_STEM
    h, w = hw
    inp = letterbox_bgr_u8(golden_image, h, w)
    batch = np.stack([inp, s_noise_batch(1, h, w, seed=3)[0], np.full_like(inp, 255)])
    tc = _engine("mnet25", h, w, RF_PREC_FP16, max_batch=3)
    simt = _engine("mnet25", h, w, RF_PREC_FP16, max_batch=3, flags=RF_FLAG_SIMT_STEM)
    try:
        tc.debug_keep_all()
        simt.debug_keep_all()
        tc.forward_heads(batch)
        simt.forward_heads(batch)
        name = "mobilenet0_relu2_fwd"
        x = np.concatenate([preprocess_bgr_u8(b) for b in batch])
        ref = MnetOracle(caffemodel("mnet25")).forward(x, want=[name])[name]
        a, b = tc.debug_tensor(name, 3), simt.debug_tensor(name, 3)
        scale = float(np.abs(ref).max())
        assert np.abs(a - ref).max() / scale < 2e-3, np.abs(a - ref).max() / scale
        assert np.abs(b - ref).max() / scale < 1e-3, np.abs(b - ref).max() / scale
        assert np.abs(a - b).max() / scale < 2e-3
    finally:
        tc.close()
        simt.close()


def test_graph_replay_equals_direct_launch(golden_image):
    from retinaface_b200 import RF_PREC_FP16
    from retinaface_b200.capi import RF_FLAG_NO_GRAPH
    inp = letterbox_bgr_u8(golden_image, 448, 448)
    batch = list(s_real_batch(inp, 5))
    a = _engine("mnet25", 448, 448, RF_PREC_FP16, max_batch=8)
    b = _engine("mnet25", 448, 448, RF_PREC_FP16, max_batch=8, flags=RF_FLAG_NO_GRAPH)
    try:
        for _ in range(3):  # replay several times, varying batch size
            for n in (5, 1, 3):
                fa = a.detect_batch(batch[:n], 0.9, 0.4)
                fb = b.detect_batch(batch[:n], 0.9, 0.4)
                for x, y in zip(fa, fb):
                    assert np.array_equal(x, y)
    finally:
        a.close()
        b.close()


def test_detector_class_mirror(golden_image):
    """RetinaFace(model_dir, "net3").detect(img, 0.9) -- the call main.cpp:15,43 makes."""
    from retinaface_b200 import RetinaFace
    rf = RetinaFace(os.path.join(GOLDEN, "weights"), "net3", net_w=448, net_h=448)
    faces = rf.detect(golden_image, 0.9)
    assert len(faces) == 5 and abs(faces[0].score - 0.9986) < 5e-3
    assert rf.detect(np.zeros((0, 0, 3), np.uint8), 0.9) == []
    per = rf.detectBatchImages([golden_image, golden_image[:400, :600]], 0.9)
    assert len(per) == 2 and len(per[0]) == 5


def test_cpp_driver_on_golden_photo(golden_image, tmp_path):
    """The C++ class shell through the main.cpp-style driver: raw BGR photo in, 5 faces out (448x448, thr 0.9)."""
    import subprocess
    from retinaface_b200.build import build_host
    exe = build_host()
    raw = tmp_path / "img.bgr"
    raw.write_bytes(np.ascontiguousarray(golden_image).tobytes())
    r = subprocess.run([exe, os.path.join(GOLDEN, "weights"), "--image", str(raw), "1280", "886", "--net", "448", "448", "--iters", "3"],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    assert "5 faces in image 0" in r.stdout and "score 0.99" in r.stdout
    # SURVEY 8f-2 through the C++ class: image-coordinate faces from 4 views (2 scales x mirrored), drawn on a clone
    vis = tmp_path / "vis.bgr"
    r = subprocess.run([exe, os.path.join(GOLDEN, "weights"), "--image", str(raw), "1280", "886", "--net", "448", "448", "--iters", "1",
                        "--tta", "--draw", str(vis)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    assert "in image coordinates (4 views)" in r.stdout
    out = np.frombuffer(vis.read_bytes(), np.uint8).reshape(886, 1280, 3)
    changed = (out != golden_image).any(axis=2)
    red = (out == (0, 0, 255)).all(axis=2) & changed
    green = (out == (0, 255, 0)).all(axis=2) & changed
    assert red.sum() > 5 * 400 and green.sum() >= 5 * 5 * 6 and (changed == (red | green)).all()
    # the reference's own input form (main.cpp:18: a JPEG file): decoded on the GPU
    r = subprocess.run([exe, os.path.join(GOLDEN, "weights"), "--jpeg", os.path.join(GOLDEN, "data", "img.jpg"), "--net", "448", "448", "--iters", "3",
                        "--batch", "2"], capture_output=True, text=True, timeout=120)
    if "libnvjpeg" in r.stderr:
        pytest.skip("libnvjpeg not present on this box")
    assert r.returncode == 0, r.stderr
    assert "5 faces in image 0" in r.stdout and "score 0.9" in r.stdout and "JPEG decoded on the GPU" in r.stdout


def test_pipelined_submit_collect_equals_blocking(golden_image):
    """rf_submit_batch / rf_collect_batch (H2D of batch i+1 overlapping the kernels of batch i) returns exactly
    what the blocking rf_detect_batch returns, RF_PIPELINE_DEPTH batches in flight over the default 8 execution contexts."""
    from retinaface_b200 import RF_PREC_FP16, RfError
    from retinaface_b200.capi import PIPELINE_DEPTH
    inp = letterbox_bgr_u8(golden_image, 448, 448)
    batches = [list(s_real_batch(np.roll(inp, 16 * k, axis=0), 4)) for k in range(PIPELINE_DEPTH + 4)]
    eng = _engine("mnet25", 448, 448, RF_PREC_FP16, max_batch=4)
    try:
        want = [eng.detect_batch(b, 0.9, 0.4) for b in batches]
        tickets = []
        got = []
        for k, b in enumerate(batches):
            if len(tickets) == PIPELINE_DEPTH:
                f, c = eng.collect(tickets.pop(0))
                got.append([f[i, :c[i]] for i in range(len(c))])
            tickets.append(eng.submit(b, 0.9, 0.4))
        assert len(tickets) == PIPELINE_DEPTH
        with pytest.raises(RfError):
            eng.submit(batches[0], 0.9, 0.4)          # one more batch in flight is refused
        while tickets:
            f, c = eng.collect(tickets.pop(0))
            got.append([f[i, :c[i]] for i in range(len(c))])
        assert len(got) == len(want)
        for g, w in zip(got, want):
            for a, b in zip(g, w):
                assert np.array_equal(a, b)
    finally:
        eng.close()


def test_int8_engine_vs_integer_oracle(golden_image, post_oracle):
    """RF_PREC_INT8 (configs[2]: mnet-deconv-0517 + its TensorRT calibration table).  TensorRT's INT8 kernels
    are closed source, so the bar has two parts: (1) the CUDA engine against the integer oracle that restates
    its quantisation scheme (oracle/mnet_int8.py): the FP32 stem within 1 LSB of its quantised output (summation
    order), and -- continuing the oracle from the engine's own stem output -- EVERY int8 tensor bit-identical
    (integer GEMMs; the FP32 depthwise / merge stages spell every rounding), heads within 1e-4; (2) the INT8
    result against the FP32 golden detections of the reference's model -- the calibration's own tolerance: same
    5 faces, boxes within 2 px, scores within 0.03."""
    from oracle.mnet_int8 import Int8Oracle
    from retinaface_b200 import RF_PREC_INT8, Engine
    table = os.path.join(GOLDEN, "weights", "mnet-deconv-0517.table.int8")
    inp = letterbox_bgr_u8(golden_image, 448, 448)
    batch = np.stack([inp, np.roll(inp, 24, axis=1)])
    eng = Engine(caffemodel("mnet-deconv-0517"), 448, 448, precision=RF_PREC_INT8, max_batch=2, int8_table=table)
    try:
        eng.debug_keep_all()
        heads = eng.forward_heads(batch)
        oracle = Int8Oracle(caffemodel("mnet-deconv-0517"), table)
        stem_gpu = eng.debug_tensor("mobilenet0_relu2_fwd", 2)
        stem_ref, _ = oracle.stem(batch)
        d = np.abs(stem_gpu - stem_ref)
        assert d.max() <= 1 and (d > 0).mean() < 1e-3, (d.max(), (d > 0).mean())
        o_heads, o_t = oracle.forward(batch, want_tensors=True, q_stem=stem_gpu)
        for name, (q, s) in o_t.items():
            if name in ("_plus0", "_plus1", "mobilenet0_relu2_fwd"):
                continue          # the FPN sums are fused into the aggr conv's staging at this batch size
            got = eng.debug_tensor(name, 2)
            assert np.array_equal(got, q), (name, np.abs(got - q).max(), (got != q).mean())
        for k in range(9):
            assert np.abs(heads[k] - o_heads[k]).max() < 1e-4, (k, np.abs(heads[k] - o_heads[k]).max())
        faces, idx = eng.detect_batch(list(batch), 0.9, 0.4, want_index=True)
        ref = post_oracle.postprocess([x[0] for x in heads], 448, 448, 0.9, 0.4)
        _compare_dets(faces[0], idx[0], ref, "int8 own heads")
        gold = np.load(os.path.join(GOLDEN, "dets_mnet-deconv-0517_448x448.npz"))["faces_thr0.9"]
        assert len(faces[0]) == len(gold) == 5
        for g in gold:      # match by nearest box centre (the order of near-equal scores may differ)
            c = faces[0][np.argmin(np.abs(faces[0][:, 1:3] - g[1:3]).sum(1))]
            assert np.abs(c[1:5] - g[1:5]).max() < 2.0 and abs(c[0] - g[0]) < 0.03, (c[:5], g[:5])
    finally:
        eng.close()


@pytest.mark.parametrize("prec", ["fp16", "int8"])
def test_large_input_and_odd_batches(prec, golden_image, post_oracle):
    """configs[3]-style input (1280x896, 47,040 anchors/image) and batch sizes that make tiles straddle image
    boundaries (1, 3, max_batch): tensor-core engines against the FP32 golden detections of the same model, and
    every batch element against its own heads through the oracle post-process (selection bit-exact)."""
    from retinaface_b200 import RF_PREC_FP16, RF_PREC_INT8, Engine
    model = "mnet-deconv-0517"
    table = os.path.join(GOLDEN, "weights", model + ".table.int8")
    h, w = 896, 1280
    inp = letterbox_bgr_u8(golden_image, h, w)
    eng = Engine(caffemodel(model), h, w, precision=RF_PREC_FP16 if prec == "fp16" else RF_PREC_INT8, max_batch=3,
                 int8_table=table if prec == "int8" else None)
    try:
        gold = np.load(os.path.join(GOLDEN, f"dets_{model}_{h}x{w}.npz"))["faces_thr0.9"]
        tol_px, tol_s = (1.0, 1e-2) if prec == "fp16" else (4.0, 0.05)
        for n in (1, 3, 2):
            batch = [inp] + [np.roll(inp, 32 * k, axis=1) for k in range(1, n)]
            faces, idx = eng.detect_batch(batch, 0.9, 0.4, want_index=True)
            assert len(faces[0]) == len(gold), (prec, n, len(faces[0]), len(gold))
            for g in gold:
                c = faces[0][np.argmin(np.abs(faces[0][:, 1:3] - g[1:3]).sum(1))]
                assert np.abs(c[1:5] - g[1:5]).max() < tol_px and abs(c[0] - g[0]) < tol_s, (prec, n, c[:5], g[:5])
            heads = eng.forward_heads(np.stack(batch))
            for i in range(n):
                ref = post_oracle.postprocess([x[i] for x in heads], h, w, 0.9, 0.4)
                _compare_dets(faces[i], idx[i], ref, f"{prec} n={n} img={i}")
                assert len(faces[i]) >= 5
    finally:
        eng.close()


def test_int8_calibrator_end_to_end(golden_image, tmp_path):
    """SURVEY 8f-3: rf_calibrate_int8 on an FP32 engine writes a TensorRT-format table for *mnet25* (the reference ships a
    table only for mnet-deconv-0517); an INT8 engine created from that table then reproduces the FP32 golden detections
    within the calibration tolerance.  Also: on mnet-deconv-0517 the scales it finds are of the same magnitude as the
    shipped TensorRT table's (different calibration images, same method family)."""
    from oracle.mnet_int8 import read_table
    from retinaface_b200 import RF_PREC_FP32, RF_PREC_INT8, Engine
    inp = letterbox_bgr_u8(golden_image, 448, 448)
    calib = np.stack([np.roll(np.roll(inp, 16 * k, axis=1), 8 * (k % 3), axis=0) for k in range(8)] + [inp[:, ::-1].copy()])
    for model in ("mnet25", "mnet-deconv-0517"):
        table = str(tmp_path / f"{model}.table.int8")
        fp32 = Engine(caffemodel(model), 448, 448, precision=RF_PREC_FP32, max_batch=4)
        try:
            fp32.calibrate_int8(calib, table)
        finally:
            fp32.close()
        t = read_table(table)
        assert open(table).readline().strip() == "TRT-5102-EntropyCalibration2" and len(t) >= 44
        if model == "mnet-deconv-0517":
            shipped = read_table(os.path.join(GOLDEN, "weights", "mnet-deconv-0517.table.int8"))
            ratios = np.array([t[k] / shipped[k] for k in t if k in shipped and k != "data"])
            assert len(ratios) >= 40 and 0.5 < np.median(ratios) < 2.0 and (np.abs(np.log2(ratios)) < 2).mean() > 0.9, np.median(ratios)
        eng = Engine(caffemodel(model), 448, 448, precision=RF_PREC_INT8, max_batch=2, int8_table=table)
        try:
            faces = eng.detect_batch([inp], 0.9, 0.4)[0]
            dets = np.load(os.path.join(GOLDEN, f"dets_{model}_448x448.npz"))
            gold, gold_lo = dets["faces_thr0.9"], dets["faces_thr0.5"]
            assert len(gold) == 5 and len(faces) >= 5
            for g in gold:          # every FP32 face is found, boxes within 3 px, scores within 0.05
                c = faces[np.argmin(np.abs(faces[:, 1:3] - g[1:3]).sum(1))]
                assert np.abs(c[1:5] - g[1:5]).max() < 3.0 and abs(c[0] - g[0]) < 0.05, (model, c[:5], g[:5])
            for c in faces:         # and nothing is invented: a face pushed over 0.9 by quantisation noise is an FP32 face at 0.5
                g = gold_lo[np.argmin(np.abs(gold_lo[:, 1:3] - c[1:3]).sum(1))]
                assert np.abs(c[1:5] - g[1:5]).max() < 3.0, (model, c[:5], g[:5])
        finally:
            eng.close()


@pytest.mark.parametrize("hw", [(416, 288), (320, 320), (96, 160)])
def test_shipped_and_odd_network_sizes(hw, golden_image, post_oracle):
    """The network sizes the reference's own prototxts carry (mnet25.prototxt:7 -> 416x288 (HxW),
    mnet-deconv-0517.prototxt:7 -> 320x320) and a small non-square one: FP32 engine heads vs the numpy oracle
    (2e-4), FP16 and INT8 tensor-core engines vs the FP32 engine's detections (same faces, 1.5 / 4 px)."""
    from retinaface_b200 import RF_PREC_FP16, RF_PREC_FP32, RF_PREC_INT8, Engine
    h, w = hw
    model = "mnet-deconv-0517"
    table = os.path.join(GOLDEN, "weights", model + ".table.int8")
    inp = letterbox_bgr_u8(golden_image, h, w)
    batch = np.stack([inp, np.roll(inp, 8, axis=1), inp[::-1].copy()])
    e32 = Engine(caffemodel(model), h, w, precision=RF_PREC_FP32, max_batch=3)
    try:
        heads = e32.forward_heads(batch)
        ref = MnetOracle(caffemodel(model)).forward(np.concatenate([preprocess_bgr_u8(b) for b in batch]))
        for k, name in enumerate(topology.OUTPUT_BLOBS):
            assert np.abs(heads[k] - ref[name]).max() < TOL_FP32, (hw, name)
        base = e32.detect_batch(list(batch), 0.8, 0.4)
    finally:
        e32.close()
    for prec, tol in ((RF_PREC_FP16, 1.5), (RF_PREC_INT8, 4.0)):
        eng = Engine(caffemodel(model), h, w, precision=prec, max_batch=3, int8_table=table if prec == RF_PREC_INT8 else None)
        try:
            faces, idx = eng.detect_batch(list(batch), 0.8, 0.4, want_index=True)
            hd = eng.forward_heads(batch)
            for i in range(3):
                _compare_dets(faces[i], idx[i], post_oracle.postprocess([x[i] for x in hd], h, w, 0.8, 0.4), f"{hw} prec={prec} img={i}")
                strong = base[i][base[i][:, 0] > 0.95]           # faces well above the threshold must survive quantisation
                for g in strong:
                    assert len(faces[i]) > 0, (hw, prec, i)
                    c = faces[i][np.argmin(np.abs(faces[i][:, 1:3] - g[1:3]).sum(1))]
                    assert np.abs(c[1:5] - g[1:5]).max() < tol, (hw, prec, i, c[:5], g[:5])
        finally:
            eng.close()


def test_detect_views_tta_and_map_back(golden_image, post_oracle):
    """SURVEY.md 8f-2 (rf_detect_views): multi-scale + mirrored views of one image run as one batch, mapped back to
    ORIGINAL IMAGE pixels (x * scale, RetinaFace.cpp:732-738) and merged by one NMS across views, all on the GPU.
    Oracle: every view built on the host (np flip + the OpenCV letter-box oracle into the view's box), detected through
    the plain batch path, mapped back / un-mirrored in float32 numpy and merged by the oracle NMS -- faces identical
    bit for bit, in order.  A single (1.0, no flip) view is detect + map-back."""
    from retinaface_b200 import RF_PREC_FP32, RfError
    h_img, w_img = golden_image.shape[:2]
    eng = _engine("mnet25", 448, 448, RF_PREC_FP32, max_batch=4, max_image=(1024, 1280))
    try:
        views = [(1.0, False), (1.0, True), (0.75, False), (0.6, True)]
        faces, view_of, scales = eng.detect_views(golden_image, views, 0.9, 0.4)
        cands = []
        for v, (s, flip) in enumerate(views):
            bw, bh = int(448 * s), int(448 * s)
            src = np.ascontiguousarray(golden_image[:, ::-1]) if flip else golden_image
            canvas = np.zeros((448, 448, 3), np.uint8)
            canvas[:bh, :bw] = letterbox_bgr_u8(src, bh, bw)
            det = eng.detect_batch([canvas], 0.9, 0.4)[0]
            sc = max(np.float32(1.0 * w_img / bw), np.float32(1.0 * h_img / bh), np.float32(1.0))
            assert scales[v] == sc
            m = det.copy()
            m[:, 1:] = det[:, 1:] * np.float32(sc)
            if flip:
                wm1 = np.float32(w_img - 1)
                f = m.copy()
                f[:, 1], f[:, 3] = wm1 - m[:, 3], wm1 - m[:, 1]
                lx = wm1 - m[:, 5:10]
                f[:, 5:10] = lx[:, [1, 0, 2, 4, 3]]
                f[:, 10:15] = m[:, 10:15][:, [1, 0, 2, 4, 3]]
                m = f
            cands.append((v, m))
        allc = np.concatenate([m for _, m in cands])
        vids = np.concatenate([np.full(len(m), v, np.int32) for v, m in cands])
        want, pos = post_oracle.nms(allc, 0.4)
        assert len(want) >= 5 and len(cands[3][1]) >= 1        # the small mirrored view still finds faces
        assert faces.shape == want.shape
        assert np.array_equal(faces, want)
        assert np.array_equal(view_of, vids[pos])
        # single plain view == detect + map-back
        one, _, sc1 = eng.detect_views(golden_image, [(1.0, False)], 0.9, 0.4)
        plain = eng.detect_batch([golden_image], 0.9, 0.4)[0]
        ref = plain.copy()
        ref[:, 1:] = plain[:, 1:] * np.float32(sc1[0])
        assert np.array_equal(one, ref)
        # faces land on the photo: boxes inside the image, mirrored views agree with the plain ones within a few pixels
        assert (faces[:, 1] >= 0).all() and (faces[:, 3] <= w_img + 2).all() and (faces[:, 4] <= h_img + 2).all()
        m0, m1 = cands[0][1], cands[1][1]

        def iou(a, b):
            iw = min(a[3], b[3]) - max(a[1], b[1]) + 1
            ih = min(a[4], b[4]) - max(a[2], b[2]) + 1
            inter = max(iw, 0) * max(ih, 0)
            return inter / ((a[3] - a[1] + 1) * (a[4] - a[2] + 1) + (b[3] - b[1] + 1) * (b[4] - b[2] + 1) - inter)
        for f0 in m0:      # the un-mirrored view sees the same faces in the same places, eyes on the same sides
            best = max(m1, key=lambda f1: iou(f0, f1))
            assert iou(f0, best) > 0.6, iou(f0, best)
            assert np.abs(best[5:15] - f0[5:15]).max() < 0.25 * (f0[3] - f0[1]), (best[5:15], f0[5:15])
        with pytest.raises(RfError):
            eng.detect_views(golden_image, [(1.5, False)], 0.9, 0.4)
        with pytest.raises(RfError):
            eng.detect_views(golden_image, [(1.0, False)] * 5, 0.9, 0.4)     # > max_batch views
    finally:
        eng.close()


def test_pinned_arbitrary_size_images_take_the_direct_copy_path(golden_image):
    """Caller images that are not network-sized: from pinned memory they are DMA-ed straight out of the caller's buffer
    (no host staging copy, no host synchronisation per image); results equal the pageable path's, image by image."""
    import torch
    from retinaface_b200 import RF_PREC_FP16
    eng = _engine("mnet25", 448, 448, RF_PREC_FP16, max_batch=4, max_image=(1024, 1280))
    try:
        other = np.ascontiguousarray(golden_image[100:700, 200:1100])           # a second size, 900x600
        want = eng.detect_batch([golden_image, other, golden_image], 0.9, 0.4)
        pins = []
        for im in (golden_image, other, golden_image):
            t = torch.empty(im.shape, dtype=torch.uint8).pin_memory()
            t.numpy()[:] = im
            pins.append(t)
        got = eng.detect_batch([t.numpy() for t in pins], 0.9, 0.4)
        assert [len(x) for x in got] == [len(x) for x in want] and len(got[0]) == 5
        for a, b in zip(got, want):
            assert np.array_equal(a, b)
    finally:
        eng.close()


@pytest.mark.parametrize("prec", ["fp16", "int8"])
@pytest.mark.parametrize("hw", [(448, 448), (288, 416)])
def test_2d_tile_kernels_equal_the_1d_ones_bit_for_bit(prec, hw, golden_image):
    """k_tc_dwpw_2d / k_tc_dwpw_2d_i8 (large maps) against the linear-tile kernels they replace (RF_FLAG_DW_1D): same
    arithmetic in the same order, so every activation downstream -- and the heads -- must be IDENTICAL, including the
    partial tiles of a 104x72 map (416x288 input)."""
    from retinaface_b200 import RF_PREC_FP16, RF_PREC_INT8, Engine
    from retinaface_b200.capi import RF_FLAG_DW_1D
    h, w = hw
    model = "mnet-deconv-0517"
    kw = dict(precision=RF_PREC_FP16) if prec == "fp16" else dict(precision=RF_PREC_INT8,
                                                                  int8_table=os.path.join(GOLDEN, "weights", model + ".table.int8"))
    inp = letterbox_bgr_u8(golden_image, h, w)
    batch = np.stack([inp, s_noise_batch(1, h, w, seed=5)[0], np.roll(inp, 16, axis=1)])
    a = Engine(caffemodel(model), h, w, max_batch=3, **kw)
    b = Engine(caffemodel(model), h, w, max_batch=3, flags=RF_FLAG_DW_1D, **kw)
    try:
        a.debug_keep_all()
        b.debug_keep_all()
        ha, hb = a.forward_heads(batch), b.forward_heads(batch)
        for name in ("mobilenet0_relu4_fwd", "mobilenet0_relu6_fwd", "mobilenet0_relu10_fwd"):
            assert np.array_equal(a.debug_tensor(name, 3), b.debug_tensor(name, 3)), name
        for k in range(9):
            assert np.array_equal(ha[k], hb[k]), k
    finally:
        a.close()
        b.close()
