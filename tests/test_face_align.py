"""Landmark-aligned face crops (insightface norm_crop on the GPU): rf_detect_align_batch / rf_align_batch_device.

CPU: the numpy oracle (oracle/align.py) against cv2.warpAffine byte for byte, the closed-form similarity fit against the SVD
Umeyama form, the align kernel's resource use, the C++ surface building.  GPU: crops byte-identical to cv2.warpAffine with the
matrix the library reports, that matrix against the oracle's fit, detection results untouched, both entry points and both
layouts, validation, and the Python / C++ class surfaces.
"""
import os
import re
import subprocess

import cv2
import numpy as np
import pytest

from conftest import GOLDEN, ROOT, WEIGHTS, caffemodel
from oracle.align import (ARCFACE_112, invert_affine, landmarks_in_image, similarity_fit, template_for, warp_affine_u8)
from oracle.inputs import letterbox_bgr_u8, s_real_batch

gpu = pytest.mark.gpu


def _random_similarity(rng, w, h, src_w, src_h):
    """A similarity of any rotation and scale whose crop centre lands anywhere in (or next to) the source image."""
    ang, s = rng.uniform(-np.pi, np.pi), rng.uniform(0.05, 3.0)
    cx, cy = rng.uniform(-0.2 * src_w, 1.2 * src_w), rng.uniform(-0.2 * src_h, 1.2 * src_h)
    a, b = s * np.cos(ang), s * np.sin(ang)
    return np.array([[a, -b, w / 2 - (a * cx - b * cy)], [b, a, h / 2 - (b * cx + a * cy)]])


def _cv2_warp(img, M, w, h):
    return cv2.warpAffine(img, np.asarray(M, np.float64).reshape(2, 3), (w, h), flags=cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT,
                          borderValue=0)


# ---------------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("size,count", [((112, 112), 100), ((96, 112), 60), ((224, 224), 60)])
def test_oracle_warp_equals_cv2_byte_for_byte(size, count, golden_image):
    """oracle.align.warp_affine_u8 == cv2.warpAffine(INTER_LINEAR, BORDER_CONSTANT 0) on seeded random similarities over the
    golden photo: crops inside, partly and wholly outside the image."""
    w, h = size
    rng = np.random.default_rng(1000 + w + h)
    outside = partial = 0
    for _ in range(count):
        M = _random_similarity(rng, w, h, golden_image.shape[1], golden_image.shape[0])
        ref = _cv2_warp(golden_image, M, w, h)
        assert np.array_equal(warp_affine_u8(golden_image, M, w, h), ref), M
        zero = (ref == 0).all(axis=2).mean()
        outside += zero == 1.0
        partial += 0.05 < zero < 1.0
    assert outside >= 1 and partial >= 5, (outside, partial)


def test_oracle_warp_singular_matrix_and_integer_shift(golden_image):
    """A singular (all-zero) M (OpenCV inverts it to zero: every pixel samples (0, 0)) and pure integer shifts (the
    fx = fy = 0 weights, where OpenCV's weight table carries its sum correction)."""
    for M in (np.zeros((2, 3)), np.array([[1.0, 0, -300], [0, 1.0, -200]]), np.array([[1.0, 0, 40], [0, 1.0, 30]])):
        assert np.array_equal(warp_affine_u8(golden_image, M, 112, 112), _cv2_warp(golden_image, M, 112, 112))


def test_similarity_fit_closed_form_equals_umeyama():
    """Closed-form least squares == skimage's SVD Umeyama (restated) within 1e-12 relative, on seeded landmark sets (with
    noise, and mirrored ones where Umeyama's reflection guard is active); the template maps onto itself exactly."""
    rng = np.random.default_rng(7)
    for k in range(300):
        ang, s = rng.uniform(-np.pi, np.pi), rng.uniform(0.1, 20)
        R = s * np.array([[np.cos(ang), -np.sin(ang)], [np.sin(ang), np.cos(ang)]])
        src = (ARCFACE_112.astype(np.float64) @ R.T) + rng.uniform(-2000, 2000, 2) + rng.normal(0, 3, (5, 2))
        if k % 5 == 0:
            src[:, 0] = -src[:, 0]
        for dst in (ARCFACE_112, template_for(224, 224)):
            a, b = similarity_fit(src, dst, "closed"), similarity_fit(src, dst, "umeyama")
            assert np.abs(a - b).max() <= 1e-12 * np.abs(b).max(), (a, b)
    ident = similarity_fit(ARCFACE_112, ARCFACE_112)
    assert np.abs(ident - np.array([[1, 0, 0], [0, 1, 0]])).max() < 1e-12
    assert np.array_equal(invert_affine(np.array([[1.0, 0, 0], [0, 1.0, 0]])), np.array([[1.0, -0.0, 0], [-0.0, 1.0, 0]]))


def test_align_kernel_compiles_without_spills(built_lib, tmp_path):
    """The align kernel compiles for sm_100a with no local-memory spills."""
    from retinaface_b200.build import ARCH, COMMON, CSRC, nvcc
    obj = str(tmp_path / "align.o")
    r = subprocess.run([nvcc()] + ARCH + COMMON + ["-fmad=false", "-Xptxas", "-v", "-c", os.path.join(CSRC, "align.cu"), "-o", obj],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    info = r.stderr[r.stderr.index("k_align"):]
    assert re.search(r"0 bytes spill stores, 0 bytes spill loads", info), info


def test_align_symbols_exported_and_spec_layout(built_lib):
    import ctypes as C
    from retinaface_b200 import capi
    lib = C.CDLL(built_lib)
    assert hasattr(lib, "rf_detect_align_batch") and hasattr(lib, "rf_align_batch_device")
    assert C.sizeof(capi._AlignSpec) == 4 * 2 + 4 * 10 + 4 * 2 + 4 * 2
    assert np.array_equal(capi.ARCFACE_112, ARCFACE_112)
    spec = capi.align_spec((224, 224))
    assert spec.crop_w == 224 and spec.max_crops == 16 and spec.layout == capi.RF_CROP_U8_BGR and list(spec.dst_x) == [0.0] * 5


def test_cpp_surface_has_detect_and_align(built_lib):
    """RetinaFace::detectAndAlign / lastCrops and rf_main --align build against the C ABI (running them needs the GPU)."""
    from retinaface_b200.build import build_host
    exe = build_host()
    assert os.access(exe, os.X_OK)
    src = open(os.path.join(ROOT, "retinaface_b200", "host", "RetinaFace.h")).read()
    assert "void detectAndAlign(vector<cv::Mat> imgs, float threshold" in src and "lastCrops(" in src


# ---------------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------------
def _engine(net_hw, prec, **kw):
    from retinaface_b200 import Engine
    kw.setdefault("max_image", (896, 1280))
    return Engine(caffemodel(kw.pop("model", "mnet25")), net_hw[0], net_hw[1], precision=prec, **kw)


def _check_crops(images, per, scales, template, crop_w, crop_h):
    """The bars of every u8 crop: the library's M == the oracle's fit (1e-9 relative); the crop == cv2.warpAffine with the
    library's M byte for byte; against cv2 with the oracle's M, <= 1 LSB on <= 0.1 % of bytes.  Returns the crop count."""
    total = 0
    for img, (faces, crops, affine), s in zip(images, per, scales):
        src = np.ascontiguousarray(img)
        assert len(crops) == len(affine) <= len(faces)
        for j in range(len(crops)):
            M = similarity_fit(landmarks_in_image(faces[j], s), template)
            assert np.abs(affine[j] - M).max() <= 1e-9 * np.abs(M).max(), (affine[j], M)
            assert np.array_equal(crops[j], _cv2_warp(src, affine[j], crop_w, crop_h)), j
            d = np.abs(crops[j].astype(np.int16) - _cv2_warp(src, M, crop_w, crop_h))
            assert d.max() <= 1 and (d > 0).mean() <= 1e-3
            total += 1
    return total


@gpu
@pytest.mark.parametrize("prec", [0, 1], ids=["fp32", "fp16"])
@pytest.mark.parametrize("net_hw", [(448, 448), (896, 1280)], ids=["448-letterbox", "1280x896-identity"])
def test_detect_align_golden_photo(net_hw, prec, golden_image):
    """Golden photo 1280x886 (letter-boxed into 448^2 / copied into 1280x896): detection results bit-equal to rf_detect_batch,
    matrices equal to the oracle's fit, crops byte-identical to cv2.warpAffine."""
    eng = _engine(net_hw, prec, max_batch=2)
    try:
        imgs = [golden_image, np.roll(golden_image, 40, axis=1)]
        want, want_idx = eng.detect_batch(imgs, 0.5, 0.4, want_index=True)
        per, scales, idx = eng.detect_align(imgs, 0.5, 0.4, want_index=True)
        for i in range(2):
            assert np.array_equal(per[i][0], want[i]) and np.array_equal(idx[i], want_idx[i])
            assert len(per[i][1]) == min(len(want[i]), 16) >= 5
        ref_scale = np.float32(max(np.float32(1280 / net_hw[1]), np.float32(886 / net_hw[0]), np.float32(1)))
        assert (scales == ref_scale).all(), scales
        assert _check_crops(imgs, per, scales, ARCFACE_112, 112, 112) >= 10
    finally:
        eng.close()


@gpu
def test_detect_align_mixed_batch(golden_image):
    """Network-sized, letter-boxed, pinned, pageable and padded-row-stride images in one call, plus a photo cut next to a face so
    its crop reaches past the image border (constant-border taps).  Same bars as the golden-photo test."""
    import torch
    eng = _engine((448, 448), 1, max_batch=8)
    try:
        net = letterbox_bgr_u8(golden_image, 448, 448)
        faces0 = eng.detect_batch([golden_image], 0.5, 0.4)[0]
        s0 = max(1280 / 448, 886 / 448)
        x1 = int(faces0[0, 1] * s0)                                  # cut the photo a few pixels left of the top face's box
        cut = np.ascontiguousarray(golden_image[:, max(x1 - 3, 0):])
        pinned_t = torch.empty(golden_image.shape, dtype=torch.uint8).pin_memory()
        pinned = pinned_t.numpy()
        pinned[:] = np.roll(golden_image, 24, axis=0)
        pinned_net_t = torch.empty(net.shape, dtype=torch.uint8).pin_memory()
        pinned_net = pinned_net_t.numpy()
        pinned_net[:] = np.roll(net, 8, axis=1)
        wide = np.zeros((886, 1400, 3), np.uint8)
        wide[:, :1280] = np.roll(golden_image, -32, axis=1)
        padded = wide[:, :1280]
        assert padded.strides[0] == 1400 * 3
        imgs = [net, golden_image, pinned, padded, cut, pinned_net, golden_image[:300, :420].copy()]
        want, want_idx = eng.detect_batch([np.ascontiguousarray(im) for im in imgs], 0.5, 0.4, want_index=True)
        per, scales, idx = eng.detect_align(imgs, 0.5, 0.4, want_index=True)
        for i in range(len(imgs)):
            assert np.array_equal(per[i][0], want[i]) and np.array_equal(idx[i], want_idx[i]), i
        assert scales[0] == 1 and scales[5] == 1 and scales[6] == 1 and scales[1] > 2
        assert _check_crops(imgs, per, scales, ARCFACE_112, 112, 112) >= 20
        # the cut photo: at least one crop samples past the left image edge
        beyond = 0
        for j, M in enumerate(per[4][2]):
            inv = invert_affine(M)
            corners = inv @ np.array([[0, 0, 1], [111, 0, 1], [0, 111, 1], [111, 111, 1]], np.float64).T
            beyond += corners[0].min() < 0
        assert beyond >= 1
    finally:
        eng.close()


@gpu
def test_max_crops_f16_layout_and_custom_template(golden_image):
    """max_crops below the face count: exactly max_crops crops, those of the top-scoring faces in score order.  RF_CROP_F16_RGB
    == ((crop_rgb - 127.5) * f32(1 / 127.5)).astype(f16) bit for bit.  A custom template on a 96 x 112 crop matches cv2."""
    from retinaface_b200 import RF_CROP_F16_RGB
    eng = _engine((448, 448), 1, max_batch=2)
    try:
        imgs = [golden_image, np.roll(golden_image, 64, axis=1)]
        full, scales = eng.detect_align(imgs, 0.5, 0.4)
        few, _ = eng.detect_align(imgs, 0.5, 0.4, max_crops=2)
        for i in range(2):
            assert len(full[i][0]) > 2 and few[i][1].shape[0] == 2
            assert np.array_equal(few[i][1], full[i][1][:2]) and np.array_equal(few[i][2], full[i][2][:2])
            assert (np.diff(full[i][0][:, 0]) <= 0).all()
        f16, _ = eng.detect_align(imgs, 0.5, 0.4, layout=RF_CROP_F16_RGB)
        for i in range(2):
            u8 = full[i][1]
            want = ((u8[..., ::-1].astype(np.float32) - np.float32(127.5)) * np.float32(1 / 127.5)).astype(np.float16).transpose(0, 3, 1, 2)
            assert f16[i][1].dtype == np.float16 and f16[i][1].view(np.uint16).tolist() == want.view(np.uint16).tolist()
        tmpl = ARCFACE_112 - np.array([8.0, 0.0], np.float32)          # the 96 x 112 variant of the ArcFace template
        cus, sc = eng.detect_align(imgs, 0.5, 0.4, crop=(96, 112), template=tmpl)
        assert cus[0][1].shape[1:] == (112, 96, 3)
        assert _check_crops(imgs, cus, sc, tmpl, 96, 112) >= 10
    finally:
        eng.close()


@gpu
def test_device_resident_align_two_contexts(golden_image):
    """torch CUDA u8 images -> rf_detect_batch_device -> rf_align_batch_device into torch FP16 tensors, two batches in flight
    on different execution contexts: equal to the host path on the same images."""
    import torch
    from retinaface_b200 import RF_CROP_F16_RGB, align_spec
    eng = _engine((448, 448), 1, max_batch=4, streams=2)
    try:
        net = letterbox_bgr_u8(golden_image, 448, 448)
        batches = [s_real_batch(net, 4), s_real_batch(np.roll(net, 16, axis=0), 4)]
        dev = [torch.from_numpy(b).cuda() for b in batches]
        torch.cuda.synchronize()
        spec = align_spec(max_crops=8, layout=RF_CROP_F16_RGB)
        outs, affs = [], []
        for d in dev:
            dets, counts = eng.detect_device(4, 0.5, 0.4, d.data_ptr())
            out = torch.full((4, 8, 3, 112, 112), float("nan"), dtype=torch.float16, device="cuda")
            aff = torch.zeros((4, 8, 2, 3), dtype=torch.float64, device="cuda")
            torch.cuda.synchronize()                # (the fills run on torch's stream, the library's streams do not wait for it)
            eng.align_device(4, d.data_ptr(), dets, counts, out.data_ptr(), spec, aff.data_ptr())
            outs.append(out)
            affs.append(aff)
        eng.synchronize()
        for b, out, aff in zip(batches, outs, affs):
            per, _ = eng.detect_align(list(b), 0.5, 0.4, max_crops=8, layout=RF_CROP_F16_RGB)
            o, a = out.cpu().numpy(), aff.cpu().numpy()
            for i in range(4):
                m = len(per[i][1])
                assert m >= 5
                assert o[i, :m].view(np.uint16).tolist() == per[i][1].view(np.uint16).tolist()
                assert np.array_equal(a[i, :m], per[i][2])
                assert np.isnan(o[i, m:].astype(np.float32)).all()        # slots past the count are not written
    finally:
        eng.close()


@gpu
def test_align_leaves_detection_unchanged_and_validates(golden_image):
    """rf_detect_batch results and rf_launches_per_batch are the same before and after alignment calls; invalid specs are
    RF_ERR_INVALID_ARG; more letter-boxed images than raw buffers is RF_ERR_CAPACITY."""
    import ctypes as C
    from retinaface_b200 import RfError, align_spec
    eng = _engine((448, 448), 1, max_batch=2)
    try:
        imgs = [golden_image, letterbox_bgr_u8(golden_image, 448, 448)]
        before = eng.detect_batch(imgs, 0.5, 0.4, want_index=True)
        launches = eng.launches_per_batch(2)
        eng.detect_align(imgs, 0.5, 0.4)
        eng.detect_align(imgs, 0.5, 0.4, crop=(224, 224), max_crops=4)
        after = eng.detect_batch(imgs, 0.5, 0.4, want_index=True)
        assert eng.launches_per_batch(2) == launches
        for a, b in zip(before, after):
            for x, y in zip(a, b):
                assert np.array_equal(x, y)
        bad = [dict(crop=(0, 112)), dict(crop=(112, 1025)), dict(crop=(100, 100)), dict(max_crops=0), dict(max_crops=eng.max_faces + 1),
               dict(layout=7)]
        for kw in bad:
            with pytest.raises(RfError) as e:
                eng.detect_align(imgs, 0.5, 0.4, spec=align_spec(**kw))
            assert e.value.status == -1, kw
            assert eng.lib.rf_align_batch_device(eng.h, eng.device_input_ptr(), 1, 1, 1, C.byref(align_spec(**kw)), 1, None) == -1
        n = 1
        ptrs = (C.c_void_p * n)(imgs[0].ctypes.data)
        ws, hs = (C.c_int * n)(1280), (C.c_int * n)(886)
        out = np.empty(16 * 112 * 112 * 3, np.uint8)
        assert eng.lib.rf_detect_align_batch(eng.h, ptrs, ws, hs, None, n, 0.5, 0.4, None, None, None, None, None, out.ctypes.data, None) == -1
    finally:
        eng.close()
    # raw buffers capped at 2 GiB: 8192^2 x 3 bytes each -> 10 of them for 11 images
    eng = _engine((448, 448), 1, max_batch=11, max_image=(8192, 8192))
    try:
        small = [np.ascontiguousarray(np.roll(golden_image, 8 * k, axis=1)[:300, :460]) for k in range(11)]
        with pytest.raises(RfError) as e:
            eng.detect_align(small, 0.5, 0.4)
        assert e.value.status == -6 and "not network-sized" in str(e.value)
        assert len(eng.detect_batch(small, 0.5, 0.4)) == 11         # the plain path still chunks through the raw buffers
        per, _ = eng.detect_align(small[:10], 0.5, 0.4)
        assert len(per) == 10
    finally:
        eng.close()


@gpu
def test_python_and_cpp_surfaces_match_the_c_abi(golden_image, tmp_path):
    """RetinaFace.detectAndAlign (Python) and rf_main --align (C++): 5 crops of the golden photo at 448^2, thr 0.9, byte-identical
    to the C-ABI crops."""
    from retinaface_b200 import Engine, RetinaFace
    from retinaface_b200.build import build_host
    rf = RetinaFace(WEIGHTS)
    try:
        got = rf.detectAndAlign([golden_image], 0.9)[0]
        assert len(got) == 5
        s = np.float32(max(1280 / 448, 886 / 448))
        faces0 = rf.detectBatchImages([golden_image], 0.9)[0]
        assert abs(got[0][0].pts_x[0] - np.float32(faces0[0].pts_x[0]) * s) <= 1e-3 * abs(got[0][0].pts_x[0])
    finally:
        rf.engine.close()
    eng = Engine(os.path.join(WEIGHTS, RetinaFace.MODEL_FILE), 448, 448, max_batch=8, max_image=(3072, 4096))
    try:
        per, _ = eng.detect_align([golden_image], 0.9, 0.4)
    finally:
        eng.close()
    abi = per[0][1]
    assert abi.shape[0] == 5
    for (_, c), a in zip(got, abi):
        assert np.array_equal(c, a)
    exe = build_host()
    raw, crops = tmp_path / "img.bgr", tmp_path / "crops.bgr"
    raw.write_bytes(np.ascontiguousarray(golden_image).tobytes())
    r = subprocess.run([exe, WEIGHTS, "--image", str(raw), "1280", "886", "--net", "448", "448", "--iters", "1", "--align", str(crops)],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    assert "aligned crops of image 0: 5" in r.stdout
    cpp = np.frombuffer(crops.read_bytes(), np.uint8).reshape(-1, 112, 112, 3)
    assert np.array_equal(cpp, abi)
