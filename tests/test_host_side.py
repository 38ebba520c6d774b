"""CPU: the C-ABI library loads, exports every declared symbol, and its host-side logic (model
front end, argument validation, error reporting) behaves -- no compute calls without a GPU."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from conftest import ROOT, caffemodel


def test_exports_every_declared_symbol(built_lib):
    hdr = open(os.path.join(ROOT, "include", "rf_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(rf_[a-z0-9_]+)\s*\(", hdr)) - {"rf_handle_s"})
    from retinaface_b200 import capi
    assert sorted(capi.EXPORTS) == declared
    lib = C.CDLL(built_lib)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.rf_abi_version() == 2


def test_product_has_no_oracle_dependency():
    """The product package must not import or link anything under oracle/ (nor any CPU fallback)."""
    pkg = os.path.join(ROOT, "retinaface_b200")
    for root, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                src = open(os.path.join(root, f), errors="ignore").read()
                assert not re.search(r"^\s*(from|import)\s+oracle", src, re.M), f          # no python import
                assert not re.search(r"#\s*include\s*[<\"][^>\"]*oracle", src), f             # no C/C++ include
                assert "liboracle" not in src and "libref_postproc" not in src and "oracle/_ref" not in src, f   # no link / dlopen


def test_model_front_end_matches_oracle_fold(built_lib):
    from oracle.mnet_numpy import folded_params
    from retinaface_b200.capi import model_inspect
    for m in ("mnet25", "mnet-deconv-0517"):
        fp = folded_params(caffemodel(m))
        n = 0
        for name, d in fp.items():
            if "b" not in d:
                continue
            w, b = model_inspect(caffemodel(m), name)
            assert np.array_equal(w, d["w"]) and np.array_equal(b, d["b"]), name
            n += 1
        assert n == 27 + 5 + 15 + 9


def test_error_paths_without_gpu(built_lib, tmp_path):
    from retinaface_b200 import Engine, RfError
    with pytest.raises(RfError) as e:
        Engine(str(tmp_path / "missing.caffemodel"), 448, 448)
    assert e.value.status == -2
    bad = tmp_path / "bad.caffemodel"
    bad.write_bytes(b"\x0a\x03abc")  # a NetParameter with only a name
    with pytest.raises(RfError) as e:
        Engine(str(bad), 448, 448)
    assert e.value.status == -3
    with pytest.raises(RfError) as e:
        Engine(caffemodel("mnet25"), 450, 448)  # not a multiple of 32
    assert e.value.status == -1
    import torch
    if not torch.cuda.is_available():
        with pytest.raises(RfError) as e:
            Engine(caffemodel("mnet25"), 448, 448)
        assert e.value.status == -5 and "no CPU path" in str(e.value)


def test_detector_mirror_rejects_unconfigured_networks(built_lib):
    from retinaface_b200 import RetinaFace
    with pytest.raises(ValueError):
        RetinaFace("tests/golden/weights", "net5")


def test_cpp_driver_builds_and_fails_loudly_without_gpu(built_lib):
    """retinaface_b200/host (RetinaFace class shell + main.cpp-style driver) compiles against the C ABI;
    without a GPU it must exit non-zero with the library's error, not fall back to anything."""
    import subprocess
    import torch
    from retinaface_b200.build import build_host
    exe = build_host()
    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the gpu test")
    r = subprocess.run([exe, os.path.join(ROOT, "tests", "golden", "weights"), "--iters", "1"], capture_output=True, text=True, timeout=60)
    assert r.returncode == 1 and "no CPU path" in r.stderr


def test_calibrator_threshold_search_matches_numpy_restatement(built_lib):
    """Host-side part of rf_calibrate_int8: the KL threshold search of the library == the numpy restatement,
    on half-normal, exponential, spiky and empty histograms (512 bins keep the O(bins^2) numpy loop short)."""
    from oracle.calibrator_ref import kl_threshold_bins as ref
    from retinaface_b200.capi import kl_threshold_bins as lib
    rng = np.random.default_rng(0)
    cases = [np.histogram(np.abs(rng.normal(0, 1, 200_000)), bins=512, range=(0, 6))[0],
             np.histogram(rng.exponential(1.0, 100_000), bins=512, range=(0, 20))[0],
             np.histogram(np.concatenate([np.abs(rng.normal(0, 0.1, 50_000)), rng.uniform(5, 10, 50)]), bins=512, range=(0, 10))[0],
             np.zeros(512, dtype=np.int64), np.r_[np.zeros(300), 5, np.zeros(211)].astype(np.int64)]
    for h in cases:
        a, b = lib(h.astype(np.uint32)), ref(h)
        assert abs(a - b) <= 2, (a, b)          # identical up to summation-order ties between neighbouring candidates
    assert 128 <= lib(cases[2].astype(np.uint32)) < 320     # most of the sparse uniform outliers in [5, 10) (bins >= 256) are clipped
    assert lib(cases[0].astype(np.uint32)) > 300            # a half-normal keeps most of its range (no over-clipping)


def test_detector_mirror_draw_is_the_references_visualisation():
    """RetinaFace.draw (SURVEY.md 8f-2; RetinaFace.cpp:730-741): red box outline of thickness 2 and green landmark dots on a
    copy; clipped at the image border; the input image is left untouched."""
    import numpy as np
    from retinaface_b200.detector import FaceDetectInfo, RetinaFace
    img = np.full((40, 60, 3), 7, np.uint8)
    f = FaceDetectInfo(0.99, (10.2, 5.0, 30.0, 25.6), (15.0, 25.0, 20.0, 16.0, 24.0), (12.0, 12.0, 16.0, 21.0, 21.0))
    g = FaceDetectInfo(0.95, (50.0, 30.0, 70.0, 50.0), (55.0,) * 5, (35.0,) * 5)          # runs over the border
    out = RetinaFace.draw(img, [f, g])
    assert (img == 7).all() and out.shape == img.shape
    red = (out == (0, 0, 255)).all(axis=2)
    green = (out == (0, 255, 0)).all(axis=2)
    assert red[4:6, 9:31].all() and red[25:27, 9:31].all() and red[4:27, 9:11].all() and red[4:27, 29:31].all()
    assert not red[8:24, 13:28].any()                      # outline only
    assert green[11:14, 14:17].all() and green[20:23, 23:26].all()
    assert red[29:31, 49:60].all() and red[29:40, 49:51].all()


def test_host_copy_pool_copies_every_band(tmp_path):
    """csrc/host_copy.h (staging of pageable caller images, SURVEY 8f-1): row-band parallel copy with 0/1/3/7 workers, packed
    and strided sources, sizes on both sides of the single-thread cut-off, reused 200 times per pool -- byte-identical to
    a plain row copy; pools shut down cleanly."""
    import subprocess
    src = tmp_path / "pool_check.cpp"
    src.write_text(r'''
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include "host_copy.h"
int main() {
    for (int workers : {0, 1, 3, 7}) {
        rf::HostCopyPool pool(workers);
        for (int rep = 0; rep < 200; rep++) {
            const int rows = 1 + rand() % 1200, rb = 3 * (1 + rand() % 1500), stride = rb + (rep % 3 ? 0 : 64);
            std::vector<uint8_t> src((size_t)rows * stride), dst((size_t)rows * rb, 0xAA), ref((size_t)rows * rb);
            for (auto &b : src) b = (uint8_t)rand();
            for (int y = 0; y < rows; y++) memcpy(&ref[(size_t)y * rb], &src[(size_t)y * stride], rb);
            pool.copy_rows(dst.data(), src.data(), rb, stride, rows);
            if (dst != ref) { printf("MISMATCH workers=%d rep=%d\n", workers, rep); return 1; }
        }
    }
    printf("pool ok\n");
    return 0;
}
''')
    exe = tmp_path / "pool_check"
    csrc = os.path.join(ROOT, "retinaface_b200", "csrc")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-pthread", "-I", csrc, str(src), "-o", str(exe)])
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "pool ok" in r.stdout, r.stdout + r.stderr


def test_capacity_guard_for_32bit_activation_offsets(built_lib):
    """ADVICE r1: the kernels index activations with 32-bit element offsets; rf_create must refuse a max_batch whose largest
    tensor (the stem output, H/2 x W/2 x 16) does not fit, with RF_ERR_CAPACITY, before any device work."""
    from retinaface_b200 import Engine, RfError
    # 468 images: 468 * 448 * 640 * 16 = 2,146,959,360 < 2^31 - 1 = 2,147,483,647 -> accepted by the guard: created where there is a
    # GPU, refused later (no device / out of memory) where there is none
    try:
        Engine(caffemodel("mnet25"), 896, 1280, max_batch=468).close()
    except RfError as e:
        assert e.status in (-5, -4), e.status
    with pytest.raises(RfError) as e:
        Engine(caffemodel("mnet25"), 896, 1280, max_batch=469)
    assert e.value.status == -6 and "32-bit" in str(e.value)
    with pytest.raises(RfError) as e:
        Engine(caffemodel("mnet25"), 448, 448, max_batch=2676)
    assert e.value.status == -6


def test_tile_plan_of_the_headline_config(built_lib, monkeypatch):
    """rf_plan_describe (host-only): the FP16 plans of BASELINE configs[1].  Every chain enabled (RF_TILE_MASK=511): at most 15
    kernel launches per forward, each chain within the 227 KB shared-memory / 512-column TMEM budget of an SM.  Defaults:
    one execution context (latency mode) -> the convolution chains (FPN merge + aggr, SSH + predictors + decode + NMS) and
    chain B; several contexts (throughput mode) -> the round-1 kernels with decode + NMS fused into one launch.  Chains
    fall back to the round-1 kernels layer by layer where they cannot fit (wide maps); RF_FLAG_LEGACY_TC = one kernel per layer."""
    from retinaface_b200.capi import RF_FLAG_LEGACY_TC, plan_describe
    monkeypatch.setenv("RF_TILE_MASK", "511")
    text = plan_describe(caffemodel("mnet25"), 448, 448, max_batch=8)
    assert int(text.split()[0]) <= 15, text
    chains = [ln for ln in text.splitlines() if ln.startswith("tile_")]
    assert len(chains) >= 8
    assert any("heads+decode" in ln for ln in chains) and any("merge+aggr" in ln for ln in chains)
    for ln in chains:
        smem = int(re.search(r"smem (\d+) B", ln).group(1))
        sets, cols = (int(x) for x in re.search(r"TMEM (\d+) x (\d+) cols", ln).groups())
        assert smem <= 227 * 1024 and sets * cols <= 512, ln
    big = plan_describe(caffemodel("mnet25"), 896, 1280, max_batch=8)
    assert int(big.split()[0]) <= 30 and "tc2d_dw3" in big          # the 640-wide level does not fit a chain
    for hw in ((288, 416), (320, 320), (96, 160)):
        assert int(plan_describe(caffemodel("mnet-deconv-0517"), hw[0], hw[1], max_batch=3).split()[0]) <= 30
    monkeypatch.delenv("RF_TILE_MASK")
    # latency mode (one execution context): SSH + predictor + NMS chains; at batch <= 2 the merge+aggr chains too
    lat = plan_describe(caffemodel("mnet25"), 448, 448, max_batch=8, streams=1)
    assert "tile_ssh_c1+heads+decode" in lat and "tile_c1_merge+aggr" not in lat and int(lat.split()[0]) == 22
    lat1 = plan_describe(caffemodel("mnet25"), 448, 448, max_batch=1, streams=1)
    assert "tile_ssh_c1+heads+decode" in lat1 and "tile_c1_merge+aggr" in lat1 and int(lat1.split()[0]) <= 21
    thr = plan_describe(caffemodel("mnet25"), 448, 448, max_batch=8)
    assert int(thr.split()[0]) == 29 and "heads_1x1+softmax+decode+nms_all_levels" in thr and "sort+nms" not in thr
    legacy = plan_describe(caffemodel("mnet25"), 448, 448, max_batch=8, flags=RF_FLAG_LEGACY_TC)
    assert int(legacy.split()[0]) == 29 and "tile_" not in legacy


def test_fast_div_multiplier_is_exact_over_the_kernels_ranges():
    """csrc/common.cuh fast_div: q = umulhi(n, ceil(2^32 / d)) replaces the run-time integer divisions of the tile / pixel index
    math.  It is exact while n * d < 2^32; the kernels divide block indices (< 2^20), padded row numbers and GEMM row numbers
    by map widths / heights / tile counts (<= a few thousand).  Restated here and checked against // over those ranges."""
    import numpy as np
    for d in [1, 2, 3, 7, 8, 14, 15, 16, 28, 29, 30, 40, 56, 57, 58, 98, 112, 114, 196, 224, 226, 449, 784, 897, 1282, 2240, 3136]:
        mul = 0 if d <= 1 else ((1 << 32) + d - 1) // d
        n = np.arange(0, min(1 << 21, (1 << 32) // d), dtype=np.uint64)
        q = n if mul == 0 else (n * np.uint64(mul)) >> np.uint64(32)
        assert np.array_equal(q, n // np.uint64(d)), d
        # floor division of negative numerators (first tile: lo = -Wp): -fast_div(-n + d - 1)
        neg = np.arange(1, 4 * d + 1, dtype=np.int64)
        qq = -(((neg + d - 1).astype(np.uint64) * np.uint64(mul)) >> np.uint64(32)).astype(np.int64) if mul else -neg
        assert np.array_equal(qq, -((neg + d - 1) // d)) and np.array_equal(qq, np.floor_divide(-neg, d)), d


def test_header_is_plain_c_and_links(built_lib, tmp_path):
    """include/rf_b200.h is the drop-in boundary for ANY FFI: it must compile as C99 (no C++, no CUDA, no torch types) and a C
    program must link against the library and run the calls that need no GPU."""
    import subprocess
    src = tmp_path / "abi.c"
    src.write_text('#include <stdio.h>\n#include <string.h>\n#include "rf_b200.h"\n'
                   'int main(void) {\n'
                   '    rf_config c; memset(&c, 0, sizeof c);\n'
                   '    int fmc = 0; int strides[8]; float anchors[64];\n'
                   '    if (rf_abi_version() != 2) return 1;\n'
                   '    if (rf_create(NULL, NULL) >= 0) return 2;                 /* argument errors are status codes, not aborts */\n'
                   '    printf("%s | %s\\n", rf_build_info(), rf_status_string(RF_ERR_INVALID_ARG));\n'
                   '    (void)c; (void)fmc; (void)strides; (void)anchors;\n'
                   '    return 0;\n}\n')
    exe = tmp_path / "abi"
    libdir = os.path.dirname(built_lib)
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe),
                           "-L", libdir, "-lrf_b200", f"-Wl,-rpath,{libdir}"])
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=60)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "sm_100a" in r.stdout
