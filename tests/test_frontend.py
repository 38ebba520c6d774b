"""CPU: the model-format front end (retinaface_b200/csrc/frontend.cpp, SURVEY.md 8f-4) through its host-only C entry points:
prototxt (protobuf text) reader, graph check against the RetinaFace mnet25 family, folding driven by the FILE's parameters,
the reference's network-name / anchor switch, and the folded-model cache with its staleness check."""
import os
import re
import shutil

import numpy as np
import pytest

from conftest import WEIGHTS, caffemodel
from oracle import topology


@pytest.fixture()
def gen_prototxt(tmp_path, built_lib):
    p = tmp_path / "generated.prototxt"
    p.write_text(topology.to_prototxt(448, 448, 1))
    return str(p)


def test_generated_prototxt_parses_and_folds_like_the_builtin_graph(gen_prototxt):
    from retinaface_b200.capi import model_inspect, model_load
    for layer in ("mobilenet0_conv0_fwd", "mobilenet0_conv13_fwd", "rf_c1_aggr", "rf_c3_det_context_conv3_2", "face_rpn_landmark_pred_stride8"):
        cs, idims, (w, b) = model_load(caffemodel("mnet25"), gen_prototxt, None, layer)
        w0, b0 = model_inspect(caffemodel("mnet25"), layer)
        assert cs == 0 and idims == (1, 3, 448, 448)
        assert np.array_equal(w, w0) and np.array_equal(b, b0), layer


@pytest.mark.parametrize("name,hw", [("mnet25", (416, 288)), ("mnet-deconv-0517", (320, 320))])
def test_reference_prototxts_are_parsed_from_text(name, hw, built_lib):
    """Both shipped prototxt files (different spellings of the reshape / crop layers, `shape: { ... }` with a colon) parse, pass the
    graph check, give the input size the reference's parseNet reads from line 7, and fold to the same weights as the built-in graph."""
    from retinaface_b200.capi import model_inspect, model_load
    proto = os.path.join(WEIGHTS, name + ".prototxt")
    cs, idims, (w, b) = model_load(caffemodel(name), proto, None, "rf_c2_aggr")
    assert idims == (1, 3) + hw
    w0, b0 = model_inspect(caffemodel(name), "rf_c2_aggr")
    assert np.array_equal(w, w0) and np.array_equal(b, b0)


def test_folding_is_driven_by_the_file(gen_prototxt, tmp_path):
    """Change what the FILE says and the folded weights follow: a BatchNorm eps, and a convolution whose bias the file switches off."""
    from retinaface_b200.capi import model_load
    text = open(gen_prototxt).read()
    _, _, (w0, b0) = model_load(caffemodel("mnet25"), gen_prototxt, None, "rf_c3_lateral")
    # (1) eps of rf_c3_lateral_bn: 2e-05 -> 0.5
    i = text.index('name: "rf_c3_lateral_bn"')
    j = text.index("eps:", i)
    edited = tmp_path / "eps.prototxt"
    edited.write_text(text[:j] + re.sub(r"eps:\s*[0-9.eE+-]+", "eps: 0.5", text[j:], count=1))
    _, _, (w1, b1) = model_load(caffemodel("mnet25"), str(edited), None, "rf_c3_lateral")
    assert not np.array_equal(w1, w0) and np.abs(w1).max() < np.abs(w0).max() * 1.0001      # a larger eps shrinks gamma / sqrt(var + eps)
    assert np.abs(w1).sum() < np.abs(w0).sum()
    # (2) a wiring change is refused with a message naming the layer
    swapped = tmp_path / "swapped.prototxt"
    a, b = 'bottom: "rf_c3_det_conv1_bn" bottom: "rf_c3_det_context_conv2_bn"', 'bottom: "rf_c3_det_context_conv2_bn" bottom: "rf_c3_det_conv1_bn"'
    assert a in text
    s = text.replace(a, b, 1)          # the SSH concat of level c3 with its first two inputs swapped
    swapped.write_text(s)
    from retinaface_b200 import RfError
    with pytest.raises(RfError) as e:
        model_load(caffemodel("mnet25"), str(swapped), None, None)
    assert e.value.status == -3 and "concat" in str(e.value)
    # (3) a different stride is refused: the plan would not match
    strided = tmp_path / "stride.prototxt"
    i3 = text.index('name: "mobilenet0_conv5_fwd"')
    j3 = text.index("stride:", i3)
    strided.write_text(text[:j3] + re.sub(r"stride:\s*\d+", "stride: 2", text[j3:], count=1))
    with pytest.raises(RfError) as e:
        model_load(caffemodel("mnet25"), str(strided), None, None)
    assert e.value.status == -3 and "mobilenet0_conv5_fwd" in str(e.value)


def test_malformed_prototxt_fails_with_a_message_not_a_hang(tmp_path, built_lib):
    """The reference's parseNet loops forever when `input_param` is missing and assumes 3-digit sizes (trtnetbase.cpp:159-187)."""
    from retinaface_b200 import RfError
    from retinaface_b200.capi import model_load
    cases = {"no_input.prototxt": 'name: "x"\nlayer { name: "c" type: "Convolution" bottom: "data" top: "c" convolution_param { num_output: 8 kernel_size: 3 } }\n',
             "unbalanced.prototxt": 'layer { name: "data" type: "Input" top: "data" input_param { shape: { dim: 1 dim: 3 dim: 64 dim: 64 } }\n',
             "garbage.prototxt": 'layer { name: "data" type: = }\n', "empty.prototxt": ""}
    for fn, text in cases.items():
        p = tmp_path / fn
        p.write_text(text)
        with pytest.raises(RfError) as e:
            model_load(caffemodel("mnet25"), str(p), None, None)
        assert e.value.status == -3, fn
    with pytest.raises(RfError) as e:
        model_load(caffemodel("mnet25"), str(tmp_path / "missing.prototxt"), None, None)
    assert e.value.status == -2


def test_model_cache_hit_and_staleness(gen_prototxt, tmp_path):
    """The reference reuses `retina.cache` whenever the file exists (trtnetbase.cpp:205-230: no staleness check).  Here: miss -> written;
    hit; another caffemodel under the same cache path -> stale -> rewritten; a truncated cache file -> stale -> rewritten; and a hit
    returns exactly the weights a fresh load folds."""
    from retinaface_b200.capi import model_inspect, model_load
    cache = str(tmp_path / "model.rfcache")
    cm = str(tmp_path / "m.caffemodel")
    shutil.copy(caffemodel("mnet25"), cm)
    st = [model_load(cm, gen_prototxt, cache, None)[0] for _ in range(3)]
    assert st == [1, 2, 2]
    _, _, (w, b) = model_load(cm, gen_prototxt, cache, "mobilenet0_conv24_fwd")
    w0, b0 = model_inspect(cm, "mobilenet0_conv24_fwd")
    assert np.array_equal(w, w0) and np.array_equal(b, b0)
    shutil.copy(caffemodel("mnet-deconv-0517"), cm)                 # same path, other weights
    assert model_load(cm, gen_prototxt, cache, None)[0] == 3
    cs, _, (w2, _) = model_load(cm, gen_prototxt, cache, "mobilenet0_conv24_fwd")
    assert cs == 2 and not np.array_equal(w2, w0)
    assert np.array_equal(w2, model_inspect(caffemodel("mnet-deconv-0517"), "mobilenet0_conv24_fwd")[0])
    data = open(cache, "rb").read()
    open(cache, "wb").write(data[: len(data) // 2])                 # truncated
    assert model_load(cm, gen_prototxt, cache, None)[0] == 3
    assert model_load(cm, gen_prototxt, cache, None)[0] == 2
    assert model_load(cm, None, cache, None)[0] == 3                # the prototxt is part of the key


def test_network_name_switch(built_lib):
    """RetinaFace.cpp:211-268: net3 -> strides 32/16/8, scales {32,16},{8,4},{2,1}, ratio 1; net3a adds ratio 1.5; the names whose
    fmc != 3 have no anchor configuration in the reference either ("please reconfig anchor_cfg"); unknown names are an error."""
    from retinaface_b200 import RfError
    from retinaface_b200.capi import network_config
    assert network_config("net3") == ([32, 16, 8], [[32, 16], [8, 4], [2, 1]], [1.0])
    assert network_config("net3a")[2] == [1.0, 1.5]
    assert network_config("ssh")[0] == [32, 16, 8]
    for bad in ("net5", "net5a", "net6", "net4", "resnet"):
        with pytest.raises(RfError) as e:
            network_config(bad)
        assert e.value.status == -7
    from retinaface_b200 import Engine
    with pytest.raises(RfError) as e:
        Engine(caffemodel("mnet25"), 448, 448, network="net3a")
    assert e.value.status == -7 and "anchor" in str(e.value)
