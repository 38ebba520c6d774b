"""retinaface_b200 -- B200-native (sm_100a) RetinaFace mnet25 detect path.

The product is ``librf_b200.so`` (CUDA kernels behind the C ABI of ``include/rf_b200.h``); this
package is the thin Python host side used by the tests and ``bench.py``: a ctypes binding
(``capi``) and ``RetinaFace``, a mirror of the reference's C++ class surface
(``retinaface/RetinaFace.h:63-70``).  There is no CPU fallback anywhere in this package.
"""
from .capi import (ARCFACE_112, RF_CROP_F16_RGB, RF_CROP_U8_BGR, RF_PREC_FP16, RF_PREC_FP32, RF_PREC_INT8, RfError, Engine,  # noqa: F401
                   align_spec, lib_path, load_library)
from .detector import FaceDetectInfo, RetinaFace  # noqa: F401

__all__ = ["Engine", "RetinaFace", "FaceDetectInfo", "RfError", "load_library", "lib_path",
           "RF_PREC_FP32", "RF_PREC_FP16", "RF_PREC_INT8", "RF_CROP_U8_BGR", "RF_CROP_F16_RGB", "ARCFACE_112", "align_spec"]
