"""Python mirror of the reference's detector class surface, over the C ABI.

Mirrors ``class RetinaFace`` (retinaface/RetinaFace.h:63-70): same constructor arguments
(model directory, network name "net3", nms threshold 0.4), ``detect(img, threshold, scales)``
and ``detectBatchImages(imgs, threshold)``.  The reference's methods return ``void`` and drop
their results (RetinaFace.cpp:665,726,747); here they return the ``FaceDetectInfo`` list that the
reference computes and discards.  The C++ twin of this file is ``retinaface_b200/host/RetinaFace.h``.
"""
from __future__ import annotations

import os
from dataclasses import dataclass
from typing import List, Sequence, Tuple

import numpy as np

from .capi import RF_PREC_FP16, Engine


@dataclass
class FaceDetectInfo:  # RetinaFace.h:37-42
    score: float
    rect: tuple   # anchor_box x1,y1,x2,y2
    pts_x: tuple  # FacePts.x[5]
    pts_y: tuple  # FacePts.y[5]

    @staticmethod
    def from_row(r: np.ndarray) -> "FaceDetectInfo":
        return FaceDetectInfo(float(r[0]), tuple(map(float, r[1:5])), tuple(map(float, r[5:10])), tuple(map(float, r[10:15])))


class RetinaFace:
    MODEL_FILE = "mnet-deconv-0517.caffemodel"  # the file the reference always loads, RetinaFace.cpp:276

    def __init__(self, model: str, network: str = "net3", nms: float = 0.4, *, net_w: int = 448, net_h: int = 448,
                 max_batch: int = 8, precision: int = RF_PREC_FP16, device: int = 0, max_faces: int = 256,
                 model_file: str = None, max_image=(3072, 4096)):
        if network != "net3":
            # RetinaFace.cpp:211-242 lists other names, but only the fmc==3 "net3" anchors are configured (:245-271)
            raise ValueError(f"network setting error {network}: only 'net3' is configured")
        self.nms_threshold = nms
        path = os.path.join(model, model_file or self.MODEL_FILE)
        self.engine = Engine(path, net_h, net_w, precision=precision, max_batch=max_batch, max_faces=max_faces,
                             device=device, max_image=max_image)

    def detect(self, img: np.ndarray, threshold: float = 0.5, scales: float = 1.0) -> List[FaceDetectInfo]:
        if img is None or img.size == 0:  # RetinaFace.cpp:578-580
            return []
        return self.detectBatchImages([img], threshold)[0]

    def detectBatchImages(self, imgs: Sequence[np.ndarray], threshold: float = 0.5) -> List[List[FaceDetectInfo]]:
        rows = self.engine.detect_batch(list(imgs), threshold, self.nms_threshold)
        return [[FaceDetectInfo.from_row(r) for r in per] for per in rows]

    def detectInImage(self, img: np.ndarray, threshold: float = 0.5, scales: Sequence[float] = (1.0,), flip: bool = False
                      ) -> List[FaceDetectInfo]:
        """SURVEY.md 8f-2: what the reference leaves commented out / unused (RetinaFace.cpp:730-746, the `scales` argument of
        RetinaFace.h:70): faces in ORIGINAL IMAGE pixels (x * scale), optionally with multi-scale + horizontal-flip test-time
        augmentation.  ``scales``: fractions (0, 1] of the network input the image is fitted into; with ``flip`` every scale
        is also run mirrored.  All views form one batch; the merge NMS across views runs on the GPU (rf_detect_views)."""
        if img is None or img.size == 0:
            return []
        views = [(float(s), f) for s in scales for f in ((False, True) if flip else (False,))]
        faces, _, _ = self.engine.detect_views(img, views, threshold, self.nms_threshold)
        return [FaceDetectInfo.from_row(r) for r in faces]

    def detectAndAlign(self, imgs: Sequence[np.ndarray], threshold: float = 0.5, crop_size: int = 112,
                       max_crops: int = 16) -> List[List[Tuple[FaceDetectInfo, np.ndarray]]]:
        """Detection + the step a recognition pipeline takes next (insightface's norm_crop): per image, up to ``max_crops``
        faces in score order as (FaceDetectInfo in ORIGINAL IMAGE pixels, aligned crop_size x crop_size u8 BGR crop).  The
        crops are warped on the GPU (rf_detect_align_batch) from the original images, byte-identical to cv2.warpAffine with
        the ArcFace-template similarity of the face's landmarks; ``crop_size`` must be a multiple of 112."""
        out: List[List[Tuple[FaceDetectInfo, np.ndarray]]] = []
        imgs = list(imgs)
        mb = self.engine.max_batch
        for start in range(0, len(imgs), mb):
            per, scales = self.engine.detect_align(imgs[start:start + mb], threshold, self.nms_threshold, crop=(crop_size, crop_size),
                                                   max_crops=max_crops)
            for (faces, crops, _), s in zip(per, scales):
                s = np.float32(s)
                rows = faces[:len(crops)].copy()
                rows[:, 1:] *= s        # network-input -> image pixels (RetinaFace.cpp:732-738), in float32 like the library
                out.append([(FaceDetectInfo.from_row(r), c) for r, c in zip(rows, crops)])
        return out

    @staticmethod
    def draw(img: np.ndarray, faces: Sequence[FaceDetectInfo]) -> np.ndarray:
        """The reference's commented-out visualisation (RetinaFace.cpp:730-741): red box outline of thickness 2, green
        landmark dots, on a copy (:744: `clone()`), for faces in image coordinates.  Plain numpy (no OpenCV needed)."""
        out = np.array(img, dtype=np.uint8, copy=True)
        hh, ww = out.shape[:2]

        def fill(x0, y0, x1, y1, colour):
            x0, y0, x1, y1 = max(x0, 0), max(y0, 0), min(x1, ww), min(y1, hh)
            if x1 > x0 and y1 > y0:
                out[y0:y1, x0:x1] = colour
        for f in faces:
            x1, y1, x2, y2 = (int(round(v)) for v in f.rect)
            for (a, b, c, d) in ((x1 - 1, y1 - 1, x2 + 1, y1 + 1), (x1 - 1, y2 - 1, x2 + 1, y2 + 1),
                                 (x1 - 1, y1 - 1, x1 + 1, y2 + 1), (x2 - 1, y1 - 1, x2 + 1, y2 + 1)):
                fill(a, b, c, d, (0, 0, 255))
            for px, py in zip(f.pts_x, f.pts_y):
                cx, cy = int(round(px)), int(round(py))
                fill(cx - 1, cy - 1, cx + 2, cy + 2, (0, 255, 0))
        return out

    @staticmethod
    def map_back_scale(img_w: int, img_h: int, net_w: int, net_h: int) -> float:
        """scale of RetinaFace.cpp:587-591: multiply coordinates by it to return to image pixels (:732-738)."""
        return max(img_w / net_w, img_h / net_h, 1.0)
