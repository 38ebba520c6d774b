"""Face alignment oracle: the 5-point similarity fit and OpenCV's fixed-point ``warpAffine`` in numpy.
Test infrastructure -- see ``oracle/__init__.py``.

What the library's align kernel (``retinaface_b200/csrc/align.cu``) restates, written independently in vectorised numpy:

* ``similarity_fit`` -- least squares of ``[a -b; b a] p + t ~ q`` over the five landmark pairs, in FP64, in two forms: the
  closed form and the SVD form of Umeyama (1991) the way ``skimage.transform.SimilarityTransform.estimate`` computes it
  (insightface's ``estimate_norm``).  In 2-D both are the optimal proper similarity, so they agree to rounding.
* ``warp_affine_u8`` -- ``cv2.warpAffine(img, M, (w, h), INTER_LINEAR, BORDER_CONSTANT, 0)`` on u8 BGR: M inverted in
  OpenCV's operation order, source coordinates in ``AB_BITS = 10`` fixed point, 5-bit fractions, the 32 x 32 bilinear weight
  table of ``initInterTab2D`` (weights rounded to 1/32768, sum fixed up), ``(sum + (1 << 14)) >> 15``, taps outside read 0.
"""
from __future__ import annotations

import numpy as np

# insightface's arcface_dst (float32): the landmark template of a 112 x 112 recognizer crop
ARCFACE_112 = np.array([[38.2946, 51.6963], [73.5318, 51.5014], [56.0252, 71.7366], [41.5493, 92.3655], [70.7299, 92.2041]],
                       dtype=np.float32)

INTER_BITS = 5
INTER_TAB_SIZE = 1 << INTER_BITS
AB_BITS = 10
AB_SCALE = 1 << AB_BITS
COEF_BITS = 15
COEF_SCALE = 1 << COEF_BITS


def template_for(crop_w: int, crop_h: int) -> np.ndarray:
    """The ArcFace template for a crop whose sides are multiples of 112 (estimate_norm: template * size / 112), float32."""
    t = ARCFACE_112.copy()
    t[:, 0] *= np.float32(crop_w / 112.0)
    t[:, 1] *= np.float32(crop_h / 112.0)
    return t


def _closed_form(src: np.ndarray, dst: np.ndarray) -> np.ndarray:
    p = src - src.mean(axis=0)
    q = dst - dst.mean(axis=0)
    den = float((p * p).sum())
    if den == 0.0:
        a = b = 0.0
    else:
        a = float((p[:, 0] * q[:, 0] + p[:, 1] * q[:, 1]).sum()) / den
        b = float((p[:, 0] * q[:, 1] - p[:, 1] * q[:, 0]).sum()) / den
    sm, dm = src.mean(axis=0), dst.mean(axis=0)
    tx = dm[0] - (a * sm[0] - b * sm[1])
    ty = dm[1] - (b * sm[0] + a * sm[1])
    return np.array([[a, -b, tx], [b, a, ty]], dtype=np.float64)


def _umeyama(src: np.ndarray, dst: np.ndarray) -> np.ndarray:
    """skimage.transform._geometric._umeyama(src, dst, estimate_scale=True), 2-D, first two rows."""
    num, dim = src.shape
    src_mean, dst_mean = src.mean(axis=0), dst.mean(axis=0)
    src_demean, dst_demean = src - src_mean, dst - dst_mean
    A = dst_demean.T @ src_demean / num
    d = np.ones((dim,), dtype=np.float64)
    if np.linalg.det(A) < 0:
        d[dim - 1] = -1
    T = np.eye(dim + 1, dtype=np.float64)
    U, S, V = np.linalg.svd(A)
    rank = np.linalg.matrix_rank(A)
    if rank == 0:
        return np.full((2, 3), np.nan)
    if rank == dim - 1:
        if np.linalg.det(U) * np.linalg.det(V) > 0:
            T[:dim, :dim] = U @ V
        else:
            s = d[dim - 1]
            d[dim - 1] = -1
            T[:dim, :dim] = U @ np.diag(d) @ V
            d[dim - 1] = s
    else:
        T[:dim, :dim] = U @ np.diag(d) @ V
    scale = 1.0 / src_demean.var(axis=0).sum() * (S @ d)
    T[:dim, dim] = dst_mean - scale * (T[:dim, :dim] @ src_mean.T)
    T[:dim, :dim] *= scale
    return T[:2].copy()


def similarity_fit(src5, dst5, method: str = "closed") -> np.ndarray:
    """2 x 3 FP64 matrix M mapping the five ``src5`` points (image pixels) onto ``dst5`` (crop pixels): what insightface
    passes to cv2.warpAffine.  method: "closed" (closed-form least squares) or "umeyama" (SVD, as skimage does it)."""
    src = np.asarray(src5, dtype=np.float64).reshape(5, 2)
    dst = np.asarray(dst5, dtype=np.float64).reshape(5, 2)
    if method == "closed":
        return _closed_form(src, dst)
    if method == "umeyama":
        return _umeyama(src, dst)
    raise ValueError(method)


def landmarks_in_image(face_row: np.ndarray, scale: float) -> np.ndarray:
    """(5, 2) float32 landmarks of one FaceDetectInfo row (score, box, lx[5], ly[5]) times the map-back factor, in float32
    (the product the library forms)."""
    r = np.asarray(face_row, dtype=np.float32)
    s = np.float32(scale)
    return np.stack([r[5:10] * s, r[10:15] * s], axis=1)


def bilinear_tab() -> np.ndarray:
    """initInterTab2D(INTER_LINEAR, fixpt=true): int16 [32*32][4] weights (y0x0, y0x1, y1x0, y1x1), row = fy * 32 + fx."""
    lin = np.empty((INTER_TAB_SIZE, 2), dtype=np.float32)
    for i in range(INTER_TAB_SIZE):
        x = np.float32(i) * np.float32(1.0 / INTER_TAB_SIZE)
        lin[i] = (np.float32(1.0) - x, x)
    tab = np.empty((INTER_TAB_SIZE * INTER_TAB_SIZE, 4), dtype=np.int32)
    for i in range(INTER_TAB_SIZE):
        for j in range(INTER_TAB_SIZE):
            w = np.empty(4, dtype=np.int32)
            for k1 in range(2):
                for k2 in range(2):
                    v = np.float32(lin[i, k1] * lin[j, k2])
                    w[2 * k1 + k2] = min(max(int(np.rint(np.float64(v) * COEF_SCALE)), -32768), 32767)   # saturate_cast<short>
            diff = int(w.sum()) - COEF_SCALE
            if diff:
                # OpenCV searches the central 2 x 2 taps starting at index (ksize/2, ksize/2); for a 2 x 2 kernel that start is
                # tap (1, 1) and the other taps it compares lie past this cell (still zero), so the fix-up lands on tap (1, 1)
                w[3] -= diff
            tab[i * INTER_TAB_SIZE + j] = w
    return tab


_TAB = None


def invert_affine(M) -> np.ndarray:
    """cv::warpAffine's inversion of a forward map (imgwarp.cpp), in its operation order."""
    m = [float(v) for v in np.asarray(M, dtype=np.float64).reshape(6)]
    D = m[0] * m[4] - m[1] * m[3]
    D = 1.0 / D if D != 0 else 0.0
    A11, A22 = m[4] * D, m[0] * D
    m[0] = A11
    m[1] *= -D
    m[3] *= -D
    m[4] = A22
    b1 = -m[0] * m[2] - m[1] * m[5]
    b2 = -m[3] * m[2] - m[4] * m[5]
    m[2], m[5] = b1, b2
    return np.array(m, dtype=np.float64).reshape(2, 3)


def warp_affine_u8(img: np.ndarray, M, w: int, h: int) -> np.ndarray:
    """cv2.warpAffine(img, M, (w, h), flags=INTER_LINEAR, borderMode=BORDER_CONSTANT, borderValue=0) for u8 HWC images,
    byte for byte (OpenCV's fixed-point path)."""
    global _TAB
    if _TAB is None:
        _TAB = bilinear_tab()
    src = np.ascontiguousarray(img, dtype=np.uint8)
    sh, sw = src.shape[:2]
    cn = src.shape[2] if src.ndim == 3 else 1
    src = src.reshape(sh, sw, cn)
    m = invert_affine(M)
    xs = np.arange(w, dtype=np.float64)
    ys = np.arange(h, dtype=np.float64)
    adelta = np.rint(m[0, 0] * xs * AB_SCALE).astype(np.int64)
    bdelta = np.rint(m[1, 0] * xs * AB_SCALE).astype(np.int64)
    round_delta = AB_SCALE // INTER_TAB_SIZE // 2
    X0 = np.rint((m[0, 1] * ys + m[0, 2]) * AB_SCALE).astype(np.int64) + round_delta
    Y0 = np.rint((m[1, 1] * ys + m[1, 2]) * AB_SCALE).astype(np.int64) + round_delta
    X = (X0[:, None] + adelta[None, :]) >> (AB_BITS - INTER_BITS)
    Y = (Y0[:, None] + bdelta[None, :]) >> (AB_BITS - INTER_BITS)
    sx = np.clip(X >> INTER_BITS, -32768, 32767)
    sy = np.clip(Y >> INTER_BITS, -32768, 32767)
    wt = _TAB[((Y & (INTER_TAB_SIZE - 1)) << INTER_BITS) | (X & (INTER_TAB_SIZE - 1))].astype(np.int64)   # (h, w, 4)
    acc = np.zeros((h, w, cn), dtype=np.int64)
    for k, (dy, dx) in enumerate(((0, 0), (0, 1), (1, 0), (1, 1))):
        ty, tx = sy + dy, sx + dx
        inside = (tx >= 0) & (tx < sw) & (ty >= 0) & (ty < sh)
        v = src[np.clip(ty, 0, sh - 1), np.clip(tx, 0, sw - 1)].astype(np.int64)
        v[~inside] = 0
        acc += v * wt[..., k:k + 1]
    out = np.clip((acc + (1 << (COEF_BITS - 1))) >> COEF_BITS, 0, 255).astype(np.uint8)
    return out if img.ndim == 3 else out[..., 0]


def norm_crop(img: np.ndarray, face_row, scale: float, crop_w: int = 112, crop_h: int = 112, template=None):
    """insightface norm_crop of one face record: (crop u8 BGR, M)."""
    dst = template_for(crop_w, crop_h) if template is None else np.asarray(template, dtype=np.float32)
    M = similarity_fit(landmarks_in_image(face_row, scale), dst)
    return warp_affine_u8(img, M, crop_w, crop_h), M
