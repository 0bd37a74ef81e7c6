"""Host-side integer coefficient tables for the two resize kernels.

The reference resizes every tile on the CPU before inference:

* ``SimpleDetector.detect`` / ``detect_batch`` call ``PIL.Image.resize((640, 640))``
  (``simple_detector.py:463``, ``:655``) -- Pillow's default filter is BICUBIC with
  antialiasing, two passes (horizontal into a uint8 temporary, then vertical),
  22-bit fixed-point coefficients;
* ``GPUHandler.preprocess_image`` calls ``cv2.resize(img, (640, 640))``
  (``_script/gpu_handler.py:74-76``) -- INTER_LINEAR, half-pixel centres, 11-bit
  coefficients, no antialias.

Both are integer algorithms once the per-output-index coefficients are known, so
the coefficients are computed here in float64/float32 exactly as the libraries do
and uploaded once per (in_size, out_size); the CUDA kernels then do only integer
multiply-accumulate and are bit-exact against Pillow / OpenCV by construction.
"""
from __future__ import annotations

import math
from functools import lru_cache
from typing import Tuple

import numpy as np

PIL_PRECISION_BITS = 32 - 8 - 2
CV_COEF_BITS = 11


def _bicubic(x: float) -> float:
    a = -0.5
    if x < 0.0:
        x = -x
    if x < 1.0:
        return ((a + 2.0) * x - (a + 3.0)) * x * x + 1
    if x < 2.0:
        return (((x - 5) * x + 8) * x - 4) * a
    return 0.0


@lru_cache(maxsize=64)
def pil_bicubic_table(in_size: int, out_size: int) -> Tuple[np.ndarray, np.ndarray, int]:
    """(bounds int32 [out,2] = (first, count), coeffs int32 [out, ksize], ksize)."""
    scale = in_size / out_size
    filterscale = max(scale, 1.0)
    support = 2.0 * filterscale
    ksize = int(math.ceil(support)) * 2 + 1
    bounds = np.zeros((out_size, 2), dtype=np.int32)
    kk = np.zeros((out_size, ksize), dtype=np.int32)
    ss = 1.0 / filterscale
    for xx in range(out_size):
        center = (xx + 0.5) * scale
        xmin = int(center - support + 0.5)
        if xmin < 0:
            xmin = 0
        xmax = int(center + support + 0.5)
        if xmax > in_size:
            xmax = in_size
        xmax -= xmin
        ws = [_bicubic((x + xmin - center + 0.5) * ss) for x in range(xmax)]
        ww = 0.0
        for w in ws:
            ww += w
        for x in range(xmax):
            w = ws[x] / ww if ww != 0.0 else ws[x]
            if w < 0:
                kk[xx, x] = int(-0.5 + w * (1 << PIL_PRECISION_BITS))
            else:
                kk[xx, x] = int(0.5 + w * (1 << PIL_PRECISION_BITS))
        bounds[xx] = (xmin, xmax)
    return bounds, kk, ksize


@lru_cache(maxsize=64)
def cv2_linear_table(in_size: int, out_size: int, vertical: bool = False) -> Tuple[np.ndarray, np.ndarray]:
    """(ofs int32 [out,2] = (i0, i1), coef int16 [out,2]) for one axis (``cv2_linear_coef`` in ``csrc/common.cuh``).

    OpenCV clamps the two passes differently.  Horizontally, a tap outside the
    image zeroes the fraction and clamps the index.  Vertically
    (``vertical=True``), the fraction is kept and the two row indices are
    clamped separately.  The tables agree on every down-scale and differ in the
    edge rows of an up-scale, where the vertical sum's two ``>> 16`` truncations
    round differently.
    """
    scale = np.float64(in_size) / np.float64(out_size)
    ofs = np.zeros((out_size, 2), dtype=np.int32)
    coef = np.zeros((out_size, 2), dtype=np.int16)
    for d in range(out_size):
        f = np.float32((d + 0.5) * scale - 0.5)
        s = int(math.floor(float(f)))
        f = np.float32(f - np.float32(s))
        if vertical:
            ofs[d] = (min(max(s, 0), in_size - 1), min(max(s + 1, 0), in_size - 1))
        else:
            if s < 0:
                f, s = np.float32(0.0), 0
            if s >= in_size - 1:
                f, s = np.float32(0.0), in_size - 1
            ofs[d] = (s, min(s + 1, in_size - 1))
        c0 = np.float32(1.0) - f
        a0 = int(np.rint(np.float32(c0 * np.float32(2048.0))))
        a1 = int(np.rint(np.float32(f * np.float32(2048.0))))
        coef[d] = (a0, a1)
    return ofs, coef


def letterbox_geometry(h: int, w: int, size: int = 640):
    """Ultralytics LetterBox (auto=False, scaleup=True, center=True) geometry:
    returns (new_w, new_h, left, top, gain).  Python ``round`` is banker's, as upstream."""
    r = min(size / h, size / w)
    new_w, new_h = int(round(w * r)), int(round(h * r))
    dw, dh = (size - new_w) / 2, (size - new_h) / 2
    top, left = int(round(dh - 0.1)), int(round(dw - 0.1))
    return new_w, new_h, left, top, r


# ---- NumPy emulations of the kernels' integer arithmetic (used by the CPU tests) -------

def emulate_pil_bicubic(img: np.ndarray, out_h: int, out_w: int) -> np.ndarray:
    h, w, c = img.shape
    src = img.astype(np.int64)
    if w != out_w:
        bounds, kk, ks = pil_bicubic_table(w, out_w)
        tmp = np.empty((h, out_w, c), dtype=np.int64)
        for xx in range(out_w):
            x0, n = bounds[xx]
            acc = (src[:, x0:x0 + n, :] * kk[xx, :n].astype(np.int64)[None, :, None]).sum(1) + (1 << (PIL_PRECISION_BITS - 1))
            tmp[:, xx, :] = np.clip(acc >> PIL_PRECISION_BITS, 0, 255)
        src = tmp
    if h != out_h:
        bounds, kk, ks = pil_bicubic_table(h, out_h)
        out = np.empty((out_h, out_w, c), dtype=np.int64)
        for yy in range(out_h):
            y0, n = bounds[yy]
            acc = (src[y0:y0 + n] * kk[yy, :n].astype(np.int64)[:, None, None]).sum(0) + (1 << (PIL_PRECISION_BITS - 1))
            out[yy] = np.clip(acc >> PIL_PRECISION_BITS, 0, 255)
        src = out
    return src.astype(np.uint8)


def emulate_cv2_linear(img: np.ndarray, out_h: int, out_w: int) -> np.ndarray:
    h, w, c = img.shape
    xo, xa = cv2_linear_table(w, out_w)
    yo, yb = cv2_linear_table(h, out_h, vertical=True)
    s = img.astype(np.int32)
    rows = s[:, xo[:, 0], :] * xa[:, 0].astype(np.int32)[None, :, None] + s[:, xo[:, 1], :] * xa[:, 1].astype(np.int32)[None, :, None]
    r0 = rows[yo[:, 0]] >> 4
    r1 = rows[yo[:, 1]] >> 4
    b0 = yb[:, 0].astype(np.int32)[:, None, None]
    b1 = yb[:, 1].astype(np.int32)[:, None, None]
    v = (((b0 * r0) >> 16) + ((b1 * r1) >> 16) + 2) >> 2
    return np.clip(v, 0, 255).astype(np.uint8)
