"""Windows of any size (mosaic.window_geometry, b2d_resize_windows) and OpenCV's vertical INTER_LINEAR rule, without a GPU."""
from __future__ import annotations

import ctypes as C
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from aerial_image_recognition_b200 import mosaic as M  # noqa: E402
from aerial_image_recognition_b200 import resample as R  # noqa: E402

cv2 = pytest.importorskip("cv2")

# (in_h, in_w) -> (out_h, out_w): up-scales (which used the horizontal clamp for rows too), exact 2x, down-scales, odd sizes
RESIZE_CASES = [
    ((320, 320), (640, 640)), ((300, 500), (640, 640)), ((500, 300), (640, 640)), ((64, 64), (640, 640)), ((7, 9), (640, 640)),
    ((480, 480), (640, 640)), ((100, 320), (200, 640)), ((1, 5), (3, 640)), ((2, 2), (640, 640)),
    ((1280, 1280), (640, 640)), ((1200, 1200), (640, 640)), ((2000, 2000), (640, 640)), ((340, 1200), (181, 640)),
    ((1200, 64), (640, 34)), ((777, 901), (613, 59)), ((33, 1001), (457, 640)),
]


@pytest.mark.parametrize("src,dst", RESIZE_CASES)
def test_emulated_cv2_linear_equals_cv2(src, dst):
    rng = np.random.default_rng(src[0] * 7919 + src[1])
    a = rng.integers(0, 256, (*src, 3), dtype=np.uint8)
    assert np.array_equal(cv2.resize(a, (dst[1], dst[0]), interpolation=cv2.INTER_LINEAR), R.emulate_cv2_linear(a, *dst))


def test_emulated_cv2_linear_random_sizes():
    rng = np.random.default_rng(5)
    for _ in range(30):
        ih, iw = (int(v) for v in rng.integers(1, 700, 2))
        oh, ow = (int(v) for v in rng.integers(1, 700, 2))
        a = rng.integers(0, 256, (ih, iw, 3), dtype=np.uint8)
        assert np.array_equal(cv2.resize(a, (ow, oh)), R.emulate_cv2_linear(a, oh, ow)), (ih, iw, oh, ow)


def test_vertical_rule_keeps_the_fraction_and_clamps_each_row():
    ofs, coef = R.cv2_linear_table(320, 640, vertical=True)
    assert tuple(ofs[0]) == (0, 0) and tuple(coef[0]) == (512, 1536)           # fy = -0.25: both rows clamp to 0
    assert tuple(ofs[-1]) == (319, 319) and tuple(coef[-1]) == (1536, 512)
    hofs, hcoef = R.cv2_linear_table(320, 640)
    assert tuple(hofs[0]) == (0, 1) and tuple(hcoef[0]) == (2048, 0)           # horizontally the fraction is zeroed
    for i, o in [(1200, 640), (1280, 640), (864, 640), (640, 640)]:            # down-scales: the two rules give the same bytes
        a = np.random.default_rng(i).integers(0, 256, (i, 3, 3), dtype=np.uint8)
        assert np.array_equal(cv2.resize(a, (3, o)), R.emulate_cv2_linear(a, o, 3))


@pytest.mark.parametrize("i,o", [(320, 640), (300, 640), (64, 640), (7, 640), (1200, 640), (1, 640), (640, 1)])
def test_c_horizontal_table_equals_python(lib, i, o):
    k = C.c_int()
    b = np.zeros((o, 2), np.int32); c = np.zeros((o, 2), np.int32)
    assert lib.b2d_resize_table(1, i, o, b.ctypes.data_as(C.c_void_p), c.ctypes.data_as(C.c_void_p), C.byref(k)) == 0
    po, pc = R.cv2_linear_table(i, o)
    assert k.value == 2 and np.array_equal(b, po) and np.array_equal(c, pc.astype(np.int32))


# ---- window geometry ----------------------------------------------------------------------------------------------
GRIDS = [(320, 256), (480, 400), (640, 512), (960, 768), (1200, 600), (1280, 640)]
MOSAICS = [(3001, 2651), (2300, 1700), (1201, 1925), (1000, 1000)]


@pytest.mark.parametrize("win,stride", GRIDS)
def test_window_geometry_is_letterbox_where_one_axis_is_clipped(win, stride):
    S = 640
    seen_single = 0
    for H, W in MOSAICS:
        wins = M.window_grid(H, W, win, stride)
        nw, nh, left, top, g = M.window_geometry(wins, win, S)
        assert g == S / win
        for k, (x0, y0, w0, h0) in enumerate(wins):
            w0, h0 = int(w0), int(h0)
            if w0 == win or h0 == win:
                lw, lh, ll, lt, r = R.letterbox_geometry(h0, w0, S)
                assert r == g
                if lw >= 1 and lh >= 1:
                    assert (nw[k], nh[k], left[k], top[k]) == (lw, lh, ll, lt), (H, W, k)
                    seen_single += 1
            # the stated rule, on every window (double-clipped corners and slivers included)
            ew, eh = max(1, round(w0 * g)), max(1, round(h0 * g))
            assert (nw[k], nh[k]) == (ew, eh)
            assert (left[k], top[k]) == (round((S - ew) / 2 - 0.1), round((S - eh) / 2 - 0.1))
            assert 0 <= left[k] and left[k] + nw[k] <= S and 0 <= top[k] and top[k] + nh[k] <= S
    assert seen_single > 0


def test_window_geometry_corner_and_sliver():
    # a 1-pixel sliver row and column: 1801 % 600 == 1
    wins = M.window_grid(1801, 1801, 1200, 600)
    assert (wins[:, 2] == 1).any() and (wins[:, 3] == 1).any()
    nw, nh, left, top, g = M.window_geometry(wins, 1200, 640)
    one = wins[:, 2] == 1
    assert (nw[one] == 1).all() and (left[one] == 319).all()                   # max(1, round(0.53)) = 1, round(319.5 - 0.1) = 319
    corner = (wins[:, 2] < 1200) & (wins[:, 3] < 1200)
    assert corner.any()
    k = int(np.flatnonzero(corner)[0])
    w0, h0 = int(wins[k, 2]), int(wins[k, 3])
    assert (nw[k], nh[k]) == (max(1, round(w0 * g)), max(1, round(h0 * g)))    # the neighbours' gain, not min(640 / h0, 640 / w0)
    nw2, nh2, _, _, _ = M.window_geometry(np.array([[0, 0, 64, 64]]), 640, 640)
    assert (nw2[0], nh2[0]) == (64, 64)                                         # g = 1: no zoom on a 64 x 64 corner


def test_check_windows_refuses_with_a_message():
    M.check_windows(M.window_grid(1000, 900, 480, 400), 480, 1000, 900)
    for bad, msg in [([[0, 0, 0, 10]], "w0, h0"), ([[0, 0, 10, 481]], "w0, h0"), ([[895, 0, 10, 10]], "inside"),
                     ([[-1, 0, 10, 10]], "inside"), ([[0, 995, 10, 10]], "inside")]:
        with pytest.raises(ValueError, match=msg):
            M.check_windows(np.array(bad), 480, 1000, 900)
    with pytest.raises(ValueError, match="positive"):
        M.check_windows(np.zeros((0, 4)), 0, 1000, 900)


def test_affine_params_default_is_unchanged():
    gt = (2335637.62, 0.1, 0.0, 6845688.78, 0.0, -0.1)
    wins = M.window_grid(1500, 1100)
    p = M.affine_params(wins, gt)
    ref = np.zeros((len(wins), 16))
    ref[:, :6] = gt
    ref[:, 6:8] = wins[:, :2]
    ref[:, 8] = (640 - wins[:, 2]) // 2
    ref[:, 9] = (640 - wins[:, 3]) // 2
    ref[:, 10] = 1.0
    ref[:, 11:13] = wins[:, 2:4]
    assert np.array_equal(p, ref) and np.array_equal(M.affine_params(wins, gt, 640), ref)
    q = M.affine_params(M.window_grid(1500, 1100, 1200, 600), gt, 1200, 640)
    assert (q[:, 10] == 640 / 1200).all()


# ---- the whole window path, emulated: cut, resample, letterbox ---------------------------------------------------------
def emulate_windows(mosaic: np.ndarray, wins: np.ndarray, win: int, imgsz: int, fill: int = 114) -> np.ndarray:
    """NumPy restatement of b2d_resize_windows(out=u8): the kernels' integer arithmetic per window."""
    nw, nh, left, top, _ = M.window_geometry(wins, win, imgsz)
    out = np.full((len(wins), imgsz, imgsz, 3), fill, np.uint8)
    for k, (x0, y0, w0, h0) in enumerate(wins):
        crop = mosaic[y0:y0 + h0, x0:x0 + w0]
        out[k, top[k]:top[k] + nh[k], left[k]:left[k] + nw[k]] = R.emulate_cv2_linear(crop, int(nh[k]), int(nw[k]))
    return out


def cv2_windows(mosaic: np.ndarray, wins: np.ndarray, win: int, imgsz: int, fill: int = 114) -> np.ndarray:
    """The same windows through cv2.resize + cv2.copyMakeBorder, as Ultralytics LetterBox does at the gain imgsz / win."""
    g = imgsz / win
    out = []
    for x0, y0, w0, h0 in wins:
        crop = np.ascontiguousarray(mosaic[y0:y0 + h0, x0:x0 + w0])
        new_w, new_h = max(1, round(int(w0) * g)), max(1, round(int(h0) * g))
        if (new_w, new_h) != (w0, h0):
            crop = cv2.resize(crop, (new_w, new_h), interpolation=cv2.INTER_LINEAR)
        dw, dh = (imgsz - new_w) / 2, (imgsz - new_h) / 2
        top, bottom = round(dh - 0.1), round(dh + 0.1)
        left, right = round(dw - 0.1), round(dw + 0.1)
        out.append(cv2.copyMakeBorder(crop, top, bottom, left, right, cv2.BORDER_CONSTANT, value=(fill, fill, fill)))
    return np.stack(out)


@pytest.mark.parametrize("win,stride", [(1200, 600), (480, 400), (320, 256), (1280, 640), (960, 768)])
def test_emulated_window_path_equals_cv2(win, stride):
    from aerial_image_recognition_b200 import synth
    H, W = 1801, 1333
    m = synth.make_mosaic(H, W, seed=3)
    wins = M.window_grid(H, W, win, stride)
    assert np.array_equal(emulate_windows(m, wins, win, 640), cv2_windows(m, wins, win, 640))
