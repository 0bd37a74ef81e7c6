"""GPU tests (-m gpu) of per-tile candidate selection -- ``head_kernel<1>`` / ``rows_filter_kernel`` -> ``sort_keys_kernel`` ->
``select_kernel`` (and the oriented-box path's shared capacity) -- bit for bit against NumPy references built so the answer is
known exactly: every sort arm and its power-of-two edges in one launch, heavy confidence ties, signed confidences, threshold and
capacity edges, tiles of more than 32 768 candidates, NMS at IoU = threshold, zero-area boxes, suppression chains across the
256-candidate chunks, class offsets up to class 79, and Ultralytics' max_nms cut."""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from aerial_image_recognition_b200 import graph as G, weights as W
from oracle import postproc as OP

F = np.float32


def _engine(*a, **k):
    from aerial_image_recognition_b200.engine import Engine
    return Engine(*a, **k)


@pytest.fixture(scope="module")
def eng():
    """Any planned engine post-processes caller-supplied rows; the small v8m one is quick to build."""
    g = G.build("yolov8m", imgsz=128)
    e = _engine("yolov8m", weights=W.make_synthetic_weights(g, 0, calibrate=False), max_batch=16, graph=g)
    yield e
    e.close()


# ---- references ------------------------------------------------------------------------------------------------
def _records(rows, idx, tile):
    """``DET_DTYPE`` records of rows[idx] as the engine writes them (conf * 1.0 is the conf; cls from column 5 when there is one)."""
    from aerial_image_recognition_b200.engine import DET_DTYPE
    r = np.zeros(len(idx), DET_DTYPE)
    for k, f in enumerate(("cx", "cy", "w", "h", "conf")):
        r[f] = rows[idx, k]
    r["cls"] = rows[idx, 5].astype(np.int32) if rows.shape[1] > 5 else 0
    r["tile"], r["anchor"] = tile, idx
    return r


def _passing(rows, thr, inclusive=True):
    c = rows[:, 4]
    return np.nonzero(c >= F(thr) if inclusive else c > F(thr))[0]


def _key_order(conf, idx):
    """Descending confidence (+0.0 and -0.0 equal), ties by ascending anchor."""
    return idx[np.lexsort((idx, -conf[idx].astype(np.float64)))]


def _offset_boxes(rows):
    """xywh -> xyxy + cls * 7680 in fp32, one rounding per operation, as select_kernel and Ultralytics compute them."""
    hw, hh = rows[:, 2] * F(0.5), rows[:, 3] * F(0.5)
    off = rows[:, 5].astype(np.int32).astype(F) * F(7680.0)
    return np.stack([(rows[:, 0] - hw) + off, (rows[:, 1] - hh) + off, (rows[:, 0] + hw) + off, (rows[:, 1] + hh) + off], 1)


def _nms_anchors(rows, thr, inclusive, iou_thr, max_det):
    idx = _passing(rows, thr, inclusive)
    keep = OP.nms_greedy_reference(_offset_boxes(rows[idx]), rows[idx, 4], iou_thr)
    return idx[keep[:max_det]]


def _same(got, exp, what):
    """Bit-exact record comparison (every field, -0.0 distinct from +0.0), with the first difference in the message."""
    assert len(got) == len(exp), f"{what}: {len(got)} records, expected {len(exp)}"
    words = got.dtype.itemsize // 4
    g, e = got.view(np.uint32).reshape(len(got), words), exp.view(np.uint32).reshape(len(exp), words)
    bad = np.nonzero((g != e).any(1))[0]
    assert not len(bad), f"{what}: {len(bad)} records differ, first at {bad[0]}: got {got[bad[0]]}, expected {exp[bad[0]]}"


def _post(eng, rows, *a, **k):
    """postprocess(rows=...) -> (list of per-tile records, the raw (dets, counts) tensors)."""
    from aerial_image_recognition_b200.engine import dets_to_numpy
    d, c = eng.postprocess(rows.shape[0], *a, rows=torch.from_numpy(np.ascontiguousarray(rows)).cuda(), **k)
    return dets_to_numpy(d, c), (d, c)


def _bytes_equal(a, b):
    (da, ca), (db, cb) = a, b
    return torch.equal(ca, cb) and all(torch.equal(da[t, :int(ca[t])], db[t, :int(cb[t])]) for t in range(len(ca)))


# ---- every sort arm and its edges ------------------------------------------------------------------------------
ARM_COUNTS = [0, 1, 2, 31, 33, 1023, 1024, 1025, 2048, 2049, 4096, 8192, 16384, 16385, 32768, 32769]
TIE_CONFS = np.array([0.3, 0.5, 0.75, 1.0], F)


def _tie_rows(rng, n, A, counts, thr=0.25):
    """Rows [n, A, 6]: in tile t, counts[t] rows at random positions pass `thr`; four fifths of them take one of four confidences
    (heavy ties), the rest a random one.  The others sit below `thr`.  Boxes and classes random."""
    rows = np.zeros((n, A, 6), F)
    rows[..., 0:2] = rng.uniform(0, 640, (n, A, 2))
    rows[..., 2:4] = rng.uniform(2, 80, (n, A, 2))
    rows[..., 4] = rng.uniform(0, thr * 0.99, (n, A))
    rows[..., 5] = rng.integers(0, 80, (n, A))
    for t, m in enumerate(counts):
        sel = rng.permutation(A)[:m]
        conf = rng.choice(TIE_CONFS, m)
        uniq = rng.random(m) < 0.2
        conf[uniq] = rng.uniform(thr, 1.0, int(uniq.sum()))
        rows[t, sel, 4] = conf
    return rows


def test_every_sort_arm_and_edge_in_one_launch(eng):
    """One tile per passing count: 0 .. 1024 keys sort in shared memory, 1025 .. 16384 in registers (2048 / 4096 / 8192 / 16384 keys),
    16385 .. 32769 in global memory; filter-only (row order), top_k >= count (the full key order) and a small top_k, each twice."""
    n, A, thr = len(ARM_COUNTS), 40000, 0.25
    rows = _tie_rows(np.random.default_rng(11), n, A, ARM_COUNTS, thr)
    for kw, order in (({}, "rows"), ({"top_k": A}, "keys"), ({"top_k": 1500}, "keys")):
        got, raw = _post(eng, rows, thr, True, **kw)
        for t in range(n):
            idx = _passing(rows[t], thr)
            assert len(idx) == ARM_COUNTS[t]
            if order == "keys":
                idx = _key_order(rows[t, :, 4], idx)[:kw["top_k"]]
            _same(got[t], _records(rows[t], idx, t), f"{kw or 'filter'}, tile {t} ({ARM_COUNTS[t]} passing)")
        assert _bytes_equal(raw, _post(eng, rows, thr, True, **kw)[1]), f"{kw}: a second identical call differs"


# ---- threshold edges and row widths ----------------------------------------------------------------------------
@pytest.mark.parametrize("ncol", [5, 6, 8])
def test_threshold_equality_and_row_width(eng, ncol):
    """conf == float32(thr) passes with inclusive=True only; ncol = 5 rows are class 0, columns past the sixth are ignored."""
    rng = np.random.default_rng(ncol)
    thr = 0.3
    t32 = F(thr)
    rows = rng.uniform(0, 100, (2, 3000, ncol)).astype(F)
    if ncol > 5:
        rows[..., 5] = rng.integers(0, 80, (2, 3000))
    rows[..., 4] = rng.choice(np.array([np.nextafter(t32, F(0)), t32, np.nextafter(t32, F(1)), F(0.1), F(0.9)], F), (2, 3000))
    for inclusive in (True, False):
        for kw in ({}, {"top_k": 3000}):
            got, _ = _post(eng, rows, thr, inclusive, **kw)
            for t in range(2):
                idx = _passing(rows[t], thr, inclusive)
                assert (rows[t, idx, 4] == t32).any() == inclusive
                if kw:
                    idx = _key_order(rows[t, :, 4], idx)
                _same(got[t], _records(rows[t], idx, t), f"ncol {ncol}, inclusive {inclusive}, {kw}")


# ---- signed confidences -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("thr", [0.0, -1.0])
def test_signed_confidences_sort_like_floats(eng, thr):
    """+0.0 and -0.0 tie (broken by anchor) and negative confidences sort below them.  The list in the rows' order is the NumPy
    counter-example [0.5, 0.0, -0.0, 0.9, -0.25, 0.25], then 4000 rows of +-0.0 and random values of both signs."""
    rng = np.random.default_rng(7)
    head = np.array([0.5, 0.0, -0.0, 0.9, -0.25, 0.25], F)
    tail = rng.choice(np.array([0.0, -0.0, -0.5, 0.5, -1.0, 1.0], F), 4000)
    tail[::3] = rng.uniform(-1, 1, len(tail[::3]))
    conf = np.concatenate([head, tail])
    rows = np.zeros((2, len(conf), 6), F)
    rows[..., :4] = rng.uniform(0, 640, (2, len(conf), 4))
    rows[..., 4] = conf
    rows[0, len(head):, 4] = -2.0              # tile 0: only the counter-example passes
    assert np.signbit(conf[conf == 0]).any() and (~np.signbit(conf[conf == 0])).any()
    got, _ = _post(eng, rows, thr, True, top_k=len(conf))
    assert got[0]["anchor"].tolist() == ([3, 0, 5, 1, 2, 4] if thr < 0 else [3, 0, 5, 1, 2])
    for t in range(2):
        idx = _key_order(rows[t, :, 4], _passing(rows[t], thr))
        _same(got[t], _records(rows[t], idx, t), f"signed confidences, thr {thr}, tile {t}")


# ---- caps --------------------------------------------------------------------------------------------------------
def test_explicit_cap_truncates_the_ordered_list(eng):
    rows = _tie_rows(np.random.default_rng(3), 2, 5000, [2600, 700])
    for kw in ({}, {"top_k": 2000}, {"top_k": 400}):
        got, (_, counts) = _post(eng, rows, 0.25, True, cap=500, **kw)
        for t in range(2):
            idx = _passing(rows[t], 0.25)
            if kw:
                idx = _key_order(rows[t, :, 4], idx)[:kw["top_k"]]
            assert int(counts[t]) == min(len(idx), 500)
            _same(got[t], _records(rows[t], idx[:500], t), f"cap 500, {kw or 'filter'}, tile {t}")


def _grid_boxes(m, spacing=30.0, size=10.0, y0=0.0, cols=40):
    """m disjoint boxes (cx, cy, w, h) on a grid."""
    k = np.arange(m)
    return np.stack([(k % cols) * spacing + size, y0 + (k // cols) * spacing + size, np.full(m, size), np.full(m, size)], 1).astype(F)


def test_nms_max_det_limits_and_caps(eng):
    """700 disjoint boxes: max_det = 512 keeps the best 512; max_det above cap keeps cap; max_det = 513 is refused."""
    from aerial_image_recognition_b200._lib import B2DError
    rng = np.random.default_rng(5)
    m = 700
    rows = np.zeros((2, m, 6), F)
    for t in range(2):
        rows[t, :, :4] = _grid_boxes(m)[rng.permutation(m)]
        rows[t, :, 4] = rng.permutation(np.linspace(0.3, 0.95, m)).astype(F)
        rows[t, :, 5] = rng.integers(0, 80, m)
    for max_det, cap in ((512, None), (300, None), (512, 100), (300, 200)):
        got, (_, counts) = _post(eng, rows, 0.25, False, iou_thr=0.7, max_det=max_det, cap=cap)
        keep = min(max_det, cap or max_det)
        for t in range(2):
            exp = _nms_anchors(rows[t], 0.25, False, 0.7, keep)
            assert len(exp) == keep and int(counts[t]) == keep
            _same(got[t], _records(rows[t], exp, t), f"max_det {max_det}, cap {cap}")
    with pytest.raises(B2DError, match="max_det 513 exceeds"):
        _post(eng, rows, 0.25, False, iou_thr=0.7, max_det=513)


# ---- NMS structure -----------------------------------------------------------------------------------------------
def _chain_tile(rng, start, m=600):
    """m candidates with unique confidences, descending with the rank r.  Ranks start, start + 1, start + 2 are a chain A, B, C in a
    row (IoU(A, B) = IoU(B, C) = 3/7 > 0.4, IoU(A, C) = 1/9): A suppresses B, so C survives.  Every other rank is a filler, in pairs
    of identical boxes (the second suppressed), so fewer than 512 are kept before rank 511.  Rows in random anchor order."""
    fill = [r for r in range(m) if r not in (start, start + 1, start + 2)]
    boxes = np.zeros((m, 4), F)
    boxes[fill] = _grid_boxes(len(fill) // 2 + 1, y0=100.0)[np.arange(len(fill)) // 2]
    for k in range(3):
        boxes[start + k] = (5.0 + 4.0 * k, 5.0, 10.0, 10.0)
    rows = np.zeros((m, 6), F)
    rows[:, :4] = boxes
    rows[:, 4] = (F(0.9) - np.arange(m, dtype=F) * F(1e-4)).astype(F)
    return rows[rng.permutation(m)]


def _edge_tile(m=600):
    """IoU exactly 0.5 ([0,0,2,1] and [0,0,1,1], in class 0 and, offset exactly, in class 3), zero-area boxes above and below a box
    they overlap, a duplicate that is suppressed, and disjoint fillers."""
    rows = np.zeros((m, 6), F)
    rows[:, :4] = _grid_boxes(m, y0=200.0)
    rows[:, 4] = np.linspace(0.5, 0.3, m).astype(F)
    special = [(1.0, 0.5, 2.0, 1.0, 0.9, 0), (0.5, 0.5, 1.0, 1.0, 0.8, 0),       # IoU == 0.5
               (1.0, 0.5, 2.0, 1.0, 0.9, 3), (0.5, 0.5, 1.0, 1.0, 0.8, 3),
               (50.5, 50.0, 0.0, 5.0, 0.95, 0),                                  # zero width, higher score than the box it crosses
               (50.0, 50.0, 10.0, 10.0, 0.7, 0), (50.0, 50.0, 10.0, 10.0, 0.65, 0),
               (50.0, 50.0, 0.0, 0.0, 0.6, 0), (52.0, 50.0, 6.0, 0.0, 0.55, 0)]  # zero area inside it
    rows[:len(special)] = np.array(special, F)
    return rows


def test_nms_equal_iou_zero_area_and_chains_across_chunks(eng):
    """Greedy NMS over 256-candidate chunks: chains starting at ranks 254, 255, 510, 511 straddle the chunk boundaries; IoU equal
    to the threshold keeps both boxes; zero-area boxes neither suppress nor are suppressed."""
    rng = np.random.default_rng(9)
    starts = [254, 255, 510, 511]
    rows = np.stack([_chain_tile(rng, s) for s in starts] + [_edge_tile()])
    got, _ = _post(eng, rows, 0.25, False, iou_thr=0.4, max_det=512)
    for t, s in enumerate(starts):
        exp = _nms_anchors(rows[t], 0.25, False, 0.4, 512)
        order = _key_order(rows[t, :, 4], np.arange(len(rows[t])))
        assert order[s + 2] in exp and order[s + 1] not in exp and order[s] in exp, s
        _same(got[t], _records(rows[t], exp, t), f"chain at rank {s}")
    t = len(starts)
    _same(got[t], _records(rows[t], _nms_anchors(rows[t], 0.25, False, 0.4, 512), t), "edge tile at iou_thr 0.4")
    got, _ = _post(eng, rows[t:t + 1], 0.25, False, iou_thr=0.5, max_det=512)
    exp = _nms_anchors(rows[t], 0.25, False, 0.5, 512)
    assert {0, 1, 2, 3, 4, 5, 7, 8} <= set(exp.tolist()) and 6 not in exp
    _same(got[0], _records(rows[t], exp, 0), "edge tile at iou_thr 0.5")


@pytest.mark.parametrize("iou_thr,max_det", [(0.7, 300), (0.45, 512)])
def test_nms_class_offsets_up_to_class_79(eng, iou_thr, max_det):
    """8400 clustered rows in classes 0 .. 79 (half in 70 .. 79, where cls * 7680 ~ 6e5 and fp32 rounds the offset boxes to 1/16 px),
    tied and unique confidences."""
    rng = np.random.default_rng(int(iou_thr * 100))
    n, A = 3, 8400
    rows = np.zeros((n, A, 6), F)
    centres = rng.uniform(20, 620, (n, 60, 2))
    pick = rng.integers(0, 60, (n, A))
    rows[..., :2] = np.take_along_axis(centres, pick[..., None].repeat(2, -1), 1) + rng.normal(0, 3, (n, A, 2))
    rows[..., 2:4] = rng.uniform(10, 60, (n, A, 2))
    rows[..., 4] = np.where(rng.random((n, A)) < 0.5, rng.choice(TIE_CONFS, (n, A)), rng.random((n, A)))
    rows[..., 5] = np.where(rng.random((n, A)) < 0.5, rng.integers(70, 80, (n, A)), rng.integers(0, 80, (n, A)))
    got, _ = _post(eng, rows, 0.25, False, iou_thr=iou_thr, max_det=max_det)
    for t in range(n):
        _same(got[t], _records(rows[t], _nms_anchors(rows[t], 0.25, False, iou_thr, max_det), t), f"classes 0..79, tile {t}")
        assert got[t]["cls"].max() >= 70


def test_nms_looks_at_the_best_max_nms_candidates_only(eng):
    """40 000 passing rows with unique confidences: the best 30 000 are copies of 50 boxes, the rest isolated boxes.  Ultralytics
    keeps the 50 (max_nms = 30000 cuts the isolated ones before NMS); without the cut 300 would be kept."""
    rng = np.random.default_rng(1)
    A, top = 40000, 30000
    rank = np.arange(A)
    rows = np.zeros((A, 6), F)
    rows[:top, :4] = _grid_boxes(50, spacing=100.0, size=20.0, cols=10)[rank[:top] % 50]
    rows[top:, :4] = _grid_boxes(A - top, spacing=20.0, size=8.0, y0=1000.0, cols=100)
    rows[:, 4] = np.linspace(0.9, 0.3, A).astype(F)
    assert len(np.unique(rows[:, 4])) == A
    rows = rows[rng.permutation(A)]
    got, _ = _post(eng, rows[None], 0.25, False, iou_thr=0.7, max_det=300)
    pred = np.ascontiguousarray(rows[:, :5].T[None])
    ref = OP.ultralytics_nms(pred, 0.25, 0.7, 300, max_nms=top)[0]
    anchor_of = {float(c): a for a, c in enumerate(rows[:, 4])}
    exp = np.array([anchor_of[float(c)] for c in ref[:, 4]])
    assert len(exp) == 50
    _same(got[0], _records(rows, exp, 0), "max_nms")


# ---- more than 32 768 candidates per tile ---------------------------------------------------------------------------
def test_rows_path_keeps_every_one_of_64512_passing_rows(eng):
    n, A = 2, 64512                   # yolov7 at 1024 x 1024
    rows = _tie_rows(np.random.default_rng(17), n, A, [A, A])
    rows[1, ::3, 4] = 0.0             # conf == thr, inclusive
    for kw in ({}, {"top_k": A}):
        got, raw = _post(eng, rows, 0.0, True, **kw)
        for t in range(n):
            idx = np.arange(A)
            if kw:
                idx = _key_order(rows[t, :, 4], idx)
            _same(got[t], _records(rows[t], idx, t), f"{A} passing rows, {kw or 'filter'}")
        assert _bytes_equal(raw, _post(eng, rows, 0.0, True, **kw)[1])


def test_more_than_65536_rows_refused(eng):
    from aerial_image_recognition_b200._lib import B2DError
    rows = np.zeros((1, 65537, 6), F)
    with pytest.raises(B2DError, match="65537 rows per tile exceed the limit of 65536"):
        _post(eng, rows, 0.5, True)


def _write_head(eng, g, n, fill):
    """Write each level's head map [n, hw, hw, c] straight into the engine's buffer: fill(level, shape) -> fp32 array."""
    for i, lv in enumerate(g.head["levels"]):
        hw, c = lv["hw"], g.bufs[lv["buf"]].c
        eng.buffer(lv["buf"], n).copy_(torch.from_numpy(fill(i, (n, hw, hw, c))).cuda())
    torch.cuda.synchronize()


def test_yolov7_1024_head_path_keeps_every_row():
    """yolov7 at 1024 x 1024 has 64 512 rows per tile.  Objectness logits of +-200 decode to exactly 1.0 and +0.0, so every row
    passes at conf_thr = 0 with real ties; postprocess equals decode_rows filtered in NumPy, in row order and in key order."""
    g = G.build("yolov7", imgsz=1024)
    n = 2
    e = _engine("yolov7", weights=W.make_synthetic_weights(g, 0, calibrate=False), max_batch=n, graph=g)
    rng = np.random.default_rng(4)
    no = g.nc + 5

    def fill(i, shape):
        m = rng.normal(0, 1.5, shape).astype(F)
        for a in range(3):
            m[..., a * no + 4] = rng.choice(np.array([-200.0, 200.0], F), shape[:3])
        return m
    _write_head(e, g, n, fill)
    dec = e.decode_rows(n).cpu().numpy()
    A = dec.shape[1]
    assert A == 64512 and set(np.unique(dec[..., 4]).tolist()) == {0.0, 1.0}
    from aerial_image_recognition_b200.engine import dets_to_numpy
    for kw in ({}, {"top_k": A}, {"top_k": 1000}):
        got = dets_to_numpy(*e.postprocess(n, 0.0, True, **kw))
        for t in range(n):
            idx = _passing(dec[t], 0.0)
            assert len(idx) == A
            if kw:
                idx = _key_order(dec[t, :, 4], idx)[:kw["top_k"]]
            _same(got[t], _records(dec[t], idx, t), f"yolov7 1024, {kw or 'filter'}, tile {t}")
    e.close()


def test_obb_1280_top_k_keeps_every_row():
    """yolov8m-obb at 1280 x 1280 has 33 600 rows per tile, all passing at conf_thr = 0; with top_k = 33600 every one comes back in
    key order (class logits of -200 / 0 / 200: scores 0, 0.5, 1, heavily tied), as regularized records."""
    from aerial_image_recognition_b200.engine import OBB_DTYPE, obbs_to_numpy
    arch = "yolov8m-obb"
    g = G.build(arch, imgsz=1280)
    n = 2
    e = _engine(arch, weights=W.make_synthetic_weights(g, 0, calibrate=False), max_batch=n, graph=g)
    rng = np.random.default_rng(8)
    nc = g.nc

    def fill(i, shape):
        m = rng.normal(0, 1.5, shape).astype(F)
        m[..., 64:64 + nc] = rng.choice(np.array([-200.0, 0.0, 200.0], F), shape[:3] + (nc,), p=[0.9, 0.07, 0.03])
        return m
    _write_head(e, g, n, fill)
    dec = e.decode_rows(n).cpu().numpy()
    A = dec.shape[1]
    assert A == 33600
    got = obbs_to_numpy(*e.postprocess(n, 0.0, True, top_k=A))
    e.close()
    pi, half_pi = F(math.pi), F(math.pi / 2)
    for t in range(n):
        idx = _key_order(dec[t, :, 4], np.arange(A))
        d = dec[t, idx]
        keep = d[:, 2] > d[:, 3]
        th = np.where(keep, d[:, 6], d[:, 6] + half_pi).astype(F)
        md = np.fmod(th, pi)
        md = np.where(md < 0, md + pi, md).astype(F)
        exp = np.zeros(A, OBB_DTYPE)
        exp["cx"], exp["cy"] = d[:, 0], d[:, 1]
        exp["w"], exp["h"] = np.where(keep, d[:, 2], d[:, 3]), np.where(keep, d[:, 3], d[:, 2])
        exp["theta"], exp["conf"], exp["cls"] = md, d[:, 4], d[:, 5].astype(np.int32)
        exp["tile"], exp["anchor"] = t, idx
        _same(got[t], exp, f"obb 1280, tile {t}")
