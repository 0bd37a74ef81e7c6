"""Windows of any size on the device (-m gpu): b2d_resize_windows against cv2 per window, the engine-input form, the
model-sized case against b2d_cut_windows, MosaicDetector end to end and sharded, and cv2 INTER_LINEAR up-scales through
b2d_preprocess."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from aerial_image_recognition_b200 import graph as G, mosaic as M, synth, weights as W
from test_cpu_window_resample import cv2_windows

GT = (2335637.62, 0.1, 0.0, 6845688.78, 0.0, -0.1)


def _engine(arch="yolov8m", imgsz=640, max_batch=4, precision="bf16"):
    from aerial_image_recognition_b200.engine import Engine
    g = G.build(arch, imgsz=imgsz)
    return Engine(arch, weights=W.make_synthetic_weights(g, 0), max_batch=max_batch, graph=g, precision=precision)


@pytest.fixture(scope="module")
def eng640():
    e = _engine()
    yield e
    e.close()


@pytest.fixture(scope="module")
def ragged():
    H, W_ = 3001, 2651
    m = synth.make_mosaic(H, W_, seed=6)
    return m, torch.from_numpy(m).cuda()


# ---- cv2 INTER_LINEAR up-scales through b2d_preprocess -----------------------------------------------------------
@pytest.mark.parametrize("h,w", [(320, 320), (300, 500), (256, 256), (512, 512), (64, 64), (7, 9), (480, 480), (100, 320)])
def test_preprocess_upscale_bit_exact_against_cv2(eng640, h, w):
    import cv2
    rng = np.random.default_rng(h * 1009 + w)
    img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    t = torch.from_numpy(img)[None].cuda()
    assert np.array_equal(eng640.preprocess(t, "cv2_linear", out="u8").cpu().numpy()[0], cv2.resize(img, (640, 640)))
    r = min(640 / h, 640 / w)
    nw, nh = int(round(w * r)), int(round(h * r))
    dw, dh = (640 - nw) / 2, (640 - nh) / 2
    res = cv2.resize(img, (nw, nh), interpolation=cv2.INTER_LINEAR) if (w, h) != (nw, nh) else img
    ref = cv2.copyMakeBorder(res, int(round(dh - 0.1)), int(round(dh + 0.1)), int(round(dw - 0.1)), int(round(dw + 0.1)),
                             cv2.BORDER_CONSTANT, value=(114, 114, 114))
    assert np.array_equal(eng640.preprocess(t, "letterbox", out="u8").cpu().numpy()[0], ref)


# ---- b2d_resize_windows ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("win,stride", [(1200, 600), (1280, 640), (960, 768), (480, 400), (320, 256)])
def test_resize_windows_bit_exact_against_cv2(eng640, ragged, win, stride):
    m, md = ragged
    wins = M.window_grid(*m.shape[:2], win, stride)
    if win == 1200:                       # 3001 % 600 == 1 gives a sliver row; add a sliver column and a 1 x 1 corner
        wins = np.concatenate([wins, [[2650, 0, 1, 1200], [2650, 3000, 1, 1]]]).astype(np.int32)
    assert ((wins[:, 2] < win) & (wins[:, 3] < win)).any()      # a corner clipped on both axes
    got = eng640.resize_windows(md, torch.from_numpy(wins).cuda(), win, out="u8").cpu().numpy()
    ref = cv2_windows(m, wins, win, 640)
    for k in range(len(wins)):
        assert np.array_equal(got[k], ref[k]), (k, wins[k])


def test_resize_windows_pitch_fill_and_bgr(eng640, ragged):
    """A column slice of the mosaic (row pitch > 3 W, rows not 16-byte aligned), another fill value, and the BGR swap."""
    m, md = ragged
    sub, subd = m[:, 37:2037], md[:, 37:2037]
    assert subd.stride(0) == 3 * m.shape[1]
    wins = M.window_grid(sub.shape[0], sub.shape[1], 1200, 600)
    got = eng640.resize_windows(subd, wins, 1200, fill=7, bgr=True, out="u8").cpu().numpy()
    assert np.array_equal(got, cv2_windows(sub, wins, 1200, 640, fill=7)[..., ::-1])


def test_resize_windows_at_model_size_equals_cut_windows(eng640, ragged):
    m, md = ragged
    wins = torch.from_numpy(M.window_grid(*m.shape[:2])).cuda()
    assert torch.equal(eng640.resize_windows(md, wins, 640, out="u8"), eng640.cut_windows(md, wins))
    assert torch.equal(eng640.resize_windows(md, wins, 640, fill=0, out="u8"), eng640.cut_windows(md, wins, fill=0))


@pytest.mark.parametrize("precision", ["bf16", "fp16", "fp16x2"])
def test_resize_windows_engine_input_is_the_u8_canvas(ragged, precision):
    m, md = ragged
    e = _engine(imgsz=256, max_batch=4, precision=precision)
    try:
        wins = M.window_grid(*m.shape[:2], 1200, 600)[-4:]          # the last row: clipped and corner windows
        u8 = e.resize_windows(md, wins, 1200, out="u8")
        assert e.resize_windows(md, wins, 1200) is None
        got = e.buffer("input", 4).float()
        assert torch.equal(got[..., :3], u8.float()) and (got[..., 3] == 0).all()
    finally:
        e.close()


def test_resize_windows_refuses_bad_input_with_a_message(eng640, ragged):
    import ctypes as C
    from aerial_image_recognition_b200._lib import B2DError
    m, md = ragged
    for bad in ([[0, 0, 0, 100]], [[0, 0, 100, 1201]], [[2600, 0, 100, 100]], [[0, -1, 100, 100]], [[0, 2950, 100, 100]]):
        with pytest.raises(ValueError, match="window 0"):
            eng640.resize_windows(md, torch.tensor(bad, dtype=torch.int32).cuda(), 1200, out="u8")
    with pytest.raises(ValueError, match="positive"):
        eng640.resize_windows(md, np.zeros((1, 4), np.int32), 0, out="u8")
    wins = M.window_grid(*m.shape[:2], 1200, 600)[:5]
    with pytest.raises(B2DError, match="max_batch"):
        eng640.resize_windows(md, wins, 1200)
    lib, org = eng640.lib, torch.from_numpy(wins).cuda()
    null = C.c_void_p(0)
    assert lib.b2d_resize_windows(eng640.h, C.c_void_p(md.data_ptr()), 3001, 2651, 2651 * 3, C.c_void_p(org.data_ptr()), 1, 0, 114,
                                  0, 2, null, eng640.stream) < 0
    assert b"window size 0" in lib.b2d_last_error()
    out = torch.empty((1, 640, 640, 3), dtype=torch.uint8, device="cuda")
    assert lib.b2d_resize_windows(eng640.h, C.c_void_p(md.data_ptr()), 3001, 2651, 2651 * 3, C.c_void_p(org.data_ptr()), 1, 1200, 114,
                                  0, 1, C.c_void_p(out.data_ptr()), eng640.stream) < 0
    assert b"out_kind" in lib.b2d_last_error()


def test_resize_windows_on_an_oriented_box_engine(ragged):
    m, md = ragged
    e = _engine("yolov8m-obb", imgsz=256, max_batch=2)
    try:
        wins = M.window_grid(*m.shape[:2], 480, 400)[:2]
        got = e.resize_windows(md, wins, 480, out="u8").cpu().numpy()
        assert np.array_equal(got, cv2_windows(m, wins, 480, 256))
    finally:
        e.close()


# ---- MosaicDetector ----------------------------------------------------------------------------------------------
def _same_records(a, b):
    """Bit-identical in every field of OUT_DTYPE (the 4 padding bytes of a record are not part of the result)."""
    assert len(a) == len(b), (len(a), len(b))
    for f in a.dtype.names:
        assert a[f].tobytes() == b[f].tobytes(), (f, int(np.sum(a[f] != b[f])), len(a))


def _host_letterbox_run(det, m, H, W_):
    """MosaicDetector's result restated: cv2 letterbox of each window on the host, infer(identity), georef(affine) with
    window_geometry's pad and gain, the notebook's conf filter and the same dedup."""
    eng = det.eng
    wins = M.window_grid(H, W_, det.win, det.stride)
    ids = np.arange(len(wins), dtype=np.int64)
    tiles = cv2_windows(m, wins, det.win, eng.imgsz, det.fill)
    params = torch.from_numpy(M.affine_params(wins, det.gt, det.win, eng.imgsz)).cuda()
    nb = -(-len(wins) // eng.max_batch)
    B = -(-len(wins) // nb)
    cols = []
    for s in range(0, len(wins), B):
        e = min(s + B, len(wins))
        dets, counts = eng.infer(torch.from_numpy(tiles[s:e]).cuda(), "identity", False, det.nms_conf, False, det.iou, 0, det.max_det)
        geo = eng.georef(dets, counts, params[s:e], "affine")
        n, cap = dets.shape[0], dets.shape[1]
        slot = torch.arange(cap, device="cuda", dtype=torch.int32)[None, :].expand(n, cap)
        conf = dets[..., 4]
        idx = ((slot < counts[:, None]) & (conf > det.conf)).reshape(-1).nonzero().squeeze(1)
        g64 = geo.view(torch.float64).view(n * cap, 5)
        wid = torch.from_numpy(ids[s:e]).cuda()[:, None].expand(n, cap).reshape(-1)
        cols.append((g64[:, 0][idx], g64[:, 1][idx], conf.reshape(-1)[idx], dets.view(torch.int32)[..., 5].reshape(-1)[idx], wid[idx],
                     slot.reshape(-1)[idx]))
    x, y, conf, cls, wid, slot = (torch.cat(c) for c in zip(*cols))
    keep = eng.dedup(x, y, conf, det.dedup_thr, True, tiebreak=det.order_key(wid, slot)).bool().nonzero().squeeze(1)
    return det._pack(x[keep], y[keep], conf[keep], cls[keep], wid[keep], slot[keep])


def test_mosaic_detector_large_windows_equals_host_letterbox(eng640):
    H, W_ = 2300, 1700
    m = synth.make_mosaic(H, W_, seed=2)
    det = M.MosaicDetector(eng640, GT, win=1200, stride=600, conf=0.3, dedup_thr=1.0)
    got = det.run(torch.from_numpy(m).cuda(), H, W_, 0, 1)
    ref = _host_letterbox_run(det, m, H, W_)
    assert len(got) > 0
    _same_records(got, ref)


@pytest.mark.parametrize("win,stride", [(1200, 600), (480, 400)])
def test_sharded_mosaic_equals_single_rank_any_window(eng640, win, stride):
    """test_sharded_mosaic_equals_single_rank at windows the model does not take as they are: 1, 2 and 3 emulated ranks."""
    H, W_ = 2300, 1700
    mosaic_np = synth.make_mosaic(H, W_, seed=2)
    mosaic = torch.from_numpy(mosaic_np).cuda()
    det = M.MosaicDetector(eng640, GT, win=win, stride=stride, conf=0.3, dedup_thr=1.0)
    single = det.run(mosaic, H, W_, 0, 1)
    assert det.last_raw > len(single) > 0
    key = lambda a: np.sort(a, order=["window", "slot"])
    for world in (2, 3):
        covers = [M.shard_windows(H, W_, r, world, win, stride)[2] for r in range(world)]
        locals_, recs = [], []
        for r in range(world):
            wins, ids, _ = M.shard_windows(H, W_, r, world, win, stride)
            lo, hi = covers[r]
            out = det.detect_windows(mosaic[lo:hi].contiguous(), wins, ids, y_offset=lo)
            loc, rec = det.seam_split(*out, r, covers)
            locals_.append(loc); recs.append(rec)
        origin = np.concatenate([np.full(len(rc), r, np.int64) for r, rc in enumerate(recs)])
        union = np.concatenate([np.concatenate([locals_[r], det.seam_merge(recs, origin, r)]) for r in range(world)])
        assert len(union) == len(single)
        a, b = key(union), key(single)
        _same_records(a, b)
