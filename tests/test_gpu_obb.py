"""GPU tests (-m gpu) of the oriented-box model ``yolov8m-obb``: every planned op against torch, the rotated decode, the ProbIoU
fast NMS and the corner georeferencing against the fp32 oracle (``_obb_oracle.py``), the fp16x2 contract on C2 tiles, batch
invariance, CUDA-graph replay and the refusal of cross-kind calls."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from aerial_image_recognition_b200 import graph as G, synth, weights as W
from _obb_oracle import YoloV8mObbOracle, batch_probiou, rows_adapter, ultralytics_nms_rotated, xywhr2xyxyxyxy
from test_gpu_parity import _check_every_op

ARCH = "yolov8m-obb"
PROB_BAND = 1e-4          # |ProbIoU - iou_thr| below which the fp32 CPU and CUDA libm may decide a pair differently


def _engine(*a, **k):
    from aerial_image_recognition_b200.engine import Engine
    return Engine(*a, **k)


# ---- every op of the graph ------------------------------------------------------------------------------------
@pytest.mark.parametrize("imgsz,n", [(128, 3), (224, 3), (640, 8), (1024, 2)])      # 224: partial tiles; 640 / 8: tiles spanning images
def test_obb_every_planned_op_matches_torch(imgsz, n):
    seen = _check_every_op(ARCH, imgsz, n)
    g = G.build(ARCH, imgsz=imgsz)
    i = next(k for k, op in enumerate(g.ops) if op.weight == "model.22.cv4.0.2")
    print(f"\nangle conv (1 output channel at channel {g.head['angle_c']} of {g.bufs['head0'].c}): {seen[i]}")


def test_obb_every_planned_op_large_batch_kernel_variants(monkeypatch):
    monkeypatch.setenv("B2D_MT", "4")
    monkeypatch.setenv("B2D_PAIR", "2")
    seen = _check_every_op(ARCH, 640, 2)
    assert any("halo-pair" in d for d in seen) and any(" x4 " in d for d in seen), seen[:8]


def test_obb_every_planned_op_split_fp16():
    _check_every_op(ARCH, 320, 2, precision="fp16x2")


# ---- decode --------------------------------------------------------------------------------------------------
def _head_maps(eng, g, n):
    """The engine's head buffers as the oracle's raw maps [n, 64 + nc + 1, h, w] (box | cls | angle)."""
    nc, ac = g.nc, g.head["angle_c"]
    out = []
    for lv in g.head["levels"]:
        b = eng.buffer(lv["buf"], n).cpu()
        out.append(torch.cat([b[..., :64 + nc], b[..., ac:ac + 1]], -1).permute(0, 3, 1, 2).contiguous())
    return out


@pytest.fixture(scope="module")
def obb640():
    g = G.build(ARCH)
    w = W.make_synthetic_weights(g, 0)
    e = _engine(ARCH, weights=w, max_batch=4, graph=g)
    e._weights = w
    yield e
    e.close()


def test_obb_decode_matches_oracle_on_identical_head_maps(obb640):
    g, n = obb640.graph, 4
    obb640.preprocess(torch.from_numpy(synth.make_tiles(n, 640, 21)).cuda(), "identity")
    obb640.forward(n)
    rows = obb640.decode_rows(n).cpu().numpy()
    ref = np.stack([rows_adapter(p) for p in YoloV8mObbOracle.decode(_head_maps(obb640, g, n)).numpy()])
    assert rows.shape == ref.shape == (n, 8400, 7)
    ds = np.abs(rows[..., 4] - ref[..., 4]).max()
    db = np.abs(rows[..., :4] - ref[..., :4]).max()
    dt = np.abs(rows[..., 6] - ref[..., 6]).max()
    print(f"\ndecode vs oracle: |d score| {ds:.2e}, |d box| {db:.2e} px, |d theta| {dt:.2e}; theta range "
          f"[{rows[..., 6].min():.3f}, {rows[..., 6].max():.3f}]")
    assert ds < 1e-6 and db < 2e-2 and dt < 1e-5, (ds, db, dt)
    assert np.array_equal(rows[..., 5], ref[..., 5])
    assert rows[..., 6].min() < -0.5 and rows[..., 6].max() > 2.0          # the calibrated angle branch really rotates boxes


# ---- rotated NMS on identical candidates -----------------------------------------------------------------------
def _synthetic_head(eng, g, n, n_pass, seed, nc_used=3):
    """Write head maps straight into the engine's head buffers: peaked DFL logits (distances 0.5 .. 5 cells, so neighbouring
    anchors form clusters of overlapping boxes), class logits from four values (exact score ties) on `n_pass` anchors per tile
    (the rest below any threshold), angle logits ~ N(0, 1.5)."""
    rng = np.random.default_rng(seed)
    nc, ac = g.nc, g.head["angle_c"]
    A = g.head["anchors_total"]
    ks = np.arange(16, dtype=np.float32)
    passing = [rng.permutation(A)[:n_pass] for _ in range(n)]
    a0 = 0
    for lv in g.head["levels"]:
        hw = lv["hw"]
        m = np.zeros((n, hw * hw, g.bufs[lv["buf"]].c), np.float32)
        d = rng.uniform(0.5, 5.0, (n, hw * hw, 4)).astype(np.float32)
        m[..., :64] = (-2.0 * (ks[None, None, None, :] - d[..., None]) ** 2).reshape(n, hw * hw, 64)
        m[..., 64:64 + nc] = -12.0
        cls = rng.integers(0, nc_used, (n, hw * hw))
        val = rng.choice(np.array([-0.5, 0.0, 0.75, 1.5], np.float32), (n, hw * hw))
        for t in range(n):
            sel = passing[t]
            local = sel[(sel >= a0) & (sel < a0 + hw * hw)] - a0
            m[t, local, 64 + cls[t, local]] = val[t, local]
        m[..., ac] = rng.normal(0.0, 1.5, (n, hw * hw)).astype(np.float32)
        eng.buffer(lv["buf"], n).copy_(torch.from_numpy(m.reshape(n, hw, hw, -1)).cuda())
        a0 += hw * hw
    torch.cuda.synchronize()


def _pred_from_rows(rows, nc):
    """Decoded rows [A, 7] -> the [4 + nc + 1, A] prediction the oracle NMS reads (one-hot class scores: max / argmax = conf / cls)."""
    A = rows.shape[0]
    p = np.zeros((4 + nc + 1, A), np.float32)
    p[:4] = rows[:, :4].T
    p[4 + rows[:, 5].astype(np.int64), np.arange(A)] = rows[:, 4]
    p[-1] = rows[:, 6]
    return p


def _near_threshold_pairs(rows, anchors, iou_thr):
    """ProbIoU (oracle arithmetic, class-offset boxes) between each anchor of `anchors` and every candidate."""
    b = np.concatenate([rows[:, :2] + rows[:, 5:6] * 7680.0, rows[:, 2:4], rows[:, 6:7]], 1).astype(np.float32)
    return batch_probiou(b, b[anchors]).numpy()


@pytest.mark.parametrize("imgsz,n_pass", [(640, 37), (640, 8400), (1024, 21504)])
def test_obb_rotated_nms_matches_oracle(imgsz, n_pass):
    g = G.build(ARCH, imgsz=imgsz)
    n = 2
    eng = _engine(ARCH, weights=W.make_synthetic_weights(g, 0, calibrate=False), max_batch=n, graph=g)
    _synthetic_head(eng, g, n, n_pass, seed=imgsz + n_pass)
    rows = eng.decode_rows(n).cpu().numpy()
    conf_thr, iou_thr = 0.25, 0.7
    from aerial_image_recognition_b200.engine import obbs_to_numpy
    full = obbs_to_numpy(*eng.postprocess(n, conf_thr, False, iou_thr, 0, 30000, cap=30000))
    top = obbs_to_numpy(*eng.postprocess(n, conf_thr, False, iou_thr, 0, 300))
    eng.close()
    flagged = 0
    for t in range(n):
        ref = ultralytics_nms_rotated(_pred_from_rows(rows[t], g.nc)[None], conf_thr, iou_thr, max_det=30000)[0]
        assert (rows[t, :, 4] > conf_thr).sum() == n_pass
        ka, kr = full[t]["anchor"].astype(np.int64), ref[:, 7].astype(np.int64)
        if not np.array_equal(ka, kr):
            diff = np.setxor1d(ka, kr)
            cand = np.nonzero(rows[t, :, 4] > conf_thr)[0]
            pi = _near_threshold_pairs(rows[t][cand], np.searchsorted(cand, diff), iou_thr)
            near = (np.abs(pi - iou_thr) < PROB_BAND).any(0)
            flagged += int(near.sum())
            assert near.all(), (t, diff[~near][:10])
            assert np.array_equal(ka[~np.isin(ka, diff)], kr[~np.isin(kr, diff)])      # the rest, in the same order
        else:
            # regularized records equal the oracle's (same fp32 inputs; theta through fmod)
            assert np.array_equal(full[t]["w"], ref[:, 2]) and np.array_equal(full[t]["h"], ref[:, 3])
            assert np.abs(full[t]["theta"] - ref[:, 4]).max(initial=0) <= 4e-7
            assert np.array_equal(full[t]["conf"], ref[:, 5]) and np.array_equal(full[t]["cls"], ref[:, 6].astype(np.int32))
        assert np.array_equal(top[t]["anchor"], full[t]["anchor"][:300])                # max_det truncates the same list
        print(f"\nA = {rows.shape[1]}, {n_pass} candidates: {len(ka)} kept ({len(top[t])} after max_det 300), classes "
              f"{np.unique(full[t]['cls']).tolist()}, conf ties {len(full[t]) - len(np.unique(full[t]['conf']))}")
    print(f"pairs within {PROB_BAND} of iou_thr that decided a difference: {flagged}")


# ---- the contract on C2 tiles ----------------------------------------------------------------------------------
SCORE_TOL, CORNER_TOL_PX, TIE_BAND, SCORE_FLOOR, PROB_CONTRACT_BAND = 1e-3, 0.5, 2e-3, 0.05, 2e-2


def test_obb_contract_split_fp16_vs_fp32_oracle():
    """fp16x2 against the fp32 oracle at 640 x 640 on C2 tiles: scores within 1e-3, the four corners within 0.5 px (corners do
    not depend on the w / h swap of regularization), keep sets identical outside the score band and the ProbIoU band."""
    g = G.build(ARCH)
    w = W.make_synthetic_weights(g, 0)
    n = 4
    tiles = synth.make_tiles(n, 640, 1000)
    x = torch.from_numpy(tiles.astype(np.float32) / 255.0).permute(0, 3, 1, 2)
    pred = YoloV8mObbOracle(w, False).forward(x).numpy()
    ref = np.stack([rows_adapter(p) for p in pred])
    eng = _engine(ARCH, weights=w, max_batch=n, graph=g, precision="fp16x2")
    dets, counts = eng.infer(torch.from_numpy(tiles).cuda(), "identity", conf_thr=0.25, inclusive=False, iou_thr=0.7, max_det=300)
    rows = eng.decode_rows(n).cpu().numpy()
    eng.close()
    from aerial_image_recognition_b200.engine import obbs_to_numpy
    got = obbs_to_numpy(dets, counts)
    sel = ref[..., 4] >= SCORE_FLOOR
    ds = np.abs(rows[..., 4] - ref[..., 4])[sel]
    cr = lambda r: xywhr2xyxyxyxy(np.concatenate([r[:, :4], r[:, 6:7]], 1))
    dc = np.abs(cr(rows[sel]) - cr(ref[sel])).max((1, 2))
    print(f"\n[obb fp16x2 vs fp32 oracle] {int(sel.sum())} anchors >= {SCORE_FLOOR}: |d score| max {ds.max():.2e}, "
          f"|d corner| max {dc.max():.3f} px, p99 {np.quantile(dc, 0.99):.3f} px")
    assert ds.max() <= SCORE_TOL and dc.max() <= CORNER_TOL_PX, (ds.max(), dc.max())
    explained = total = 0
    for t in range(n):
        kr = ultralytics_nms_rotated(pred[t:t + 1], 0.25, 0.7, 300)[0][:, 7].astype(np.int64)
        ka = got[t]["anchor"].astype(np.int64)
        total += len(kr)
        diff = np.setxor1d(ka, kr)
        if not len(diff):
            continue
        cand = np.nonzero(ref[t, :, 4] > 0.25 - TIE_BAND)[0]
        pi = _near_threshold_pairs(ref[t][cand], np.searchsorted(cand, diff), 0.7)
        sc = ref[t][cand][:, 4]
        for k, a in enumerate(diff):
            near_score = abs(ref[t, a, 4] - 0.25) < TIE_BAND
            near_iou = (np.abs(pi[:, k] - 0.7) < PROB_CONTRACT_BAND).any()
            swap = ((pi[:, k] > 0.7 - PROB_CONTRACT_BAND) & (np.abs(sc - ref[t, a, 4]) < TIE_BAND)).sum() > 1
            assert near_score or near_iou or swap, (t, a, ref[t, a, 4])
            explained += 1
    print(f"keep sets: {explained} anchors of {total} differ, each within the score band {TIE_BAND} or the ProbIoU band {PROB_CONTRACT_BAND}")


# ---- georeferencing ------------------------------------------------------------------------------------------
def _corners_f32(cx, cy, w, h, th):
    """xywhr2xyxyxyxy in fp32 with the device's cos / sin (torch's CUDA kernels call the same precise cosf / sinf)."""
    t = torch.from_numpy(th.astype(np.float32)).cuda()
    cs, sn = torch.cos(t).cpu().numpy(), torch.sin(t).cpu().numpy()
    f = np.float32
    w2, h2n, h2 = w / f(2), -h / f(2), h / f(2)
    v1x, v1y, v2x, v2y = w2 * cs, w2 * sn, h2n * sn, h2 * cs
    px = np.stack([(cx + v1x) + v2x, (cx + v1x) - v2x, (cx - v1x) - v2x, (cx - v1x) + v2x], 1)
    py = np.stack([(cy + v1y) + v2y, (cy + v1y) - v2y, (cy - v1y) - v2y, (cy - v1y) + v2y], 1)
    return px.astype(np.float32), py.astype(np.float32)


def test_obb_georef_bit_exact_against_numpy_float64(obb640):
    from aerial_image_recognition_b200.engine import GEO_PARAMS, geoobbs_to_numpy, obbs_to_numpy
    n = 4
    dets, counts = obb640.infer(torch.from_numpy(synth.make_tiles(n, 640, 33)).cuda(), "identity", conf_thr=0.25, inclusive=False,
                                iou_thr=0.7, max_det=300)
    got = obbs_to_numpy(dets, counts)
    assert sum(len(d) for d in got) > 50
    rng = np.random.default_rng(5)
    P = np.zeros((n, GEO_PARAMS))
    P[:, :6] = np.stack([rng.uniform(20, 21, n), rng.uniform(21.001, 21.01, n), rng.uniform(52, 52.1, n), rng.uniform(52.2, 52.3, n),
                         np.full(n, 864.0), np.full(n, 640.0)], 1)
    bounds = geoobbs_to_numpy(obb640.georef(dets, counts, torch.from_numpy(P).cuda(), "bounds"), counts)
    A = np.zeros((n, GEO_PARAMS))
    A[:, :6] = np.stack([rng.uniform(3e5, 4e5, n), np.full(n, 0.3), rng.uniform(-1e-3, 1e-3, n), rng.uniform(5e6, 6e6, n),
                         rng.uniform(-1e-3, 1e-3, n), np.full(n, -0.3)], 1)
    A[:, 6:11] = np.stack([rng.integers(0, 5000, n), rng.integers(0, 5000, n), rng.integers(0, 80, n), rng.integers(0, 80, n),
                           rng.uniform(0.5, 1.0, n)], 1)
    affine = geoobbs_to_numpy(obb640.georef(dets, counts, torch.from_numpy(A).cuda(), "affine"), counts)
    f = np.float32
    for t in range(n):
        d = got[t]
        # bounds: every point interpolated in float64 (simple_detector.py:487-494)
        px, py = _corners_f32(d["cx"], d["cy"], d["w"], d["h"], d["theta"])
        west, east, south, north, crop, ms = P[t, :6]
        lon = lambda v: west + (v.astype(np.float64) / ms) * (east - west)
        lat = lambda v: north - (v.astype(np.float64) / ms) * (north - south)
        b = bounds[t]
        assert np.array_equal(b["x"], lon(d["cx"])) and np.array_equal(b["y"], lat(d["cy"]))
        assert np.array_equal(b["corners"][..., 0], lon(px)) and np.array_equal(b["corners"][..., 1], lat(py))
        assert np.array_equal(b["w"], ((d["w"].astype(np.float64) / ms) * crop).astype(np.float32))
        assert np.array_equal(b["theta"], d["theta"]) and np.array_equal(b["cls"], d["cls"]) and np.array_equal(b["conf"], d["conf"])
        # affine: letterbox undone in fp32 (no clipping), corners in fp32, offset + geotransform in float64
        gt = A[t, :6]
        padx, pady, gain = f(A[t, 8]), f(A[t, 9]), f(A[t, 10])
        cx, cy = (d["cx"] - padx) / gain, (d["cy"] - pady) / gain
        w, h = d["w"] / gain, d["h"] / gain
        px, py = _corners_f32(cx, cy, w, h, d["theta"])
        X = lambda v: v.astype(np.float64) + A[t, 6]
        Y = lambda v: v.astype(np.float64) + A[t, 7]
        gx = lambda vx, vy: (gt[0] + X(vx) * gt[1]) + Y(vy) * gt[2]
        gy = lambda vx, vy: (gt[3] + X(vx) * gt[4]) + Y(vy) * gt[5]
        a = affine[t]
        assert np.array_equal(a["x"], gx(cx, cy)) and np.array_equal(a["y"], gy(cx, cy))
        assert np.array_equal(a["corners"][..., 0], gx(px, py)) and np.array_equal(a["corners"][..., 1], gy(px, py))
        assert np.array_equal(a["w"], w) and np.array_equal(a["h"], h)
    for mode in ("gpuhandler", "tensor_f32"):
        from aerial_image_recognition_b200._lib import B2DError
        with pytest.raises(B2DError, match="no oriented-box variant"):
            obb640.georef(dets, counts, torch.from_numpy(P).cuda(), mode)


# ---- batch invariance and graph replay ----------------------------------------------------------------------
def test_obb_batch_subsets_and_permutation_bit_identical():
    from aerial_image_recognition_b200.engine import obbs_to_numpy
    g = G.build(ARCH)
    eng = _engine(ARCH, weights=W.make_synthetic_weights(g, 0), max_batch=64, graph=g)
    tiles = torch.from_numpy(synth.make_tiles(64, 640, 55)).cuda()
    run = lambda x: obbs_to_numpy(*eng.infer(x, "identity", conf_thr=0.25, inclusive=False, iou_thr=0.7, max_det=300))
    fields = ("cx", "cy", "w", "h", "theta", "conf", "cls", "anchor")
    same = lambda a, b: all(np.array_equal(a[f], b[f]) for f in fields)
    full = run(tiles)
    assert sum(len(d) for d in full) > 64
    for lo, hi in ((0, 1), (5, 12), (17, 50)):
        sub = run(tiles[lo:hi].contiguous())
        assert all(same(sub[k], full[lo + k]) for k in range(hi - lo)), (lo, hi)
    perm = torch.from_numpy(np.random.default_rng(3).permutation(64))
    pm = run(tiles[perm.cuda()].contiguous())
    assert all(same(pm[k], full[int(perm[k])]) for k in range(64))
    eng.close()


def test_obb_graph_replay_equals_eager_forward(obb640):
    g, n = obb640.graph, 3
    obb640.preprocess(torch.from_numpy(synth.make_tiles(n, 640, 77)).cuda(), "identity")
    maps = []
    for _ in range(3):             # eager, captured + launched, replayed
        for lv in g.head["levels"]:
            obb640.buffer(lv["buf"], n).zero_()
        obb640.forward(n)
        torch.cuda.synchronize()
        maps.append([obb640.buffer(lv["buf"], n).clone() for lv in g.head["levels"]])
    for k in (1, 2):
        assert all(torch.equal(a, b) for a, b in zip(maps[0], maps[k])), k


# ---- cross-kind calls ---------------------------------------------------------------------------------------
def test_obb_and_axis_aligned_entry_points_refuse_the_other_kind(obb640):
    from aerial_image_recognition_b200 import _lib
    from aerial_image_recognition_b200.engine import GEO_PARAMS
    lib = _lib.load()
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    buf = torch.zeros(1 << 20, dtype=torch.float32, device="cuda")
    cnt = torch.ones(4, dtype=torch.int32, device="cuda")
    par = torch.zeros((4, GEO_PARAMS), dtype=torch.float64, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr())
    tiles = torch.zeros((1, 640, 640, 3), dtype=torch.uint8, device="cuda")

    def refused(rc, what):
        assert rc < 0, what
        assert b"oriented-box head" in lib.b2d_last_error(), (what, lib.b2d_last_error())

    aa = _engine("yolov8m", imgsz=128, max_batch=1)
    for e, calls in ((obb640, [("b2d_decode_rows", (1, p(buf), s)),
                               ("b2d_postprocess", (1, 0.25, 0, 0.7, 0, 300, p(buf), p(cnt), 300, s)),
                               ("b2d_postprocess_rows", (p(buf), 1, 100, 6, 0.25, 0, 0.7, 0, 300, p(buf), p(cnt), 300, s)),
                               ("b2d_georef", (p(buf), p(cnt), 1, 10, 0, p(par), p(buf), s)),
                               ("b2d_infer_tiles", (p(tiles), 1, 640, 640, 1920, 640 * 1920, 0, 0, 0.25, 0, 0.7, 0, 300, p(buf), p(cnt), 300, s))]),
                     (aa, [("b2d_decode_rows_obb", (1, p(buf), s)),
                           ("b2d_postprocess_obb", (1, 0.25, 0, 0.7, 0, 300, p(buf), p(cnt), 300, s)),
                           ("b2d_georef_obb", (p(buf), p(cnt), 1, 10, 0, p(par), p(buf), s))])):
        for name, args in calls:
            refused(getattr(lib, name)(e.h, *args), name)
    aa.close()
    from aerial_image_recognition_b200.mosaic import MosaicDetector
    from aerial_image_recognition_b200.session import InferenceSession
    with pytest.raises(ValueError, match="oriented-box"):
        InferenceSession(engine=obb640)
    with pytest.raises(ValueError, match="oriented-box"):
        MosaicDetector(obb640, (0.0, 1.0, 0.0, 0.0, 0.0, -1.0))
    with pytest.raises(_lib.B2DError, match="oriented-box"):
        obb640.detect_host(np.zeros((1, 640, 640, 3), np.uint8), np.zeros((1, GEO_PARAMS)))
