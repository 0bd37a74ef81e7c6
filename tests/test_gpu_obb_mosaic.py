"""GPU tests (-m gpu) of the mosaic-wide oriented-box merge (``b2d_mosaic_nms_obb``, ``ObbMosaicDetector``): the kernel against
the all-pairs statement of its rule (``_obb_merge_oracle``) on constructed record sets, at C4 scale against a k-d-tree oracle,
the detector end to end against separate steps, and the refusals."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from _obb_merge_oracle import PROB_BAND, _dev, bound_coef, fate_of, frame, merge_oracle, records, to_device

ARCH = "yolov8m-obb"
CONF_THR = 0.4
GT = (2335637.62, 0.1, 0.0, 6845688.78, 0.0, -0.1)


@pytest.fixture(scope="module")
def obb():
    from aerial_image_recognition_b200 import graph as G, weights as W
    from aerial_image_recognition_b200.engine import Engine
    g = G.build(ARCH)
    e = Engine(ARCH, weights=W.make_synthetic_weights(g, 0), max_batch=8, graph=g)
    yield e
    e.close()


def _place(rec, counts, params, r, boxes):
    """Append merge-frame boxes (X, Y, w', h', theta, conf, cls) to window r as the model-input records that map onto them."""
    f = np.float32
    s0 = counts[r]
    m = min(len(boxes), rec.shape[1] - s0)
    b = boxes[:m]
    gain, padx, pady = params[r, 10], params[r, 8], params[r, 9]
    sl = slice(s0, s0 + m)
    with np.errstate(all="ignore"):
        rec[r, sl]["cx"] = ((b[:, 0] - params[r, 6]) * gain + padx).astype(f)
        rec[r, sl]["cy"] = ((b[:, 1] - params[r, 7]) * gain + pady).astype(f)
        rec[r, sl]["w"] = (b[:, 2] * gain).astype(f)
        rec[r, sl]["h"] = (b[:, 3] * gain).astype(f)
    rec[r, sl]["theta"] = b[:, 4]
    rec[r, sl]["conf"] = b[:, 5]
    rec[r, sl]["cls"] = b[:, 6].astype(np.int32)
    rec[r, sl]["anchor"] = np.arange(s0, s0 + m)
    counts[r] += m


def _constructed(seed, clusters=40, cap=256, extent=40000.0, nc=15):
    """~20 k records: clusters of 2 x 2 overlapping windows (640 / 512 at gain 1, or 1024 / 824 resampled at gain 0.625) placed
    in a 40 000 px frame, objects seen by every window of their cluster that contains them; 15 classes, confidences from a few
    values (ties across windows and slots) including CONF_THR itself, sides 1 to 1 800 px; pairs just inside and just outside
    the bound radius; and zero-area, needle, tiny, huge, out-of-range and non-finite records far apart."""
    rng = np.random.default_rng(seed)
    n = 4 * clusters + 1
    rec = records(n, cap)
    # slots past counts hold garbage that must be ignored
    for name in ("cx", "cy", "w", "h", "theta", "conf"):
        rec[name] = rng.uniform(-5, 700, rec.shape).astype(np.float32)
    rec["cls"] = rng.integers(0, nc, rec.shape)
    counts = np.zeros(n, np.int32)
    params = np.zeros((n, 16))
    params[:, :6] = GT
    confs = np.array([CONF_THR, 0.45, 0.5, 0.6, 0.75, 0.9], np.float32)
    for c in range(clusters):
        gain = 1.0 if c % 2 == 0 else 0.625
        win, stride = (640, 512) if gain == 1.0 else (1024, 824)
        ox, oy = rng.uniform(0, extent - win - stride, 2).round()
        ws = range(4 * c, 4 * c + 4)
        for q, r in enumerate(ws):
            params[r, 6], params[r, 7] = ox + stride * (q % 2), oy + stride * (q // 2)
            params[r, 8], params[r, 9] = rng.integers(0, 3, 2)
            params[r, 10] = gain
        m = 360
        L = np.exp(rng.uniform(0, np.log(1800), m))
        small = rng.random(m) < 0.7
        L[small] = np.exp(rng.uniform(np.log(8), np.log(120), int(small.sum())))
        h = np.maximum(1.0, L / np.exp(rng.uniform(0, np.log(200), m)))
        X = ox + rng.uniform(0, win + stride, m)
        Y = oy + rng.uniform(0, win + stride, m)
        objs = np.stack([X, Y, L, h, rng.uniform(0, np.pi, m), rng.choice(confs, m), rng.integers(0, nc, m)], 1)
        # pairs at the bound radius: two boxes of one class, long axes along d, at R (1 -+ 1e-3)
        for _ in range(6):
            Li = float(np.exp(rng.uniform(np.log(4), np.log(600))))
            hi = max(1.0, Li / float(rng.uniform(1, 128)))
            thr = 0.3
            R = math.sqrt(bound_coef(thr) * 2 * Li * Li)
            phi = float(rng.uniform(0, np.pi))
            x0, y0 = ox + rng.uniform(100, win), oy + rng.uniform(100, win)
            for fct in (1 - 1e-3, 1 + 1e-3):
                objs = np.concatenate([objs, [[x0, y0, Li, hi, phi, 0.9, 3], [x0 + fct * R * math.cos(phi), y0 + fct * R * math.sin(phi), Li, hi, phi, 0.75, 3]]])
        for r in ws:
            lo_x, lo_y = params[r, 6], params[r, 7]
            inside = (objs[:, 0] >= lo_x) & (objs[:, 0] < lo_x + win) & (objs[:, 1] >= lo_y) & (objs[:, 1] < lo_y + win)
            o = objs[inside].copy()
            o[:, :2] += rng.normal(0, 1.0, (len(o), 2))                  # each window sees the object a little differently
            o[:, 2:4] *= rng.uniform(0.97, 1.03, (len(o), 1))
            o[:, 4] += rng.normal(0, 0.02, len(o))
            _place(rec, counts, params, r, o)
    # degenerate records, far apart, in the last window (and a few in the others): brute force decides them all
    last = n - 1
    params[last, 6], params[last, 7], params[last, 10] = 0.0, 0.0, 1.0
    inf, nan = np.inf, np.nan
    deg = [[500, 500, 0, 0, 0, 0.9, 5], [39000, 39000, 0, 0, 0, 0.8, 5],            # zero-area, kilometres apart
           [1000, 30000, 500, 0.01, 0.3, 0.9, 6], [30000, 1000, 800, 0.01, 1.2, 0.7, 6],  # needles
           [2000, 2000, 0.5, 0.5, 0, 0.9, 7], [2001, 2000.4, 0.5, 0.5, 0, 0.6, 7],       # sub-pixel boxes
           [20000, 20000, 6000, 3000, 0.4, 0.6, 8], [23000, 21000, 5000, 4000, 0.1, 0.9, 8],  # beyond the grid's reach
           [nan, 100, 10, 5, 0, 0.95, 9], [100, 100, 10, 5, 0, 0.5, 9], [5000, 5000, inf, 5, 0, 0.9, 9],
           [7000, 7000, 10, 5, nan, 0.9, 9], [8000, 8000, 10, 5, inf, 0.8, 9], [9000, 9000, -4, 3, 0.2, 0.85, 9],
           [inf, 9000, 10, 5, 0, 0.7, 10], [3000, 3000, 10, 5, 0, inf, 10], [3000, 3000, 10, 5, 0, 0.5, 10],
           [2.5e9, 100, 10, 5, 0, 0.8, 11], [2.5e9 + 3, 100, 10, 5, 0, 0.7, 11], [150, 150, 10, 5, 0, 0.6, 11]]
    _place(rec, counts, params, last, np.asarray(deg, np.float64))
    for r in rng.choice(n - 1, 6, replace=False):
        _place(rec, counts, params, r, np.array([[rng.uniform(0, extent), rng.uniform(0, extent), 0, 0, 0, 0.55, 12],
                                                 [rng.uniform(0, extent), rng.uniform(0, extent), 300, 0.001, 0.7, 0.65, 12]]))
    return rec, counts, params


def _kernel_keep(eng, rec, counts, params, conf_thr, iou_thr):
    keep = eng.mosaic_nms_obb(to_device(rec), torch.from_numpy(counts).cuda(), torch.from_numpy(params).cuda(), conf_thr, iou_thr)
    torch.cuda.synchronize()
    return keep.cpu().numpy()


@pytest.mark.parametrize("seed,iou_thr", [(0, 0.3), (1, 0.3), (2, 0.1), (3, 0.7)])
def test_merge_kernel_matches_all_pairs_oracle(obb, seed, iou_thr):
    rec, counts, params = _constructed(seed)
    got = _kernel_keep(obb, rec, counts, params, CONF_THR, iou_thr)
    ref, near = merge_oracle(rec, counts, params, CONF_THR, iou_thr, device="cuda")
    diff = got != ref
    elig = int(frame(rec, counts, params, CONF_THR)["elig"].sum())
    print(f"\n{int(counts.sum())} records, {elig} eligible, {int(ref.sum())} kept by the oracle, {int(got.sum())} by the kernel; "
          f"{int(diff.sum())} differ, all within {PROB_BAND} of iou_thr; {int(near.sum())} records have such a pair")
    assert not (diff & ~near).any(), np.argwhere(diff & ~near)[:10]
    assert 0 < ref.sum() < elig
    assert np.array_equal(got, _kernel_keep(obb, rec, counts, params, CONF_THR, iou_thr))
    # the degenerate window: zero-area boxes kilometres apart suppress each other, as brute force says
    last = len(counts) - 1
    assert ref[last, 0] == 1 and ref[last, 1] == 0 and got[last, 1] == 0


def _c4_records(seed=11, cap=300):
    """C4 scale: the 79 x 79 grid of 640 / 512 windows over 40 000 px, ~1.2 M objects each seen by every window containing it
    (about 1.9 M records, at most 300 per window), sides mostly 8 - 120 px plus some up to 1 800 px, and a few irregular ones."""
    from aerial_image_recognition_b200 import mosaic as M
    rng = np.random.default_rng(seed)
    H = W = 40000
    win = M.window_grid(H, W, 640, 512)
    rows, cols = M.grid_shape(H, W, 512)
    n = len(win)
    params = M.affine_params(win, GT, 640)
    m = 1_200_000
    X, Y = rng.uniform(0, W, m), rng.uniform(0, H, m)
    L = np.exp(rng.uniform(np.log(8), np.log(120), m))
    big = rng.random(m) < 2e-4
    L[big] = rng.uniform(300, 1800, int(big.sum()))
    h = np.maximum(1.0, L / rng.uniform(1, 8, m))
    th = rng.uniform(0, np.pi, m)
    conf = rng.choice(np.linspace(0.3, 0.95, 27, dtype=np.float32), m)
    cls = rng.integers(0, 15, m)
    obj, wid = [], []
    ix, iy = (X // 512).astype(np.int64), (Y // 512).astype(np.int64)
    for dx in (0, -1):
        for dy in (0, -1):
            cx, cy = ix + dx, iy + dy
            ok = (cx >= 0) & (cy >= 0) & (cx < cols) & (cy < rows) & (X - 512 * cx < 640) & (Y - 512 * cy < 640)
            obj.append(np.flatnonzero(ok))
            wid.append((cy * cols + cx)[ok])
    obj, wid = np.concatenate(obj), np.concatenate(wid)
    o = np.lexsort((obj, wid))
    obj, wid = obj[o], wid[o]
    start = np.searchsorted(wid, np.arange(n))
    slot = np.arange(len(wid)) - start[wid]
    sel = slot < cap
    obj, wid, slot = obj[sel], wid[sel], slot[sel]
    rec = records(n, cap)
    f = np.float32
    jit = rng.normal(0, 0.7, (len(obj), 2))
    rec["cx"][wid, slot] = (X[obj] + jit[:, 0] - params[wid, 6] + params[wid, 8]).astype(f)
    rec["cy"][wid, slot] = (Y[obj] + jit[:, 1] - params[wid, 7] + params[wid, 9]).astype(f)
    rec["w"][wid, slot] = L[obj].astype(f)
    rec["h"][wid, slot] = h[obj].astype(f)
    rec["theta"][wid, slot] = th[obj].astype(f)
    rec["conf"][wid, slot] = conf[obj]
    rec["cls"][wid, slot] = cls[obj]
    counts = np.bincount(wid, minlength=n).astype(np.int32)
    # irregular records: zero-area, needles and a non-finite one in the first windows' last slots
    for r in range(12):
        s = counts[r]
        if s < cap:
            rec[r, s] = (rng.uniform(0, 640), rng.uniform(0, 640), [0, 400, np.nan][r % 3], [0, 0.02, 4][r % 3], 0.5, 0.8, r % 15 if r % 3 else 1, 0, s)
            counts[r] += 1
    return rec, counts, params


def test_merge_kernel_at_c4_scale_against_kdtree_oracle(obb):
    from scipy.spatial import cKDTree
    rec, counts, params = _c4_records()
    total = int(counts.sum())
    assert total > 1_800_000
    d, c, p = to_device(rec), torch.from_numpy(counts).cuda(), torch.from_numpy(params).cuda()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    k1 = obb.mosaic_nms_obb(d, c, p, CONF_THR, 0.3)
    e0.record()
    k2 = obb.mosaic_nms_obb(d, c, p, CONF_THR, 0.3)
    e1.record()
    torch.cuda.synchronize()
    assert torch.equal(k1, k2)
    keep = k1.cpu().numpy().reshape(-1)
    fr = frame(rec, counts, params, CONF_THR, "cuda")
    cache = _dev(fr, "cuda")
    Lw = np.maximum(fr["w"], fr["h"])           # NaN propagates: a NaN side makes the record irregular
    sh = np.minimum(fr["w"], fr["h"])
    with np.errstate(invalid="ignore"):
        regular = (fr["elig"] & np.isfinite(fr["X"]) & np.isfinite(fr["Y"]) & np.isfinite(Lw) & np.isfinite(rec["theta"].reshape(-1))
                   & (sh >= 1) & (Lw <= 128 * sh) & (Lw <= 2000))
    irregular = np.flatnonzero(fr["elig"] & ~regular)
    reg = np.flatnonzero(regular)
    Lmax = float(Lw[reg].max())
    tree = cKDTree(np.stack([fr["X"][reg], fr["Y"][reg]], 1))
    K = bound_coef(0.3)
    rng = np.random.default_rng(2)
    sample = rng.choice(np.flatnonzero(fr["elig"]), 2000, replace=False)
    mism = near_n = 0
    for j in sample:
        if regular[j]:          # the bound holds for regular pairs only: any other partner of j is a candidate
            cand = reg[tree.query_ball_point([fr["X"][j], fr["Y"][j]], 2 * math.sqrt(K * (float(Lw[j]) ** 2 + Lmax ** 2)))]
        else:
            cand = reg
        kept, near = fate_of(fr, int(j), np.concatenate([cand, irregular]), 0.3, "cuda", cache)
        near_n += near
        if bool(keep[j]) != kept:
            mism += 1
            assert near, (int(j), kept)
    print(f"\n{total} records, {int(fr['elig'].sum())} eligible, {int(keep.sum())} kept, {len(irregular)} irregular; "
          f"merge {e0.elapsed_time(e1):.2f} ms; sample of 2000: {mism} differ within the band ({near_n} have a pair in it)")


# ---- end to end ---------------------------------------------------------------------------------------------------
def _corners_f32(cx, cy, w, h, th):
    t = torch.from_numpy(th.astype(np.float32)).cuda()
    cs, sn = torch.cos(t).cpu().numpy(), torch.sin(t).cpu().numpy()
    f = np.float32
    w2, h2n, h2 = w / f(2), -h / f(2), h / f(2)
    v1x, v1y, v2x, v2y = w2 * cs, w2 * sn, h2n * sn, h2 * cs
    px = np.stack([(cx + v1x) + v2x, (cx + v1x) - v2x, (cx - v1x) - v2x, (cx - v1x) + v2x], 1)
    py = np.stack([(cy + v1y) + v2y, (cy + v1y) - v2y, (cy - v1y) - v2y, (cy - v1y) + v2y], 1)
    return px.astype(np.float32), py.astype(np.float32)


@pytest.mark.parametrize("H,W,win,stride", [(1300, 1500, 640, 512), (1700, 1900, 1024, 824)])
def test_obb_mosaic_detector_equals_separate_steps(obb, H, W, win, stride):
    from aerial_image_recognition_b200 import mosaic as M, synth
    from aerial_image_recognition_b200.engine import OBB_DTYPE
    conf, merge_iou = 0.3, 0.3
    mos = torch.from_numpy(synth.make_mosaic(H, W, seed=3)).cuda()
    det = M.ObbMosaicDetector(obb, GT, win=win, stride=stride, conf=conf, merge_iou=merge_iou)
    out = det.run(mos, H, W)
    windows = M.window_grid(H, W, win, stride)
    params = M.affine_params(windows, GT, win, obb.imgsz if win != obb.imgsz else None)
    recs, cnts = [], []
    for i in range(len(windows)):
        if win == obb.imgsz:
            tile = obb.cut_windows(mos, torch.from_numpy(windows[i:i + 1]).cuda(), win, 114)
        else:
            tile = obb.resize_windows(mos, windows[i:i + 1], win, 114, out="u8")
        dets, counts = obb.infer(tile, "identity", False, 0.25, False, 0.7, 0, 300)
        recs.append(dets.cpu().numpy().view(np.uint8).reshape(1, dets.shape[1], 36).view(OBB_DTYPE)[..., 0])
        cnts.append(counts.cpu().numpy())
    rec, counts = np.concatenate(recs), np.concatenate(cnts)
    keep, near = merge_oracle(rec, counts, params, conf, merge_iou, device="cuda")
    n, cap = rec.shape
    got_ids = out["window"] * cap + out["slot"]
    exp_ids = np.flatnonzero(keep.reshape(-1))
    assert np.all(np.diff(got_ids) > 0)
    diff = np.setxor1d(got_ids, exp_ids)
    assert near.reshape(-1)[diff].all(), diff[:10]
    both = np.intersect1d(got_ids, exp_ids)
    print(f"\n{len(windows)} windows, {det.last_raw} records with conf > {conf}, {len(out)} after the merge, {len(diff)} differ in the band")
    assert len(both) > 20 and det.last_raw > len(out)
    g = out[np.isin(got_ids, both)]
    d = rec.reshape(-1)[both]
    r = both // cap
    f = np.float32
    padx, pady, gain = params[r, 8].astype(f), params[r, 9].astype(f), params[r, 10].astype(f)
    cx, cy = (d["cx"] - padx) / gain, (d["cy"] - pady) / gain
    w, h = d["w"] / gain, d["h"] / gain
    px, py = _corners_f32(cx, cy, w, h, d["theta"])
    gt = np.asarray(GT)
    X = lambda v: v.astype(np.float64) + params[r, 6][:, None] if v.ndim == 2 else v.astype(np.float64) + params[r, 6]
    Y = lambda v: v.astype(np.float64) + params[r, 7][:, None] if v.ndim == 2 else v.astype(np.float64) + params[r, 7]
    gx = lambda vx, vy: (gt[0] + X(vx) * gt[1]) + Y(vy) * gt[2]
    gy = lambda vx, vy: (gt[3] + X(vx) * gt[4]) + Y(vy) * gt[5]
    assert np.array_equal(g["x"], gx(cx, cy)) and np.array_equal(g["y"], gy(cx, cy))
    assert np.array_equal(g["corners"][..., 0], gx(px, py)) and np.array_equal(g["corners"][..., 1], gy(px, py))
    assert np.array_equal(g["w"], w) and np.array_equal(g["h"], h) and np.array_equal(g["theta"], d["theta"])
    assert np.array_equal(g["conf"], d["conf"]) and np.array_equal(g["cls"], d["cls"])
    assert np.array_equal(g["window"], r) and np.array_equal(g["slot"], both % cap)


# ---- refusals -----------------------------------------------------------------------------------------------------
def test_merge_refuses_axis_aligned_engines_bad_thresholds_and_overflow(obb):
    from aerial_image_recognition_b200 import _lib
    from aerial_image_recognition_b200.engine import Engine
    from aerial_image_recognition_b200.mosaic import ObbMosaicDetector
    lib = _lib.load()
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    rec, counts, params = records(2, 8), np.zeros(2, np.int32), np.zeros((2, 16))
    d, c, p = to_device(rec), torch.from_numpy(counts).cuda(), torch.from_numpy(params).cuda()
    aa = Engine("yolov8m", imgsz=128, max_batch=1)
    with pytest.raises(_lib.B2DError, match="oriented-box head"):
        aa.mosaic_nms_obb(d, c, p, 0.4, 0.3)
    with pytest.raises(ValueError, match="oriented-box engine"):
        ObbMosaicDetector(aa, GT)
    aa.close()
    for thr in (0.0, 1.0, -0.2, 1.5, float("nan")):
        with pytest.raises(_lib.B2DError, match="outside"):
            obb.mosaic_nms_obb(d, c, p, 0.4, thr)
    ptr = lambda t: C.c_void_p(t.data_ptr())
    rc = lib.b2d_mosaic_nms_obb(obb.h, ptr(d), ptr(c), ptr(p), 1 << 16, 1 << 15, 0.4, 0.3, ptr(d), s)
    assert rc < 0 and b"exceed" in lib.b2d_last_error()
    # the engine still merges after the refusals
    assert obb.mosaic_nms_obb(d, c, p, 0.4, 0.3).sum().item() == 0
