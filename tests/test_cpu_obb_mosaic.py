"""CPU tests of the mosaic-wide oriented-box merge: the all-pairs restatement of its rule (``_obb_merge_oracle``) against
Ultralytics' ``nms_rotated`` run one class at a time, the neighbour bound the kernel's search rests on, and the result layout of
``ObbMosaicDetector``."""
import math

import numpy as np
import torch

from _obb_merge_oracle import bound_coef, merge_oracle, records
from _obb_oracle import batch_probiou, nms_rotated


def _frames(seed, n=12, cap=40, extent=40000, nc=4):
    """Windows of records whose merge-frame centres are multiples of 1/8 px below 2^19 (exact in fp32), gain 1, pad 0."""
    rng = np.random.default_rng(seed)
    rec = records(n, cap)
    params = np.zeros((n, 16))
    params[:, 6] = rng.integers(0, extent - 640, n)
    params[:, 7] = rng.integers(0, extent - 640, n)
    params[:, 10] = 1.0
    # objects shared by several windows: each record is an object seen from one window, with a jitter of a few px
    objs = rng.uniform(0, 640, (60, 2)) + params[rng.integers(0, n, 60), 6:8]
    for r in range(n):
        o = objs[rng.integers(0, len(objs), cap)]
        rec[r]["cx"] = np.round((o[:, 0] - params[r, 6] + rng.normal(0, 3, cap)) * 8) / 8
        rec[r]["cy"] = np.round((o[:, 1] - params[r, 7] + rng.normal(0, 3, cap)) * 8) / 8
    L = np.exp(rng.uniform(np.log(4), np.log(300), rec.shape)).astype(np.float32)
    rec["w"] = L
    rec["h"] = L / rng.uniform(1, 6, rec.shape).astype(np.float32)
    rec["theta"] = rng.uniform(0, np.pi, rec.shape)
    rec["conf"] = rng.choice(np.linspace(0.3, 0.95, 14, dtype=np.float32), rec.shape)       # many exact ties
    rec["cls"] = rng.integers(0, nc, rec.shape)
    counts = rng.integers(cap // 2, cap + 1, n).astype(np.int32)
    return rec, counts, params


def test_restated_rule_equals_nms_rotated_per_class():
    for seed in range(4):
        rec, counts, params = _frames(seed)
        conf_thr, iou_thr = 0.4, [0.3, 0.1, 0.7, 0.5][seed]
        keep, _ = merge_oracle(rec, counts, params, conf_thr, iou_thr)
        n, cap = rec.shape
        flat = rec.reshape(-1)
        k = np.arange(n * cap)
        elig = (k % cap < counts[k // cap]) & (flat["conf"] > np.float32(conf_thr))
        X = flat["cx"] + params[k // cap, 6]
        Y = flat["cy"] + params[k // cap, 7]
        assert np.array_equal(X.astype(np.float32), X) and np.array_equal(Y.astype(np.float32), Y)
        ref = np.zeros(n * cap, bool)
        for c in np.unique(flat["cls"][elig]):
            sel = np.flatnonzero(elig & (flat["cls"] == c))                 # ascending record index: the stable sort's tie rule
            boxes = torch.from_numpy(np.stack([X[sel], Y[sel], flat["w"][sel], flat["h"][sel], flat["theta"][sel]], 1).astype(np.float32))
            ref[sel[nms_rotated(boxes, torch.from_numpy(flat["conf"][sel]), iou_thr).numpy()]] = True
        assert np.array_equal(keep.reshape(-1).astype(bool), ref), (seed, np.flatnonzero(keep.reshape(-1).astype(bool) != ref)[:10])
        assert 0 < ref.sum() < elig.sum()             # the merge really suppresses, and keeps


def _pairs_for(rng, Li, hi, thr, m):
    """m partners of a box with long side Li and short side hi: random and adversarial (needles along d, equal boxes)."""
    Lj = np.exp(rng.uniform(0, np.log(2000), m))
    Lj[: m // 4] = Li                                                        # same size
    rho = np.exp(rng.uniform(0, np.log(128), m))
    hj = np.maximum(1.0, Lj / rho)
    hj = np.minimum(hj, Lj)
    hj[: m // 8] = np.maximum(1.0, Lj[: m // 8] / 128)                       # the thinnest regular boxes
    R = np.sqrt(bound_coef(thr) * (Li ** 2 + Lj ** 2))
    dist = R * rng.uniform(0, 1.3, m)
    dist[m // 2: m // 2 + m // 8] = R[m // 2: m // 2 + m // 8] * rng.uniform(0.98, 1.02, m // 8)
    phi = rng.uniform(0, np.pi, m)
    aligned = rng.random(m) < 0.5                                            # long axes of both along d
    thj = np.where(aligned, phi, rng.uniform(0, np.pi, m))
    return Lj, hj, thj, dist, phi, aligned


def test_regular_pair_bound_holds_in_fp32_probiou():
    rng = np.random.default_rng(7)
    checked = inside = 0
    worst = 0.0
    for trial in range(240):
        thr = float(rng.uniform(0.05, 0.95))
        Li = float(np.exp(rng.uniform(0, np.log(2000))))
        hi = max(1.0, Li / float(np.exp(rng.uniform(0, np.log(128)))))
        m = 512
        Lj, hj, thj, dist, phi, aligned = _pairs_for(rng, Li, hi, thr, m)
        thi = float(rng.uniform(0, np.pi))
        xi, yi = float(rng.uniform(0, 40000)), float(rng.uniform(0, 40000))
        thi_row = np.where(aligned, phi, thi)
        # one obb1 per distinct orientation would be [m, m]; instead each pair is its own 1 x 1 product, batched as m x m diag
        ob1 = np.stack([np.full(m, xi), np.full(m, yi), np.full(m, Li), np.full(m, hi), thi_row], 1).astype(np.float32)
        ob2 = np.stack([xi + dist * np.cos(phi), yi + dist * np.sin(phi), Lj, hj, thj], 1).astype(np.float32)
        iou = torch.diagonal(batch_probiou(ob1, ob2)).numpy()
        d = ob2[:, :2].astype(np.float64) - ob1[:, :2].astype(np.float64)
        d2 = (d ** 2).sum(1)
        lim = bound_coef(thr) * (ob1[:, 2].astype(np.float64) ** 2 + ob2[:, 2].astype(np.float64) ** 2)
        hit = iou >= np.float32(thr)
        assert (d2[hit] <= lim[hit]).all(), (trial, thr, Li, hi, np.flatnonzero(hit & (d2 > lim))[:5])
        checked += m
        inside += int(hit.sum())
        if hit.any():
            worst = max(worst, float(np.sqrt(d2[hit] / lim[hit]).max()))
    assert inside > 1000
    print(f"\n{checked} regular pairs, {inside} with ProbIoU >= thr; largest |d| / bound radius among them {worst:.3f}")


def test_bound_coefficient_at_the_dota_merge_threshold():
    # exact arithmetic: |d| <= sqrt(2 bd* / 3) max(L_i, L_j) = 0.67 max(L_i, L_j) at thr 0.3; the fp32 margins widen it to 0.72
    bd = -math.log(1 + 1e-7 - 0.7 ** 2)
    assert 0.66 < math.sqrt(2 * bd / 3) < 0.68
    assert math.sqrt(2 * bd / 3) < math.sqrt(2 * bound_coef(0.3)) < 0.73
    assert all(bound_coef(a) > bound_coef(b) for a, b in ((0.05, 0.3), (0.3, 0.7), (0.7, 0.95)))


def test_obb_mosaic_result_layout_relabels_geoobb_records():
    from aerial_image_recognition_b200.engine import GEOOBB_DTYPE
    from aerial_image_recognition_b200.mosaic import ObbMosaicDetector
    out = ObbMosaicDetector.OUT_DTYPE
    for name in ("x", "y", "corners", "conf", "w", "h", "theta", "cls"):
        assert out.fields[name] == GEOOBB_DTYPE.fields[name], name
    assert out.fields["window"][0] == np.dtype("<i8") and out.fields["slot"][0] == np.dtype("<i4")
    assert out.itemsize == 112 and out.fields["window"][1] % 8 == 0
