"""ORACLE (test infrastructure) of the mosaic-wide oriented-box merge (``b2d_mosaic_nms_obb``): the rule of ``include/b2det.h``
restated all-pairs in NumPy / torch fp32, and the neighbour bound of DESIGN.md section 6.

The pair arithmetic is ``_obb_oracle.batch_probiou`` with the centre difference handed in (fp64 difference rounded once to
fp32) and C's ``fmaxf`` / ``fminf`` for the clamp (a NaN sum clamps to eps).  Every division is tensor / tensor: torch divides
a CUDA tensor by a Python scalar through the reciprocal, which is not the kernel's division.
"""
from __future__ import annotations

import math

import numpy as np
import torch

EPS = 1e-7
PROB_BAND = 1e-4          # |ProbIoU - iou_thr| below which the CPU and CUDA libm may decide a pair differently (test_gpu_obb.py)
OBB_FIELDS = ("cx", "cy", "w", "h", "theta", "conf", "cls", "tile", "anchor")


def bound_coef(thr: float) -> float:
    """K of the regular-pair bound: ProbIoU(i, j) >= thr only if |d|^2 <= K (L_i^2 + L_j^2)."""
    u = 2.0 ** -24
    hm = 1.0 - thr + 4 * u
    arg = 1.0 + float(np.float32(EPS)) - hm * hm * (1 + 2 * u) - 8 * u
    bd_lim = min(-math.log(arg), 100.0) if arg > math.exp(-100.0) else 100.0
    return (bd_lim + 1.0 / 16) * 17.0 / 48.0


def gaussian(w: np.ndarray, h: np.ndarray, th: np.ndarray, device="cpu"):
    """(A, B, C, P) fp32 NumPy arrays, as ``obb_gaussian``: cos / sin from torch on ``device`` (CUDA's are the kernel's)."""
    f = np.float32
    t = torch.from_numpy(np.ascontiguousarray(th, dtype=f)).to(device)
    cs, sn = torch.cos(t).cpu().numpy(), torch.sin(t).cpu().numpy()
    with np.errstate(all="ignore"):
        w, h = w.astype(f), h.astype(f)
        a, b = (w * w) / f(12), (h * h) / f(12)
        c2, s2 = cs * cs, sn * sn
        A = a * c2 + b * s2
        B = a * s2 + b * c2
        C = ((a - b) * cs) * sn
        P = np.fmax(A * B - C * C, f(0))
    return A, B, C, P


def probiou(dx, dy, gi, gj):
    """ProbIoU(obb1 = i, obb2 = j) of fp32 tensors (broadcasting), gi / gj = (A, B, C, P)."""
    Ai, Bi, Ci, Pi = gi
    Aj, Bj, Cj, Pj = gj
    eps = torch.tensor(EPS, dtype=torch.float32, device=dx.device)
    a12, b12, c12 = Ai + Aj, Bi + Bj, Ci + Cj
    den = a12 * b12 - c12 * c12
    dene = den + eps
    t1 = ((a12 * (dy * dy) + b12 * (dx * dx)) / dene) * 0.25
    t2 = (((c12 * (-dx)) * dy) / dene) * 0.5
    t3 = torch.log(den / (4.0 * torch.sqrt(Pi * Pj) + eps) + eps) * 0.5
    bd = torch.fmin(torch.fmax((t1 + t2) + t3, eps), torch.tensor(100.0, device=dx.device))
    hd = torch.sqrt((1.0 - torch.exp(-bd)) + eps)
    return 1.0 - hd


def frame(rec: np.ndarray, counts: np.ndarray, params: np.ndarray, conf_thr: float, device="cpu"):
    """Flat per-record merge inputs of ``rec`` (OBB_DTYPE [n, cap]): eligible, X, Y (fp64), w', h' (fp32), the Gaussian, conf, cls."""
    n, cap = rec.shape
    f = np.float32
    r = np.repeat(np.arange(n), cap)
    s = np.tile(np.arange(cap), n)
    d = rec.reshape(-1)
    conf = d["conf"].astype(f)
    with np.errstate(invalid="ignore"):
        elig = (s < np.asarray(counts)[r]) & (conf > f(conf_thr))
    P = params[r]
    padx, pady, gain = P[:, 8].astype(f), P[:, 9].astype(f), P[:, 10].astype(f)
    with np.errstate(all="ignore"):
        cx = (d["cx"].astype(f) - padx) / gain
        cy = (d["cy"].astype(f) - pady) / gain
        w, h = d["w"].astype(f) / gain, d["h"].astype(f) / gain
        X = cx.astype(np.float64) + P[:, 6]
        Y = cy.astype(np.float64) + P[:, 7]
    g = gaussian(w, h, d["theta"], device)
    return dict(elig=elig, X=X, Y=Y, w=w, h=h, g=np.stack(g, 1), conf=conf, cls=d["cls"].astype(np.int64), idx=np.arange(n * cap))


def pair_iou(fr, I: np.ndarray, J: np.ndarray, device="cpu", dev_cache=None):
    """[len(I), len(J)] ProbIoU with the records of I as obb1, from the frame ``fr``."""
    c = dev_cache if dev_cache is not None else _dev(fr, device)
    Ii, Jj = torch.from_numpy(I).to(device), torch.from_numpy(J).to(device)
    dx = (c["X"][Ii][:, None] - c["X"][Jj][None, :]).float()
    dy = (c["Y"][Ii][:, None] - c["Y"][Jj][None, :]).float()
    gi = [c["g"][Ii, q][:, None] for q in range(4)]
    gj = [c["g"][Jj, q][None, :] for q in range(4)]
    with torch.no_grad():
        return probiou(dx, dy, gi, gj)


def _dev(fr, device):
    return {"X": torch.from_numpy(fr["X"]).to(device), "Y": torch.from_numpy(fr["Y"]).to(device), "g": torch.from_numpy(fr["g"]).to(device)}


def priority_order(fr, sel: np.ndarray) -> np.ndarray:
    """Indices of ``sel`` in merge priority: confidence descending (floats compare, +0 == -0), then the lower record index."""
    return sel[np.lexsort((sel, -fr["conf"][sel].astype(np.float64)))]


def merge_oracle(rec, counts, params, conf_thr, iou_thr, device="cpu", chunk=512, band=PROB_BAND):
    """All-pairs statement of the rule.  Returns keep uint8 [n, cap] and near bool [n, cap]: a higher-priority record of the same
    class has |ProbIoU - iou_thr| < band with this one (its fate may differ by an ulp of libm)."""
    n, cap = rec.shape
    fr = frame(rec, counts, params, conf_thr, device)
    c = _dev(fr, device)
    keep = fr["elig"].copy()
    near = np.zeros(n * cap, bool)
    thr = np.float32(iou_thr)
    for k in np.unique(fr["cls"][fr["elig"]]):
        order = priority_order(fr, np.flatnonzero(fr["elig"] & (fr["cls"] == k)))
        m = len(order)
        for j0 in range(0, m, chunk):
            J = order[j0:j0 + chunk]
            I = order[:j0 + len(J)]
            iou = pair_iou(fr, I, J, device, c)
            earlier = torch.arange(len(I), device=device)[:, None] < torch.arange(j0, j0 + len(J), device=device)[None, :]
            sup = ((iou >= float(thr)) & earlier).any(0).cpu().numpy()
            nb = (((iou - float(thr)).abs() < band) & earlier).any(0).cpu().numpy()
            keep[J[sup]] = False
            near[J] |= nb
    return keep.reshape(n, cap).astype(np.uint8), near.reshape(n, cap)


def fate_of(fr, j: int, candidates: np.ndarray, iou_thr: float, device="cpu", dev_cache=None, band=PROB_BAND):
    """(kept, near) of record j against ``candidates`` (a superset of the records that can suppress it)."""
    if not fr["elig"][j]:
        return False, False
    cand = candidates[fr["elig"][candidates] & (fr["cls"][candidates] == fr["cls"][j]) & (candidates != j)]
    cj = fr["conf"][j]
    cand = cand[(fr["conf"][cand] > cj) | ((fr["conf"][cand] == cj) & (cand < j))]
    if not len(cand):
        return True, False
    iou = pair_iou(fr, cand, np.array([j]), device, dev_cache)[:, 0]
    return not bool((iou >= float(np.float32(iou_thr))).any()), bool(((iou - float(np.float32(iou_thr))).abs() < band).any())


def records(n: int, cap: int) -> np.ndarray:
    """A zeroed OBB_DTYPE [n, cap] array."""
    from aerial_image_recognition_b200.engine import OBB_DTYPE
    return np.zeros((n, cap), OBB_DTYPE)


def to_device(rec: np.ndarray, device="cuda"):
    """OBB_DTYPE [n, cap] -> float32 [n, cap, 9] CUDA tensor (the layout Engine.postprocess returns)."""
    n, cap = rec.shape
    return torch.from_numpy(np.ascontiguousarray(rec).view(np.float32).reshape(n, cap, 9).copy()).to(device)
