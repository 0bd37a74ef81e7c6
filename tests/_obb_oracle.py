"""ORACLE (test infrastructure) for the oriented-box model ``yolov8m-obb``: a conventionally written PyTorch fp32 CPU network
(NCHW, explicit ``torch.cat``) and the Ultralytics >= 8.1 [EXT] oriented-box post-processing restated from its published
semantics -- ``OBB.forward`` + ``dist2rbox``, ``non_max_suppression(rotated=True)`` -> ``nms_rotated`` -> ``batch_probiou``,
``regularize_rboxes`` and ``xywhr2xyxyxyxy``.  No Ultralytics is installed to check against; the hand cases in
``test_cpu_obb.py`` pin the arithmetic.  It is independent of the engine's offset-write graph (``graph.build_yolov8m_obb``).
"""
from __future__ import annotations

import math
from typing import List

import numpy as np
import torch
import torch.nn.functional as F

from oracle.yolo_torch import YoloV8mOracle

EPS = 1e-7
MAX_WH = 7680


class YoloV8mObbOracle(YoloV8mOracle):
    """YOLOv8m backbone / neck + the OBB head (dense cls branch, angle branch cv4), deploy (BN-folded) form."""

    def neck(self, x):
        x0 = self.conv("model.0", x, 3, 2)
        x1 = self.conv("model.1", x0, 3, 2)
        x2 = self.c2f("model.2", x1, 2, True)
        x3 = self.conv("model.3", x2, 3, 2)
        x4 = self.c2f("model.4", x3, 4, True)
        x5 = self.conv("model.5", x4, 3, 2)
        x6 = self.c2f("model.6", x5, 4, True)
        x7 = self.conv("model.7", x6, 3, 2)
        x8 = self.c2f("model.8", x7, 2, True)
        x9 = self.sppf("model.9", x8)
        x12 = self.c2f("model.12", torch.cat([F.interpolate(x9, scale_factor=2, mode="nearest"), x6], 1), 2, False)
        x15 = self.c2f("model.15", torch.cat([F.interpolate(x12, scale_factor=2, mode="nearest"), x4], 1), 2, False)
        x18 = self.c2f("model.18", torch.cat([self.conv("model.16", x15, 3, 2), x12], 1), 2, False)
        x21 = self.c2f("model.21", torch.cat([self.conv("model.19", x18, 3, 2), x9], 1), 2, False)
        return x15, x18, x21

    def branch(self, name, f):
        y = self.conv(f"{name}.0", f, 3)
        y = self.conv(f"{name}.1", y, 3)
        return self.conv(f"{name}.2", y, 1, act=False, out_f32=True)

    @torch.no_grad()
    def raw_head(self, x: torch.Tensor) -> List[torch.Tensor]:
        """x: [B,3,H,W] fp32 in [0,1].  Returns per level [B, 64 + nc + 1, h, w] fp32 raw (box DFL logits | cls logits | angle logit)."""
        feats = self.neck(x)
        ang = [self.branch(f"model.22.cv4.{i}", f) for i, f in enumerate(feats)]
        return [torch.cat([self.branch(f"model.22.cv2.{i}", f), self.branch(f"model.22.cv3.{i}", f), ang[i]], 1)
                for i, f in enumerate(feats)]

    @staticmethod
    def decode(raw: List[torch.Tensor], strides=(8, 16, 32)) -> torch.Tensor:
        """``OBB.forward`` inference path -> [B, 4 + nc + 1, A]: cx, cy, w, h, class sigmoids, theta."""
        B, no = raw[0].shape[:2]
        x_cat = torch.cat([r.reshape(B, no, -1) for r in raw], 2)
        box, cls, angle = x_cat[:, :64], x_cat[:, 64:no - 1], x_cat[:, no - 1:]
        angle = (angle.sigmoid() - 0.25) * math.pi
        anchors, svec = [], []
        for r, s in zip(raw, strides):
            h, w = r.shape[2:]
            yy, xx = torch.meshgrid(torch.arange(h, dtype=torch.float32) + 0.5, torch.arange(w, dtype=torch.float32) + 0.5, indexing="ij")
            anchors.append(torch.stack((xx, yy), -1).view(-1, 2))
            svec.append(torch.full((h * w, 1), float(s)))
        anchors = torch.cat(anchors).transpose(0, 1)
        svec = torch.cat(svec).transpose(0, 1)
        b, _, a = box.shape
        dist = box.view(b, 4, 16, a).transpose(2, 1).softmax(1)
        dist = (dist * torch.arange(16, dtype=torch.float32).view(1, 16, 1, 1)).sum(1)      # the DFL conv
        # dist2rbox
        lt, rb = dist.split(2, dim=1)
        cos, sin = torch.cos(angle), torch.sin(angle)
        xf, yf = ((rb - lt) / 2).split(1, dim=1)
        x, y = xf * cos - yf * sin, xf * sin + yf * cos
        xy = torch.cat([x, y], dim=1) + anchors.unsqueeze(0)
        dbox = torch.cat([xy, lt + rb], dim=1) * svec
        return torch.cat((dbox, cls.sigmoid(), angle), 1)

    @torch.no_grad()
    def forward(self, x):
        return self.decode(self.raw_head(x))


def rows_adapter(pred_b: np.ndarray) -> np.ndarray:
    """[4 + nc + 1, A] -> [A, 7] rows (cx, cy, w, h, conf = max class, cls, theta): the layout of ``Engine.decode_rows`` on an OBB engine."""
    cls = pred_b[4:-1]
    return np.concatenate([pred_b[:4].T, cls.max(0)[:, None], cls.argmax(0)[:, None].astype(np.float32), pred_b[-1:].T], 1)


# ---- ProbIoU and rotated NMS ---------------------------------------------------------------------------------
def _covariance(boxes: torch.Tensor):
    gbbs = torch.cat((boxes[:, 2:4].pow(2) / 12, boxes[:, 4:]), dim=-1)
    a, b, c = gbbs.split(1, dim=-1)
    cos, sin = c.cos(), c.sin()
    cos2, sin2 = cos.pow(2), sin.pow(2)
    return a * cos2 + b * sin2, a * sin2 + b * cos2, (a - b) * cos * sin


def batch_probiou(obb1, obb2, eps: float = EPS) -> torch.Tensor:
    """Ultralytics ``batch_probiou``: [N, 5] x [M, 5] (cx, cy, w, h, theta) -> [N, M] probabilistic IoU, fp32."""
    obb1 = torch.as_tensor(obb1, dtype=torch.float32)
    obb2 = torch.as_tensor(obb2, dtype=torch.float32)
    x1, y1 = obb1[..., :2].split(1, dim=-1)
    x2, y2 = (x.squeeze(-1)[None] for x in obb2[..., :2].split(1, dim=-1))
    a1, b1, c1 = _covariance(obb1)
    a2, b2, c2 = (x.squeeze(-1)[None] for x in _covariance(obb2))
    t1 = (((a1 + a2) * (y1 - y2).pow(2) + (b1 + b2) * (x1 - x2).pow(2)) / ((a1 + a2) * (b1 + b2) - (c1 + c2).pow(2) + eps)) * 0.25
    t2 = (((c1 + c2) * (x2 - x1) * (y1 - y2)) / ((a1 + a2) * (b1 + b2) - (c1 + c2).pow(2) + eps)) * 0.5
    t3 = (((a1 + a2) * (b1 + b2) - (c1 + c2).pow(2))
          / (4 * ((a1 * b1 - c1.pow(2)).clamp_(0) * (a2 * b2 - c2.pow(2)).clamp_(0)).sqrt() + eps) + eps).log() * 0.5
    bd = (t1 + t2 + t3).clamp(eps, 100.0)
    hd = (1.0 - (-bd).exp() + eps).sqrt()
    return 1 - hd


def nms_rotated(boxes: torch.Tensor, scores: torch.Tensor, threshold: float, chunk: int = 512) -> torch.Tensor:
    """Ultralytics ``nms_rotated`` ("fast NMS"): sort by score, keep j iff ProbIoU(i, j) < thr for every earlier i -- a box that
    was itself suppressed still suppresses.  The sort is stable (equal scores keep input order), which is the engine's tie rule.
    The [N, N] ProbIoU matrix is built ``chunk`` columns at a time (same elements, bounded memory)."""
    order = torch.sort(scores, descending=True, stable=True).indices
    b = boxes[order]
    n = b.shape[0]
    colmax = torch.zeros(n)
    for j0 in range(0, n, chunk):
        ious = batch_probiou(b, b[j0:j0 + chunk])
        ious = torch.where(torch.arange(n)[:, None] < torch.arange(j0, min(n, j0 + chunk))[None], ious, torch.zeros(()))
        colmax[j0:j0 + chunk] = ious.max(dim=0)[0]
    pick = torch.nonzero(colmax < threshold).squeeze_(-1)
    return order[pick]


def fast_nms_loop(boxes: np.ndarray, scores: np.ndarray, threshold: float) -> np.ndarray:
    """Plain-loop statement of the same rule (cross-check of ``nms_rotated``)."""
    order = np.lexsort((np.arange(len(scores)), -np.asarray(scores, np.float32)))
    iou = batch_probiou(boxes[order], boxes[order]).numpy()
    keep = []
    for jj in range(len(order)):
        if all(iou[ii, jj] < np.float32(threshold) for ii in range(jj)):
            keep.append(order[jj])
    return np.asarray(keep, np.int64)


def ultralytics_nms_rotated(pred: np.ndarray, conf_thres=0.25, iou_thres=0.7, max_det=300, max_nms=30000) -> List[np.ndarray]:
    """``non_max_suppression(rotated=True)`` then ``regularize_rboxes``.  pred: [B, 4 + nc + 1, A].  Returns per image
    [n, 7] = (cx, cy, w, h, theta, conf, cls) regularized, plus the anchor index of each kept row as column 7."""
    p = torch.from_numpy(np.ascontiguousarray(pred)).float()
    nc = p.shape[1] - 5
    out = []
    for xi in range(p.shape[0]):
        x = p[xi].transpose(0, 1)                                         # [A, 4 + nc + 1]
        anchor = torch.arange(x.shape[0])
        conf, j = x[:, 4:4 + nc].max(1, keepdim=True)
        m = conf.view(-1) > conf_thres
        x = torch.cat((x[:, :4], conf, j.float(), x[:, -1:]), 1)[m]
        anchor = anchor[m]
        if x.shape[0] > max_nms:
            o = torch.sort(x[:, 4], descending=True, stable=True).indices[:max_nms]
            x, anchor = x[o], anchor[o]
        c = x[:, 5:6] * MAX_WH
        boxes = torch.cat((x[:, :2] + c, x[:, 2:4], x[:, -1:]), dim=-1)
        i = nms_rotated(boxes, x[:, 4], iou_thres)[:max_det]
        x, anchor = x[i], anchor[i]
        r = regularize_rboxes(torch.cat([x[:, :4], x[:, -1:]], 1).numpy())
        out.append(np.concatenate([r, x[:, 4:6].numpy(), anchor[:, None].numpy().astype(np.float32)], 1))
    return out


def regularize_rboxes(rboxes: np.ndarray) -> np.ndarray:
    """Ultralytics ``regularize_rboxes``: w >= h, theta in [0, pi) (torch's floor-mod)."""
    t = torch.as_tensor(np.asarray(rboxes, np.float32))
    x, y, w, h, th = t.unbind(-1)
    swap = (w > h)
    w_ = torch.where(swap, w, h)
    h_ = torch.where(swap, h, w)
    th = torch.where(swap, th, th + math.pi / 2) % math.pi
    return torch.stack([x, y, w_, h_, th], -1).numpy()


def xywhr2xyxyxyxy(rboxes: np.ndarray) -> np.ndarray:
    """Ultralytics ``xywhr2xyxyxyxy``: [N, 5] -> [N, 4, 2] corners c+v1+v2, c+v1-v2, c-v1-v2, c-v1+v2."""
    t = torch.as_tensor(np.asarray(rboxes, np.float32))
    ctr, w, h, th = t[:, :2], t[:, 2:3], t[:, 3:4], t[:, 4:5]
    cos, sin = torch.cos(th), torch.sin(th)
    vec1 = torch.cat([w / 2 * cos, w / 2 * sin], -1)
    vec2 = torch.cat([-h / 2 * sin, h / 2 * cos], -1)
    return torch.stack([ctr + vec1 + vec2, ctr + vec1 - vec2, ctr - vec1 - vec2, ctr - vec1 + vec2], -2).numpy()
