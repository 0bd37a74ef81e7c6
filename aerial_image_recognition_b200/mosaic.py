"""Sliding-window detection over a large georeferenced mosaic, tile-sharded across GPUs (``MosaicDetector``), and oriented-box
detection over a whole mosaic on one GPU, merged by a mosaic-wide ProbIoU fast NMS (``ObbMosaicDetector``).

Ancestor in the reference: the notebook loop at ``x_arch/02_analyze_images:1 (cell 6)`` --
``for y in range(0,h,stride): for x in range(0,w,stride): model(window)`` -> boxes with
``conf > 0.4`` -> centroid + window origin -> ``pixel_to_geo`` -- and the production tiling
``TileGenerator.generate_tiles`` (``_script/utils.py:26-65``) with ``tile_overlap 0.2``
(``_script/config.py:15``) followed by the centre-distance dedup
(``simple_detector.py:540-596``).  BASELINE config C4: 40k x 40k, window 640, stride 512.

Decisions where the reference leaves a choice (stated in DESIGN.md):
* windows are model-sized (640) by default, so no resampling happens; edge windows are clipped like the
  notebook's ``min()`` and centred on a 114 canvas (Ultralytics LetterBox without up-scaling).  Any other
  window size is resampled by one gain ``imgsz / win`` for every window (``window_geometry``), so an object
  has the same size in the network input wherever it lies in the mosaic;
* the window grid is y-outer / x-inner, and that order is the global tie-break of the dedup;
* shards are contiguous bands of window rows (fewest seams).  Each window belongs to exactly one
  rank, so the only cross-rank interaction is the dedup of detections that sit in the overlap
  between two bands; only those (closed under the within-threshold relation) are exchanged.
"""
from __future__ import annotations

from typing import Callable, List, Optional, Sequence, Tuple

import numpy as np


def window_grid(h: int, w: int, win: int = 640, stride: int = 512) -> np.ndarray:
    """int32 [n, 4] = (x0, y0, w0, h0), y outer / x inner, clipped at the mosaic edge."""
    ys = np.arange(0, h, stride, dtype=np.int64)
    xs = np.arange(0, w, stride, dtype=np.int64)
    yy, xx = np.meshgrid(ys, xs, indexing="ij")
    x0 = xx.reshape(-1); y0 = yy.reshape(-1)
    return np.stack([x0, y0, np.minimum(x0 + win, w) - x0, np.minimum(y0 + win, h) - y0], 1).astype(np.int32)


def grid_shape(h: int, w: int, stride: int = 512) -> Tuple[int, int]:
    return (h + stride - 1) // stride, (w + stride - 1) // stride


def band_rows(n_rows: int, world: int) -> List[Tuple[int, int]]:
    """Contiguous window-row bands, sizes differing by at most one (larger bands first)."""
    base, extra = divmod(n_rows, world)
    out, r = [], 0
    for k in range(world):
        m = base + (1 if k < extra else 0)
        out.append((r, r + m))
        r += m
    return out


def shard_windows(h: int, w: int, rank: int, world: int, win: int = 640, stride: int = 512):
    """(windows of this rank int32 [m,4], global ids int64 [m], pixel-row coverage (y_lo, y_hi))."""
    grid = window_grid(h, w, win, stride)
    rows, cols = grid_shape(h, w, stride)
    r0, r1 = band_rows(rows, world)[rank]
    ids = np.arange(r0 * cols, r1 * cols, dtype=np.int64)
    mine = grid[ids]
    if len(mine):
        cover = (int(mine[:, 1].min()), int((mine[:, 1] + mine[:, 3]).max()))
    else:
        cover = (0, 0)
    return mine, ids, cover


def seam_flags(py: np.ndarray, rank: int, covers: Sequence[Tuple[int, int]], margin_px: float) -> np.ndarray:
    """uint8 flags: detection (mosaic pixel row ``py``) lies within ``margin_px`` of the pixel rows
    covered by another rank's windows."""
    flag = np.zeros(len(py), dtype=np.uint8)
    for r, (lo, hi) in enumerate(covers):
        if r == rank or hi <= lo:
            continue
        flag |= ((py >= lo - margin_px) & (py < hi + margin_px)).astype(np.uint8)
    return flag


def seam_flags_device(py, rank: int, covers: Sequence[Tuple[int, int]], margin_px: float):
    """``seam_flags`` on the device: ``py`` is a CUDA float tensor, the result a CUDA uint8 tensor (no host round trip)."""
    import torch
    flag = torch.zeros(py.shape, dtype=torch.bool, device=py.device)
    for r, (lo, hi) in enumerate(covers):
        if r == rank or hi <= lo:
            continue
        flag |= (py >= lo - margin_px) & (py < hi + margin_px)
    return flag.to(torch.uint8)


def window_geometry(windows: np.ndarray, win: int, imgsz: int):
    """Letterbox geometry of every window at one gain ``g = imgsz / win``: (new_w, new_h, left, top) int64 [n] each, and g.

    Ultralytics LetterBox (center=True) with ``r = g``: ``new = max(1, round(w0 * g))``, ``left = round((imgsz - new_w) / 2 - 0.1)``
    (Python ``round`` = ``rint``).  This is Ultralytics' own ``r = min(imgsz / h0, imgsz / w0)`` on every window clipped on at
    most one axis; a corner window clipped on both keeps the gain of its neighbours, so objects keep one scale across the
    mosaic.  ``max(1, ...)`` keeps the one-pixel slivers of a grid with ``W % stride == 1``.  ``b2d_resize_windows`` restates it."""
    w = np.asarray(windows)
    g = imgsz / win
    new_w = np.maximum(1, np.rint(w[:, 2].astype(np.float64) * g)).astype(np.int64)
    new_h = np.maximum(1, np.rint(w[:, 3].astype(np.float64) * g)).astype(np.int64)
    left = np.rint((imgsz - new_w) / 2 - 0.1).astype(np.int64)
    top = np.rint((imgsz - new_h) / 2 - 0.1).astype(np.int64)
    return new_w, new_h, left, top, g


def check_windows(windows: np.ndarray, win: int, height: int, width: int) -> None:
    """Raise ValueError unless every window has 1 <= w0, h0 <= win and lies inside a height x width mosaic."""
    if win <= 0:
        raise ValueError(f"window size {win} must be positive")
    w = np.asarray(windows, dtype=np.int64).reshape(-1, 4)
    x0, y0, w0, h0 = w.T
    bad = (w0 < 1) | (w0 > win) | (h0 < 1) | (h0 > win) | (x0 < 0) | (y0 < 0) | (x0 + w0 > width) | (y0 + h0 > height)
    if bad.any():
        k = int(np.flatnonzero(bad)[0])
        raise ValueError(f"window {k} (x0, y0, w0, h0) = {tuple(int(v) for v in w[k])} needs 1 <= w0, h0 <= {win} and to lie "
                         f"inside the {height} x {width} mosaic")


def affine_params(windows: np.ndarray, geotransform: Sequence[float], win: int = 640, imgsz: Optional[int] = None) -> np.ndarray:
    """float64 [n,16] georef parameters for B2D_GEO_AFFINE: gt[6], win_x, win_y, pad_x, pad_y, gain,
    w0, h0 (the letterbox undo of Ultralytics ``scale_boxes``).  ``imgsz=None`` means model-sized windows: gain 1 and the
    centring pad.  With ``imgsz`` the pad and gain are ``window_geometry``'s."""
    n = len(windows)
    p = np.zeros((n, 16), dtype=np.float64)
    p[:, 0:6] = np.asarray(geotransform, dtype=np.float64)
    p[:, 6] = windows[:, 0]
    p[:, 7] = windows[:, 1]
    if imgsz is None:
        p[:, 8] = (win - windows[:, 2]) // 2
        p[:, 9] = (win - windows[:, 3]) // 2
        p[:, 10] = 1.0
    else:
        _, _, left, top, g = window_geometry(windows, win, imgsz)
        p[:, 8] = left
        p[:, 9] = top
        p[:, 10] = g
    p[:, 11] = windows[:, 2]
    p[:, 12] = windows[:, 3]
    return p


def run_windows(eng, mosaic, windows: np.ndarray, y_offset: int, gt: Sequence[float], win: int, fill: int, nms_conf: float, iou: float,
                max_det: int):
    """Detection on every window (x0, y0, w0, h0) of ``windows`` (mosaic coordinates; ``mosaic`` is the uint8 CUDA tensor of pixel
    rows [y_offset, ...)): cut (win = the model input) or resampled windows, network, per-window NMS and affine georef, batch
    by batch with nothing read back.  Returns device tensors (geo records [n, cap, *], dets [n, cap, *], counts [n], affine params
    [n, 16]) in window order -- records of ``eng``'s kind, axis-aligned or oriented -- or None for no windows."""
    import torch
    dev = eng.device
    if not len(windows):
        return None
    # equal batches: 780 windows at max_batch 64 are 13 launches either way, but 13 x 60 keeps every step full
    # where 12 x 64 + 12 ends a band on a step that is four fifths empty
    nb = -(-len(windows) // eng.max_batch)
    B = -(-len(windows) // nb)
    local = windows.copy()
    local[:, 1] -= y_offset
    # every per-window table goes to the device once; the batch loop below queues kernels only (no host
    # synchronisation: a boolean-mask gather per batch would stall the launch queue ~100 times per mosaic)
    resample = win != eng.imgsz
    if resample:
        # windows of another size are resampled from the mosaic straight into the network input: checked once here,
        # since the per-batch launches below leave the origins on the device
        check_windows(local, win, mosaic.shape[0], mosaic.shape[1])
    params_all = torch.from_numpy(affine_params(windows, gt, win, eng.imgsz if resample else None)).to(dev)
    org_all = torch.from_numpy(local).to(dev)
    outs = []
    for s in range(0, len(windows), B):
        e = min(s + B, len(windows))
        n = e - s
        if resample:
            eng.resize_windows(mosaic, org_all[s:e], win, fill, checked=True)
            eng.forward(n)
            dets, counts = eng.postprocess(n, nms_conf, False, iou, 0, max_det)
        else:
            tiles = eng.cut_windows(mosaic, org_all[s:e], win, fill)
            dets, counts = eng.infer(tiles, "identity", False, nms_conf, False, iou, 0, max_det)
        geo = eng.georef(dets, counts, params_all[s:e], "affine")
        outs.append((geo, dets, counts))
    return (torch.cat([o[0] for o in outs]), torch.cat([o[1] for o in outs]), torch.cat([o[2] for o in outs]), params_all)


# -------------------------------------------------------------------------------------------------
# seam exchange: host-side protocol, independent of the device (tested on CPU with gloo)
# -------------------------------------------------------------------------------------------------
# One exchanged seam record = 4 x 8 bytes: x (f64), y (f64), [conf (f32) | class (i32)], order key (i64 = window * 65536 +
# slot).  SURVEY 8e sketches 24 bytes {x, y, conf, tile id}; the slot inside the window is needed too -- it is the last
# component of the total order every rank must agree on -- so the id word is 64-bit and the record 32 bytes.
RECORD_WORDS = 4


def pack_records(x, y, conf, cls, key):
    """Device tensors -> int64 [k, RECORD_WORDS] (bit patterns; see RECORD_WORDS)."""
    import torch
    w2 = (conf.contiguous().view(torch.int32).long() & 0xFFFFFFFF) | (cls.long() << 32)
    return torch.stack([x.contiguous().view(torch.int64), y.contiguous().view(torch.int64), w2, key.long()], 1)


def unpack_records(rec):
    """int64 [k, RECORD_WORDS] -> (x f64, y f64, conf f32, cls i32, key i64)."""
    import torch
    x = rec[:, 0].contiguous().view(torch.float64)
    y = rec[:, 1].contiguous().view(torch.float64)
    bits = rec[:, 2] & 0xFFFFFFFF                                                  # the float's bit pattern as 0 .. 2^32 - 1
    conf = torch.where(bits >= 2 ** 31, bits - 2 ** 32, bits).to(torch.int32).view(torch.float32)
    cls = (rec[:, 2] >> 32).to(torch.int32)
    return x, y, conf, cls, rec[:, 3].contiguous()


def exchange_seam(records, world: int, all_gather_counts: Callable, all_gather_padded: Callable):
    """records: [k, RECORD_WORDS] int64 array/tensor of this rank's flagged detections.
    Returns the per-rank parts in rank order (same on every rank) and the rank of origin
    of each row.  Two collectives: counts (world x int64), then a padded payload."""
    k = int(records.shape[0])
    counts = all_gather_counts(k)                       # list[int], length world
    cap = max(max(counts), 1)
    gathered = all_gather_padded(records, cap)          # list of [cap, RECORD_WORDS]
    parts, origin = [], []
    for r in range(world):
        parts.append(gathered[r][:counts[r]])
        origin.append(np.full(counts[r], r, dtype=np.int64))
    return parts, np.concatenate(origin) if origin else np.zeros(0, np.int64)


class MosaicDetector:
    """Runs config C4 on one rank; ``run`` returns this rank's share of the globally deduplicated
    detections as a structured array (x, y, conf, cls, window, slot)."""

    # one result record = five 8-byte words, laid out so that the device writes it and the host only re-labels it (no per-field
    # unpacking of up to a million records): x | y | conf, cls | window | slot, 4 bytes of padding
    OUT_DTYPE = np.dtype({"names": ["x", "y", "conf", "cls", "window", "slot"], "formats": ["<f8", "<f8", "<f4", "<i4", "<i8", "<i4"],
                          "offsets": [0, 8, 16, 20, 24, 32], "itemsize": 40})
    OUT_WORDS = 5

    def __init__(self, engine, geotransform: Sequence[float], win: int = 640, stride: int = 512, conf: float = 0.4,
                 nms_conf: float = 0.25, iou: float = 0.7, max_det: int = 300, dedup_thr: float = 1.0, fill: int = 114):
        from .engine import require_axis_aligned
        require_axis_aligned(engine, "MosaicDetector")
        self.eng = engine
        self.gt = tuple(float(v) for v in geotransform)
        self.win, self.stride = win, stride
        self.conf, self.nms_conf, self.iou, self.max_det = conf, nms_conf, iou, max_det
        self.dedup_thr = dedup_thr
        self.fill = fill
        self.profile = False            # True: synchronise around the phases of `dedup` and keep their wall times in `self.timings` (ms)
        self.timings = {}
        assert self.gt[2] == 0.0 and self.gt[4] == 0.0, "seam margins assume an axis-aligned geotransform"

    # ---- per-rank detection over its windows --------------------------------------------------
    def detect_windows(self, mosaic, windows: np.ndarray, ids: np.ndarray, y_offset: int = 0):
        """mosaic: uint8 CUDA tensor holding pixel rows [y_offset, y_offset + H_local) of the mosaic.
        Returns device tensors (x, y, conf, cls, window id, slot, pixel row)."""
        import torch
        eng = self.eng
        dev = eng.device
        out = run_windows(eng, mosaic, windows, y_offset, self.gt, self.win, self.fill, self.nms_conf, self.iou, self.max_det)
        if out is None:
            z = torch.zeros(0, device=dev)
            return z.double(), z.double(), z.float(), z.int(), z.long(), z.int(), z.float()
        geo, dets, counts, _ = out
        wid_n = torch.from_numpy(ids).to(dev)
        n, cap = dets.shape[0], dets.shape[1]
        slot = torch.arange(cap, device=dev, dtype=torch.int32)[None, :].expand(n, cap)
        conf = dets[..., 4]
        valid = (slot < counts[:, None]) & (conf > self.conf)            # notebook: box.conf > 0.4
        idx = valid.reshape(-1).nonzero().squeeze(1)                     # ONE compaction (one host sync); the columns are gathers
        g64 = geo.view(torch.float64).view(n * cap, 5)                    # x, y, then packed floats
        gf = geo.view(torch.float32).view(n * cap, 10)
        wid = wid_n[:, None].expand(n, cap).reshape(-1)
        cls = dets.view(torch.int32)[..., 5].reshape(-1)
        return (g64[:, 0][idx], g64[:, 1][idx], conf.reshape(-1)[idx], cls[idx], wid[idx], slot.reshape(-1)[idx], gf[:, 6][idx])

    # ---- dedup with seam exchange --------------------------------------------------------------
    @staticmethod
    def order_key(wid, slot):
        """Global total order among equal confidences: window order, then rank inside the window."""
        return wid * 65536 + slot.long()

    def _tick(self, name, t0):
        if self.profile:
            import time
            import torch
            torch.cuda.synchronize()
            self.timings[name] = self.timings.get(name, 0.0) + (time.perf_counter() - t0) * 1e3
            return time.perf_counter()
        return t0

    def seam_split(self, x, y, conf, cls, wid, slot, py, rank: int, covers, pack: bool = True):
        """Dedup everything that cannot interact with another shard; return (local survivors,
        records [k, RECORD_WORDS] float64 on device that must be exchanged).  ``pack=False`` leaves the local survivors on the
        device as the column tuple ``_pack`` takes (``dedup`` packs them together with the seam survivors: one read-back)."""
        import torch
        eng = self.eng
        import time
        t0 = time.perf_counter()
        key = self.order_key(wid, slot)
        margin_px = self.dedup_thr / min(abs(self.gt[1]), abs(self.gt[5])) + 1.0
        flag = seam_flags_device(py, rank, covers, margin_px)
        t0 = self._tick("flags", t0)
        eng.seam_closure(x, y, flag, self.dedup_thr, True)
        t0 = self._tick("closure", t0)
        seam = flag.bool()
        li, si = (~seam).nonzero().squeeze(1), seam.nonzero().squeeze(1)      # two compactions; everything below is a gather
        lx, ly, lc, lk = x[li], y[li], conf[li], key[li]
        t0 = self._tick("split", t0)
        lkeep = eng.dedup(lx, ly, lc, self.dedup_thr, True, tiebreak=lk)
        t0 = self._tick("local_dedup", t0)
        kept = li[lkeep.bool().nonzero().squeeze(1)]
        cols = (x[kept], y[kept], conf[kept], cls[kept], wid[kept], slot[kept])
        local = self._pack(*cols) if pack else cols
        rec = pack_records(x[si], y[si], conf[si], cls[si], key[si])
        self._tick("pack", t0)
        return local, rec

    def seam_merge(self, parts, origin: np.ndarray, rank: int, pack: bool = True):
        """The identical greedy pass every rank runs on the gathered seam records; returns the
        survivors that originated on ``rank`` (``pack=False``: as device columns, see ``seam_split``)."""
        import torch
        eng = self.eng
        allrec = torch.cat([torch.as_tensor(p).to(eng.device) for p in parts]) if parts else torch.zeros((0, RECORD_WORDS), dtype=torch.int64, device=eng.device)
        self.last_seam_records = int(allrec.shape[0])
        if not allrec.shape[0]:
            return np.zeros(0, self.OUT_DTYPE) if pack else None
        gx, gy, gc, gcls, gk = unpack_records(allrec)
        gkeep = eng.dedup(gx, gy, gc, self.dedup_thr, True, tiebreak=gk).bool()
        mine = (gkeep & torch.from_numpy(origin == rank).to(eng.device)).nonzero().squeeze(1)
        cols = (gx[mine], gy[mine], gc[mine], gcls[mine], gk[mine] >> 16, (gk[mine] & 0xFFFF).int())
        return self._pack(*cols) if pack else cols

    def dedup(self, x, y, conf, cls, wid, slot, py, rank: int, world: int, covers, group=None):
        import torch
        import torch.distributed as dist
        eng = self.eng
        if world == 1:
            keep = eng.dedup(x, y, conf, self.dedup_thr, True, tiebreak=self.order_key(wid, slot)).bool().nonzero().squeeze(1)
            return self._pack(x[keep], y[keep], conf[keep], cls[keep], wid[keep], slot[keep])
        local, rec = self.seam_split(x, y, conf, cls, wid, slot, py, rank, covers, pack=False)     # survivors stay on the device ...

        # seam part: NCCL all-gather over NVLink -- the counts as one [world] tensor read back once, then the padded payload
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]

        def gather_counts(k):
            out = torch.empty((world,), dtype=torch.int64, device=eng.device)
            dist.all_gather_into_tensor(out, torch.full((1,), k, dtype=torch.int64, device=eng.device), group=group)
            return out.tolist()

        def gather_padded(r, cap):
            pad = torch.zeros((cap, RECORD_WORDS), dtype=torch.int64, device=eng.device)
            pad[:r.shape[0]] = r
            out = torch.empty((world, cap, RECORD_WORDS), dtype=torch.int64, device=eng.device)
            ev[0].record()
            dist.all_gather_into_tensor(out, pad, group=group)
            ev[1].record()
            return list(out.unbind(0))

        import time
        t0 = time.perf_counter()
        parts, origin = exchange_seam(rec, world, gather_counts, gather_padded)
        t0 = self._tick("exchange", t0)
        out = self.finish(local, parts, origin, rank)
        self.last_allgather_us = ev[0].elapsed_time(ev[1]) * 1e3      # both events have completed: the read-back synchronised the stream
        return out

    def finish(self, local, parts, origin: np.ndarray, rank: int) -> np.ndarray:
        """Second half of the sharded dedup: ``local`` = the device columns ``seam_split(..., pack=False)`` left, ``parts`` /
        ``origin`` = the gathered seam records.  The merge is queued behind the local dedup without a host synchronisation in
        between, and everything comes back in ONE packed read-back (local survivors first, then this rank's seam survivors)."""
        import time
        import torch
        t0 = time.perf_counter()
        merged = self.seam_merge(parts, origin, rank, pack=False)
        t0 = self._tick("merge", t0)
        cols = local if merged is None else tuple(torch.cat([a, b.to(a.dtype)]) for a, b in zip(local, merged))
        out = self._pack(*cols)
        self._tick("read_back", t0)
        return out

    def _pack(self, x, y, conf, cls, wid, slot) -> np.ndarray:
        """Device columns -> one structured host array, through ONE device->host copy of 40-byte records that already have
        ``OUT_DTYPE``'s layout (the host side is a view plus one copy out of the reused pinned buffer)."""
        import torch
        n = int(x.numel())
        W = self.OUT_WORDS
        rec = torch.empty((n, W), dtype=torch.int64, device=x.device)
        rec[:, 0] = x.contiguous().view(torch.int64)
        rec[:, 1] = y.contiguous().view(torch.int64)
        rec[:, 2] = (conf.contiguous().view(torch.int32).long() & 0xFFFFFFFF) | (cls.long() << 32)
        rec[:, 3] = wid.long()
        rec[:, 4] = slot.long() & 0xFFFFFFFF
        stage = getattr(self, "_pack_stage", None)          # pinned staging: the copy runs at PCIe rate instead of through pageable memory
        if stage is None or stage.shape[0] < n:
            stage = self._pack_stage = torch.empty((max(n, 1 << 16), W), dtype=torch.int64).pin_memory()
        stage[:n].copy_(rec, non_blocking=True)
        torch.cuda.current_stream(x.device).synchronize()
        return stage[:n].numpy().view(self.OUT_DTYPE).reshape(n).copy()

    def run(self, mosaic, height: int, width: int, rank: int = 0, world: int = 1, y_offset: int = 0, group=None) -> np.ndarray:
        windows, ids, _ = shard_windows(height, width, rank, world, self.win, self.stride)
        covers = [shard_windows(height, width, r, world, self.win, self.stride)[2] for r in range(world)]
        x, y, conf, cls, wid, slot, py = self.detect_windows(mosaic, windows, ids, y_offset)
        self.last_raw = int(x.numel())
        return self.dedup(x, y, conf, cls, wid, slot, py, rank, world, covers, group)


class ObbMosaicDetector:
    """Oriented-box detection over a whole orthomosaic on one GPU: every window of the y-outer / x-inner grid through an
    oriented-box engine (``Engine("yolov8m-obb")``), then ONE mosaic-wide merge on the device (``Engine.mosaic_nms_obb``):
    Ultralytics' DOTA slice merge, ProbIoU fast NMS at ``merge_iou`` one class at a time over the records with
    ``conf > conf``, in the mosaic's pixel frame, so an object seen by two to four overlapping windows is reported once.
    Priority ties go to the earlier window, then the lower slot.  ``run`` returns the survivors' georeferenced footprints."""

    # GEOOBB_DTYPE with the global window (int64) in place of the batch-local tile, and the slot inside the window; the device
    # writes these 112-byte records and the host only re-labels them
    OUT_DTYPE = np.dtype({"names": ["x", "y", "corners", "conf", "w", "h", "theta", "cls", "slot", "window"],
                          "formats": ["<f8", "<f8", ("<f8", (4, 2)), "<f4", "<f4", "<f4", "<f4", "<i4", "<i4", "<i8"],
                          "offsets": [0, 8, 16, 80, 84, 88, 92, 96, 100, 104], "itemsize": 112})

    def __init__(self, engine, geotransform: Sequence[float], win: int = 640, stride: int = 512, conf: float = 0.4,
                 nms_conf: float = 0.25, iou: float = 0.7, max_det: int = 300, merge_iou: float = 0.3, fill: int = 114):
        if not getattr(engine, "is_obb", False):
            raise ValueError(f"ObbMosaicDetector needs an oriented-box engine (e.g. Engine('yolov8m-obb')); {engine.arch!r} is "
                             "axis-aligned: use MosaicDetector")
        self.eng = engine
        self.gt = tuple(float(v) for v in geotransform)
        self.win, self.stride = win, stride
        self.conf, self.nms_conf, self.iou, self.max_det = conf, nms_conf, iou, max_det
        self.merge_iou = merge_iou
        self.fill = fill
        assert self.gt[2] == 0.0 and self.gt[4] == 0.0, "the merge frame is the mosaic's pixel grid: an axis-aligned geotransform"

    def run(self, mosaic, height: int, width: int) -> np.ndarray:
        """mosaic: uint8 CUDA tensor [height, width, 3].  Returns ``OUT_DTYPE`` records of the merge's survivors in ascending
        (window, slot) order; ``last_raw`` is the number of records with ``conf > conf`` before the merge."""
        import torch
        eng = self.eng
        windows = window_grid(height, width, self.win, self.stride)
        out = run_windows(eng, mosaic, windows, 0, self.gt, self.win, self.fill, self.nms_conf, self.iou, self.max_det)
        if out is None:
            self.last_raw = 0
            return np.zeros(0, self.OUT_DTYPE)
        geo, dets, counts, params = out
        keep = eng.mosaic_nms_obb(dets, counts, params, self.conf, self.merge_iou)
        n, cap = keep.shape
        slot = torch.arange(cap, device=eng.device, dtype=torch.int32)[None, :].expand(n, cap)
        self.last_raw = int(((slot < counts[:, None]) & (dets[..., 5] > self.conf)).sum())
        idx = keep.reshape(-1).nonzero().squeeze(1)                   # ascending record index = (window, slot) order
        m = int(idx.numel())
        words = geo.view(torch.int32).view(n * cap, -1)                 # 26 words: x, y, corners, conf, w, h, theta, cls, tile
        rec = torch.empty((m, 28), dtype=torch.int32, device=eng.device)
        rec[:, :25] = words[idx, :25]
        rec[:, 25] = (idx % cap).int()
        rec.view(torch.int64)[:, 13] = idx // cap
        host = torch.empty((m, 28), dtype=torch.int32).pin_memory() if m else torch.empty((0, 28), dtype=torch.int32)
        host.copy_(rec, non_blocking=True)
        torch.cuda.current_stream(eng.device).synchronize()
        return host.numpy().view(self.OUT_DTYPE).reshape(m).copy()
