"""Drop-in for the reference's ``_script/gpu_handler.py::GPUHandler``.

Same constructor, attributes and methods (``gpu_handler.py:16-23``, ``:67-92``,
``:151-218``, ``:287-290``); the body is the device-memory and stream manager in
front of the C-ABI engine instead of an onnxruntime session:

* ``process_batch`` keeps the reference's input contract -- a list of *lists* whose
  element ``[0]`` is ``(PIL.Image, (lon_min, lat_min, lon_max, lat_max), _)``;
  anything else is skipped (``gpu_handler.py:156-161``) -- but runs all tiles of a
  call as device batches: cv2-linear resize when the tile is not 640x640
  (``:74-76``), ``conf >= threshold`` (``:166-170``), the ten best per tile
  (``:173``), and the ``x/640*864/864`` georeferencing (``:182-190``) in fp64;
* per-batch exceptions propagate by default.  The reference swallows them and returns
  ``[]`` (``:215-218``); pass ``swallow_errors=True`` for that behaviour.
"""
from __future__ import annotations

import gc
import os
from typing import Dict, List, Optional

import numpy as np
import torch

from . import tta as _tta
from .engine import GEO_PARAMS, GEODET_BYTES, GEODET_DTYPE, Engine, geodets_to_numpy, require_axis_aligned
from .session import InferenceSession, arch_from_model_path, resolve_weights


def _as_u8_hwc(img) -> np.ndarray:
    a = np.asarray(img)
    if a.ndim == 2:
        a = np.repeat(a[..., None], 3, 2)
    if a.shape[2] == 4:
        a = a[..., :3]
    a = np.ascontiguousarray(a, dtype=np.uint8)
    return a if a.flags.writeable else a.copy()      # np.asarray(PIL image) is read-only; torch.from_numpy wants a writable array


def _rgbx_view(img) -> Optional[np.ndarray]:
    """Zero-copy uint8 [h, w, 4] view of a PIL ``RGB`` image's own storage, or None.  Pillow keeps RGB pixels as 4 bytes
    (R, G, B, pad) and exports that block through the Arrow C data interface (Pillow >= 11.2); ``np.asarray(img)`` instead
    re-packs the image to 3 bytes per pixel through ``tobytes()`` -- 0.8 ms per 640 x 640 tile on one core, the cost that bounded
    ``process_batch``.  Images of another mode, images Pillow stores in several blocks and environments without the interface
    or without pyarrow give None and take the ``np.asarray`` route."""
    if getattr(img, "mode", None) != "RGB" or not hasattr(img, "__arrow_c_array__"):
        return None
    try:
        import pyarrow as pa
        flat = pa.array(img).flatten().to_numpy(zero_copy_only=True)
    except Exception:
        return None
    w, h = img.size
    return flat.reshape(h, w, 4) if flat.size == h * w * 4 else None


def _shape_of(img):
    """(h, w, 3) of a PIL image / array without converting it."""
    if hasattr(img, "size") and hasattr(img, "mode") and not isinstance(img, np.ndarray):
        return (img.size[1], img.size[0], 3)
    a = np.asarray(img)
    return (a.shape[0], a.shape[1], 3)


class TileStager:
    """Host images -> one device batch ``uint8 [n, h, w, 3]`` through reused page-locked buffers (no ``np.stack`` +
    ``pin_memory`` per batch: allocating pinned memory costs more than the copy).  PIL RGB images are staged as the 4-byte
    pixels Pillow holds (``_rgbx_view``: one memcpy per image, no re-packing on the host) and the pad byte is dropped on the
    device; anything else goes through ``np.asarray`` into a 3-byte buffer.  Two buffers per shape alternate, each guarded by
    the event of the copy that last read it, so the host fills batch i+1 while batch i is in flight."""

    def __init__(self, engine):
        require_axis_aligned(engine, "TileStager")
        self.engine = engine
        self._stage = {}            # (h, w, channels) -> two pinned uint8 [max_batch, h, w, channels] buffers
        self._free = {}             # same key -> the events after which they may be overwritten
        self._turn = 0
        self.threads = max(1, int(os.environ.get("B2D_STAGE_THREADS", "4")))      # host threads copying images into the pinned buffer
        self._pool = None

    def _executor(self):
        if self._pool is None:
            from concurrent.futures import ThreadPoolExecutor
            self._pool = ThreadPoolExecutor(self.threads, thread_name_prefix="b2d-stage")
        return self._pool

    def upload(self, imgs, shape) -> torch.Tensor:
        eng = self.engine
        n = len(imgs)
        assert 0 < n <= eng.max_batch
        views = [_rgbx_view(im) for im in imgs]
        rgbx = all(v is not None for v in views)
        key = (int(shape[0]), int(shape[1]), 4 if rgbx else 3)
        if key not in self._stage:
            self._stage[key] = [torch.empty((eng.max_batch,) + key, dtype=torch.uint8).pin_memory() for _ in range(2)]
            self._free[key] = [None, None]
        slot = self._turn % 2
        self._turn += 1
        host, free = self._stage[key][slot], self._free[key]
        if free[slot] is not None:
            free[slot].synchronize()                    # the copy that last read this buffer has finished
        hv = host.numpy()
        if rgbx and n >= 2 * self.threads and self.threads > 1:
            # plain memcpys of 1.6 MB each: NumPy releases the GIL for them, so a few threads copy at several times one core's rate
            def copy(t):
                for k in range(t, n, self.threads):
                    hv[k] = views[k]
            list(self._executor().map(copy, range(self.threads)))
        else:
            for k in range(n):
                hv[k] = views[k] if rgbx else _as_u8_hwc(imgs[k])
        tiles = host[:n].to(eng.device, non_blocking=True)
        free[slot] = torch.cuda.Event()
        free[slot].record()
        return tiles[..., :3].contiguous() if rgbx else tiles


class GPUHandler:
    def __init__(self, model_path, max_gpu_memory=5.0, confidence_threshold=0.3, output_dir=None, *,
                 arch: Optional[str] = None, weights=None, max_batch: int = 64,
                 top_k: int = 10, bgr: bool = False, device: int = 0, seed: int = 0, swallow_errors: bool = False,
                 precision: str = "bf16"):
        self.model_path = model_path
        self.max_gpu_memory = max_gpu_memory
        self.confidence_threshold = confidence_threshold
        self.output_dir = output_dir
        self.top_k = top_k
        self.bgr = bgr                      # the archived code fed BGR (gpu_handler.py:145); current code feeds RGB
        self.swallow_errors = swallow_errors
        self.session = None
        self._setup_gpu()
        arch = arch or arch_from_model_path(model_path)
        weights = resolve_weights(model_path, arch, weights)     # FileNotFoundError unless weights="synthetic" (session.py)
        self.engine = Engine(arch, weights=weights, max_batch=max_batch, device=device, seed=seed, precision=precision)
        self.session = InferenceSession(engine=self.engine)
        self._stager = TileStager(self.engine)      # pinned input staging, reused across calls
        self._stage = {}                            # ("out", cap) -> two pinned result buffers

    def _result_staging(self, cap, k):
        key = ("out", cap)
        if key not in self._stage:
            self._stage[key] = [(torch.empty((self.engine.max_batch, cap, GEODET_BYTES), dtype=torch.uint8).pin_memory(),
                                 torch.empty((self.engine.max_batch,), dtype=torch.int32).pin_memory()) for _ in range(2)]
        return self._stage[key][k % 2]

    def _setup_gpu(self):
        if not torch.cuda.is_available():
            raise RuntimeError("CUDA is not available!")       # gpu_handler.py:27-28

    # -- gpu_handler.py:67-92 -------------------------------------------------------------
    def preprocess_image(self, img):
        a = _as_u8_hwc(img)
        t = torch.from_numpy(a)[None].to(self.engine.device)
        S = self.engine.imgsz
        mode = "identity" if a.shape[:2] == (S, S) else "cv2_linear"
        return self.engine.preprocess(t, mode, out="f32").cpu().numpy()

    # -- gpu_handler.py:151-218 -----------------------------------------------------------
    def process_batch(self, images, queue_size=16):
        try:
            return self._process_batch(images)
        except Exception:
            if self.swallow_errors:
                import traceback
                traceback.print_exc()
                return []
            raise

    def _process_batch(self, images) -> List[dict]:
        eng = self.engine
        items = []
        for img_set in images:
            if not img_set or not isinstance(img_set, list) or not img_set[0]:
                continue
            img, bbox, _ = img_set[0]
            items.append((img, tuple(float(v) for v in bbox)))
        shapes = [_shape_of(it[0]) for it in items]
        pending = []                                   # (pinned records, pinned counts, n, event) of the batches in flight
        out: List[dict] = []

        def drain(upto):                               # results are read one batch behind, while the next batch computes
            while len(pending) > upto:
                geo_h, cnt_h, n, ev = pending.pop(0)
                ev.synchronize()
                recs = geo_h.numpy().view(GEODET_DTYPE)[..., 0]
                for t, c in enumerate(cnt_h.numpy()[:n].tolist()):
                    g = recs[t, :c]
                    x, y, cf = g["x"].tolist(), g["y"].tolist(), g["conf"].tolist()
                    out.extend({"lon": x[r], "lat": y[r], "confidence": cf[r]} for r in range(c))

        i = b = 0
        while i < len(items):
            # consecutive tiles of one shape form a device batch
            shape = shapes[i]
            j = i
            while j < len(items) and j - i < eng.max_batch and shapes[j] == shape:
                j += 1
            n = j - i
            tiles = self._stager.upload([it[0] for it in items[i:j]], shape)
            S = eng.imgsz
            mode = "identity" if shape[:2] == (S, S) else "cv2_linear"
            dets, counts = eng.infer(tiles, mode, self.bgr, self.confidence_threshold, True, 0.0, self.top_k)
            params = np.zeros((n, GEO_PARAMS), dtype=np.float64)
            params[:, :4] = [it[1] for it in items[i:j]]
            geo = eng.georef(dets, counts, torch.from_numpy(params).to(eng.device), "gpuhandler")
            geo_h, cnt_h = self._result_staging(geo.shape[1], b)
            geo_h[:n].copy_(geo, non_blocking=True)
            cnt_h[:n].copy_(counts, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record()
            pending.append((geo_h, cnt_h, n, ev))
            drain(1)
            i = j
            b += 1
        drain(0)
        return out

    def process_tiles(self, tiles: torch.Tensor, bboxes) -> List[dict]:
        """``process_batch`` for tiles that are already one uint8 tensor [B, H, W, 3] (device-resident or CPU) with
        ``bboxes`` float64 [B, 4] = (lon_min, lat_min, lon_max, lat_max): same filter, top-k and georeferencing, same
        records, without the per-image host staging (SURVEY.md section 8b input contract)."""
        eng = self.engine
        assert tiles.dtype == torch.uint8 and tiles.dim() == 4 and tiles.shape[3] == 3
        bb = np.asarray(bboxes, dtype=np.float64).reshape(tiles.shape[0], 4)
        tiles = tiles.to(eng.device, non_blocking=True)
        S = eng.imgsz
        mode = "identity" if tuple(tiles.shape[1:3]) == (S, S) else "cv2_linear"
        out: List[dict] = []
        for i in range(0, tiles.shape[0], eng.max_batch):
            chunk = tiles[i:i + eng.max_batch]
            n = chunk.shape[0]
            dets, counts = eng.infer(chunk, mode, self.bgr, self.confidence_threshold, True, 0.0, self.top_k)
            params = np.zeros((n, GEO_PARAMS), dtype=np.float64)
            params[:, :4] = bb[i:i + n]
            geo = eng.georef(dets, counts, torch.from_numpy(params).to(eng.device), "gpuhandler")
            for g in geodets_to_numpy(geo, counts):
                out.extend({"lon": x, "lat": y, "confidence": c} for x, y, c in zip(g["x"].tolist(), g["y"].tolist(), g["conf"].tolist()))
        return out

    # -- test-time augmentation: gpu_handler.py:94-149, :220-285 ------------------------------
    def _views_u8(self, img, views):
        t = torch.from_numpy(_as_u8_hwc(img))[None].to(self.engine.device)
        return self.engine.tta_views(t, views)

    def _prepare_tensor(self, img):
        """gpu_handler.py:142-149: uint8 RGB -> float32 CHW **BGR** / 255 on the device (no resize).  ``img`` may be a
        PIL image, a uint8 HWC array, or a uint8 device tensor [1,h,w,3] produced by the view kernels."""
        t = img if isinstance(img, torch.Tensor) else torch.from_numpy(_as_u8_hwc(img))[None].to(self.engine.device)
        # RGB -> BGR is a channel flip of the CHW tensor; x / 255 is torch's own float32 division, as in the reference
        return t[0].flip(-1).to(dtype=torch.float32).permute(2, 0, 1) / 255.0

    def _get_lighting_variations(self, img):
        """gpu_handler.py:94-123: original, CLAHE(3.0, 8x8) on L of LAB, brightness x2.0, gamma 2.0."""
        return [self._prepare_tensor(v) for v in self._views_u8(img, _tta.LIGHTING_VIEWS)]

    def _get_occlusion_variations(self, img):
        """gpu_handler.py:125-140: CLAHE(4.0, 4x4)."""
        return [self._prepare_tensor(v) for v in self._views_u8(img, _tta.OCCLUSION_VIEWS)]

    def preprocess_variations(self, img):
        """The archived handler's ``preprocess_image`` (gpu_handler_archive.py:57-67): lighting + occlusion views."""
        return self._get_lighting_variations(img) + self._get_occlusion_variations(img)

    def _get_confidence_adjustment(self, variation_index, total_variations):
        return _tta.confidence_adjustment(variation_index, total_variations)

    def _process_tensors(self, tensor_batch):
        """gpu_handler.py:220-270: ``tensor_batch`` = [(tensor_variations, bbox), ...] with float32 [3,S,S] device tensors.
        Per view: network, ``conf *= adjustment`` (float32), ``conf > threshold`` (strict); the kept rows of a tile are
        concatenated in view order and georeferenced in float32 (the reference's CUDA-tensor arithmetic).  The views of
        all tiles run as device batches; the output order is the reference's (tile, then view, then row)."""
        eng = self.engine
        tiles = [(list(v), tuple(float(b) for b in bbox)) for v, bbox in tensor_batch]
        nviews = max((len(v) for v, _ in tiles), default=0)
        per = {}                                   # (tile, view) -> structured geodet array
        for i in range(nviews):
            idx = [t for t, (v, _) in enumerate(tiles) if i < len(v)]
            for c0 in range(0, len(idx), eng.max_batch):
                chunk = idx[c0:c0 + eng.max_batch]
                eng.set_input_f32(torch.stack([tiles[t][0][i] for t in chunk]).to(eng.device))
                eng.forward(len(chunk))
                eng.set_conf_scale(self._get_confidence_adjustment(i, nviews))
                try:
                    dets, counts = eng.postprocess(len(chunk), self.confidence_threshold, False)
                finally:
                    eng.set_conf_scale(1.0)
                params = np.zeros((len(chunk), GEO_PARAMS), dtype=np.float64)
                for k, t in enumerate(chunk):
                    params[k, :4] = tiles[t][1]
                geo = eng.georef(dets, counts, torch.from_numpy(params).to(eng.device), "tensor_f32")
                for k, g in enumerate(geodets_to_numpy(geo, counts)):
                    per[(chunk[k], i)] = g
        out: List[dict] = []
        for t, (v, _) in enumerate(tiles):
            for i in range(len(v)):
                g = per[(t, i)]                      # lon / lat are float32 in this path (gpu_handler.py:247-253), widened on output
                out.extend({"lon": x, "lat": y, "confidence": c} for x, y, c in
                           zip(g["x"].astype(np.float32).tolist(), g["y"].astype(np.float32).tolist(), g["conf"].tolist()))
        return out

    def process_batch_tta(self, images, views=None):
        """``process_batch`` with the five views per tile, entirely on uint8 device batches: same input contract as
        ``process_batch`` (gpu_handler.py:156-161), the views of gpu_handler.py:94-140, ``_prepare_tensor``'s BGR order,
        then ``_process_tensors``' filter and float32 georeferencing.  Equivalent to
        ``_process_tensors([(preprocess_variations(img), bbox), ...])`` for model-sized tiles, without the float32
        round trip of the views."""
        eng = self.engine
        views = views or (_tta.LIGHTING_VIEWS + _tta.OCCLUSION_VIEWS)
        items = []
        for img_set in images:
            if not img_set or not isinstance(img_set, list) or not img_set[0]:
                continue
            img, bbox, _ = img_set[0]
            items.append((_as_u8_hwc(img), tuple(float(v) for v in bbox)))
        S = eng.imgsz
        per = {}
        for c0 in range(0, len(items), eng.max_batch):
            chunk = items[c0:c0 + eng.max_batch]
            for a, _ in chunk:
                if a.shape[:2] != (S, S):
                    raise ValueError(f"test-time augmentation needs {S}x{S} tiles (the reference does not resize here), got {a.shape}")
            tiles = torch.from_numpy(np.stack([a for a, _ in chunk])).pin_memory().to(eng.device, non_blocking=True)
            params = np.zeros((len(chunk), GEO_PARAMS), dtype=np.float64)
            for k, (_, bbox) in enumerate(chunk):
                params[k, :4] = bbox
            params_dev = torch.from_numpy(params).to(eng.device)
            for i, view in enumerate(eng.tta_views(tiles, views)):
                dets, counts = eng.infer(view, "identity", True, self.confidence_threshold, False,
                                         conf_scale=self._get_confidence_adjustment(i, len(views)))
                geo = eng.georef(dets, counts, params_dev, "tensor_f32")
                for k, g in enumerate(geodets_to_numpy(geo, counts)):
                    per[(c0 + k, i)] = g
        out: List[dict] = []
        for t in range(len(items)):
            for i in range(len(views)):
                g = per[(t, i)]                      # lon / lat are float32 in this path (gpu_handler.py:247-253), widened on output
                out.extend({"lon": x, "lat": y, "confidence": c} for x, y, c in
                           zip(g["x"].astype(np.float32).tolist(), g["y"].astype(np.float32).tolist(), g["conf"].tolist()))
        return out

    def cleanup(self):
        torch.cuda.empty_cache()
        gc.collect()
