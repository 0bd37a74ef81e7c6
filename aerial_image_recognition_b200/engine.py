"""Python owner of one ``b2d_engine`` (one GPU): builds the plan from a ``Graph`` and
weights, and exposes the stages as methods on torch CUDA tensors.

This is what ``GPUHandler._load_model`` / ``ort.InferenceSession`` is in the
reference (``_script/gpu_handler.py:39-65``, ``simple_detector.py:38-47``): the
object that owns the model on the device.  torch is used for device memory,
streams and host<->device copies only; every kernel is in ``libb2det.so``.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from . import tta as _tta
from .graph import ACT_SILU, Graph, build, op_weights
from .weights import make_synthetic_weights

RESIZE = {"identity": 0, "cv2_linear": 1, "pil_bicubic": 2, "letterbox": 3}
GEO = {"bounds": 0, "gpuhandler": 1, "affine": 2, "tensor_f32": 3}
CONV_IMPL = {"auto": 0, "tcgen05": 1}
PRECISION = {"bf16": 0, "fp16": 1, "fp16x2": 2}
DET_WORDS = 8          # b2d_det = 8 x 4 bytes
GEODET_BYTES = 40
GEO_PARAMS = 16

GEODET_DTYPE = np.dtype([("x", "<f8"), ("y", "<f8"), ("conf", "<f4"), ("x_img", "<f4"), ("y_img", "<f4"),
                         ("x_yolo", "<f4"), ("y_yolo", "<f4"), ("tile", "<i4")])
DET_DTYPE = np.dtype([("cx", "<f4"), ("cy", "<f4"), ("w", "<f4"), ("h", "<f4"), ("conf", "<f4"),
                      ("cls", "<i4"), ("tile", "<i4"), ("anchor", "<i4")])
assert GEODET_DTYPE.itemsize == GEODET_BYTES and DET_DTYPE.itemsize == 4 * DET_WORDS
# oriented boxes (arch "yolov8m-obb"): b2d_obb / b2d_geoobb
OBB_WORDS = 9
GEOOBB_BYTES = 104
OBB_DTYPE = np.dtype([("cx", "<f4"), ("cy", "<f4"), ("w", "<f4"), ("h", "<f4"), ("theta", "<f4"), ("conf", "<f4"),
                      ("cls", "<i4"), ("tile", "<i4"), ("anchor", "<i4")])
GEOOBB_DTYPE = np.dtype([("x", "<f8"), ("y", "<f8"), ("corners", "<f8", (4, 2)), ("conf", "<f4"), ("w", "<f4"), ("h", "<f4"),
                         ("theta", "<f4"), ("cls", "<i4"), ("tile", "<i4")])
assert OBB_DTYPE.itemsize == 4 * OBB_WORDS and GEOOBB_DTYPE.itemsize == GEOOBB_BYTES
HEAD_KIND = {"v8_dfl": 0, "v7_anchor": 1, "v8_obb": 2}


def _ptr(t: Optional[torch.Tensor]):
    return C.c_void_p(0 if t is None else t.data_ptr())


def _default_cap(iou_thr: float, top_k: int, max_det: int, rows: int) -> int:
    """Output records per tile when the caller gives no cap: max_det with NMS, else top_k, else one per row (every row may pass;
    post-processing refuses tiles of more than 65536 rows)."""
    return max_det if iou_thr > 0 else (top_k if top_k > 0 else rows)


class Engine:
    def __init__(self, arch: str = "yolov8m", weights: Optional[Dict[str, np.ndarray]] = None, max_batch: int = 64,
                 device: int = 0, seed: int = 0, conv_impl: str = "auto", imgsz: int = 640, nc: Optional[int] = None,
                 graph: Optional[Graph] = None, precision: str = "bf16"):
        """``precision``: storage format of activations and weights -- "bf16" (default, the configuration BASELINE.json
        is quoted on), "fp16" (three more mantissa bits, same tensor-core rate; closer to the reference's fp32 results) or
        "fp16x2" (every activation as an fp16 high + low part, ~22 mantissa bits: the mode that meets the 1e-3 score /
        0.5 px box bound against an fp32 runtime, at about half the throughput)."""
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise _lib.B2DError("CUDA is not available: the B200 engine has no CPU fallback")
        self.device = torch.device("cuda", device)
        torch.cuda.set_device(self.device)
        self.graph = graph if graph is not None else build(arch, nc, imgsz)
        self.arch = self.graph.arch
        self.is_obb = self.graph.head.get("kind") == "v8_obb"     # oriented boxes: the *_obb entry points, OBB_DTYPE records
        self.imgsz = self.graph.imgsz
        self.max_batch = int(max_batch)
        self.weights_seed = seed if weights is None else None
        w = weights if weights is not None else make_synthetic_weights(self.graph, seed)
        handle = C.c_void_p()
        _lib.check(self.lib.b2d_create(device, self.max_batch, C.byref(handle)), "b2d_create")
        self.h = handle
        self.precision = precision
        _lib.check(self.lib.b2d_set_precision(self.h, PRECISION[precision]), "b2d_set_precision")
        self._build(w, CONV_IMPL[conv_impl])
        self.num_rows = self.lib.b2d_num_anchors(self.h)
        self.num_ops = self.lib.b2d_num_ops(self.h)
        self.num_kernels = self.lib.b2d_num_kernels_per_forward(self.h)     # ops minus those fused into a neighbour
        self.sm_count = self.lib.b2d_device_sm_count(self.h)

    # ---- plan ------------------------------------------------------------------------
    def _build(self, w: Dict[str, np.ndarray], impl: int) -> None:
        g, lib = self.graph, self.lib
        self.buf_id: Dict[str, int] = {}
        for name, b in g.bufs.items():      # "input" is first by construction
            self.buf_id[name] = _lib.check(lib.b2d_plan_buffer(self.h, b.h, b.w, b.c, int(b.f32)), f"plan_buffer {name}", index=True)
        assert self.buf_id["input"] == 0
        self.op_names = []
        for op in g.ops:
            s, d = op.src, op.dst
            if op.kind in ("conv", "dwconv"):
                wt, bs = op_weights(op, w)             # the model's weights in the buffers' channel order
                wt = np.ascontiguousarray(wt, dtype=np.float32)
                bs = np.ascontiguousarray(bs, dtype=np.float32)
                cout, cing, k, groups = g.wshapes[op.weight]
                assert wt.shape == (cout, cing, k, k), (op.weight, wt.shape)
                wp, bp = wt.ctypes.data_as(C.c_void_p), bs.ctypes.data_as(C.c_void_p)
                if op.kind == "conv":
                    res_id, res_c0 = (-1, 0) if op.res is None else (self.buf_id[op.res.buf], op.res.c0)
                    _lib.check(lib.b2d_plan_conv(self.h, self.buf_id[s.buf], s.c0, cing, self.buf_id[d.buf], d.c0, cout,
                                                 k, op.s, op.act, wp, bp, res_id, res_c0, impl), f"plan_conv {op.weight}", index=True)
                else:
                    _lib.check(lib.b2d_plan_dwconv(self.h, self.buf_id[s.buf], s.c0, self.buf_id[d.buf], d.c0, d.c,
                                                   op.act, wp, bp), f"plan_dwconv {op.weight}", index=True)
            elif op.kind == "maxpool":
                _lib.check(lib.b2d_plan_maxpool(self.h, self.buf_id[s.buf], s.c0, self.buf_id[d.buf], d.c0, d.c, op.k, op.s),
                           f"plan_maxpool {op.tag}", index=True)
            elif op.kind == "upsample2x":
                _lib.check(lib.b2d_plan_upsample2x(self.h, self.buf_id[s.buf], s.c0, self.buf_id[d.buf], d.c0, d.c),
                           f"plan_upsample {op.tag}", index=True)
            else:
                raise ValueError(op.kind)
            self.op_names.append(op.tag or op.weight)
        kind = HEAD_KIND.get(g.head["kind"], -1)                 # "seg" (config C5) has no detection levels: see segment()
        for lv in g.head["levels"]:
            anc = None
            if "anchors" in lv:
                anc = np.asarray(lv["anchors"], dtype=np.float32)
            _lib.check(lib.b2d_plan_head_level(self.h, kind, self.buf_id[lv["buf"]], lv["stride"], g.nc,
                                               None if anc is None else anc.ctypes.data_as(C.c_void_p)), "plan_head_level")
        _lib.check(lib.b2d_plan_finalize(self.h), "plan_finalize")

    def close(self) -> None:
        if getattr(self, "h", None):
            self.lib.b2d_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def describe_op(self, i: int) -> str:
        buf = C.create_string_buffer(512)
        self.lib.b2d_describe_op(self.h, i, buf, 512)
        return f"{self.op_names[i]}: {buf.value.decode()}"

    def buffer(self, name: str, n: Optional[int] = None) -> torch.Tensor:
        """Zero-copy torch view [max_batch, H, W, C] of an engine buffer (tests / debugging)."""
        b = self.graph.bufs[name]
        ptr = self.lib.b2d_buffer_ptr(self.h, self.buf_id[name])
        half = torch.bfloat16 if self.precision == "bf16" else torch.float16
        split = self.precision == "fp16x2" and not b.f32 and name != "input"
        numel = self.max_batch * b.h * b.w * b.c * (2 if split else 1)

        class _Holder:
            pass
        hold = _Holder()
        hold.__cuda_array_interface__ = {"shape": (numel,), "typestr": "<f4" if b.f32 else "<u2", "data": (ptr, False),
                                         "version": 3}
        t = torch.as_tensor(hold, device=self.device)
        if not b.f32:
            t = t.view(half)
        if split:       # [hi x 8 | lo x 8] groups -> the fp32 value hi + lo (a copy, not a view)
            t = t.view(self.max_batch, b.h, b.w, b.c // 8, 2, 8).float().sum(4).view(self.max_batch, b.h, b.w, b.c)
        else:
            t = t.view(self.max_batch, b.h, b.w, b.c)
        return t if n is None else t[:n]

    # ---- stages ------------------------------------------------------------------------
    def preprocess(self, images: torch.Tensor, mode: str = "identity", bgr: bool = False, out: str = "engine"):
        """images: uint8 CUDA tensor [n, h, w, 3] (contiguous).  out='engine' fills the network
        input; 'f32' returns float32 [n,3,S,S] (what the reference feeds session.run); 'u8'
        returns the resized uint8 image (bit-exactness tests against PIL / cv2)."""
        assert images.dtype == torch.uint8 and images.is_cuda and images.dim() == 4 and images.shape[3] == 3
        images = images.contiguous()
        n, h, w, _ = images.shape
        S = self.imgsz
        dst, kind = None, 0
        if out == "f32":
            dst, kind = torch.empty((n, 3, S, S), dtype=torch.float32, device=self.device), 1
        elif out == "u8":
            dst, kind = torch.empty((n, S, S, 3), dtype=torch.uint8, device=self.device), 2
        _lib.check(self.lib.b2d_preprocess(self.h, _ptr(images), n, h, w, w * 3, h * w * 3, RESIZE[mode], int(bgr), kind,
                                           _ptr(dst), self.stream), "preprocess")
        return dst

    def set_input_f32(self, x: torch.Tensor) -> None:
        assert x.dtype == torch.float32 and x.is_cuda and tuple(x.shape[1:]) == (3, self.imgsz, self.imgsz)
        x = x.contiguous()
        _lib.check(self.lib.b2d_set_input_f32(self.h, _ptr(x), x.shape[0], self.stream), "set_input_f32")

    def forward(self, n: int) -> None:
        _lib.check(self.lib.b2d_forward(self.h, n, self.stream), "forward")

    def run_op(self, i: int, n: int) -> None:
        _lib.check(self.lib.b2d_run_op(self.h, i, n, self.stream), f"run_op {i}")

    def fused_with_next(self, i: int) -> bool:
        """forward() runs op i and op i + 1 (depthwise 3x3 -> 1x1) as one kernel."""
        return self.lib.b2d_fused_with_next(self.h, i) == 1

    def run_op_fused(self, i: int, n: int) -> None:
        _lib.check(self.lib.b2d_run_op_fused(self.h, i, n, self.stream), f"run_op_fused {i}")

    def segment(self, n: int, with_conf: bool = True):
        """Per-pixel class of the segmentation stand-in (config C5): argmax over the ``nc`` fp32 logits of the head buffer (first
        maximum wins, like ``numpy.argmax``) as uint8 ``[n, H, W]`` and, optionally, the softmax probability of that class."""
        g = self.graph
        if g.head.get("kind") != "seg":
            raise ValueError("segment() needs a segmentation graph (arch='xunet')")
        b = g.bufs[g.head["buf"]]
        labels = torch.empty((n, b.h, b.w), dtype=torch.uint8, device=self.device)
        conf = torch.empty((n, b.h, b.w), dtype=torch.float32, device=self.device) if with_conf else None
        _lib.check(self.lib.b2d_segment(self.h, self.buf_id[g.head["buf"]], n, g.nc, _ptr(labels), _ptr(conf), self.stream), "b2d_segment")
        return (labels, conf) if with_conf else labels

    def decode_rows(self, n: int) -> torch.Tensor:
        """Dense rows [n, A, 6] (cx, cy, w, h, conf, cls); on an oriented-box engine [n, A, 7] with theta (radians, not
        regularized) as the last column."""
        if self.is_obb:
            rows = torch.empty((n, self.num_rows, 7), dtype=torch.float32, device=self.device)
            _lib.check(self.lib.b2d_decode_rows_obb(self.h, n, _ptr(rows), self.stream), "decode_rows_obb")
            return rows
        rows = torch.empty((n, self.num_rows, 6), dtype=torch.float32, device=self.device)
        _lib.check(self.lib.b2d_decode_rows(self.h, n, _ptr(rows), self.stream), "decode_rows")
        return rows

    def postprocess(self, n: int, conf_thr: float = 0.3, inclusive: bool = True, iou_thr: float = 0.0, top_k: int = 0,
                    max_det: int = 300, cap: Optional[int] = None, rows: Optional[torch.Tensor] = None
                    ) -> Tuple[torch.Tensor, torch.Tensor]:
        """Returns (dets float32 [n, cap, 8] -- view ints with .view(torch.int32) --, counts int32 [n]).  On an oriented-box engine
        dets is [n, cap, 9] ``OBB_DTYPE`` records (regularized boxes after Ultralytics' rotated NMS when iou_thr > 0)."""
        if cap is None:
            cap = _default_cap(iou_thr, top_k, max_det, self.num_rows if rows is None else rows.shape[1])
        if self.is_obb:
            if rows is not None:
                raise ValueError("postprocess(rows=...) takes axis-aligned rows; an oriented-box engine post-processes its own head maps")
            dets = torch.empty((n, cap, OBB_WORDS), dtype=torch.float32, device=self.device)
            counts = torch.empty((n,), dtype=torch.int32, device=self.device)
            _lib.check(self.lib.b2d_postprocess_obb(self.h, n, conf_thr, int(inclusive), iou_thr, top_k, max_det, _ptr(dets),
                                                    _ptr(counts), cap, self.stream), "postprocess_obb")
            return dets, counts
        dets = torch.empty((n, cap, DET_WORDS), dtype=torch.float32, device=self.device)
        counts = torch.empty((n,), dtype=torch.int32, device=self.device)
        if rows is None:
            _lib.check(self.lib.b2d_postprocess(self.h, n, conf_thr, int(inclusive), iou_thr, top_k, max_det, _ptr(dets),
                                                _ptr(counts), cap, self.stream), "postprocess")
        else:
            rows = rows.contiguous()
            assert rows.dtype == torch.float32 and rows.shape[0] == n
            _lib.check(self.lib.b2d_postprocess_rows(self.h, _ptr(rows), n, rows.shape[1], rows.shape[2], conf_thr,
                                                     int(inclusive), iou_thr, top_k, max_det, _ptr(dets), _ptr(counts), cap,
                                                     self.stream), "postprocess_rows")
        return dets, counts

    def georef(self, dets: torch.Tensor, counts: torch.Tensor, params: torch.Tensor, mode: str = "bounds") -> torch.Tensor:
        """params: float64 CUDA [n, 16].  Returns uint8 [n, cap, 40] (``GEODET_DTYPE`` records); on an oriented-box engine uint8
        [n, cap, 104] (``GEOOBB_DTYPE``: centre and four corners), forms "bounds" and "affine" only."""
        n, cap = dets.shape[0], dets.shape[1]
        assert params.dtype == torch.float64 and tuple(params.shape) == (n, GEO_PARAMS) and params.is_cuda
        if self.is_obb:
            out = torch.zeros((n, cap, GEOOBB_BYTES), dtype=torch.uint8, device=self.device)
            _lib.check(self.lib.b2d_georef_obb(self.h, _ptr(dets), _ptr(counts), n, cap, GEO[mode], _ptr(params.contiguous()), _ptr(out),
                                               self.stream), "georef_obb")
            return out
        out = torch.zeros((n, cap, GEODET_BYTES), dtype=torch.uint8, device=self.device)
        _lib.check(self.lib.b2d_georef(self.h, _ptr(dets), _ptr(counts), n, cap, GEO[mode], _ptr(params.contiguous()), _ptr(out),
                                       self.stream), "georef")
        return out

    def mosaic_nms_obb(self, dets: torch.Tensor, counts: torch.Tensor, params: torch.Tensor, conf_thr: float, iou_thr: float) -> torch.Tensor:
        """Mosaic-wide ProbIoU fast NMS of an oriented-box engine's window records (``b2d_mosaic_nms_obb``): dets float32
        [n, cap, 9] ``OBB_DTYPE`` records and counts int32 [n] as ``postprocess`` returns them, params float64 [n, 16] in the
        "affine" form of each window.  Returns keep uint8 [n, cap]: 1 for a record with ``conf > conf_thr`` that no record of
        its class with higher priority (confidence, then lower row, then lower slot) overlaps by ProbIoU >= ``iou_thr``."""
        n, cap = dets.shape[0], dets.shape[1]
        assert dets.dtype == torch.float32 and dets.is_cuda and dets.dim() == 3 and dets.shape[2] == OBB_WORDS
        assert counts.dtype == torch.int32 and tuple(counts.shape) == (n,) and counts.is_cuda
        assert params.dtype == torch.float64 and tuple(params.shape) == (n, GEO_PARAMS) and params.is_cuda
        keep = torch.empty((n, cap), dtype=torch.uint8, device=self.device)
        _lib.check(self.lib.b2d_mosaic_nms_obb(self.h, _ptr(dets.contiguous()), _ptr(counts.contiguous()), _ptr(params.contiguous()), n, cap,
                                               float(conf_thr), float(iou_thr), _ptr(keep), self.stream), "mosaic_nms_obb")
        return keep

    def dedup(self, x: torch.Tensor, y: torch.Tensor, conf: torch.Tensor, thr: float, inclusive: bool = True,
              tiebreak: Optional[torch.Tensor] = None) -> torch.Tensor:
        n = x.numel()
        keep = torch.zeros((n,), dtype=torch.uint8, device=self.device)
        if n:
            assert x.dtype == torch.float64 and y.dtype == torch.float64 and conf.dtype == torch.float32
            assert tiebreak is None or (tiebreak.dtype == torch.int64 and tiebreak.numel() == n)
            tb = None if tiebreak is None else tiebreak.contiguous()
            _lib.check(self.lib.b2d_dedup(self.h, _ptr(x.contiguous()), _ptr(y.contiguous()), _ptr(conf.contiguous()), _ptr(tb), n,
                                          float(thr), int(inclusive), _ptr(keep), self.stream), "dedup")
        return keep

    def seam_closure(self, x: torch.Tensor, y: torch.Tensor, flag: torch.Tensor, thr: float, inclusive: bool = True) -> torch.Tensor:
        """In place: closes the uint8 seam flag under the within-thr relation."""
        n = x.numel()
        if n:
            assert flag.dtype == torch.uint8 and flag.is_contiguous() and flag.numel() == n
            _lib.check(self.lib.b2d_seam_closure(self.h, _ptr(x.contiguous()), _ptr(y.contiguous()), n, float(thr), int(inclusive),
                                                 _ptr(flag), self.stream), "seam_closure")
        return flag

    def utm_forward(self, lon: torch.Tensor, lat: torch.Tensor, zone: int, north: bool):
        n = lon.numel()
        x = torch.empty_like(lon); y = torch.empty_like(lat)
        if n:
            _lib.check(self.lib.b2d_utm_forward(self.h, _ptr(lon.contiguous()), _ptr(lat.contiguous()), n, zone, int(north), _ptr(x),
                                                _ptr(y), self.stream), "utm_forward")
        return x, y

    def cut_windows(self, mosaic: torch.Tensor, origins: torch.Tensor, win: Optional[int] = None, fill: int = 114) -> torch.Tensor:
        """mosaic uint8 CUDA [H, W, 3]; origins int32 CUDA [n, 4] = (x0, y0, w0, h0)."""
        win = win or self.imgsz
        n = origins.shape[0]
        out = torch.empty((n, win, win, 3), dtype=torch.uint8, device=self.device)
        _lib.check(self.lib.b2d_cut_windows(self.h, _ptr(mosaic), mosaic.shape[0], mosaic.shape[1], mosaic.stride(0),
                                            _ptr(origins.contiguous()), n, win, fill, _ptr(out), self.stream), "cut_windows")
        return out

    def resize_windows(self, mosaic: torch.Tensor, origins, win: int, fill: int = 114, bgr: bool = False, out: str = "engine", *,
                       checked: bool = False) -> Optional[torch.Tensor]:
        """Windows of any size ``win`` resampled from the mosaic into ``imgsz`` x ``imgsz`` canvases in one launch
        (``mosaic.window_geometry``: one gain ``imgsz / win``, cv2 INTER_LINEAR, centred on ``fill``).  mosaic uint8 CUDA
        [H, W, 3] (row pitch may exceed 3 W); origins int32 [n, 4] = (x0, y0, w0, h0), NumPy or CUDA.  out='engine' fills the
        network input (n <= max_batch) and returns None; 'u8' returns uint8 [n, imgsz, imgsz, 3].  The windows are checked
        against ``win`` and the mosaic first (which reads CUDA origins back to the host); ``checked=True`` skips that for
        origins the caller has already checked with ``mosaic.check_windows``."""
        from .mosaic import check_windows
        assert mosaic.dtype == torch.uint8 and mosaic.is_cuda and mosaic.dim() == 3 and mosaic.shape[2] == 3
        assert mosaic.stride(2) == 1 and mosaic.stride(1) == 3
        if win <= 0:
            raise ValueError(f"resize_windows: window size {win} must be positive")
        if not checked:
            check_windows(origins.cpu().numpy() if isinstance(origins, torch.Tensor) else np.asarray(origins), win,
                          mosaic.shape[0], mosaic.shape[1])
        if not isinstance(origins, torch.Tensor):
            origins = torch.from_numpy(np.ascontiguousarray(origins, dtype=np.int32)).to(self.device)
        assert origins.dtype == torch.int32 and origins.is_cuda and origins.dim() == 2 and origins.shape[1] == 4
        origins = origins.contiguous()
        n = origins.shape[0]
        S = self.imgsz
        if out == "u8":
            dst, kind = torch.empty((n, S, S, 3), dtype=torch.uint8, device=self.device), 2
        elif out == "engine":
            dst, kind = None, 0
        else:
            raise ValueError(f"resize_windows: out must be 'engine' or 'u8', not {out!r}")
        _lib.check(self.lib.b2d_resize_windows(self.h, _ptr(mosaic), mosaic.shape[0], mosaic.shape[1], mosaic.stride(0), _ptr(origins),
                                               n, win, fill, int(bgr), kind, _ptr(dst), self.stream), "resize_windows")
        return dst

    # ---- test-time-augmentation views (gpu_handler.py:94-140, gpu_handler_archive.py:67-122) ---------
    def _u8(self, images: torch.Tensor) -> torch.Tensor:
        assert images.dtype == torch.uint8 and images.is_cuda and images.dim() == 4 and images.shape[3] == 3
        return images.contiguous()

    def tta_clahe(self, images: torch.Tensor, clip_limit: float, grid) -> torch.Tensor:
        """RGB2LAB -> CLAHE(clip_limit, tileGridSize) on L -> LAB2RGB, uint8 [n,h,w,3] -> same (bit-exact with cv2).
        ``grid``: an int (square grid) or cv2's ``(tiles_x, tiles_y)``."""
        images = self._u8(images)
        n, h, w, _ = images.shape
        tx, ty = (grid, grid) if isinstance(grid, int) else (int(grid[0]), int(grid[1]))
        out = torch.empty_like(images)
        _lib.check(self.lib.b2d_tta_clahe(self.h, _ptr(images), n, h, w, float(clip_limit), tx, ty, _ptr(out), self.stream),
                   "tta_clahe")
        return out

    def tta_lut(self, images: torch.Tensor, lut: np.ndarray) -> torch.Tensor:
        """Per-byte curve (brightness / gamma): out = lut[images]."""
        images = self._u8(images)
        key = bytes(np.asarray(lut, dtype=np.uint8))
        assert len(key) == 256
        cache = self.__dict__.setdefault("_lut_cache", {})
        if key not in cache:
            cache[key] = torch.from_numpy(np.frombuffer(key, dtype=np.uint8).copy()).to(self.device)
        out = torch.empty_like(images)
        n = images.shape[0]
        _lib.check(self.lib.b2d_tta_lut(self.h, _ptr(images), n, images[0].numel(), _ptr(cache[key]), 0, _ptr(out), self.stream),
                   "tta_lut")
        return out

    def tta_contrast(self, images: torch.Tensor, factor: float) -> torch.Tensor:
        """PIL ImageEnhance.Contrast(img).enhance(factor) per image."""
        images = self._u8(images)
        n, h, w, _ = images.shape
        out = torch.empty_like(images)
        _lib.check(self.lib.b2d_tta_contrast(self.h, _ptr(images), n, h, w, float(factor), _ptr(out), self.stream), "tta_contrast")
        return out

    def colour_convert(self, pixels: torch.Tensor, code: str) -> torch.Tensor:
        """cv2.cvtColor on uint8 [..., 3]: code 'rgb2lab' or 'lab2rgb'."""
        assert pixels.dtype == torch.uint8 and pixels.is_cuda and pixels.shape[-1] == 3
        pixels = pixels.contiguous()
        out = torch.empty_like(pixels)
        _lib.check(self.lib.b2d_colour_convert(self.h, _ptr(pixels), pixels.numel() // 3, {"rgb2lab": 0, "lab2rgb": 1}[code],
                                               _ptr(out), self.stream), "colour_convert")
        return out

    def tta_views(self, images: torch.Tensor, views: Sequence[Tuple[str, tuple]]) -> list:
        """The uint8 views of a batch of tiles, in the reference's order (``tta.LIGHTING_VIEWS + tta.OCCLUSION_VIEWS``
        for gpu_handler.py:94-140; ``tta.ARCHIVE_VIEWS`` for the archived handler)."""
        images = self._u8(images)
        out, chain = [], images
        for kind, args in views:
            if kind == "original":
                out.append(images)
            elif kind == "clahe":
                out.append(self.tta_clahe(images, args[0], args[1]))
            elif kind == "brightness":
                out.append(self.tta_lut(images, _tta.brightness_lut(args[0])))
            elif kind == "gamma":
                out.append(self.tta_lut(images, _tta.gamma_lut(args[0])))
            elif kind == "chain":       # cumulative brightness -> contrast (gpu_handler_archive.py:79-84)
                chain = self.tta_contrast(self.tta_lut(chain, _tta.brightness_lut(args[0])), args[1])
                out.append(chain)
            else:
                raise ValueError(kind)
        return out

    def set_conf_scale(self, scale: float) -> None:
        _lib.check(self.lib.b2d_set_conf_scale(self.h, float(scale)), "set_conf_scale")

    # ---- whole path ----------------------------------------------------------------------
    def detect_host(self, tiles, params, resize: str = "identity", bgr: bool = False, conf_thr: float = 0.3, inclusive: bool = True,
                    iou_thr: float = 0.0, top_k: int = 0, max_det: int = 300, cap: Optional[int] = None, geo: str = "bounds"):
        """Host tiles in, host records out, in ONE C call (``b2d_detect_host``): ``tiles`` uint8 [n,h,w,3] (NumPy array or CPU
        tensor; any n, pinned memory overlaps the copies), ``params`` float64 [n,16].  Returns one ``GEODET_DTYPE`` array per tile."""
        if self.is_obb:
            raise _lib.B2DError("detect_host returns axis-aligned records; on an oriented-box engine use infer() + georef()")
        t = _host_array(tiles, np.uint8)
        p = _host_array(params, np.float64)
        n, h, w, _ = t.shape
        assert p.shape == (n, GEO_PARAMS)
        if cap is None:
            cap = _default_cap(iou_thr, top_k, max_det, self.num_rows)
        out = np.zeros((n, cap), dtype=GEODET_DTYPE)
        counts = np.zeros((n,), dtype=np.int32)
        _lib.check(self.lib.b2d_detect_host(self.h, C.c_void_p(t.ctypes.data), n, h, w, RESIZE[resize], int(bgr), conf_thr,
                                            int(inclusive), iou_thr, top_k, max_det, GEO[geo], C.c_void_p(p.ctypes.data),
                                            C.c_void_p(out.ctypes.data), C.c_void_p(counts.ctypes.data), cap, self.stream),
                   "detect_host")
        return [out[i, :counts[i]].copy() for i in range(n)]

    def infer(self, images: torch.Tensor, resize: str = "identity", bgr: bool = False, conf_thr: float = 0.3,
              inclusive: bool = True, iou_thr: float = 0.0, top_k: int = 0, max_det: int = 300, cap: Optional[int] = None,
              conf_scale: float = 1.0):
        """uint8 CUDA tiles -> (dets, counts) on device: preprocess + network + decode/filter(/NMS)."""
        n = images.shape[0]
        assert n <= self.max_batch
        self.preprocess(images, resize, bgr)
        self.forward(n)
        if conf_scale == 1.0:
            return self.postprocess(n, conf_thr, inclusive, iou_thr, top_k, max_det, cap)
        self.set_conf_scale(conf_scale)
        try:
            return self.postprocess(n, conf_thr, inclusive, iou_thr, top_k, max_det, cap)
        finally:
            self.set_conf_scale(1.0)


def require_axis_aligned(engine, who: str) -> None:
    """The front-ends that mirror the reference (GPUHandler and its test-time augmentation, SimpleDetector, InferenceSession,
    MosaicDetector) return axis-aligned records; built on an oriented-box engine they stop here instead of misreading its output."""
    if getattr(engine, "is_obb", False):
        raise ValueError(f"{who} handles axis-aligned detections only; {engine.arch!r} is an oriented-box model: "
                         "use Engine.infer / Engine.postprocess and Engine.georef, which return OBB_DTYPE / GEOOBB_DTYPE records")


def _host_array(x, dtype) -> np.ndarray:
    a = x.numpy() if isinstance(x, torch.Tensor) else np.asarray(x)
    assert a.dtype == dtype
    return np.ascontiguousarray(a)


def dets_to_numpy(dets: torch.Tensor, counts: torch.Tensor):
    """Device (dets, counts) -> list of structured arrays (``DET_DTYPE``), one per tile."""
    d = dets.cpu().numpy().view(np.uint8).reshape(dets.shape[0], dets.shape[1], 32).view(DET_DTYPE)[..., 0]
    c = counts.cpu().numpy()
    return [d[i, :c[i]].copy() for i in range(len(c))]


def geodets_to_numpy(geo: torch.Tensor, counts: torch.Tensor):
    g = geo.cpu().numpy().view(GEODET_DTYPE)[..., 0]
    c = counts.cpu().numpy()
    return [g[i, :c[i]].copy() for i in range(len(c))]


def obbs_to_numpy(dets: torch.Tensor, counts: torch.Tensor):
    """Device (dets, counts) of an oriented-box engine -> list of structured arrays (``OBB_DTYPE``), one per tile."""
    d = dets.cpu().numpy().view(np.uint8).reshape(dets.shape[0], dets.shape[1], 4 * OBB_WORDS).view(OBB_DTYPE)[..., 0]
    c = counts.cpu().numpy()
    return [d[i, :c[i]].copy() for i in range(len(c))]


def geoobbs_to_numpy(geo: torch.Tensor, counts: torch.Tensor):
    g = geo.cpu().numpy().view(GEOOBB_DTYPE)[..., 0]
    c = counts.cpu().numpy()
    return [g[i, :c[i]].copy() for i in range(len(c))]
