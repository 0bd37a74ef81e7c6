"""Seeded synthetic deploy-form weights for the detector graphs.

Every model blob the reference loads is absent (``.MISSING_LARGE_BLOBS:2-5``;
``_script/config.py:25``, ``simple_detector.py:710``), and there is no network,
so throughput and parity are measured with random-init weights of the right
architecture.  The generator is deterministic in ``(arch, nc, seed)``.

* conv weights are He-style, rounded to bf16-representable fp32 so the 16-bit
  engine and the fp32 oracle see *the same* weights (what is compared is the
  arithmetic, not a quantiser); BatchNorm is already folded (``.weight`` / ``.bias``);
* every conv is rescaled, layer by layer in graph order, so that its
  pre-activation has standard deviation ``PREACT_STD`` = 4 on two seeded 640x640
  tiles.  4, not 1: the map "input std -> output std" of a SiLU layer has
  elasticity 1.10 at std 1 (a tile with 6 % more contrast ends 60 layers later
  with 8x the logit spread -- measured) and 0.99 at std 4, so the statistics of
  the head stay put from tile to tile, as a trained network's do;
* the detect head is calibrated like a trained one (SURVEY.md section 7 step 1a):
  DFL logits are peaked -- bin k of a box side gets ``2 k d - k^2`` where the
  distance ``d`` (in cells, mean 1.5, std 1) is one linear feature of the branch,
  i.e. a discrete Gaussian around ``d`` with std 0.7, plus a small random part --
  and the last cls / objectness bias is placed so that about 6 % of the v8
  anchors (~500 of 8400 per tile) clear conf 0.25 (2 % of the 25200 v7 rows
  clear the reference's 0.3, ``simple_detector.py:30``);
* the oriented-box head's angle logits (``yolov8m-obb``, cv4) get mean 0 and std ``ANGLE_STD`` = 1.5, so that the decoded
  angle (sigmoid(z) - 0.25) * pi covers most of (-pi/4, 3pi/4) and the rotated NMS sees truly rotated boxes.
"""
from __future__ import annotations

import os
import sys
from typing import Dict, Tuple

import numpy as np

from .graph import Graph, op_weights

PREACT_STD = 4.0          # LSUV target of every SiLU conv (see the module docstring)
CAL_SIZE, CAL_TILES = 640, 2
DFL_SIGMA_D, DFL_D0, DFL_NOISE = 1.0, 1.5, 0.25
CLS_STD, V8_PASS_FRACTION, V7_PASS_FRACTION = 2.0, 0.06, 0.02
ANGLE_STD = 1.5                # OBB angle logits (yolov8m-obb)
GENERATOR_VERSION = 2          # part of the seed: bump when the recipe changes

_CACHE: Dict[Tuple, Dict[str, np.ndarray]] = {}


def round_to_bf16(x: np.ndarray) -> np.ndarray:
    """Round-to-nearest-even fp32 -> bf16 -> fp32 (NaN-free inputs)."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    u = x.view(np.uint32).astype(np.uint64)
    u = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000
    return u.astype(np.uint32).view(np.float32).reshape(x.shape)


def f32_to_bf16_bits(x: np.ndarray) -> np.ndarray:
    x = np.ascontiguousarray(x, dtype=np.float32)
    u = x.view(np.uint32).astype(np.uint64)
    u = (u + 0x7FFF + ((u >> 16) & 1)) >> 16
    return u.astype(np.uint16).reshape(x.shape)


def _quantised_scale(s: float) -> float:
    """Snap a calibration scale to 2**(j/8) so last-bit differences in the CPU
    conv used for calibration cannot change the generated weights."""
    return float(2.0 ** (np.round(np.log2(max(s, 1e-12)) * 8.0) / 8.0))


def _snap(v, bits: int = 12):
    """Round calibration-derived biases to multiples of 2**-bits.  They come out of CPU reductions whose last bits depend on
    the thread count (torchrun sets OMP_NUM_THREADS=1): un-snapped, two ranks of one job would run weights that differ in
    the last ulp.  The statistics themselves are taken in float64 with NumPy's (single-threaded) reductions."""
    return np.round(np.asarray(v, dtype=np.float64) * (1 << bits)) / (1 << bits)


def _final_layers(graph: Graph):
    if graph.head["kind"] == "seg":        # segmentation stand-in: the logits layer is scaled like every other conv
        return set(), set()
    if graph.head["kind"] in ("v8_dfl", "v8_obb"):
        return {f"model.22.cv2.{i}.2" for i in range(3)}, {f"model.22.cv3.{i}.2" for i in range(3)}
    return set(), {f"model.105.m.{i}" for i in range(3)}


def _angle_layers(graph: Graph):
    return {f"model.22.cv4.{i}.2" for i in range(3)} if graph.head["kind"] == "v8_obb" else set()


def make_synthetic_weights(graph: Graph, seed: int = 0, calibrate: bool = True) -> Dict[str, np.ndarray]:
    """Deterministic deploy-form weights for ``graph`` (independent of ``graph.imgsz``).

    ``calibrate=False`` skips the layer-sequential rescale and the head calibration (shape-only
    uses: the ONNX reader tests)."""
    key = (graph.arch, graph.nc, seed, calibrate)
    if key in _CACHE:
        return {k: v.copy() for k, v in _CACHE[key].items()}
    disk = _disk_cache_path(key) if calibrate else None
    if disk and os.path.exists(disk):
        try:
            with np.load(disk) as z:
                w = {k: z[k] for k in z.files}
            _CACHE[key] = {k: v.copy() for k, v in w.items()}
            return w
        except Exception:
            pass                      # unreadable cache file: regenerate
    rng = np.random.default_rng([seed, 0xB200, GENERATOR_VERSION])
    w: Dict[str, np.ndarray] = {}
    box_final, _ = _final_layers(graph)
    for name, (cout, cing, k, groups) in graph.wshapes.items():
        fan_in = cing * k * k
        std = (2.0 / fan_in) ** 0.5
        wt = rng.standard_normal((cout, cing, k, k), dtype=np.float32) * np.float32(std)
        b = rng.standard_normal(cout, dtype=np.float32) * np.float32(0.1)
        if name in box_final:
            # DFL rows of one box side share a direction v (the "distance" feature): row k = k * v + noise
            for side in range(4):
                v = rng.standard_normal(cing).astype(np.float32) / np.float32(np.sqrt(cing))
                for kk in range(16):
                    r = wt[side * 16 + kk, :, 0, 0]
                    wt[side * 16 + kk, :, 0, 0] = kk * v + DFL_NOISE * r / np.linalg.norm(r) * np.linalg.norm(v)
        w[name + ".weight"] = round_to_bf16(wt)
        w[name + ".bias"] = b.astype(np.float32)
    if calibrate:
        _calibrate(graph, w, seed)
    _CACHE[key] = {k: v.copy() for k, v in w.items()}
    if disk:
        try:                          # the calibration takes ~10 s on one thread; every process of a job wants the same tensors
            os.makedirs(os.path.dirname(disk), exist_ok=True)
            tmp = f"{disk}.{os.getpid()}.tmp.npz"
            np.savez(tmp, **w)
            os.replace(tmp, disk)
        except OSError:
            pass
    return w


def _disk_cache_path(key) -> str:
    """Generated weights are cached on disk, keyed by the arguments and by a hash of this generator's own source (and of the
    graph / tile generators it calibrates on), so an edit to any of them invalidates the cache."""
    import hashlib
    import tempfile
    from . import graph as _g, synth as _s
    h = hashlib.sha256()
    for mod in (sys.modules[__name__], _g, _s):
        with open(mod.__file__, "rb") as f:
            h.update(f.read())
    root = os.environ.get("B2D_WEIGHT_CACHE", os.path.join(tempfile.gettempdir(), "b2det_weights"))
    return os.path.join(root, f"{key[0]}_nc{key[1]}_seed{key[2]}_{h.hexdigest()[:16]}.npz")


def _calibrate(graph: Graph, w: Dict[str, np.ndarray], seed: int) -> None:
    """Layer-sequential rescale on two calibration tiles (CPU torch; this is weight *generation*,
    not the inference path)."""
    import torch
    import torch.nn.functional as F
    from .graph import build
    from .synth import make_tiles

    # One CPU thread: the blocking (hence the summation order) of the CPU convolutions depends on the thread count, and the
    # head biases below are derived from their outputs -- every process of a job (torchrun sets OMP_NUM_THREADS=1, a plain
    # `python bench.py` does not) must generate bit-identical weights, or shards of one mosaic disagree in the last ulp.
    threads = torch.get_num_threads()
    torch.set_num_threads(1)
    try:
        _calibrate_single_thread(graph, w, seed)
    finally:
        torch.set_num_threads(threads)


def _calibrate_single_thread(graph: Graph, w: Dict[str, np.ndarray], seed: int) -> None:
    import torch
    import torch.nn.functional as F
    from .graph import build
    from .synth import make_tiles

    g = build(graph.arch, graph.nc, 256 if graph.arch == "xunet" else CAL_SIZE)
    cal_size = g.imgsz
    box_final, cls_final = _final_layers(g)
    v8 = g.head["kind"] in ("v8_dfl", "v8_obb")
    angle_final = _angle_layers(g)
    x = torch.from_numpy(make_tiles(CAL_TILES, cal_size, seed=seed + 7919).astype(np.float32) / 255.0).permute(0, 3, 1, 2)
    bufs = {n: torch.zeros(CAL_TILES, b.c, b.h, b.w) for n, b in g.bufs.items()}
    bufs["input"][:, :3] = x
    inv = lambda op, a: a if op.out_perm is None else a[np.argsort(np.asarray(op.out_perm))]    # buffer order -> model order
    with torch.no_grad():
        for op in g.ops:
            src = bufs[op.src.buf][:, op.src.c0:op.src.c0 + op.src.c]
            if op.kind in ("conv", "dwconv"):
                if op.src.buf == "input":
                    src = src[:, :3]
                name = op.weight
                groups = g.wshapes[name][3]
                wt, b = (np.ascontiguousarray(a) for a in op_weights(op, w))          # buffer channel order
                y = F.conv2d(src, torch.from_numpy(wt), None, stride=op.s, padding=op.k // 2, groups=groups)
                cout = wt.shape[0]
                sc = np.ones(cout, dtype=np.float32)
                if name in box_final:
                    # logit of bin k = 2 k d - k^2 (+ noise), d = D0 + SIGMA_D * (feature - mean) / std per side
                    ks = np.arange(16, dtype=np.float32)
                    for side in range(4):
                        rows = slice(side * 16, side * 16 + 16)
                        f1 = y[:, side * 16 + 1]                                       # row 1 = v . x (+ its noise)
                        s1 = _quantised_scale(2.0 * DFL_SIGMA_D / float(f1.std()))
                        sc[rows] = s1
                        mean = y[:, rows].numpy().astype(np.float64).mean(axis=(0, 2, 3))
                        b[rows] = _snap(b[rows] - mean * s1 + 2.0 * ks * DFL_D0 - ks * ks)
                elif name in cls_final:
                    s1 = _quantised_scale(CLS_STD / float(y.std()))
                    sc[:] = s1
                    z = y * s1
                    if v8:
                        score = z.amax(1)                                               # conf = max class logit
                        thr, frac = float(np.log(0.25 / 0.75)), V8_PASS_FRACTION
                        shift = thr - float(np.quantile(score.numpy().ravel().astype(np.float64), 1.0 - frac))
                        b[:] = _snap(b + shift)
                    else:
                        no = g.nc + 5
                        obj = z.view(z.shape[0], 3, no, z.shape[2], z.shape[3])[:, :, 4]
                        thr, frac = float(np.log(0.3 / 0.7)), V7_PASS_FRACTION
                        shift = thr - float(np.quantile(obj.numpy().ravel().astype(np.float64), 1.0 - frac))
                        bb = b.reshape(3, no)
                        bb[:, 4] = _snap(bb[:, 4] + shift)
                        b = bb.reshape(-1)
                elif name in angle_final:
                    # theta = (sigmoid(z) - 0.25) pi: logits of std ANGLE_STD around 0 spread theta over most of (-pi/4, 3pi/4)
                    s1 = _quantised_scale(ANGLE_STD / float(y.std()))
                    sc[:] = s1
                    b[:] = _snap(-float(y.numpy().astype(np.float64).mean()) * s1)
                else:
                    sc[:] = _quantised_scale(PREACT_STD / float(y.std()))
                w[name + ".weight"] = round_to_bf16(w[name + ".weight"] * inv(op, sc)[:, None, None, None])   # model order
                w[name + ".bias"] = inv(op, b).astype(np.float32)
                wt, b = (torch.from_numpy(np.ascontiguousarray(a)) for a in op_weights(op, w))
                y = F.conv2d(src, wt, b, stride=op.s, padding=op.k // 2, groups=groups)
                if op.act:
                    y = y * torch.sigmoid(y)
                if op.res is not None:
                    y = y + bufs[op.res.buf][:, op.res.c0:op.res.c0 + op.res.c]
            elif op.kind == "maxpool":
                y = F.max_pool2d(src, op.k, op.s, op.k // 2 if op.s == 1 else 0)
            else:
                y = F.interpolate(src, scale_factor=2, mode="nearest")
            bufs[op.dst.buf][:, op.dst.c0:op.dst.c0 + op.dst.c] = y


def weights_fingerprint(w: Dict[str, np.ndarray]) -> str:
    import hashlib
    h = hashlib.sha256()
    for k in sorted(w):
        h.update(k.encode())
        h.update(np.ascontiguousarray(w[k]).tobytes())
    return h.hexdigest()[:16]
