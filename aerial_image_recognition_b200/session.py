"""``onnxruntime.InferenceSession``-shaped front of the engine.

Reference code talks to its model through three calls only --
``session.run(None, {session.get_inputs()[0].name: ndarray})`` and
``session.get_providers()`` (``simple_detector.py:470-477``, ``:663-669``;
``_script/gpu_handler.py:165``) -- so this object provides exactly those, backed
by the B200 engine.  ``run`` takes the float32 ``[B,3,640,640]`` tensor the
reference builds, and returns ``[rows]`` with ``rows`` float32 ``[B, N, 6]`` =
``(cx, cy, w, h, conf, cls)`` so that ``outputs[0][0]`` and ``boxes[:, 4]`` keep
their meaning (``simple_detector.py:479-480``).
"""
from __future__ import annotations

import os
from typing import Dict, List, Optional, Union

import numpy as np
import torch

from .engine import Engine, require_axis_aligned


class _Input:
    def __init__(self, name, shape):
        self.name = name
        self.shape = shape
        self.type = "tensor(float)"


def arch_from_model_path(model_path: Optional[str]) -> str:
    """The reference selects the network by file name only (``_script/config.py:25``,
    ``simple_detector.py:710``)."""
    name = os.path.basename(model_path or "").lower()
    if "yolov8" in name or "tokyo" in name or "v8" in name:
        return "yolov8m"
    if "yolo7" in name or "yolov7" in name or "itcvd" in name:
        return "yolov7"
    return "yolov8m"


SYNTHETIC = "synthetic"      # explicit opt-in for seeded random weights (bench, tests): ``weights="synthetic"``


def resolve_weights(model_path: Optional[str], arch: str, weights: Union[None, str, Dict[str, np.ndarray]]
                    ) -> Optional[Dict[str, np.ndarray]]:
    """What ``GPUHandler`` / ``SimpleDetector`` / ``InferenceSession`` hand to the engine: the caller's tensors, the
    tensors of ``model_path``, or ``None`` (= the engine's seeded synthetic weights) only for ``weights="synthetic"``."""
    if isinstance(weights, str):
        if weights != SYNTHETIC:
            raise ValueError(f"weights={weights!r}: expected a dict of tensors or {SYNTHETIC!r}")
        return None
    if weights is not None:
        return weights
    return load_weights(model_path, arch)


def load_weights(model_path: Optional[str], arch: Optional[str] = None) -> Dict[str, np.ndarray]:
    """Deploy-form tensors (``model.N....weight`` / ``.bias``) from ``model_path``:

    * ``.onnx`` -- what the reference loads (``_script/config.py:25``, ``simple_detector.py:710``): the
      convolution weights are read straight from the protobuf (``onnx_reader.py``, no ``onnx`` package)
      and checked against the engine's graph for ``arch``;
    * ``.npz`` -- the same tensors saved with ``numpy.savez``.

    A missing file raises ``FileNotFoundError``, as ``ort.InferenceSession(model_path)`` does in the reference
    (``_script/gpu_handler.py:61-65``): a mistyped path must not silently produce detections from random weights.
    The reference's own blobs are absent (``.MISSING_LARGE_BLOBS:2-5``), so benchmarks and tests opt in to seeded
    synthetic weights explicitly with ``weights="synthetic"`` (``resolve_weights``)."""
    if model_path and os.path.exists(model_path):
        if model_path.endswith(".npz"):
            with np.load(model_path) as z:
                return {k: z[k] for k in z.files}
        if model_path.endswith(".onnx"):
            from .graph import build
            from .onnx_reader import load_onnx_weights
            return load_onnx_weights(model_path, build(arch or arch_from_model_path(model_path)))
        raise ValueError(f"{model_path}: unknown model file type (expected .onnx or .npz)")
    raise FileNotFoundError(f"model file {model_path!r} not found (pass weights=\"synthetic\" to run seeded synthetic "
                            f"weights of the architecture instead)")


class InferenceSession:
    def __init__(self, model_path: Optional[str] = None, sess_options=None, providers=None, *, arch: Optional[str] = None,
                 weights: Union[None, str, Dict[str, np.ndarray]] = None, max_batch: int = 8, device: int = 0, seed: int = 0,
                 engine: Optional[Engine] = None, precision: str = "bf16"):
        if engine is None:
            arch = arch or arch_from_model_path(model_path)
            weights = resolve_weights(model_path, arch, weights)
            engine = Engine(arch, weights=weights, max_batch=max_batch, device=device, seed=seed, precision=precision)
        require_axis_aligned(engine, "InferenceSession")
        self.engine = engine
        self._inputs = [_Input("images", [None, 3, engine.imgsz, engine.imgsz])]

    def get_inputs(self) -> List[_Input]:
        return self._inputs

    def get_providers(self) -> List[str]:
        # the reference only tests for 'CUDAExecutionProvider' to decide whether to synchronise
        return ["B200ExecutionProvider", "CUDAExecutionProvider"]

    def run(self, output_names, feed: Dict[str, np.ndarray]):
        (x,) = feed.values()
        x = np.ascontiguousarray(x, dtype=np.float32)
        eng = self.engine
        outs = []
        for i in range(0, x.shape[0], eng.max_batch):
            xb = torch.from_numpy(x[i:i + eng.max_batch]).to(eng.device, non_blocking=False)
            eng.set_input_f32(xb)
            eng.forward(xb.shape[0])
            outs.append(eng.decode_rows(xb.shape[0]).cpu().numpy())
        return [np.concatenate(outs, 0)]
