"""Weights out of an ``.onnx`` file without the ``onnx`` package (SURVEY.md section 8f-1).

The reference hands its model to onnxruntime by path -- ``ort.InferenceSession(model_path, ...)``
(``_script/gpu_handler.py:61-65``, ``simple_detector.py:39-46``), the path coming from
``_script/config.py:25`` / ``simple_detector.py:710``.  The engine executes its own fixed graph
(``graph.py``), so all it needs from the file are the convolution weights.  ``onnx`` is not
installable here; an ONNX file is a protobuf ``ModelProto``, and the handful of fields needed
(``graph.node``, ``graph.initializer``, tensor ``dims / data_type / raw_data / float_data``) are
read with a ~100-line wire-format walker.

Mapping onto the engine's conv names (``model.2.m.0.cv1`` ...):

1. by initializer name -- an Ultralytics export of a fused model keeps the module path
   (``model.2.m.0.cv1.conv.weight``; the head's plain ``nn.Conv2d`` are ``model.22.cv2.0.2.weight``);
2. otherwise by order -- the ``Conv`` nodes of the file in graph order against the engine's conv
   ops in execution order (both follow the module's forward), for exporters that rename folded
   weights to ``onnx::Conv_123``.

Either way every tensor is checked against the shape the engine's graph expects, the DFL
``arange`` conv (fixed weights, part of the decode kernel here) is skipped, and a file of another
architecture fails loudly instead of running with wrong weights.
"""
from __future__ import annotations

import struct
from typing import Dict, Iterator, List, Optional, Tuple

import numpy as np

from .graph import Graph

# ---- protobuf wire format -------------------------------------------------------------------------


def _varint(buf: memoryview, pos: int) -> Tuple[int, int]:
    result = shift = 0
    while True:
        b = buf[pos]
        pos += 1
        result |= (b & 0x7F) << shift
        if not b & 0x80:
            return result, pos
        shift += 7


def _fields(buf: memoryview) -> Iterator[Tuple[int, int, object]]:
    """Yields (field number, wire type, value); length-delimited values are memoryviews."""
    pos, n = 0, len(buf)
    while pos < n:
        key, pos = _varint(buf, pos)
        fno, wt = key >> 3, key & 7
        if wt == 0:
            v, pos = _varint(buf, pos)
        elif wt == 1:
            v = bytes(buf[pos:pos + 8]); pos += 8
        elif wt == 2:
            ln, pos = _varint(buf, pos)
            v = buf[pos:pos + ln]; pos += ln
        elif wt == 5:
            v = bytes(buf[pos:pos + 4]); pos += 4
        else:
            raise ValueError(f"unsupported protobuf wire type {wt}")
        yield fno, wt, v


def _packed_varints(v, wt) -> List[int]:
    if wt == 0:
        return [v]
    out, pos = [], 0
    while pos < len(v):
        x, pos = _varint(v, pos)
        out.append(x)
    return out


# TensorProto.DataType -> numpy
_DTYPES = {1: np.float32, 2: np.uint8, 3: np.int8, 5: np.int16, 6: np.int32, 7: np.int64, 10: np.float16, 11: np.float64}


def _tensor(buf: memoryview) -> Tuple[str, Optional[np.ndarray]]:
    """TensorProto -> (name, array); bf16 (16) is widened to float32; external data is rejected."""
    dims: List[int] = []
    dtype, name, raw = 1, "", None
    floats: List[float] = []
    int64s: List[int] = []
    for fno, wt, v in _fields(buf):
        if fno == 1:
            dims += _packed_varints(v, wt)
        elif fno == 2:
            dtype = v
        elif fno == 8:
            name = bytes(v).decode()
        elif fno == 9:
            raw = bytes(v)
        elif fno == 4:                       # float_data, packed or not
            floats += list(struct.unpack(f"<{len(v) // 4}f", bytes(v))) if wt == 2 else [struct.unpack("<f", v)[0]]
        elif fno == 7:
            int64s += _packed_varints(v, wt)
        elif fno == 14 and v:                # data_location = EXTERNAL
            raise ValueError(f"initializer {name!r} uses external data; export with the weights inside the .onnx file")
    if raw is not None:
        if dtype == 16:                      # bfloat16
            a = (np.frombuffer(raw, dtype=np.uint16).astype(np.uint32) << 16).view(np.float32)
        elif dtype in _DTYPES:
            a = np.frombuffer(raw, dtype=_DTYPES[dtype])
        else:
            return name, None
    elif floats:
        a = np.asarray(floats, dtype=np.float32)
    elif int64s:
        a = np.asarray(int64s, dtype=np.int64)
    else:
        a = np.zeros(0, dtype=_DTYPES.get(dtype, np.float32))
    return name, a.reshape(dims) if dims else a


class OnnxNode:
    __slots__ = ("op_type", "name", "inputs", "outputs", "attrs")

    def __init__(self):
        self.op_type, self.name, self.inputs, self.outputs, self.attrs = "", "", [], [], {}


def _node(buf: memoryview) -> OnnxNode:
    nd = OnnxNode()
    for fno, wt, v in _fields(buf):
        if fno == 1:
            nd.inputs.append(bytes(v).decode())
        elif fno == 2:
            nd.outputs.append(bytes(v).decode())
        elif fno == 3:
            nd.name = bytes(v).decode()
        elif fno == 4:
            nd.op_type = bytes(v).decode()
        elif fno == 5:                       # AttributeProto: name 1, i 3, ints 8
            an, ai, ais = "", None, []
            for f2, w2, v2 in _fields(v):
                if f2 == 1:
                    an = bytes(v2).decode()
                elif f2 == 3:
                    ai = v2
                elif f2 == 8:
                    ais += _packed_varints(v2, w2)
            nd.attrs[an] = ais if ais else ai
    return nd


def read_onnx(path: str) -> Tuple[List[OnnxNode], Dict[str, np.ndarray]]:
    """(nodes in graph order, initializers by name) of an ONNX ModelProto file."""
    with open(path, "rb") as f:
        data = memoryview(f.read())
    graph = None
    for fno, wt, v in _fields(data):
        if fno == 7 and wt == 2:             # ModelProto.graph
            graph = v
    if graph is None:
        raise ValueError(f"{path}: no graph in the file (not an ONNX model?)")
    nodes: List[OnnxNode] = []
    inits: Dict[str, np.ndarray] = {}
    for fno, wt, v in _fields(graph):
        if fno == 1 and wt == 2:             # GraphProto.node
            nodes.append(_node(v))
        elif fno == 5 and wt == 2:           # GraphProto.initializer
            name, arr = _tensor(v)
            if arr is not None:
                inits[name] = arr
    return nodes, inits


# ---- mapping onto the engine's graph --------------------------------------------------------------


def _conv_names(g: Graph) -> List[str]:
    return [op.weight for op in g.ops if op.kind in ("conv", "dwconv")]


def _expected_shape(g: Graph, name: str) -> Tuple[int, int, int, int]:
    cout, cing, k, _groups = g.wshapes[name]
    return (cout, cing, k, k)


def _check_conv_node(path: str, g: Graph, name: str, nd: "OnnxNode") -> None:
    """The file's Conv node for ``name`` must be the convolution the engine's graph runs: kernel, stride, groups."""
    op = next(o for o in g.ops if o.kind in ("conv", "dwconv") and o.weight == name)
    _cout, _cing, k, groups = g.wshapes[name]
    ks, st, gr = nd.attrs.get("kernel_shape"), nd.attrs.get("strides"), nd.attrs.get("group")
    if ks is not None and list(ks) != [k, k]:
        raise ValueError(f"{path}: Conv node {nd.name!r} has kernel_shape {list(ks)}, the {g.arch} graph runs {name} with {k}x{k}")
    if st is not None and list(st) != [op.s, op.s]:
        raise ValueError(f"{path}: Conv node {nd.name!r} has strides {list(st)}, the {g.arch} graph runs {name} with stride {op.s}")
    if (gr or 1) != groups:
        raise ValueError(f"{path}: Conv node {nd.name!r} has group {gr or 1}, the {g.arch} graph runs {name} with {groups} groups")


def load_onnx_weights(path: str, g: Graph, by_name: bool = True) -> Dict[str, np.ndarray]:
    """Deploy-form weights ``{name + '.weight', name + '.bias'}`` (float32, the model's own channel
    order) for every conv of ``g`` from the ONNX file at ``path``.  ``by_name=False`` skips the name
    mapping and goes by graph order (what happens anyway when an exporter has renamed the weights)."""
    nodes, inits = read_onnx(path)
    names = _conv_names(g)
    out: Dict[str, np.ndarray] = {}
    # The engine runs deploy-form convolutions (BatchNorm folded into weight + bias, as Ultralytics / YOLOv7 exports are):
    # a file that still carries BatchNormalization nodes would silently lose its scale and shift.
    bn = [nd.name or nd.outputs[0] for nd in nodes if nd.op_type == "BatchNormalization"]
    if bn:
        raise ValueError(f"{path}: {len(bn)} BatchNormalization nodes (e.g. {bn[0]!r}); export the fused (eval-mode) model -- the engine "
                         f"runs convolutions with BatchNorm folded in")
    consumer = {nd.inputs[1]: nd for nd in nodes if nd.op_type == "Conv" and len(nd.inputs) > 1}

    def put(name: str, wt: np.ndarray, bs: Optional[np.ndarray], where: str) -> None:
        exp = _expected_shape(g, name)
        if tuple(wt.shape) != exp:
            raise ValueError(f"{path}: {where} has shape {tuple(wt.shape)}, the {g.arch} graph expects {exp} for {name}")
        out[name + ".weight"] = np.ascontiguousarray(wt, dtype=np.float32)
        out[name + ".bias"] = (np.zeros(exp[0], np.float32) if bs is None else np.ascontiguousarray(bs, dtype=np.float32).reshape(exp[0]))

    # 1. by initializer name (Ultralytics keeps the module path; Conv modules add '.conv')
    found = 0
    for name in names if by_name else []:
        for stem in (name + ".conv", name):
            if stem + ".weight" in inits:
                put(name, inits[stem + ".weight"], inits.get(stem + ".bias"), f"initializer {stem}.weight")
                if stem + ".weight" in consumer:
                    _check_conv_node(path, g, name, consumer[stem + ".weight"])
                found += 1
                break
    by_name = found
    if by_name == len(names):
        return out
    if by_name:
        missing = [n for n in names if n + ".weight" not in out][:4]
        raise ValueError(f"{path}: only {by_name} of {len(names)} convolutions found by name (missing e.g. {missing}); "
                         f"is this a {g.arch} export?")

    # 2. by order: Conv nodes of the file against the engine's conv ops; the DFL arange conv (1 x 16 x 1 x 1) is not a layer here
    convs = []
    for nd in nodes:
        if nd.op_type != "Conv" or len(nd.inputs) < 2 or nd.inputs[1] not in inits:
            continue
        wt = inits[nd.inputs[1]]
        if wt.ndim == 4 and wt.shape[0] == 1 and wt.shape[1] == 16 and wt.shape[2:] == (1, 1):
            continue
        convs.append((nd, wt, inits.get(nd.inputs[2]) if len(nd.inputs) > 2 else None))
    if len(convs) != len(names):
        # name the first layer where the file and the graph part ways (e.g. a depthwise cls branch, or no OBB angle branch cv4)
        k = next((i for i, (name, (_nd, wt, _bs)) in enumerate(zip(names, convs)) if tuple(wt.shape) != _expected_shape(g, name)),
                 min(len(names), len(convs)))
        where = (f"; the first that differs is Conv node {convs[k][0].name or convs[k][0].outputs[0]!r} with shape {tuple(convs[k][1].shape)} "
                 f"where the graph runs {names[k]} {_expected_shape(g, names[k])}") if k < min(len(names), len(convs)) else ""
        raise ValueError(f"{path}: {len(convs)} Conv nodes with weights in the file, the {g.arch} graph has {len(names)} convolutions{where}")
    for name, (nd, wt, bs) in zip(names, convs):
        put(name, wt, bs, f"Conv node {nd.name or nd.outputs[0]!r}")
        _check_conv_node(path, g, name, nd)
    return out


# ---- minimal writer (tests and tooling: synthetic checkpoints in the reference's file format) --------


def _enc_varint(x: int) -> bytes:
    out = bytearray()
    while True:
        b = x & 0x7F
        x >>= 7
        out.append(b | (0x80 if x else 0))
        if not x:
            return bytes(out)


def _enc_field(fno: int, payload: bytes) -> bytes:
    return _enc_varint((fno << 3) | 2) + _enc_varint(len(payload)) + payload


def _enc_tensor(name: str, a: np.ndarray) -> bytes:
    code = {np.dtype(np.float32): 1, np.dtype(np.float16): 10, np.dtype(np.int64): 7}[a.dtype]
    body = b"".join(_enc_varint((1 << 3) | 0) + _enc_varint(int(d)) for d in a.shape)
    body += _enc_varint((2 << 3) | 0) + _enc_varint(code)
    body += _enc_field(8, name.encode()) + _enc_field(9, np.ascontiguousarray(a).tobytes())
    return body


def _enc_attr_int(name: str, v: int) -> bytes:       # AttributeProto: name 1, i 3, type 20 (INT = 2)
    return _enc_field(5, _enc_field(1, name.encode()) + _enc_varint((3 << 3) | 0) + _enc_varint(v) + _enc_varint((20 << 3) | 0) + _enc_varint(2))


def _enc_attr_ints(name: str, vs) -> bytes:          # ints 8 (unpacked), type INTS = 7
    body = _enc_field(1, name.encode()) + b"".join(_enc_varint((8 << 3) | 0) + _enc_varint(int(v)) for v in vs)
    return _enc_field(5, body + _enc_varint((20 << 3) | 0) + _enc_varint(7))


def write_conv_onnx(path: str, g: Graph, w: Dict[str, np.ndarray], named: bool = True, half: bool = False) -> None:
    """Writes an ONNX file holding one ``Conv`` node (+ weight / bias initializers) per convolution of
    ``g`` in execution order, plus the DFL arange conv for ``yolov8m`` -- the part of an Ultralytics
    export that ``load_onnx_weights`` reads.  ``named=False`` mimics exporters that rename folded
    weights (``onnx::Conv_<n>``); ``half=True`` stores fp16 like ``export(half=True)``."""
    parts: List[bytes] = []
    dt = np.float16 if half else np.float32
    k = 0
    prev = "images"
    ops = {op.weight: op for op in g.ops if op.kind in ("conv", "dwconv")}
    for name in _conv_names(g):
        wn, bn = (f"{name}.conv.weight", f"{name}.conv.bias") if named else (f"onnx::Conv_{700 + 2 * k}", f"onnx::Conv_{701 + 2 * k}")
        if named and name.startswith("model.22.") and name.endswith(".2"):
            wn, bn = f"{name}.weight", f"{name}.bias"            # the head's last convs are plain nn.Conv2d
        outn = f"/{name.replace('.', '/')}/Conv_output_0"
        node = _enc_field(1, prev.encode()) + _enc_field(1, wn.encode()) + _enc_field(1, bn.encode()) + _enc_field(2, outn.encode())
        node += _enc_field(3, f"/{name.replace('.', '/')}/conv/Conv".encode()) + _enc_field(4, b"Conv")
        kk, st, groups = g.wshapes[name][2], ops[name].s, g.wshapes[name][3]
        node += _enc_attr_int("group", groups) + _enc_attr_ints("kernel_shape", (kk, kk)) + _enc_attr_ints("strides", (st, st))
        node += _enc_attr_ints("pads", (kk // 2,) * 4) + _enc_attr_ints("dilations", (1, 1))
        parts.append(_enc_field(1, node))
        parts.append(_enc_field(5, _enc_tensor(wn, w[name + ".weight"].astype(dt))))
        parts.append(_enc_field(5, _enc_tensor(bn, w[name + ".bias"].astype(dt))))
        prev = outn
        k += 1
    if g.arch in ("yolov8m", "yolov8m-obb"):
        node = _enc_field(1, prev.encode()) + _enc_field(1, b"model.22.dfl.conv.weight") + _enc_field(2, b"/model.22/dfl/conv/Conv_output_0")
        node += _enc_field(3, b"/model.22/dfl/conv/Conv") + _enc_field(4, b"Conv")
        parts.append(_enc_field(1, node))
        parts.append(_enc_field(5, _enc_tensor("model.22.dfl.conv.weight", np.arange(16, dtype=np.float32).reshape(1, 16, 1, 1).astype(dt))))
    graph = b"".join(parts) + _enc_field(2, b"b2det_synthetic")
    model = _enc_varint((1 << 3) | 0) + _enc_varint(8) + _enc_field(2, b"b2det") + _enc_field(7, graph)
    with open(path, "wb") as f:
        f.write(model)
