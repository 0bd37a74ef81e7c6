"""Detector graphs as a flat op list over NHWC activation buffers.

The reference never builds a graph itself: it hands an ``.onnx`` file to
``onnxruntime.InferenceSession`` (``_script/gpu_handler.py:61-65``,
``simple_detector.py:39-46``) and calls ``.run`` (``gpu_handler.py:165``,
``simple_detector.py:474``).  The engine replaces that runtime, so the graph has
to be stated somewhere; this module states it as data that the C-ABI plan
builder (``engine.py`` -> ``b2d_plan_*``) consumes one op at a time.

Four architectures are described:

* ``yolov8m`` with ``nc=2`` and the Ultralytics 8.3.x depthwise cls branch -- the
  "tokyo" checkpoint, recovered from the training log in
  ``x_arch/01_train_tokyo.ipynb:1 (cell 15 output)`` (SURVEY.md Appendix A.1).
* ``yolov8m-obb`` -- the same backbone and neck with Ultralytics' oriented-box head (``build_yolov8m_obb``), the family of
  the published overhead-imagery (DOTAv1) checkpoints.
* ``yolov7`` canonical deploy graph -- the stand-in for the missing ITCVD
  model named at ``_script/config.py:25`` (SURVEY.md Appendix A.4).

* ``xunet`` -- a stated EfficientNet-B0-shaped U-Net stand-in for the "ramp XUnet 256" blob of BASELINE config C5, of which the
  reference holds only the name (``build_xunet``).

Design rules (B200-first, not ONNX-shaped):

* activations are NHWC so a pixel's channels are one contiguous K-run for the
  implicit-GEMM conv and one TMA box row;
* ``Concat`` never runs: every producer writes at a channel offset into the
  consumer's buffer, every consumer reads a channel slice through its own
  tensor map;
* ``Split`` never runs for the same reason;
* weights keep the Ultralytics module path as their name (``model.2.m.0.cv1``)
  in deploy form (BN folded: ``.weight`` [Cout, Cin/groups, k, k], ``.bias``
  [Cout]) so a real checkpoint can be dropped in later.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

ACT_NONE = 0
ACT_SILU = 1


@dataclass
class Buf:
    """One NHWC activation buffer (batch dimension supplied at plan time)."""
    name: str
    h: int
    w: int
    c: int
    f32: bool = False  # head outputs stay fp32; everything else is bf16


@dataclass
class Ref:
    """A channel slice [c0, c0+c) of a buffer."""
    buf: str
    c0: int
    c: int


@dataclass
class Op:
    kind: str                 # conv | dwconv | maxpool | upsample2x
    src: Ref
    dst: Ref
    k: int = 1
    s: int = 1
    act: int = ACT_NONE
    weight: Optional[str] = None   # weight name (conv / dwconv)
    res: Optional[Ref] = None      # residual added after the activation
    tag: str = ""
    # Channel placement: the buffers may hold a concat's segments in another order than the model's
    # (see _c2f).  out_perm[j] / in_perm[j] = the model's output / input channel that lives at
    # channel j of the destination / source slice; None = the model's own order.
    out_perm: Optional[List[int]] = None
    in_perm: Optional[List[int]] = None


@dataclass
class Graph:
    arch: str
    nc: int
    imgsz: int
    bufs: Dict[str, Buf] = field(default_factory=dict)
    ops: List[Op] = field(default_factory=list)
    # conv name -> (cout, cin_per_group, k, groups)
    wshapes: Dict[str, Tuple[int, int, int, int]] = field(default_factory=dict)
    # head description consumed by the decode kernel
    head: Dict = field(default_factory=dict)
    in_c: int = 4  # stem input is RGB padded to 4 channels (8 B per pixel)

    def buf(self, name, h, w, c, f32=False) -> str:
        assert name not in self.bufs, name
        self.bufs[name] = Buf(name, h, w, c, f32)
        return name

    def conv(self, name, src: Ref, dst: Ref, k=1, s=1, act=ACT_SILU, res=None, groups=1, out_perm=None, in_perm=None):
        sb, db = self.bufs[src.buf], self.bufs[dst.buf]
        pad = k // 2
        assert (sb.h + 2 * pad - k) // s + 1 == db.h, (name, sb.h, db.h)
        assert src.c0 + src.c <= sb.c and dst.c0 + dst.c <= db.c, name
        if groups == 1:
            cin = 3 if (src.buf == "input") else src.c
            self.wshapes[name] = (dst.c, cin, k, 1)
            self.ops.append(Op("conv", src, dst, k, s, act, name, res, name, out_perm, in_perm))
        else:
            assert groups == src.c == dst.c and k == 3 and s == 1
            self.wshapes[name] = (dst.c, 1, k, groups)
            self.ops.append(Op("dwconv", src, dst, k, s, act, name, None, name))

    def maxpool(self, src: Ref, dst: Ref, k, s, tag=""):
        self.ops.append(Op("maxpool", src, dst, k, s, tag=tag))

    def upsample(self, src: Ref, dst: Ref, tag=""):
        self.ops.append(Op("upsample2x", src, dst, tag=tag))

    # ---- accounting (SURVEY.md Appendix A.2 / D.7) -------------------------------
    def macs_per_tile(self) -> int:
        total = 0
        for op in self.ops:
            if op.kind in ("conv", "dwconv"):
                cout, cing, k, g = self.wshapes[op.weight]
                db = self.bufs[op.dst.buf]
                total += db.h * db.w * cout * cing * k * k
        return total

    def fused_param_count(self) -> int:
        n = 0
        for cout, cing, k, g in self.wshapes.values():
            n += cout * cing * k * k + cout
        return n + (16 if self.arch in ("yolov8m", "yolov8m-obb") else 0)  # + the DFL arange conv


def op_weights(op: Op, w) -> Tuple:
    """(weight [Cout, Cin/g, k, k], bias [Cout]) of a conv op in the channel order of the buffers it
    reads and writes: the model's weights with the op's channel placement applied."""
    wt, bs = w[op.weight + ".weight"], w[op.weight + ".bias"]
    if op.out_perm is not None:
        wt, bs = wt[op.out_perm], bs[op.out_perm]
    if op.in_perm is not None:
        wt = wt[:, op.in_perm]
    return wt, bs


def _c2f(g: Graph, name, src: Ref, dst: Ref, n, shortcut, hw, order=None):
    """Ultralytics C2f with the concat realised as channel offsets.

    The model's cat = [y0 | y1 | m0(y1) | m1(m0) ...]: cv1 produces [y0 | y1], bottleneck i reads
    segment i+1 and writes segment i+2, cv2 reads everything.  ``order[j]`` = the segment stored in
    slot j of the buffer (default: the model's order).  The placement matters when a segment is
    narrower than a 128-byte L2 line: TMA fetches whole lines, so a 96-byte (48-channel) segment
    that straddles two lines costs 2.7x its bytes in DRAM reads (measured, profiles/), one that sits
    inside a line 1.3x.  cv1's output rows and cv2's input columns are permuted to match
    (``Op.out_perm`` / ``Op.in_perm``); results are identical.
    """
    c = dst.c // 2
    order = list(range(n + 2)) if order is None else list(order)
    assert sorted(order) == list(range(n + 2))
    slot = {seg: j for j, seg in enumerate(order)}
    assert abs(slot[0] - slot[1]) == 1, "cv1 writes y0 and y1 with one store: they must be neighbours"
    cat = g.buf(f"{name}.cat", hw, hw, (2 + n) * c)
    tmp = g.buf(f"{name}.tmp", hw, hw, c)
    swap = slot[1] < slot[0]
    g.conv(f"{name}.cv1", src, Ref(cat, min(slot[0], slot[1]) * c, 2 * c), 1, 1,
           out_perm=(list(range(c, 2 * c)) + list(range(c))) if swap else None)
    for i in range(n):
        x = Ref(cat, slot[i + 1] * c, c)
        g.conv(f"{name}.m.{i}.cv1", x, Ref(tmp, 0, c), 3, 1)
        g.conv(f"{name}.m.{i}.cv2", Ref(tmp, 0, c), Ref(cat, slot[i + 2] * c, c), 3, 1,
               res=x if shortcut else None)
    in_perm = None if order == list(range(n + 2)) else [seg * c + k for seg in order for k in range(c)]
    g.conv(f"{name}.cv2", Ref(cat, 0, (2 + n) * c), dst, 1, 1, in_perm=in_perm)


def build_yolov8m(nc: int = 2, imgsz: int = 640) -> Graph:
    """YOLOv8m, Ultralytics 8.3.4 head (SURVEY.md Appendix A.1)."""
    g, feats = _yolov8m_body("yolov8m", nc, imgsz)
    # Detect head (8.3.x: box branch dense, cls branch depthwise-separable)
    levels = []
    c2, c3 = 64, 192
    for i, (feat, ch, hw, stride) in enumerate(feats):
        # box 64 | cls nc | padding up to a multiple of 32 fp32 channels: a pixel is then a whole number of 128-byte lines and the box
        # branch's 256-byte rows start on a line (with 68 channels = 272 bytes every store straddled three lines: cv2.0.2 50 -> 35 us)
        hc = ((64 + nc + 31) // 32) * 32
        out = g.buf(f"head{i}", hw, hw, hc, f32=True)
        _v8_box_branch(g, i, feat, ch, hw, out)
        d0 = g.buf(f"h{i}.d0", hw, hw, ch)
        e0 = g.buf(f"h{i}.e0", hw, hw, c3)
        d1 = g.buf(f"h{i}.d1", hw, hw, c3)
        e1 = g.buf(f"h{i}.e1", hw, hw, c3)
        g.conv(f"model.22.cv3.{i}.0.0", Ref(feat, 0, ch), Ref(d0, 0, ch), 3, 1, groups=ch)
        g.conv(f"model.22.cv3.{i}.0.1", Ref(d0, 0, ch), Ref(e0, 0, c3), 1, 1)
        g.conv(f"model.22.cv3.{i}.1.0", Ref(e0, 0, c3), Ref(d1, 0, c3), 3, 1, groups=c3)
        g.conv(f"model.22.cv3.{i}.1.1", Ref(d1, 0, c3), Ref(e1, 0, c3), 1, 1)
        g.conv(f"model.22.cv3.{i}.2", Ref(e1, 0, c3), Ref(out, 64, nc), 1, 1, act=ACT_NONE)
        levels.append({"buf": out, "hw": hw, "stride": stride, "c": hc})
    g.head = {"kind": "v8_dfl", "levels": levels, "reg_max": 16, "nc": nc,
              "anchors_total": sum(l["hw"] ** 2 for l in levels)}
    return g


def obb_angle_channel(nc: int) -> int:
    """Channel of the angle logit in a ``yolov8m-obb`` head map: the first 16-byte-aligned fp32 channel after box 64 | cls nc
    (a conv writes its output slice through a tensor map whose base must be 16-byte aligned).  The C library places it the same way."""
    return (64 + nc + 3) // 4 * 4


def build_yolov8m_obb(nc: int = 15, imgsz: int = 640) -> Graph:
    """YOLOv8m-OBB, the oriented-box head of Ultralytics >= 8.1 [EXT] on the YOLOv8m backbone and neck (identical to
    ``build_yolov8m`` up to model.21).  Per level: the box branch cv2 as in v8, a dense cls branch cv3 (Conv 3x3, Conv 3x3,
    Conv2d 1x1 with c3 = max(192, min(nc, 100)) channels, as in the published v8 OBB checkpoints) and an angle branch cv4 (Conv 3x3,
    Conv 3x3, Conv2d 1x1 -> 1 with 48 = max(192 // 4, 1) channels).  The head map of a level is fp32 [box 64 | cls nc | pad | angle | pad]
    (angle at ``obb_angle_channel(nc)``, width a multiple of 32 channels).  Ultralytics' ``OBB.forward`` runs cv4 over all three
    levels before ``Detect.forward`` runs cv2 / cv3, and the ops are listed in that order (the ONNX reader maps by order)."""
    g, feats = _yolov8m_body("yolov8m-obb", nc, imgsz)
    c3, c4 = max(192, min(nc, 100)), 48
    ac = obb_angle_channel(nc)
    hc = ((ac + 1 + 31) // 32) * 32
    outs = [g.buf(f"head{i}", hw, hw, hc, f32=True) for i, (_, _, hw, _) in enumerate(feats)]
    for i, (feat, ch, hw, _) in enumerate(feats):
        a = g.buf(f"h{i}.a0", hw, hw, c4)
        b = g.buf(f"h{i}.a1", hw, hw, c4)
        g.conv(f"model.22.cv4.{i}.0", Ref(feat, 0, ch), Ref(a, 0, c4), 3, 1)
        g.conv(f"model.22.cv4.{i}.1", Ref(a, 0, c4), Ref(b, 0, c4), 3, 1)
        g.conv(f"model.22.cv4.{i}.2", Ref(b, 0, c4), Ref(outs[i], ac, 1), 1, 1, act=ACT_NONE)
    levels = []
    for i, (feat, ch, hw, stride) in enumerate(feats):
        _v8_box_branch(g, i, feat, ch, hw, outs[i])
        a = g.buf(f"h{i}.c0", hw, hw, c3)
        b = g.buf(f"h{i}.c1", hw, hw, c3)
        g.conv(f"model.22.cv3.{i}.0", Ref(feat, 0, ch), Ref(a, 0, c3), 3, 1)
        g.conv(f"model.22.cv3.{i}.1", Ref(a, 0, c3), Ref(b, 0, c3), 3, 1)
        g.conv(f"model.22.cv3.{i}.2", Ref(b, 0, c3), Ref(outs[i], 64, nc), 1, 1, act=ACT_NONE)
        levels.append({"buf": outs[i], "hw": hw, "stride": stride, "c": hc})
    g.head = {"kind": "v8_obb", "levels": levels, "reg_max": 16, "nc": nc, "angle_c": ac,
              "anchors_total": sum(l["hw"] ** 2 for l in levels)}
    return g


def _v8_box_branch(g: Graph, i: int, feat: str, ch: int, hw: int, out: str) -> None:
    c2 = 64
    a = g.buf(f"h{i}.b0", hw, hw, c2)
    b = g.buf(f"h{i}.b1", hw, hw, c2)
    g.conv(f"model.22.cv2.{i}.0", Ref(feat, 0, ch), Ref(a, 0, c2), 3, 1)
    g.conv(f"model.22.cv2.{i}.1", Ref(a, 0, c2), Ref(b, 0, c2), 3, 1)
    g.conv(f"model.22.cv2.{i}.2", Ref(b, 0, c2), Ref(out, 0, 64), 1, 1, act=ACT_NONE)


def _yolov8m_body(arch: str, nc: int, imgsz: int):
    """YOLOv8m backbone and neck (model.0 - model.21); returns the graph and (buffer, channels, size, stride) of P3, P4, P5."""
    assert imgsz % 32 == 0
    g = Graph(arch, nc, imgsz)
    s1, s2, s3, s4, s5 = (imgsz // 2, imgsz // 4, imgsz // 8, imgsz // 16, imgsz // 32)
    g.buf("input", imgsz, imgsz, 4)
    # concat buffers of the FPN/PAN, allocated up front so producers can target them
    cat11 = g.buf("cat11", s4, s4, 576 + 384)   # [up(9) | 6]
    cat14 = g.buf("cat14", s3, s3, 384 + 192)   # [up(12) | 4]
    cat17 = g.buf("cat17", s4, s4, 192 + 384)   # [16 | 12]
    cat20 = g.buf("cat20", s5, s5, 384 + 576)   # [19 | 9]

    x0 = g.buf("x0", s1, s1, 48)
    g.conv("model.0", Ref("input", 0, 4), Ref(x0, 0, 48), 3, 2)
    x1 = g.buf("x1", s2, s2, 96)
    g.conv("model.1", Ref(x0, 0, 48), Ref(x1, 0, 96), 3, 2)
    x2 = g.buf("x2", s2, s2, 96)
    # 48-channel segments (96 B): y1 and m0, the two that are read as slices, go to the ends of the 384-byte pixel
    _c2f(g, "model.2", Ref(x1, 0, 96), Ref(x2, 0, 96), 2, True, s2, order=(1, 0, 3, 2))
    x3 = g.buf("x3", s3, s3, 192)
    g.conv("model.3", Ref(x2, 0, 96), Ref(x3, 0, 192), 3, 2)
    p4 = Ref(cat14, 384, 192)                               # layer 4 output
    _c2f(g, "model.4", Ref(x3, 0, 192), p4, 4, True, s3)
    x5 = g.buf("x5", s4, s4, 384)
    g.conv("model.5", p4, Ref(x5, 0, 384), 3, 2)
    p6 = Ref(cat11, 576, 384)                               # layer 6 output
    _c2f(g, "model.6", Ref(x5, 0, 384), p6, 4, True, s4)
    x7 = g.buf("x7", s5, s5, 576)
    g.conv("model.7", p6, Ref(x7, 0, 576), 3, 2)
    x8 = g.buf("x8", s5, s5, 576)
    _c2f(g, "model.8", Ref(x7, 0, 576), Ref(x8, 0, 576), 2, True, s5)
    # SPPF: cat = [x | m(x) | m(m(x)) | m(m(m(x)))]
    sp = g.buf("model.9.cat", s5, s5, 4 * 288)
    g.conv("model.9.cv1", Ref(x8, 0, 576), Ref(sp, 0, 288), 1, 1)
    for i in range(3):
        g.maxpool(Ref(sp, i * 288, 288), Ref(sp, (i + 1) * 288, 288), 5, 1, tag=f"model.9.m{i}")
    p9 = Ref(cat20, 384, 576)                               # layer 9 output
    g.conv("model.9.cv2", Ref(sp, 0, 1152), p9, 1, 1)
    g.upsample(p9, Ref(cat11, 0, 576), tag="model.10")
    p12 = Ref(cat17, 192, 384)                              # layer 12 output
    _c2f(g, "model.12", Ref(cat11, 0, 960), p12, 2, False, s4)
    g.upsample(p12, Ref(cat14, 0, 384), tag="model.13")
    x15 = g.buf("x15", s3, s3, 192)                         # P3 out
    _c2f(g, "model.15", Ref(cat14, 0, 576), Ref(x15, 0, 192), 2, False, s3)
    g.conv("model.16", Ref(x15, 0, 192), Ref(cat17, 0, 192), 3, 2)
    x18 = g.buf("x18", s4, s4, 384)                         # P4 out
    _c2f(g, "model.18", Ref(cat17, 0, 576), Ref(x18, 0, 384), 2, False, s4)
    g.conv("model.19", Ref(x18, 0, 384), Ref(cat20, 0, 384), 3, 2)
    x21 = g.buf("x21", s5, s5, 576)                         # P5 out
    _c2f(g, "model.21", Ref(cat20, 0, 960), Ref(x21, 0, 576), 2, False, s5)
    return g, ((x15, 192, s3, 8), (x18, 384, s4, 16), (x21, 576, s5, 32))


# ---------------------------------------------------------------------------------
# canonical YOLOv7 deploy graph (SURVEY.md Appendix A.4)
# ---------------------------------------------------------------------------------
V7_ANCHORS = (
    (12, 16, 19, 36, 40, 28),
    (36, 75, 76, 55, 72, 146),
    (142, 110, 192, 243, 459, 401),
)


def build_yolov7(nc: int = 1, imgsz: int = 640) -> Graph:
    assert imgsz % 32 == 0
    g = Graph("yolov7", nc, imgsz)
    s0, s1, s2, s3, s4, s5 = (imgsz, imgsz // 2, imgsz // 4, imgsz // 8, imgsz // 16, imgsz // 32)
    g.buf("input", imgsz, imgsz, 4)
    idx = [0]

    def nm():
        n = f"model.{idx[0]}"
        idx[0] += 1
        return n

    def skip(n=1):
        idx[0] += n

    def elan(src: Ref, c, cout, hw, dst: Optional[Ref] = None):
        """backbone ELAN: out = Conv(4c,cout,1)(cat[b4,b2,b,a])  (8 module slots)."""
        cat = g.buf(f"elan{idx[0]}.cat", hw, hw, 4 * c)
        t = g.buf(f"elan{idx[0]}.t", hw, hw, c)
        a, b, b2, b4 = Ref(cat, 3 * c, c), Ref(cat, 2 * c, c), Ref(cat, c, c), Ref(cat, 0, c)
        g.conv(nm(), src, a, 1, 1)
        g.conv(nm(), src, b, 1, 1)
        g.conv(nm(), b, Ref(t, 0, c), 3, 1)
        g.conv(nm(), Ref(t, 0, c), b2, 3, 1)
        g.conv(nm(), b2, Ref(t, 0, c), 3, 1)
        g.conv(nm(), Ref(t, 0, c), b4, 3, 1)
        skip()  # Concat
        if dst is None:
            o = g.buf(f"elan{idx[0]}.out", hw, hw, cout)
            dst = Ref(o, 0, cout)
        g.conv(nm(), Ref(cat, 0, 4 * c), dst, 1, 1)
        return dst

    def mpblk(src: Ref, c, hw_in, dst: Ref):
        """cat[ Conv(c,c,3,2)(Conv(cin,c,1)(x)), Conv(cin,c,1)(MP(x)) ] -> dst [0,2c) (5 slots)."""
        hw = hw_in // 2
        mp = g.buf(f"mp{idx[0]}.p", hw, hw, src.c)
        t = g.buf(f"mp{idx[0]}.t", hw_in, hw_in, c)
        skip()  # MP
        g.maxpool(src, Ref(mp, 0, src.c), 2, 2, tag=f"model.{idx[0]-1}")
        g.conv(nm(), Ref(mp, 0, src.c), Ref(dst.buf, dst.c0 + c, c), 1, 1)
        g.conv(nm(), src, Ref(t, 0, c), 1, 1)
        g.conv(nm(), Ref(t, 0, c), Ref(dst.buf, dst.c0, c), 3, 2)
        skip()  # Concat
        return dst

    def elan_h(src: Ref, c, cout, hw, dst: Optional[Ref] = None):
        """head ELAN-H: cat[b4,b3,b2,b1,b,a] with b* of width c/2 (8 slots)."""
        h = c // 2
        cat = g.buf(f"elanh{idx[0]}.cat", hw, hw, 2 * c + 4 * h)
        b4, b3, b2, b1 = (Ref(cat, i * h, h) for i in range(4))
        b, a = Ref(cat, 4 * h, c), Ref(cat, 4 * h + c, c)
        g.conv(nm(), src, a, 1, 1)
        g.conv(nm(), src, b, 1, 1)
        g.conv(nm(), b, b1, 3, 1)
        g.conv(nm(), b1, b2, 3, 1)
        g.conv(nm(), b2, b3, 3, 1)
        g.conv(nm(), b3, b4, 3, 1)
        skip()
        if dst is None:
            o = g.buf(f"elanh{idx[0]}.out", hw, hw, cout)
            dst = Ref(o, 0, cout)
        g.conv(nm(), Ref(cat, 0, 2 * c + 4 * h), dst, 1, 1)
        return dst

    # backbone
    t0 = g.buf("b0", s0, s0, 32); g.conv(nm(), Ref("input", 0, 4), Ref(t0, 0, 32), 3, 1)
    t1 = g.buf("b1", s1, s1, 64); g.conv(nm(), Ref(t0, 0, 32), Ref(t1, 0, 64), 3, 2)
    t2 = g.buf("b2", s1, s1, 64); g.conv(nm(), Ref(t1, 0, 64), Ref(t2, 0, 64), 3, 1)
    t3 = g.buf("b3", s2, s2, 128); g.conv(nm(), Ref(t2, 0, 64), Ref(t3, 0, 128), 3, 2)
    e11 = elan(Ref(t3, 0, 128), 64, 256, s2)                       # 4-11
    m16 = g.buf("m16", s3, s3, 256); mpblk(e11, 128, s2, Ref(m16, 0, 256))   # 12-16
    p3 = elan(Ref(m16, 0, 256), 128, 512, s3)                      # 17-24  (#24)
    m29 = g.buf("m29", s4, s4, 512); mpblk(p3, 256, s3, Ref(m29, 0, 512))    # 25-29
    p4 = elan(Ref(m29, 0, 512), 256, 1024, s4)                     # 30-37  (#37)
    m42 = g.buf("m42", s5, s5, 1024); mpblk(p4, 512, s4, Ref(m42, 0, 1024))  # 38-42
    p5 = elan(Ref(m42, 0, 1024), 256, 1024, s5)                    # 43-50
    # 51 SPPCSPC(1024 -> 512), c_ = 512
    assert idx[0] == 51
    cat93 = g.buf("cat93", s5, s5, 1024)        # [MPblk(88) 512 | #51 512]
    sp = "model.51"
    c_ = 512
    a1 = g.buf("spp.a1", s5, s5, c_); a3 = g.buf("spp.a3", s5, s5, c_)
    spcat = g.buf("spp.cat", s5, s5, 4 * c_)
    a5 = g.buf("spp.a5", s5, s5, c_)
    ycat = g.buf("spp.ycat", s5, s5, 2 * c_)
    g.conv(f"{sp}.cv1", p5, Ref(a1, 0, c_), 1, 1)
    g.conv(f"{sp}.cv3", Ref(a1, 0, c_), Ref(a3, 0, c_), 3, 1)
    g.conv(f"{sp}.cv4", Ref(a3, 0, c_), Ref(spcat, 0, c_), 1, 1)
    for j, k in enumerate((5, 9, 13)):
        g.maxpool(Ref(spcat, 0, c_), Ref(spcat, (j + 1) * c_, c_), k, 1, tag=f"{sp}.m{k}")
    g.conv(f"{sp}.cv5", Ref(spcat, 0, 4 * c_), Ref(a5, 0, c_), 1, 1)
    g.conv(f"{sp}.cv6", Ref(a5, 0, c_), Ref(ycat, 0, c_), 3, 1)
    g.conv(f"{sp}.cv2", p5, Ref(ycat, c_, c_), 1, 1)
    n51 = Ref(cat93, 512, 512)
    g.conv(f"{sp}.cv7", Ref(ycat, 0, 2 * c_), n51, 1, 1)
    idx[0] = 52
    # top-down
    cat55 = g.buf("cat55", s4, s4, 512)         # [conv54(from 37) 256 | up(52) 256]
    u52 = g.buf("u52", s5, s5, 256); g.conv(nm(), n51, Ref(u52, 0, 256), 1, 1)      # 52
    skip(); g.upsample(Ref(u52, 0, 256), Ref(cat55, 256, 256), tag="model.53")      # 53
    g.conv(nm(), p4, Ref(cat55, 0, 256), 1, 1)                                      # 54
    skip()                                                                           # 55 concat [54, 53]
    cat80 = g.buf("cat80", s4, s4, 512)         # [MPblk(75) 256 | #63 256]
    n63 = elan_h(Ref(cat55, 0, 512), 256, 256, s4, Ref(cat80, 256, 256))            # 56-63
    cat67 = g.buf("cat67", s3, s3, 256)         # [conv66(from 24) 128 | up(64) 128]
    u64 = g.buf("u64", s4, s4, 128); g.conv(nm(), n63, Ref(u64, 0, 128), 1, 1)      # 64
    skip(); g.upsample(Ref(u64, 0, 128), Ref(cat67, 128, 128), tag="model.65")      # 65
    g.conv(nm(), p3, Ref(cat67, 0, 128), 1, 1)                                      # 66
    skip()                                                                           # 67
    n75 = elan_h(Ref(cat67, 0, 256), 128, 128, s3)                                   # 68-75
    mpblk(n75, 128, s3, Ref(cat80, 0, 256))                                          # 76-80 (concat with 63)
    n88 = elan_h(Ref(cat80, 0, 512), 256, 256, s4)                                   # 81-88
    mpblk(n88, 256, s4, Ref(cat93, 0, 512))                                          # 89-93 (concat with 51)
    n101 = elan_h(Ref(cat93, 0, 1024), 512, 512, s5)                                 # 94-101
    assert idx[0] == 102, idx[0]
    levels = []
    no = nc + 5
    for i, (feat, cin, cout, hw, stride) in enumerate(((n75, 128, 256, s3, 8), (n88, 256, 512, s4, 16), (n101, 512, 1024, s5, 32))):
        r = g.buf(f"rep{i}", hw, hw, cout)
        g.conv(f"model.{102 + i}", feat, Ref(r, 0, cout), 3, 1)          # RepConv, deploy form
        hc = ((3 * no + 3) // 4) * 4
        out = g.buf(f"head{i}", hw, hw, hc, f32=True)
        g.conv(f"model.105.m.{i}", Ref(r, 0, cout), Ref(out, 0, 3 * no), 1, 1, act=ACT_NONE)
        levels.append({"buf": out, "hw": hw, "stride": stride, "c": hc, "anchors": V7_ANCHORS[i]})
    g.head = {"kind": "v7_anchor", "levels": levels, "nc": nc, "na": 3,
              "anchors_total": 3 * sum(l["hw"] ** 2 for l in levels)}
    return g


# EfficientNet-B0 stage table (expand ratio, output channels, repeats, stride) with the widths of stages 2-5 rounded up to
# multiples of 32 (24 -> 32, 40 -> 64, 80 -> 96, 112 -> 128) so that every 6x expanded width is a whole number of the engine's
# 64-channel K chunks (the depthwise kernel tiles wide layers by chunk).
XUNET_STAGES = ((1, 16, 1, 1), (6, 32, 2, 2), (6, 64, 2, 2), (6, 96, 3, 2), (6, 128, 3, 1), (6, 192, 4, 2), (6, 320, 1, 1))
XUNET_DECODER = (256, 128, 64, 32, 16)


def build_xunet(nc: int = 4, imgsz: int = 256) -> Graph:
    """Encoder-decoder segmentation stand-in for BASELINE config C5 ("ramp XUnet 256").

    The reference holds only the blob's name (``.MISSING_LARGE_BLOBS:3``) -- no code, no architecture (SURVEY.md A.5, 8f-5).
    [EXT] ramp's model is an EfficientNet-B0-encoder U-Net with a 4-class softmax on 256 x 256 tiles; this graph is a STATED
    stand-in of that shape built from the ops the engine has, not a reproduction:

    * encoder: stem 3x3 s2 -> 32, then the seven EfficientNet-B0 stages as MBConv blocks (1x1 expand + SiLU, depthwise 3x3 + SiLU,
      1x1 linear projection, identity shortcut where shapes allow).  Differences from B0, all forced by the op set: stage widths
      rounded up to multiples of 32, every depthwise kernel is 3x3 (B0 mixes 3x3 and 5x5), a stride-2 block runs its depthwise conv at
      stride 1 followed by a 2x2 max-pool, no squeeze-and-excitation;
    * decoder: the segmentation_models U-Net -- five blocks of nearest 2x upsample, concat with the encoder skip (a channel
      offset, never a copy), two 3x3 convs (SiLU instead of BatchNorm + ReLU) with 256 / 128 / 64 / 32 / 16 channels;
    * head: 3x3 conv to ``nc`` logits (fp32 NHWC, padded to 4 channels = 16 bytes); argmax / softmax are the segment kernel's.
    """
    assert imgsz % 32 == 0
    g = Graph("xunet", nc, imgsz)
    g.buf("input", imgsz, imgsz, 4)
    hw = imgsz // 2
    # decoder concat buffers [upsampled | skip], allocated first so the encoder can write its skips into them
    skips_c = tuple(XUNET_STAGES[i][1] for i in (0, 1, 2, 4))     # encoder outputs at imgsz / 2, / 4, / 8, / 16: 16, 32, 64, 128
    dec_in = (XUNET_STAGES[-1][1],) + XUNET_DECODER[:-1]          # channels arriving from below: 320, 256, 128, 64, 32
    cats = []
    for lvl in range(4):                            # lvl 0 = imgsz / 16 ... lvl 3 = imgsz / 2
        size = imgsz // (16 >> lvl)
        cats.append(g.buf(f"dec{lvl}.cat", size, size, dec_in[lvl] + skips_c[3 - lvl]))
    skip_ref = {imgsz // 2: Ref(cats[3], dec_in[3], skips_c[0]), imgsz // 4: Ref(cats[2], dec_in[2], skips_c[1]),
                imgsz // 8: Ref(cats[1], dec_in[1], skips_c[2]), imgsz // 16: Ref(cats[0], dec_in[0], skips_c[3])}
    x = Ref(g.buf("enc.stem", hw, hw, 32), 0, 32)
    g.conv("encoder.stem", Ref("input", 0, 4), x, 3, 2)
    last_of_size = {1: 0, 2: 1, 3: 2, 5: 4}         # stage index (1-based) whose output is the skip of its resolution
    for si, (e, c, r, s) in enumerate(XUNET_STAGES, start=1):
        for bi in range(r):
            name = f"encoder.s{si}.b{bi}"
            cin, stride = x.c, (s if bi == 0 else 1)
            mid = cin * e
            t = x
            if e != 1:
                t = Ref(g.buf(f"{name}.exp", hw, hw, mid), 0, mid)
                g.conv(f"{name}.expand", x, t, 1, 1)
            d = Ref(g.buf(f"{name}.dw", hw, hw, mid), 0, mid)
            g.conv(f"{name}.dw", t, d, 3, 1, groups=mid)
            if stride == 2:
                hw //= 2
                pd = Ref(g.buf(f"{name}.pool", hw, hw, mid), 0, mid)
                g.maxpool(d, pd, 2, 2, tag=f"{name}.pool")
                d = pd
            is_skip = si in last_of_size and bi == r - 1
            out = skip_ref[hw] if is_skip else Ref(g.buf(f"{name}.out", hw, hw, c), 0, c)
            g.conv(f"{name}.project", d, out, 1, 1, act=ACT_NONE, res=x if (stride == 1 and cin == c) else None)
            x = out
    # decoder
    for lvl in range(5):
        name = f"decoder.b{lvl}"
        cdec = XUNET_DECODER[lvl]
        hw *= 2
        if lvl < 4:
            g.upsample(x, Ref(cats[lvl], 0, x.c), tag=f"{name}.up")
            src = Ref(cats[lvl], 0, g.bufs[cats[lvl]].c)
        else:
            up = g.buf(f"{name}.up", hw, hw, x.c)
            g.upsample(x, Ref(up, 0, x.c), tag=f"{name}.up")
            src = Ref(up, 0, x.c)
        a = Ref(g.buf(f"{name}.c1", hw, hw, cdec), 0, cdec)
        g.conv(f"{name}.conv1", src, a, 3, 1)
        b = Ref(g.buf(f"{name}.c2", hw, hw, cdec), 0, cdec)
        g.conv(f"{name}.conv2", a, b, 3, 1)
        x = b
    hc = ((nc + 3) // 4) * 4
    logits = g.buf("logits", imgsz, imgsz, hc, f32=True)
    g.conv("segmentation_head", x, Ref(logits, 0, nc), 3, 1, act=ACT_NONE)
    g.head = {"kind": "seg", "levels": [], "buf": logits, "nc": nc, "c": hc, "anchors_total": 0}
    return g


def build(arch: str, nc: Optional[int] = None, imgsz: int = 640) -> Graph:
    if arch in ("yolov8m", "v8", "yolov8m_tokyo"):
        return build_yolov8m(2 if nc is None else nc, imgsz)
    if arch in ("yolov8m-obb", "yolov8m_obb"):
        return build_yolov8m_obb(15 if nc is None else nc, imgsz)
    if arch in ("yolov7", "v7", "yolov7_itcvd"):
        return build_yolov7(1 if nc is None else nc, imgsz)
    if arch in ("xunet", "ramp_xunet"):
        return build_xunet(4 if nc is None else nc, 256 if imgsz == 640 else imgsz)
    raise ValueError(f"unknown architecture {arch!r}")
