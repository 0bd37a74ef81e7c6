"""CPU tests of the oriented-box model ``yolov8m-obb``: graph pins, the offset-write graph against the conventional oracle,
unchanged existing architectures, and the restated Ultralytics post-processing on hand cases."""
import math

import numpy as np
import pytest
import torch

from aerial_image_recognition_b200 import graph as G, weights as W
from _ir_cpu import run_graph_cpu
from _obb_oracle import (YoloV8mObbOracle, batch_probiou, fast_nms_loop, nms_rotated, regularize_rboxes, ultralytics_nms_rotated,
                         xywhr2xyxyxyxy)


def test_obb_graph_parameter_and_flop_pins():
    g = G.build("yolov8m-obb")
    assert g.nc == 15 and g.head["kind"] == "v8_obb"
    assert g.fused_param_count() == 26_408_752                 # published: 26.4 M [EXT]
    assert 2 * g.macs_per_tile() == 80_866_752_000             # 80.87 GFLOP per 640^2 tile (v8m of config C2: 67.43)
    assert 2 * G.build("yolov8m-obb", imgsz=1024).macs_per_tile() == 207_018_885_120   # Ultralytics' own counter says 208.6 [EXT]
    assert 2 * G.build("yolov8m").macs_per_tile() == 67_425_792_000


@pytest.mark.parametrize("nc", [1, 2, 15, 16, 80])
def test_obb_head_layout(nc):
    g = G.build("yolov8m-obb", nc=nc, imgsz=128)
    ac = g.head["angle_c"]
    assert ac == G.obb_angle_channel(nc) and ac >= 64 + nc and (ac * 4) % 16 == 0
    for lv in g.head["levels"]:
        assert g.bufs[lv["buf"]].c % 32 == 0 and g.bufs[lv["buf"]].c > ac
    names = [op.weight for op in g.ops if op.weight and op.weight.startswith("model.22")]
    assert names[:9] == [f"model.22.cv4.{i}.{j}" for i in range(3) for j in range(3)]       # OBB.forward runs cv4 first
    assert g.wshapes["model.22.cv3.0.0"] == (max(192, min(nc, 100)), 192, 3, 1) and g.wshapes["model.22.cv4.2.0"] == (48, 576, 3, 1)
    angle = [op for op in g.ops if op.weight and op.weight.startswith("model.22.cv4") and op.weight.endswith(".2")]
    assert all(op.dst.c0 == ac and op.dst.c == 1 for op in angle)


def test_obb_offset_write_graph_equals_oracle():
    g = G.build("yolov8m-obb", imgsz=64)
    w = W.make_synthetic_weights(g, 0, calibrate=False)
    x = torch.rand(2, 3, 64, 64, generator=torch.Generator().manual_seed(0))
    bufs = run_graph_cpu(g, w, x)
    raw = YoloV8mObbOracle(w, False).raw_head(x)
    ac = g.head["angle_c"]
    for lv, r in zip(g.head["levels"], raw):
        b = bufs[lv["buf"]]
        got = torch.cat([b[:, :64 + g.nc], b[:, ac:ac + 1]], 1)
        assert got.shape == r.shape and torch.allclose(got, r, rtol=1e-4, atol=1e-4), (got - r).abs().max()


# weights_fingerprint of the parent commit's generator, and a digest of the op list: adding the OBB model changes neither
PARENT = {"yolov8m": ("1374ec94878a720c", "93fb569c2ca4c60e"), "yolov7": ("86b7522752dc30c2", "752ecbf68c07f536"),
          "xunet": ("d5d699d5fb439fca", "a8ab925dfb86996d")}


@pytest.mark.parametrize("arch", sorted(PARENT))
def test_existing_architectures_unchanged(arch):
    import hashlib
    g = G.build(arch)
    ops = hashlib.sha256(repr([(o.kind, o.src, o.dst, o.k, o.s, o.act, o.weight, o.res, o.tag, o.out_perm, o.in_perm) for o in g.ops]).encode()
                         + repr(g.bufs).encode() + repr(g.head).encode()).hexdigest()[:16]
    assert ops == PARENT[arch][1]
    assert W.weights_fingerprint(W.make_synthetic_weights(g, 0)) == PARENT[arch][0]


def test_obb_angle_calibration_rotates_boxes():
    g = G.build("yolov8m-obb", imgsz=128)
    w = W.make_synthetic_weights(g, 0)
    from aerial_image_recognition_b200 import synth
    x = torch.from_numpy(synth.make_tiles(2, 128, 4).astype(np.float32) / 255.0).permute(0, 3, 1, 2)
    th = YoloV8mObbOracle(w, False).forward(x)[:, -1].numpy()
    assert th.min() < -0.4 and th.max() > 1.9 and 0.5 < th.std() < 1.2, (th.min(), th.max(), th.std())


# ---- ProbIoU, fast NMS, regularization, corners --------------------------------------------------------------
def test_probiou_hand_cases():
    a = np.array([[10, 20, 8, 3, 0.3]], np.float32)
    assert abs(batch_probiou(a, a)[0, 0].item() - 1.0) < 1e-3
    sq = np.array([[0, 0, 5, 5, 0.0]], np.float32)
    sq90 = np.array([[0, 0, 5, 5, math.pi / 2]], np.float32)
    assert abs(batch_probiou(sq, sq90)[0, 0].item() - batch_probiou(sq, sq)[0, 0].item()) < 1e-6
    rng = np.random.default_rng(0)
    b = np.concatenate([rng.uniform(0, 50, (20, 2)), rng.uniform(2, 20, (20, 2)), rng.uniform(-1, 3, (20, 1))], 1).astype(np.float32)
    m = batch_probiou(b, b).numpy()
    assert np.abs(m - m.T).max() < 1e-6
    far = np.array([[0, 0, 4, 2, 0.1], [1000, 1000, 4, 2, 0.1]], np.float32)
    assert batch_probiou(far[:1], far[1:])[0, 0].item() <= 1e-6


def test_fast_nms_chain_drops_the_third_box():
    """A suppresses B, B suppresses C, A does not suppress C: fast NMS drops C (a suppressed box still suppresses); greedy NMS
    would keep it."""
    boxes = np.array([[0, 0, 10, 4, 0], [2, 0, 10, 4, 0], [4, 0, 10, 4, 0]], np.float32)
    scores = np.array([0.9, 0.8, 0.7], np.float32)
    m = batch_probiou(boxes, boxes).numpy()
    thr = 0.6
    assert m[0, 1] >= thr and m[1, 2] >= thr and m[0, 2] < thr, m
    keep = nms_rotated(torch.from_numpy(boxes), torch.from_numpy(scores), thr).numpy()
    assert keep.tolist() == [0] and fast_nms_loop(boxes, scores, thr).tolist() == [0]
    greedy = [i for i in range(3) if all(m[k, i] < thr for k in range(i) if k in (0,))]
    assert greedy == [0, 2]


@pytest.mark.parametrize("seed", range(4))
def test_oracle_nms_equals_plain_loop_with_ties(seed):
    rng = np.random.default_rng(seed)
    n = 120
    ctr = rng.uniform(0, 60, (n, 2))
    b = np.concatenate([ctr, rng.uniform(3, 15, (n, 2)), rng.uniform(-0.8, 2.4, (n, 1))], 1).astype(np.float32)
    scores = rng.choice(np.array([0.3, 0.5, 0.5, 0.7, 0.9], np.float32), n)            # exact ties
    a = nms_rotated(torch.from_numpy(b), torch.from_numpy(scores), 0.5, chunk=37).numpy()
    assert a.tolist() == fast_nms_loop(b, scores, 0.5).tolist()


def test_ultralytics_nms_rotated_pipeline():
    pred = np.zeros((1, 4 + 2 + 1, 4), np.float32)
    pred[0, :4] = np.array([[10, 11, 100, 10], [10, 10, 100, 10], [8, 8, 30, 30], [5, 5, 20, 20]], np.float32).T
    pred[0, 4] = [0.9, 0.0, 0.0, 0.2]
    pred[0, 5] = [0.0, 0.8, 0.6, 0.0]
    pred[0, 6] = [0.0, 0.0, 2.0, 0.0]
    out = ultralytics_nms_rotated(pred, 0.25, 0.7)[0]
    # anchors 0 and 1 overlap but carry different classes (class offset), anchor 3 is under conf; anchor 2 keeps its own box
    assert out[:, 7].tolist() == [0, 1, 2]
    assert out[:, 6].tolist() == [0, 1, 1]
    assert np.allclose(out[2, :5], regularize_rboxes(np.array([[8, 8, 30, 30, 2.0]], np.float32))[0])


def test_regularize_rboxes_and_corners_hand_cases():
    r = regularize_rboxes(np.array([[0, 0, 4, 2, 0.5], [0, 0, 2, 4, 0.5], [0, 0, 3, 3, -0.2], [0, 0, 5, 1, 4.0]], np.float32))
    assert np.allclose(r[0], [0, 0, 4, 2, 0.5])
    assert np.allclose(r[1], [0, 0, 4, 2, 0.5 + math.pi / 2])
    assert np.allclose(r[2], [0, 0, 3, 3, (-0.2 + math.pi / 2) % math.pi])        # w == h swaps (w > h is strict)
    assert np.allclose(r[3], [0, 0, 5, 1, 4.0 - math.pi], atol=1e-6)
    assert (r[:, 4] >= 0).all() and (r[:, 4] < math.pi).all()
    c = xywhr2xyxyxyxy(np.array([[10, 20, 4, 2, 0.0], [0, 0, 4, 2, math.pi / 2]], np.float32))
    assert np.allclose(c[0], [[12, 21], [12, 19], [8, 19], [8, 21]])
    assert np.allclose(c[1], [[-1, 2], [1, 2], [1, -2], [-1, -2]], atol=1e-6)
    # corners do not depend on the w / h swap of regularization (as a set)
    b = np.array([[3, 4, 2, 7, 0.4]], np.float32)
    c0, c1 = xywhr2xyxyxyxy(b)[0], xywhr2xyxyxyxy(regularize_rboxes(b))[0]
    assert np.allclose(np.sort(c0, 0), np.sort(c1, 0), atol=1e-5)


# ---- ONNX: a torch export of a conventional OBB module ----------------------------------------------------------
def _obb_module(nc, depthwise_cls=False, angle=True):
    import torch.nn as nn
    import _export_onnx as E

    class OBB(nn.Module):
        """Ultralytics >= 8.1 OBB head on the v8 Detect branches: cv4 runs over all levels before cv2 / cv3."""

        def __init__(self, ch):
            super().__init__()
            c3 = max(192, min(nc, 100))
            self.cv2 = nn.ModuleList(nn.Sequential(E.Conv(x, 64, 3), E.Conv(64, 64, 3), nn.Conv2d(64, 64, 1)) for x in ch)
            if depthwise_cls:
                self.cv3 = nn.ModuleList(nn.Sequential(nn.Sequential(E.Conv(x, x, 3, g=x), E.Conv(x, c3, 1)),
                                                       nn.Sequential(E.Conv(c3, c3, 3, g=c3), E.Conv(c3, c3, 1)), nn.Conv2d(c3, nc, 1)) for x in ch)
            else:
                self.cv3 = nn.ModuleList(nn.Sequential(E.Conv(x, c3, 3), E.Conv(c3, c3, 3), nn.Conv2d(c3, nc, 1)) for x in ch)
            if angle:
                self.cv4 = nn.ModuleList(nn.Sequential(E.Conv(x, 48, 3), E.Conv(48, 48, 3), nn.Conv2d(48, 1, 1)) for x in ch)
            self.dfl = E.DFL()

        def forward(self, xs):
            b = xs[0].shape[0]
            ang = [self.cv4[i](x).view(b, 1, -1) for i, x in enumerate(xs)] if hasattr(self, "cv4") else []
            outs = [torch.cat((self.cv2[i](x), self.cv3[i](x)), 1).view(b, 64 + nc, -1) for i, x in enumerate(xs)]
            cat = torch.cat(outs, 2)
            box = self.dfl(cat[:, :64])
            return torch.cat([box, cat[:, 64:].sigmoid()] + ([(torch.cat(ang, 2).sigmoid() - 0.25) * math.pi] if ang else []), 1)

    m = E.YoloV8m(nc)
    m.model[22] = OBB((192, 384, 576))
    return m


@pytest.fixture(scope="module")
def obb_export(tmp_path_factory):
    import _export_onnx as E
    g = G.build("yolov8m-obb", imgsz=64)
    w = W.make_synthetic_weights(g, 0, calibrate=False)
    m = _obb_module(g.nc)
    E.load_deploy_weights(m, w)
    d = tmp_path_factory.mktemp("obb_onnx")
    E.export(m, str(d / "yolov8m-obb.onnx"))
    return g, w, d


def test_onnx_reader_loads_a_torch_exported_obb_model_by_name_and_by_order(obb_export):
    from aerial_image_recognition_b200 import onnx_reader as R
    g, w, d = obb_export
    path = str(d / "yolov8m-obb.onnx")
    _nodes, inits = R.read_onnx(path)
    assert "model.22.cv4.2.2.weight" in inits and "model.22.cv3.0.1.conv.weight" in inits
    for by_name in (True, False):
        got = R.load_onnx_weights(path, g, by_name=by_name)
        assert set(got) == set(w) and all(np.array_equal(got[k], w[k]) for k in w), by_name


@pytest.mark.parametrize("variant,layer", [("depthwise", "model.22.cv3.0.0"), ("no_angle", "model.22.cv4.0.0")])
def test_onnx_reader_refuses_the_wrong_obb_head(tmp_path, variant, layer):
    import _export_onnx as E
    from aerial_image_recognition_b200 import onnx_reader as R
    g = G.build("yolov8m-obb", imgsz=64)
    m = _obb_module(g.nc, depthwise_cls=variant == "depthwise", angle=variant != "no_angle")
    path = str(tmp_path / f"{variant}.onnx")
    E.export(m, path)
    for by_name in (True, False):
        with pytest.raises(ValueError, match=layer.replace(".", r"\.")):
            R.load_onnx_weights(path, g, by_name=by_name)
