"""GPU parity tests (-m gpu): the CUDA path, called through the C ABI (ctypes -> libb2det.so),
against the CPU oracle on the same seeded inputs.  Integer / byte / index work must be bit-exact;
bf16 network outputs are compared with the tolerances written in each test."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from aerial_image_recognition_b200 import graph as G, mosaic as M, synth, weights as W
from oracle import postproc as OP
from oracle.yolo_torch import make_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _engine(*a, **k):
    from aerial_image_recognition_b200.engine import Engine
    return Engine(*a, **k)


@pytest.fixture(scope="module")
def eng640():
    g = G.build("yolov8m")
    w = W.make_synthetic_weights(g, 0)
    e = _engine("yolov8m", weights=w, max_batch=4, graph=g)
    e._weights = w
    yield e
    e.close()


@pytest.fixture(scope="module")
def tiles4():
    return synth.make_tiles(4, 640, 5)


# ---- K1 ---------------------------------------------------------------------------------------
def _images():
    from PIL import Image
    rng = np.random.default_rng(0)
    out = [np.array(Image.open(os.path.join(ROOT, "tests/golden/test_tile_864.png")).convert("RGB"))]
    for shape in [(864, 864), (1280, 1280), (1000, 1300), (700, 640), (640, 1200)]:
        out.append(rng.integers(0, 256, (*shape, 3), dtype=np.uint8))
    return out


def test_preprocess_bit_exact_against_pillow_and_opencv(eng640):
    import cv2
    from PIL import Image
    for img in _images():
        t = torch.from_numpy(img)[None].cuda()
        pil = np.array(Image.fromarray(img).resize((640, 640)))
        cv = cv2.resize(img, (640, 640))
        assert np.array_equal(eng640.preprocess(t, "pil_bicubic", out="u8").cpu().numpy()[0], pil)
        assert np.array_equal(eng640.preprocess(t, "cv2_linear", out="u8").cpu().numpy()[0], cv)
        # the f32 tensor the reference feeds session.run (simple_detector.py:465-467)
        ref = np.expand_dims((pil.astype(np.float32) / 255.0).transpose(2, 0, 1), 0)
        assert np.array_equal(eng640.preprocess(t, "pil_bicubic", out="f32").cpu().numpy(), ref)
        assert np.array_equal(eng640.preprocess(t, "cv2_linear", bgr=True, out="u8").cpu().numpy()[0], cv[..., ::-1])


def test_preprocess_identity_and_engine_input(eng640, tiles4):
    t = torch.from_numpy(tiles4).cuda()
    assert np.array_equal(eng640.preprocess(t, "identity", out="u8").cpu().numpy(), tiles4)
    eng640.preprocess(t, "identity")
    got = eng640.buffer("input", 4).float().cpu().numpy()
    # the network input is the raw pixel value (exact in bf16); `/ 255.0` is the stem's accumulator scale
    assert np.array_equal(got[..., :3], tiles4.astype(np.float32)) and (got[..., 3] == 0).all()


@pytest.mark.parametrize("h,w", [(600, 1200), (601, 1203), (333, 640), (1200, 601), (640, 333), (777, 500), (64, 640), (640, 64)])
def test_letterbox_matches_ultralytics_letterbox(eng640, h, w):
    """Ultralytics LetterBox(auto=False, scaleup=True, center=True) restated with cv2 itself: r = min(640/h, 640/w), resize to
    (round(w r), round(h r)) with INTER_LINEAR, then ``top, bottom = round(dh - 0.1), round(dh + 0.1)`` (same for left / right)
    rows of 114 -- odd paddings (601x1203 -> 320 rows + 1 odd, 333x640, 777x500 ...) put the extra row / column at the bottom / right."""
    import cv2
    rng = np.random.default_rng(h * 10007 + w)
    img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    got = eng640.preprocess(torch.from_numpy(img)[None].cuda(), "letterbox", out="u8").cpu().numpy()[0]
    r = min(640 / h, 640 / w)
    nw, nh = int(round(w * r)), int(round(h * r))
    dw, dh = (640 - nw) / 2, (640 - nh) / 2
    res = cv2.resize(img, (nw, nh), interpolation=cv2.INTER_LINEAR) if (w, h) != (nw, nh) else img
    top, bottom = int(round(dh - 0.1)), int(round(dh + 0.1))
    left, right = int(round(dw - 0.1)), int(round(dw + 0.1))
    ref = cv2.copyMakeBorder(res, top, bottom, left, right, cv2.BORDER_CONSTANT, value=(114, 114, 114))
    assert ref.shape == (640, 640, 3) and np.array_equal(got, ref)


def test_session_input_path_equals_preprocess_path(eng640, tiles4):
    t = torch.from_numpy(tiles4[:2]).cuda()
    eng640.preprocess(t, "identity")
    a = eng640.buffer("input", 2).clone()
    eng640.set_input_f32(eng640.preprocess(t, "identity", out="f32"))
    assert torch.equal(a, eng640.buffer("input", 2))


# ---- K2/K3: every op of the graph against torch on the engine's own inputs -------------------------
@pytest.mark.parametrize("arch,imgsz,n", [("yolov8m", 128, 3), ("yolov8m", 320, 2), ("yolov7", 128, 2),
                                          ("yolov8m", 224, 3), ("yolov7", 160, 2), ("xunet", 96, 2)])     # the last three: partial tiles in x and y
def test_every_planned_op_matches_torch(arch, imgsz, n):
    _check_every_op(arch, imgsz, n)


@pytest.mark.parametrize("arch,imgsz,n", [("yolov8m", 640, 2), ("yolov7", 256, 2)])
def test_every_planned_op_large_batch_kernel_variants(arch, imgsz, n, monkeypatch):
    """The planner only picks multi-tile rounds (mt = 2 / 4) and CTA pairs when a layer has enough tiles to
    balance 148 SMs, i.e. at bench batch sizes.  Force them (B2D_MT, B2D_PAIR=2 are read at plan time) so the
    kernels the benchmark runs -- the CTA-pair forms of the halo and generic kernels, two-tile halo/generic rounds, four-tile
    stem -- are the ones checked."""
    monkeypatch.setenv("B2D_MT", "4")
    monkeypatch.setenv("B2D_PAIR", "2")
    seen = _check_every_op(arch, imgsz, n)
    assert any("halo-pair" in d for d in seen) and any("tcgen05-pair conv" in d for d in seen), seen[:8]
    assert any(" x2 " in d for d in seen) and any(" x4 " in d for d in seen), seen[:8]


def test_every_planned_op_matches_torch_split_fp16():
    """B2D_PREC_FP16X2: every op on its own inputs (hi + lo read back as fp32) to ~fp32 accuracy."""
    _check_every_op("yolov8m", 320, 2, precision="fp16x2")
    _check_every_op("yolov7", 128, 2, precision="fp16x2")


def test_every_planned_op_at_full_size_with_tiles_spanning_images():
    """At 640x640 the 20x20 layers run 4x4-pixel x 8-image M tiles and the 40x40 ones 8x8 x 2: n = 8 fills such tiles with
    eight different images (n = 2 leaves six of the eight image slots of a tile empty)."""
    seen = _check_every_op("yolov8m", 640, 8)
    assert any("tile 4x4x8" in d for d in seen) and any("tile 8x8x2" in d for d in seen), [d for d in seen if "20x20" in d][:3]


def _check_every_op(arch, imgsz, n, precision="bf16"):
    from _ir_cpu import run_graph_cpu  # noqa: F401  (same arithmetic, per-op form below)
    import torch.nn.functional as F
    seen = []
    g = G.build(arch, imgsz=imgsz)
    w = W.make_synthetic_weights(g, 2)
    eng = _engine(arch, weights=w, max_batch=n, imgsz=imgsz, graph=g, precision=precision)
    eng.preprocess(torch.from_numpy(synth.make_tiles(n, imgsz, 9)).cuda(), "identity")
    # one ulp of the storage format: 2^-8 (bf16), 2^-11 (fp16); split fp16 keeps ~22 bits, the bound is fp32 summation order
    rel16 = {"bf16": 4e-3, "fp16": 5e-4, "fp16x2": 2e-5}[precision]
    for i, op in enumerate(g.ops):
        eng.run_op(i, n)
        torch.cuda.synchronize()
        src = eng.buffer(op.src.buf, n).float().cpu()[..., op.src.c0:op.src.c0 + op.src.c].permute(0, 3, 1, 2)
        if op.kind in ("conv", "dwconv"):
            if op.src.buf == "input":
                src = src[:, :3] / 255.0                 # the input buffer holds raw pixel values; this is the reference's tensor
            wt, bs = (torch.from_numpy(np.ascontiguousarray(a)) for a in G.op_weights(op, w))
            y = F.conv2d(src, wt, bs,
                         stride=op.s, padding=op.k // 2, groups=g.wshapes[op.weight][3])
            if op.act:
                y = y * torch.sigmoid(y)
            if op.res is not None:
                y = y + eng.buffer(op.res.buf, n).float().cpu()[..., op.res.c0:op.res.c0 + op.res.c].permute(0, 3, 1, 2)
        elif op.kind == "maxpool":
            y = F.max_pool2d(src, op.k, op.s, op.k // 2 if op.s == 1 else 0)
        else:
            y = F.interpolate(src, scale_factor=2, mode="nearest")
        got = eng.buffer(op.dst.buf, n).float().cpu()[..., op.dst.c0:op.dst.c0 + op.dst.c].permute(0, 3, 1, 2)
        err = (got - y).abs().max().item()
        # bf16 output rounding is 2^-9 relative; fp32 head outputs and pools/upsamples are far tighter
        tol = (rel16 if not g.bufs[op.dst.buf].f32 else min(2e-4, 10 * rel16)) * y.abs().max().item() + 1e-5
        if op.kind in ("maxpool", "upsample2x"):
            tol = 0.0
        assert err <= tol, (i, eng.describe_op(i), err, tol)
        seen.append(eng.describe_op(i))
    eng.close()
    return seen


@pytest.mark.parametrize("arch,imgsz,n,precision", [("yolov8m", 128, 3, "bf16"), ("yolov8m", 320, 2, "bf16"), ("yolov8m", 640, 2, "bf16"),
                                                     ("yolov8m", 640, 8, "bf16"), ("yolov8m", 320, 2, "fp16")])
def test_fused_depthwise_pointwise_kernel_matches_torch(arch, imgsz, n, precision):
    """forward() runs DWConv 3x3 -> Conv 1x1 of the cls branch as one kernel (conv_tc_dwpw_kernel): on the engine's own input
    the pair kernel must equal torch's dwconv -> SiLU -> (rounded to the storage format, as the unfused pair stores it) ->
    1x1 -> SiLU to one ulp of the storage format, and agree with the two single-op kernels to the same bound."""
    import torch.nn.functional as F
    g = G.build(arch, imgsz=imgsz)
    w = W.make_synthetic_weights(g, 2)
    eng = _engine(arch, weights=w, max_batch=n, imgsz=imgsz, graph=g, precision=precision)
    eng.preprocess(torch.from_numpy(synth.make_tiles(n, imgsz, 9)).cuda(), "identity")
    eng.forward(n)
    torch.cuda.synchronize()
    rel16 = {"bf16": 4e-3, "fp16": 5e-4}[precision]
    store = torch.bfloat16 if precision == "bf16" else torch.float16
    pairs = [i for i in range(len(g.ops) - 1) if eng.fused_with_next(i)]
    assert len(pairs) == 6, pairs                      # cv3.{0,1,2}.{0,1}: two pairs per head level
    for i in pairs:
        a, b = g.ops[i], g.ops[i + 1]
        assert a.kind == "dwconv" and b.kind == "conv" and b.k == 1
        src = eng.buffer(a.src.buf, n).float().cpu()[..., a.src.c0:a.src.c0 + a.src.c].permute(0, 3, 1, 2)
        wa, ba = (torch.from_numpy(np.ascontiguousarray(x)) for x in G.op_weights(a, w))
        wb, bb = (torch.from_numpy(np.ascontiguousarray(x)) for x in G.op_weights(b, w))
        mid = F.conv2d(src, wa, ba, padding=1, groups=a.src.c)
        mid = (mid * torch.sigmoid(mid)).to(store).float()
        y = F.conv2d(mid, wb, bb)
        y = y * torch.sigmoid(y)
        def out():
            torch.cuda.synchronize()
            return eng.buffer(b.dst.buf, n).float().cpu()[..., b.dst.c0:b.dst.c0 + b.dst.c].permute(0, 3, 1, 2).clone()
        eng.buffer(b.dst.buf, n).zero_()
        eng.run_op_fused(i, n)
        fused = out()
        eng.buffer(b.dst.buf, n).zero_()
        eng.run_op(i, n)
        eng.run_op(i + 1, n)
        single = out()
        tol = 2 * rel16 * y.abs().max().item() + 1e-5
        assert (fused - y).abs().max().item() <= tol, (i, eng.describe_op(i), (fused - y).abs().max().item(), tol)
        assert (fused - single).abs().max().item() <= tol, (i, (fused - single).abs().max().item(), tol)
    assert eng.num_kernels == sum(1 for _ in g.ops) - 2 - len(pairs), eng.num_kernels     # SPPF pool chain (3 -> 1) and the six pairs
    eng.close()


# ---- config C5: the segmentation stand-in ("ramp XUnet 256") -------------------------------------------
def test_xunet_every_planned_op_matches_torch():
    seen = _check_every_op("xunet", 128, 3)
    assert any("stem-s2d" in d for d in seen) and any("depthwise" in d for d in seen)
    _check_every_op("xunet", 256, 2)


def test_xunet_logits_and_labels_vs_oracle():
    """Whole stand-in network at 256 x 256: logits against the oracle with the same storage rounding (kernels' arithmetic) and against
    the fp32 oracle (storage format's deviation), labels / softmax kernel exact on the engine's own logits, and label agreement."""
    from oracle.xunet_torch import XUnetOracle
    n = 3
    g = G.build("xunet")
    w = W.make_synthetic_weights(g, 0)
    tiles = synth.make_tiles(n, 256, 77)
    x = torch.from_numpy(tiles.astype(np.float32) / 255.0).permute(0, 3, 1, 2)
    ref16 = XUnetOracle(w, emulate_bf16=True).logits(x)
    ref32 = XUnetOracle(w, emulate_bf16=False).logits(x)
    eng = _engine("xunet", weights=w, max_batch=n, graph=g)
    eng.preprocess(torch.from_numpy(tiles).cuda(), "identity")
    eng.forward(n)
    z = eng.buffer("logits", n).float().cpu()[..., :4].permute(0, 3, 1, 2)
    scale = ref32.abs().max().item()
    e16, e32 = (z - ref16).abs().max().item() / scale, (z - ref32).abs().max().item() / scale
    print(f"xunet logits: max |d| / max |z| = {e16:.2e} vs bf16-emulating oracle, {e32:.2e} vs fp32 oracle")
    assert e16 < 3e-2 and e32 < 6e-2, (e16, e32)
    labels, conf = eng.segment(n)
    torch.cuda.synchronize()
    zz = eng.buffer("logits", n).float()[:n, ..., :4]
    assert torch.equal(labels.cpu(), zz.argmax(-1).to(torch.uint8).cpu())                # first maximum wins, like argmax
    assert (conf.cpu() - torch.softmax(zz, -1).amax(-1).cpu()).abs().max().item() < 1e-6
    agree = (labels.cpu() == ref32.argmax(1).to(torch.uint8)).float().mean().item()
    assert agree > 0.97, agree
    eng.close()


# ---- whole network vs the oracle -------------------------------------------------------------------
# Contract (BASELINE.json north_star; the reference's fp32 `session.run`, simple_detector.py:474-481): scores within 1e-3
# absolute, boxes within 0.5 px, identical keep set away from score ties.  Asserted at 640x640 on C2 tiles (the bench's
# generator) against the fp32 oracle, over every anchor with score >= 0.05, and the keep set (`score >= thr`, thr = the
# reference's 0.3 and the bench's 0.25) must be identical outside the band |score - thr| < 2e-3.
SCORE_TOL, BOX_TOL_PX, TIE_BAND, SCORE_FLOOR = 1e-3, 0.5, 2e-3, 0.05


@pytest.fixture(scope="module")
def c2_reference():
    """Four C2 tiles and the fp32 oracle's rows for them (cx, cy, w, h, conf, cls)."""
    g = G.build("yolov8m")
    w = W.make_synthetic_weights(g, 0)
    tiles = synth.make_tiles(4, 640, 1000)
    x = torch.from_numpy(tiles.astype(np.float32) / 255.0).permute(0, 3, 1, 2)
    ref = np.stack([OP.v8_rows_adapter(r.numpy()) for r in make_oracle("yolov8m", w, False).forward(x)])
    return g, w, tiles, x, ref


def _rows_of(precision, g, w, tiles):
    eng = _engine("yolov8m", weights=w, max_batch=len(tiles), graph=g, precision=precision)
    eng.preprocess(torch.from_numpy(tiles).cuda(), "identity")
    eng.forward(len(tiles))
    rows = eng.decode_rows(len(tiles)).cpu().numpy()
    eng.close()
    return rows


def _deviation(rows, ref, tag):
    sel = ref[..., 4] >= SCORE_FLOOR
    ds = np.abs(rows[..., 4] - ref[..., 4])[sel]
    db = np.abs(rows[..., :4] - ref[..., :4]).max(-1)[sel]
    q = lambda a: tuple(float(np.quantile(a, p)) for p in (0.5, 0.99, 0.999, 1.0))
    worst = {}
    for thr in (0.3, 0.25):
        dis = (rows[..., 4] >= thr) != (ref[..., 4] >= thr)
        worst[thr] = (int(dis.sum()), int((ref[..., 4] >= thr).sum()), float(np.abs(ref[..., 4] - thr)[dis].max()) if dis.any() else 0.0)
    print(f"\n[{tag}] {int(sel.sum())} anchors with score >= {SCORE_FLOOR}: |d score| median / p99 / p99.9 / max = %.2e %.2e %.2e %.2e ; "
          "|d box| px = %.3f %.3f %.3f %.3f ; keep set: " % (q(ds) + q(db)) +
          ", ".join(f"thr {t}: {n} of {m} differ, farthest from thr {d:.1e}" for t, (n, m, d) in worst.items()))
    return q(ds), q(db), worst


def test_contract_scores_boxes_keep_set_split_fp16_vs_fp32_oracle(c2_reference):
    """The configuration that meets the contract: B2D_PREC_FP16X2 (activations as fp16 hi + lo, fp32 accumulate)."""
    g, w, tiles, x, ref = c2_reference
    ds, db, worst = _deviation(_rows_of("fp16x2", g, w, tiles), ref, "fp16x2 vs fp32 oracle")
    assert ds[3] <= SCORE_TOL, ds
    assert db[3] <= BOX_TOL_PX, db
    for thr, (n, m, far) in worst.items():
        assert far < TIE_BAND, (thr, n, m, far)          # every disagreement is a tie with the threshold


def test_fast_storage_modes_stated_deviation_from_fp32_oracle(c2_reference):
    """bf16 (the BASELINE configuration) and fp16 store one 16-bit value per activation: 2^-9 / 2^-12 relative rounding at
    each of ~60 layers.  That is NOT within the 1e-3 contract at the tail; the bounds the test pins are the measured ones
    (DESIGN.md section 2 has the table), and the deviation is shown to be the storage format's, not the kernels': a CPU model
    that only rounds its stored activations the same way is as far from fp32 as the engine is."""
    g, w, tiles, x, ref = c2_reference
    bounds = {"fp16": dict(p99=6e-3, smax=1.5e-2, bmax=1.5, band=1.5e-2), "bf16": dict(p99=5e-2, smax=0.15, bmax=12.0, band=0.15)}
    for prec, emu in (("fp16", "fp16"), ("bf16", True)):
        rows = _rows_of(prec, g, w, tiles)
        ds, db, worst = _deviation(rows, ref, f"{prec} vs fp32 oracle")
        b = bounds[prec]
        assert ds[1] <= b["p99"] and ds[3] <= b["smax"] and db[3] <= b["bmax"], (prec, ds, db)
        for thr, (n, m, far) in worst.items():
            assert far < b["band"] and n <= 0.05 * m, (prec, thr, n, m, far)
        emu_rows = np.stack([OP.v8_rows_adapter(r.numpy()) for r in make_oracle("yolov8m", w, emu).forward(x)])
        d_eng, d_emu = np.abs(rows[..., 4] - ref[..., 4]), np.abs(emu_rows[..., 4] - ref[..., 4])
        assert d_eng.mean() < 1.25 * d_emu.mean() + 1e-5 and np.quantile(d_eng, 0.99) < 1.25 * np.quantile(d_emu, 0.99) + 1e-4, (
            prec, d_eng.mean(), d_emu.mean(), np.quantile(d_eng, 0.99), np.quantile(d_emu, 0.99))


def test_contract_yolov7_split_fp16_vs_fp32_oracle():
    """The same contract on the canonical YOLOv7 graph (BASELINE config C3; the reference's own filter reads column 4 = objectness,
    simple_detector.py:479-481): rows (cx, cy, w, h, obj, cls) at 640 x 640 against the fp32 oracle."""
    g = G.build("yolov7")
    w = W.make_synthetic_weights(g, 0)
    tiles = synth.make_tiles(2, 640, 3000)
    x = torch.from_numpy(tiles.astype(np.float32) / 255.0).permute(0, 3, 1, 2)
    ref = make_oracle("yolov7", w, False).forward(x).numpy()
    eng = _engine("yolov7", weights=w, max_batch=2, graph=g, precision="fp16x2")
    eng.preprocess(torch.from_numpy(tiles).cuda(), "identity")
    eng.forward(2)
    rows = eng.decode_rows(2).cpu().numpy()
    eng.close()
    sel = ref[..., 4] >= SCORE_FLOOR
    ds = np.abs(rows[..., 4] - ref[..., 4])[sel]
    db = np.abs(rows[..., :4] - ref[..., :4]).max(-1)[sel]
    dis = (rows[..., 4] >= 0.3) != (ref[..., 4] >= 0.3)
    far = float(np.abs(ref[..., 4] - 0.3)[dis].max()) if dis.any() else 0.0
    print(f"\n[yolov7 fp16x2 vs fp32 oracle] {int(sel.sum())} rows with obj >= {SCORE_FLOOR}: |d obj| max {ds.max():.2e} p99 {np.quantile(ds, 0.99):.2e}; "
          f"|d box| px max {db.max():.3f}; keep set (obj >= 0.3): {int(dis.sum())} of {int((ref[..., 4] >= 0.3).sum())} differ, farthest {far:.1e}")
    assert ds.max() <= SCORE_TOL and db.max() <= BOX_TOL_PX and far < TIE_BAND, (ds.max(), db.max(), far)


def test_split_fp16_whole_pipeline_matches_oracle_detections(c2_reference):
    """Decode + Ultralytics NMS on the precise rows: the detections of every tile are the oracle's (same anchors kept, in the
    same order) unless a competing pair sits within the tie band."""
    g, w, tiles, x, ref = c2_reference
    n = len(tiles)
    eng = _engine("yolov8m", weights=w, max_batch=n, graph=g, precision="fp16x2")
    dets, counts = eng.infer(torch.from_numpy(tiles).cuda(), "identity", False, 0.25, False, 0.7, 0, 300)
    from aerial_image_recognition_b200.engine import dets_to_numpy
    got = dets_to_numpy(dets, counts)
    pred = make_oracle("yolov8m", w, False).forward(x).numpy()
    agree = total = 0
    for i in range(n):
        ref_det = OP.ultralytics_nms(pred[i:i + 1], 0.25, 0.7, 300)[0]
        ga = set(int(a) for a in got[i]["anchor"])
        # map the oracle's kept boxes back to anchors through their (unique) scores + centres
        rs = ref[i]
        ra = set()
        for d in ref_det:
            cx, cy = (d[0] + d[2]) / 2, (d[1] + d[3]) / 2
            k = np.argmin(np.abs(rs[:, 0] - cx) + np.abs(rs[:, 1] - cy) + 1e3 * np.abs(rs[:, 4] - d[4]))
            ra.add(int(k))
        agree += len(ga & ra); total += len(ga | ra)
    eng.close()
    assert agree / total > 0.995, (agree, total)


def test_decode_kernel_matches_oracle_decode_on_identical_head_maps(eng640, tiles4):
    """Isolates K4: feed the oracle decode the engine's own raw head maps."""
    n = 2
    eng640.preprocess(torch.from_numpy(tiles4[:n]).cuda(), "identity")
    eng640.forward(n)
    rows = eng640.decode_rows(n).cpu().numpy()
    raw = [eng640.buffer(lv["buf"], n).float().cpu()[..., :66].permute(0, 3, 1, 2).contiguous() for lv in eng640.graph.head["levels"]]
    from oracle.yolo_torch import YoloV8mOracle
    ref = np.stack([OP.v8_rows_adapter(r.numpy()) for r in YoloV8mOracle.decode(raw)])
    assert np.abs(rows[..., :4] - ref[..., :4]).max() < 2e-2        # px; expf / reduction-order noise only
    assert np.abs(rows[..., 4] - ref[..., 4]).max() < 1e-6
    assert np.array_equal(rows[..., 5], ref[..., 5])


def test_v7_decode_kernel_matches_oracle():
    g = G.build("yolov7", imgsz=256)
    w = W.make_synthetic_weights(g, 0)
    eng = _engine("yolov7", weights=w, max_batch=2, imgsz=256, graph=g)
    t = synth.make_tiles(2, 256, 3)
    eng.preprocess(torch.from_numpy(t).cuda(), "identity")
    eng.forward(2)
    rows = eng.decode_rows(2).cpu().numpy()
    from oracle.yolo_torch import YoloV7Oracle
    raw = [eng.buffer(lv["buf"], 2).float().cpu()[..., :18].permute(0, 3, 1, 2).contiguous() for lv in g.head["levels"]]
    ref = YoloV7Oracle.decode(raw).numpy()
    assert rows.shape == (2, 3 * (32 * 32 + 16 * 16 + 8 * 8), 6)
    assert np.abs(rows[..., :5] - ref[..., :5]).max() < 1e-3 * max(1.0, np.abs(ref[..., :4]).max())
    full = make_oracle("yolov7", w, emulate_bf16=True).forward(torch.from_numpy(t.astype(np.float32) / 255).permute(0, 3, 1, 2)).numpy()
    assert np.median(np.abs(rows[..., 4] - full[..., 4])) < 2e-3
    eng.close()


# ---- K4' / K5: filter, top-k, NMS are exact on identical rows ------------------------------------------
def _synthetic_rows(n, A, seed=3):
    rng = np.random.default_rng(seed)
    rows = np.zeros((n, A, 6), np.float32)
    centers = rng.uniform(20, 620, (n, 40, 2)).astype(np.float32)
    idx = rng.integers(0, 40, (n, A))
    rows[..., 0:2] = np.take_along_axis(centers, idx[..., None].repeat(2, -1), 1) + rng.normal(0, 3, (n, A, 2)).astype(np.float32)
    rows[..., 2:4] = rng.uniform(15, 50, (n, A, 2)).astype(np.float32)
    rows[..., 4] = (rng.random((n, A)) ** 6).astype(np.float32)
    rows[..., 5] = rng.integers(0, 2, (n, A)).astype(np.float32)
    rows[0, :50, 4] = 0.5
    return rows


@pytest.mark.parametrize("A", [8400, 25200, 37])
def test_filter_topk_and_nms_exact(eng640, A):
    from aerial_image_recognition_b200.engine import dets_to_numpy
    n = 3
    rows = _synthetic_rows(n, A)
    rt = torch.from_numpy(rows).cuda()
    got = dets_to_numpy(*eng640.postprocess(n, 0.3, True, rows=rt))
    for i in range(n):
        ref = OP.filter_rows(rows[i], 0.3)
        assert len(ref) == len(got[i]) and np.array_equal(ref[:, :5], np.stack([got[i][k] for k in ("cx", "cy", "w", "h", "conf")], 1))
    got = dets_to_numpy(*eng640.postprocess(n, 0.3, True, top_k=10, rows=rt))
    for i in range(n):
        ref = OP.top_k_rows(OP.filter_rows(rows[i], 0.3), 10)
        assert np.array_equal(ref[:, 4], got[i]["conf"])
    pred = np.zeros((n, 6, A), np.float32)
    pred[:, :4] = rows[..., :4].transpose(0, 2, 1)
    cls = rows[..., 5].astype(int)
    for c in range(2):
        pred[:, 4 + c] = np.where(cls == c, rows[..., 4], rows[..., 4] * 0.5)
    ref = OP.ultralytics_nms(pred, 0.25, 0.7, 300)
    rows_nms = np.stack([OP.v8_rows_adapter(p) for p in pred])
    got = dets_to_numpy(*eng640.postprocess(n, 0.25, False, iou_thr=0.7, max_det=300, rows=torch.from_numpy(rows_nms).cuda()))
    for i in range(n):
        assert len(ref[i]) == len(got[i])
        assert np.array_equal(ref[i][:, 4], got[i]["conf"]) and np.array_equal(ref[i][:, 5].astype(np.int32), got[i]["cls"])
        x1 = got[i]["cx"] - got[i]["w"] / np.float32(2)
        assert np.array_equal(ref[i][:, 0], x1)


def test_postprocess_empty_and_all_pass(eng640):
    from aerial_image_recognition_b200.engine import dets_to_numpy
    rows = np.zeros((2, 100, 6), np.float32)
    rows[1, :, 4] = 0.9
    rows[1, :, :4] = np.arange(400, dtype=np.float32).reshape(100, 4)
    got = dets_to_numpy(*eng640.postprocess(2, 0.3, True, rows=torch.from_numpy(rows).cuda()))
    assert len(got[0]) == 0 and len(got[1]) == 100 and np.array_equal(got[1]["cx"], rows[1, :, 0])


def test_fused_head_postprocess_equals_rows_postprocess(eng640, tiles4):
    """The fused decode+filter kernel and decode_rows -> filter_rows give the same detections."""
    from aerial_image_recognition_b200.engine import dets_to_numpy
    n = 4
    dets, counts = eng640.infer(torch.from_numpy(tiles4).cuda(), "identity", conf_thr=0.3, inclusive=True)
    rows = eng640.decode_rows(n).cpu().numpy()
    got = dets_to_numpy(dets, counts)
    for i in range(n):
        ref = OP.filter_rows(rows[i], 0.3)
        assert len(ref) == len(got[i]) and np.array_equal(ref[:, 4], got[i]["conf"]) and np.array_equal(ref[:, 0], got[i]["cx"])
    d2, c2 = eng640.postprocess(n, 0.25, False, iou_thr=0.7, max_det=300)
    pred = np.concatenate([rows[..., :4], np.where(np.arange(2)[None, None] == rows[..., 5:6], rows[..., 4:5], 0)], -1).transpose(0, 2, 1)
    ref = OP.ultralytics_nms(np.ascontiguousarray(pred), 0.25, 0.7, 300)
    got = dets_to_numpy(d2, c2)
    for i in range(n):
        assert len(ref[i]) == len(got[i]) and np.array_equal(ref[i][:, 4], got[i]["conf"])


# ---- K6 georef: bit-exact fp64 ---------------------------------------------------------------------------
def test_georef_three_forms_bit_exact(eng640):
    from aerial_image_recognition_b200.engine import dets_to_numpy, geodets_to_numpy
    n = 3
    rows = _synthetic_rows(n, 4000, seed=8)
    dets, counts = eng640.postprocess(n, 0.3, True, rows=torch.from_numpy(rows).cuda(), cap=1024)
    dd = dets_to_numpy(dets, counts)
    P = np.zeros((n, 16))
    for i in range(n):
        P[i, :6] = (-118.2503 + i * 1e-3, -118.2497 + i * 1e-3, 34.0497, 34.0503, 864, 640)
    gg = geodets_to_numpy(eng640.georef(dets, counts, torch.from_numpy(P).cuda(), "bounds"), counts)
    for i in range(n):
        for k in range(len(dd[i])):
            lon, lat, xi, yi = OP.georef_bounds(dd[i]["cx"][k], dd[i]["cy"][k], *P[i, :4], 640, 864)
            assert (lon, lat) == (gg[i]["x"][k], gg[i]["y"][k]) and np.float32(xi) == gg[i]["x_img"][k]
    P2 = np.zeros((n, 16)); P2[:, :4] = P[:, [0, 2, 1, 3]]
    gg = geodets_to_numpy(eng640.georef(dets, counts, torch.from_numpy(P2).cuda(), "gpuhandler"), counts)
    for i in range(n):
        for k in range(len(dd[i])):
            assert OP.georef_gpuhandler(dd[i]["cx"][k], dd[i]["cy"][k], *P2[i, :4]) == (gg[i]["x"][k], gg[i]["y"][k])
    gt = (2335637.62, 0.1, 0.0, 6845688.78, 0.0, -0.1)
    wins = np.array([[0, 0, 640, 640], [39936, 512, 64, 640], [1024, 39936, 640, 64]], np.int32)
    P3 = M.affine_params(wins, gt)
    gg = geodets_to_numpy(eng640.georef(dets, counts, torch.from_numpy(P3).cuda(), "affine"), counts)
    for i in range(n):
        d = dd[i]
        b = np.stack([d["cx"] - d["w"] / np.float32(2), d["cy"] - d["h"] / np.float32(2),
                      d["cx"] + d["w"] / np.float32(2), d["cy"] + d["h"] / np.float32(2)], 1)
        w0, h0 = int(wins[i, 2]), int(wins[i, 3])
        # Ultralytics scale_boxes for a model-sized letterbox (gain 1), then the notebook's centroid
        b[:, [0, 2]] -= np.float32((640 - w0) // 2); b[:, [1, 3]] -= np.float32((640 - h0) // 2)
        b[:, [0, 2]] = b[:, [0, 2]].clip(0, w0); b[:, [1, 3]] = b[:, [1, 3]].clip(0, h0)
        for k in range(len(d)):
            cx = float(np.float32(b[k, 0] + b[k, 2])) / 2 + int(wins[i, 0])
            cy = float(np.float32(b[k, 1] + b[k, 3])) / 2 + int(wins[i, 1])
            assert OP.georef_affine(cx, cy, gt) == (gg[i]["x"][k], gg[i]["y"][k])


# ---- K5' dedup / closure / UTM ----------------------------------------------------------------------------
@pytest.mark.parametrize("m", [0, 1, 2000, 60000])
def test_dedup_identical_to_sequential_greedy(eng640, m):
    rng = np.random.default_rng(m)
    x = rng.uniform(0, 40 * max(m, 1) ** 0.5 / 10, m); y = rng.uniform(0, 40 * max(m, 1) ** 0.5 / 10, m)
    conf = rng.random(m).astype(np.float32)
    conf[: m // 10] = 0.5
    for incl in (True, False):
        keep = eng640.dedup(torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda(), torch.from_numpy(conf).cuda(), 1.0, incl).cpu().numpy()
        ref = np.zeros(m, bool); ref[OP.dedup_greedy(x, y, conf, 1.0, incl)] = True
        assert np.array_equal(ref, keep.astype(bool))
    if m:  # idempotent: deduplicating the survivors removes nothing
        k = keep.astype(bool)
        again = eng640.dedup(torch.from_numpy(x[k]).cuda(), torch.from_numpy(y[k]).cuda(), torch.from_numpy(conf[k]).cuda(), 1.0, False)
        assert again.all()


def test_dedup_negative_and_origin_cells(eng640):
    """Points in grid cell (-1, -1) and around the origin (negative-coordinate CRS, raw lon/lat near 0): with plain
    two's-complement packing that cell's key was the hash table's empty-slot sentinel and its points were invisible."""
    rng = np.random.default_rng(12)
    x = rng.uniform(-3.0, 3.0, 4000); y = rng.uniform(-3.0, 3.0, 4000)
    conf = rng.random(4000).astype(np.float32)
    for incl in (True, False):
        keep = eng640.dedup(torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda(), torch.from_numpy(conf).cuda(), 1.0, incl).cpu().numpy()
        ref = np.zeros(4000, bool); ref[OP.dedup_greedy(x, y, conf, 1.0, incl)] = True
        assert np.array_equal(ref, keep.astype(bool))
    from aerial_image_recognition_b200._lib import B2DError
    far = torch.tensor([0.0, 1e13], dtype=torch.float64).cuda()       # |x / thr| >= 2^31: refused, not truncated
    with pytest.raises(B2DError, match="outside the grid"):
        eng640.dedup(far, far.clone(), torch.ones(2).cuda(), 1.0, True)


def test_dedup_chain_and_exact_threshold(eng640):
    # a 500-long chain at spacing exactly thr: inclusive keeps every second, strict keeps all
    x = np.arange(500, dtype=np.float64); y = np.zeros(500)
    conf = np.linspace(1.0, 0.5, 500).astype(np.float32)
    k = eng640.dedup(torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda(), torch.from_numpy(conf).cuda(), 1.0, True).cpu().numpy()
    assert np.array_equal(k, (np.arange(500) % 2 == 0).astype(np.uint8))
    k = eng640.dedup(torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda(), torch.from_numpy(conf).cuda(), 1.0, False).cpu().numpy()
    assert k.all()


def test_utm_forward_and_simple_detector_remove_duplicates(eng640):
    rng = np.random.default_rng(1)
    lon = rng.uniform(-118.3, -118.2, 3000); lat = rng.uniform(34.0, 34.1, 3000)
    ux, uy = eng640.utm_forward(torch.from_numpy(lon).cuda(), torch.from_numpy(lat).cuda(), 11, True)
    rx, ry = OP.utm_forward(lon, lat, 11, True)
    assert np.abs(ux.cpu().numpy() - rx).max() < 1e-6 and np.abs(uy.cpu().numpy() - ry).max() < 1e-6


# ---- mosaic: sharded == unsharded -----------------------------------------------------------------------------
def test_sharded_mosaic_equals_single_rank(eng640):
    """Emulates 1, 2 and 3 ranks on one GPU (ranks run one after the other; the all-gather is a list):
    the union of the per-rank outputs must be the single-rank result, bit for bit."""
    H, W_ = 2300, 1700
    mosaic_np = synth.make_mosaic(H, W_, seed=2)
    mosaic = torch.from_numpy(mosaic_np).cuda()
    gt = (2335637.62, 0.1, 0.0, 6845688.78, 0.0, -0.1)
    det = M.MosaicDetector(eng640, gt, conf=0.3, dedup_thr=1.0)
    single = det.run(mosaic, H, W_, 0, 1)
    assert det.last_raw > len(single) > 0            # the overlap produced duplicates and dedup removed them
    key = lambda a: np.sort(a, order=["window", "slot"])
    for world in (2, 3):
        covers = [M.shard_windows(H, W_, r, world)[2] for r in range(world)]
        locals_, recs, cols_ = [], [], []
        for r in range(world):
            wins, ids, _ = M.shard_windows(H, W_, r, world)
            lo, hi = covers[r]
            band = mosaic[lo:hi].contiguous()                      # each rank holds only its band (+ overlap)
            out = det.detect_windows(band, wins, ids, y_offset=lo)
            loc, rec = det.seam_split(*out, r, covers)
            cols, rec2 = det.seam_split(*out, r, covers, pack=False)   # the form `dedup` uses under torchrun: columns stay on the device
            assert torch.equal(rec, rec2)
            locals_.append(loc); recs.append(rec); cols_.append(cols)
        origin = np.concatenate([np.full(len(rc), r, np.int64) for r, rc in enumerate(recs)])
        merged = [np.concatenate([locals_[r], det.seam_merge(recs, origin, r)]) for r in range(world)]
        for r in range(world):                                      # ... and its one packed read-back gives the same records
            assert np.array_equal(det.finish(cols_[r], recs, origin, r), merged[r])
        union = np.concatenate(merged)
        assert len(union) == len(single)
        a, b = key(union), key(single)
        assert np.array_equal(a["window"], b["window"]) and np.array_equal(a["slot"], b["slot"])
        assert np.array_equal(a["x"], b["x"]) and np.array_equal(a["y"], b["y"]) and np.array_equal(a["conf"], b["conf"])
        assert sum(len(rc) for rc in recs) < det.last_raw           # only seam records were exchanged


def test_cut_windows_matches_numpy(eng640):
    H, W_ = 1500, 1100
    m = synth.make_mosaic(H, W_, seed=4)
    wins = M.window_grid(H, W_)
    got = eng640.cut_windows(torch.from_numpy(m).cuda(), torch.from_numpy(wins).cuda()).cpu().numpy()
    for i, (x0, y0, w0, h0) in enumerate(wins):
        ref = np.full((640, 640, 3), 114, np.uint8)
        left, top = (640 - w0) // 2, (640 - h0) // 2
        ref[top:top + h0, left:left + w0] = m[y0:y0 + h0, x0:x0 + w0]
        assert np.array_equal(got[i], ref), i


# ---- the reference-facing classes -------------------------------------------------------------------------------
def _preview(west, south, size_deg=0.0006, crop=864):
    return {"spatial_info": {"bounds": {"west": west, "east": west + size_deg, "south": south, "north": south + size_deg}},
            "image_info": {"crop_size": crop}}


def test_simple_detector_matches_reference_restatement():
    """C1: the 864x864 reference tile through SimpleDetector.detect, against the oracle restatement of
    simple_detector.py:456-504 fed the engine's own rows (pre/post-processing exact) and against
    the full CPU oracle (network tolerance)."""
    from PIL import Image
    from aerial_image_recognition_b200.simple_detector import SimpleDetector
    g = G.build("yolov8m")
    w = W.make_synthetic_weights(g, 0)
    det = SimpleDetector("models/yolov8_tokyo_checkpoint.onnx", None, weights=w, max_batch=2)
    img = Image.open(os.path.join(ROOT, "tests/golden/test_tile_864.png")).convert("RGB")
    info = _preview(-118.2503, 34.0497)
    out = det.detect(img, info)
    # reference restatement on the rows the session returns for the reference's own preprocessing
    arr = np.expand_dims((np.array(img.resize((640, 640))).astype(np.float32) / 255.0).transpose(2, 0, 1), 0)
    rows = det.model.run(None, {det.model.get_inputs()[0].name: arr})[0][0]
    boxes = rows[rows[:, 4] >= det.confidence_threshold]
    b = info["spatial_info"]["bounds"]
    assert len(out) == len(boxes) > 0
    for o, r in zip(out, boxes):
        lon, lat, xi, yi = OP.georef_bounds(r[0], r[1], b["west"], b["east"], b["south"], b["north"], 640, 864)
        assert o["lon"] == lon and o["lat"] == lat and o["confidence"] == float(r[4])
        assert o["image"]["x"] == float(np.float32(xi)) and o["yolo"]["x"] == float(r[0])
    assert set(out[0]) == {"lon", "lat", "confidence", "image", "yolo"}
    # _process_detections on host rows gives the same records; detect_batch concatenates in order
    assert det._process_detections(rows, info) == out
    two = det.detect_batch([img, img], [info, _preview(-118.24, 34.05)])
    assert two[:len(out)] == out and len(two) == 2 * len(out)
    # the tensor input forms of SURVEY 8b: one uint8 tensor [B,H,W,3], on the device or on the host (3 tiles > max_batch 2)
    t3 = torch.from_numpy(np.stack([np.array(img)] * 3))
    infos = [info, _preview(-118.24, 34.05), info]
    ref3 = det.detect_batch([img, img, img], infos)
    assert det.detect_batch(t3.cuda(), infos) == ref3 and det.detect_batch(t3, infos) == ref3
    # network tolerance against the independent CPU oracle on the same preprocessed tensor
    ref_rows = OP.v8_rows_adapter(make_oracle("yolov8m", w, True).forward(torch.from_numpy(arr))[0].numpy())
    assert np.median(np.abs(rows[:, 4] - ref_rows[:, 4])) < 1e-3
    # _remove_duplicates == greedy oracle in UTM
    dd = det._remove_duplicates(out, 1.0)
    z, north = OP.utm_zone(out[0]["lon"], out[0]["lat"])
    ex, ny = OP.utm_forward([o["lon"] for o in out], [o["lat"] for o in out], z, north)
    keep = OP.dedup_greedy(ex, ny, np.array([o["confidence"] for o in out]), 1.0, True)
    assert dd == [out[i] for i in keep]
    det.engine.close()


def test_gpu_handler_process_batch_matches_reference_restatement():
    import cv2
    from PIL import Image
    from aerial_image_recognition_b200.gpu_handler import GPUHandler
    g = G.build("yolov7")
    w = W.make_synthetic_weights(g, 0)
    h = GPUHandler("car_aerial_detection_yolo7_ITCVD_deepness.onnx", confidence_threshold=0.3, weights=w, max_batch=4)
    rng = np.random.default_rng(5)
    imgs = [Image.fromarray(synth.make_tiles(1, 864, 40 + i)[0]) for i in range(3)] + [Image.fromarray(synth.make_tiles(1, 640, 50)[0])]
    bboxes = [(21.0 + 0.001 * i, 52.0, 21.0006 + 0.001 * i, 52.0004) for i in range(4)]
    batch = [[(im, bb, None)] for im, bb in zip(imgs, bboxes)]
    batch.insert(1, (imgs[0], bboxes[0]))        # WMS-style bare tuple: silently skipped (gpu_handler.py:157-158)
    out = h.process_batch(batch)
    ref = []
    for im, bb in zip(imgs, bboxes):
        a = np.array(im)
        if a.shape[0] != 640:
            a = cv2.resize(a, (640, 640))
        x = np.expand_dims((a.astype(np.float32) / 255.0).transpose(2, 0, 1), 0)
        assert np.array_equal(h.preprocess_image(im), x)
        rows = h.session.run(None, {h.session.get_inputs()[0].name: x})[0][0]
        f = rows[rows[:, 4] >= 0.3]
        for r in f[np.argsort(-f[:, 4], kind="stable")[:10]]:
            lon, lat = OP.georef_gpuhandler(r[0], r[1], *bb)
            ref.append({"lon": lon, "lat": lat, "confidence": float(r[4])})
    assert len(out) == len(ref) > 0
    assert out == ref
    # tensor input form (SURVEY 8b): uint8 [B,H,W,3] + float64 [B,4]
    same = [np.array(im) for im in imgs[:3]]
    assert h.process_tiles(torch.from_numpy(np.stack(same)).cuda(), bboxes[:3]) == h.process_batch([[(im, bb, None)] for im, bb in zip(imgs[:3], bboxes[:3])])
    h.cleanup()
    h.engine.close()


def test_detect_host_one_call_equals_the_staged_path(eng640):
    # b2d_detect_host (host buffers in and out, chunks of max_batch double-buffered) against preprocess / forward /
    # postprocess / georef called one by one on device tensors; 10 tiles through a max_batch-4 engine = 2.5 chunks
    from aerial_image_recognition_b200.engine import GEO_PARAMS, geodets_to_numpy
    tiles = synth.make_tiles(10, 640, 61)
    params = np.zeros((10, GEO_PARAMS))
    for k in range(10):
        params[k, :6] = (21.0 + 0.001 * k, 21.0006 + 0.001 * k, 52.0, 52.0004, 864, 640)
    for kw in (dict(conf_thr=0.3, inclusive=True), dict(conf_thr=0.25, inclusive=False, iou_thr=0.7, max_det=300)):
        got = eng640.detect_host(torch.from_numpy(tiles).pin_memory(), params, **kw)
        got2 = eng640.detect_host(tiles, params, **kw)            # pageable memory
        ref = []
        for c0 in range(0, 10, 4):
            d = torch.from_numpy(tiles[c0:c0 + 4]).cuda()
            dets, counts = eng640.infer(d, "identity", False, kw["conf_thr"], kw["inclusive"], kw.get("iou_thr", 0.0), 0, 300)
            geo = eng640.georef(dets, counts, torch.from_numpy(params[c0:c0 + 4]).cuda(), "bounds")
            ref += geodets_to_numpy(geo, counts)
        assert len(got) == len(ref) == 10 and sum(len(r) for r in ref) > 0
        for a, b, c in zip(got, got2, ref):
            assert a.tobytes() == c.tobytes() and b.tobytes() == c.tobytes()


# ---- size-independent properties at BASELINE batch size ----------------------------------------------------------------
def test_full_batch_determinism_and_batch_invariance():
    eng = _engine("yolov8m", max_batch=64)
    t = synth.make_tiles(8, 640, 21)
    big = torch.from_numpy(np.concatenate([t] * 8)).cuda()
    d1, c1 = eng.infer(big, "identity", conf_thr=0.25, inclusive=False, iou_thr=0.7)
    d2, c2 = eng.infer(big, "identity", conf_thr=0.25, inclusive=False, iou_thr=0.7)
    assert torch.equal(c1, c2) and torch.equal(d1.view(torch.int32)[..., :6], d2.view(torch.int32)[..., :6])    # run-to-run
    # a tile's result does not depend on its position in the batch or on the batch size
    assert torch.equal(c1[:8], c1[8:16]) and torch.equal(c1[:8], c1[56:64])
    for i in range(8):
        k = int(c1[i])
        assert torch.equal(d1[i, :k, :6], d1[56 + i, :k, :6])
    d3, c3 = eng.infer(big[:5].contiguous(), "identity", conf_thr=0.25, inclusive=False, iou_thr=0.7)
    assert torch.equal(c3, c1[:5])
    for i in range(5):
        assert torch.equal(d3[i, :int(c3[i]), :6], d1[i, :int(c3[i]), :6])
    eng.close()


def test_bench_dump_outputs_are_the_last_timed_step(tmp_path):
    # bench.py --dump-outputs DIR: the records its timed path (Engine.infer + Engine.georef) returned in the last of --steps
    # steps; the same inputs through a fresh engine in this process give them bit for bit, so dumps of two builds compare
    import json
    import subprocess
    import sys
    import bench
    from aerial_image_recognition_b200.engine import GEODET_DTYPE, geodets_to_numpy
    steps = 3
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1", "--legs", "",
                        "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps
    assert sorted(p.name for p in tmp_path.iterdir()) == sorted([f"{n}.npy" for n in GEODET_DTYPE.names] + ["counts.npy"])
    got = {p.stem: np.load(p) for p in tmp_path.iterdir()}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values()) and sum(a.nbytes for a in got.values()) <= 64 << 20
    assert got["counts"].sum() == line["config"]["detections_last_step"] > 0
    eng = _engine("yolov8m", max_batch=bench.BATCH, seed=0)
    tiles = bench.input_batches(0)[(steps - 1) % bench.NPOOL].cuda()
    dets, counts = eng.infer(tiles, "identity", False, bench.CONF, False, bench.IOU, 0, bench.MAX_DET)
    geo = eng.georef(dets, counts, torch.from_numpy(bench._geo_params(bench.BATCH)).cuda(), "bounds")
    ref = np.concatenate(geodets_to_numpy(geo, counts))
    eng.close()
    assert np.array_equal(got["counts"], counts.cpu().numpy())
    for name in GEODET_DTYPE.names:
        assert np.array_equal(got[name], ref[name]), name


# ---- SURVEY 8f-1: the model arrives as an .onnx path, as in the reference ---------------------------------------
def test_detector_built_from_onnx_file_equals_detector_built_from_tensors(tmp_path):
    """``SimpleDetector(model_path)`` / ``GPUHandler(model_path)`` with a real file at the path
    (``simple_detector.py:710``, ``_script/config.py:25``): weights read from the ONNX protobuf give
    bit-identical rows to the same tensors handed over directly."""
    from aerial_image_recognition_b200 import onnx_reader as R
    from aerial_image_recognition_b200.gpu_handler import GPUHandler
    from aerial_image_recognition_b200.simple_detector import SimpleDetector
    g = G.build("yolov8m")
    w = W.make_synthetic_weights(g, 3)
    path = str(tmp_path / "yolov8_tokyo_checkpoint.onnx")
    R.write_conv_onnx(path, g, w, named=False)                  # anonymous initializers: matched by graph order
    x = (synth.make_tiles(2, 640, 8).astype(np.float32) / 255.0).transpose(0, 3, 1, 2)
    a = SimpleDetector(path, None, max_batch=2)
    b = SimpleDetector("absent.onnx", None, weights=w, max_batch=2)
    with pytest.raises(FileNotFoundError):                     # a mistyped path fails like ort.InferenceSession does: no silent random weights
        SimpleDetector(str(tmp_path / "absent.onnx"), None, max_batch=2)
    with pytest.raises(FileNotFoundError):
        GPUHandler(str(tmp_path / "absent.onnx"), max_batch=2)
    ra = a.model.run(None, {"images": x})[0]
    rb = b.model.run(None, {"images": x})[0]
    assert ra.shape == (2, 8400, 6) and np.array_equal(ra, rb)
    h = GPUHandler(path, max_batch=2)
    assert np.array_equal(h.session.run(None, {"images": x})[0], rb)


@pytest.mark.parametrize("arch,imgsz", [("yolov8m", 320), ("yolov7", 256)])
def test_graph_replay_with_parallel_branches_equals_eager_forward(arch, imgsz):
    """forward() runs eagerly on its first call, is captured into a CUDA graph (independent ops on parallel capture
    streams, edges from the buffer read/write analysis) on the second and replayed afterwards: all three must leave
    bit-identical head maps -- a missing dependency edge would show up as a race here."""
    g = G.build(arch, imgsz=imgsz)
    w = W.make_synthetic_weights(g, 4)
    eng = _engine(arch, weights=w, max_batch=3, imgsz=imgsz, graph=g)
    tiles = torch.from_numpy(synth.make_tiles(3, imgsz, 21)).cuda()
    outs = []
    for _ in range(4):
        eng.preprocess(tiles, "identity")
        eng.forward(3)
        torch.cuda.synchronize()
        outs.append([eng.buffer(lv["buf"], 3).float().cpu().clone() for lv in g.head["levels"]])
    for k in range(1, 4):
        for a, b in zip(outs[0], outs[k]):
            assert torch.equal(a, b)
    eng.close()


# ---- SURVEY 8f-2 / 8f-3: the production loop and its files ---------------------------------------------------------
def test_results_manager_remove_duplicates_matches_reference_semantics(eng640, tmp_path):
    """``ResultsManager.remove_duplicates`` (``_script/utils.py:212-274``): zone from the mean longitude, strict ``<``,
    survivors in descending confidence with coordinates out of a UTM round trip."""
    from aerial_image_recognition_b200 import geo, utils as U
    rng = np.random.default_rng(3)
    base = np.array([21.0, 52.2])
    pts = base + rng.uniform(0, 0.002, (400, 2))
    pts = np.concatenate([pts, pts[:120] + rng.normal(0, 4e-6, (120, 2))])          # near-duplicates within ~0.5 m
    conf = rng.uniform(0.3, 0.95, len(pts)).astype(np.float32)
    dets = [{'lon': float(p[0]), 'lat': float(p[1]), 'confidence': float(c)} for p, c in zip(pts, conf)]
    rm = U.ResultsManager(str(tmp_path), duplicate_distance=2.0, engine=eng640)
    got = rm.remove_duplicates(dets)
    zone = geo.utm_zone_of(float(pts[:, 0].mean()))
    x, y = geo.utm_forward(pts[:, 0], pts[:, 1], zone, True)
    order = np.argsort(-conf, kind="stable")
    keep = OP.dedup_greedy(x[order], y[order], conf[order], 2.0, inclusive=False)
    ref_idx = order[keep]
    assert len(got) == len(ref_idx) < len(dets)
    assert [g['confidence'] for g in got] == [float(conf[i]) for i in ref_idx]
    for g, i in zip(got, ref_idx):
        assert abs(g['lon'] - pts[i, 0]) < 1e-9 and abs(g['lat'] - pts[i, 1]) < 1e-9     # round trip: ~1e-12 deg
    rm0 = U.ResultsManager(str(tmp_path), duplicate_distance=0, engine=eng640)                # the default: nothing removed
    assert len(rm0.remove_duplicates(dets)) == len(dets)


def test_car_detector_production_loop(tmp_path):
    """``CarDetector(base_dir, custom_config).detect()`` (``_script/detector.py:156-237``) against the same steps done
    by hand: tiles in generation order, batches of ``batch_size``, final duplicate removal, results GeoJSON; then a
    resume from a checkpoint."""
    import json
    from aerial_image_recognition_b200 import utils as U
    from aerial_image_recognition_b200.detector import CarDetector
    g = G.build("yolov7")
    w = W.make_synthetic_weights(g, 0)
    cfg = {'frame_path': 'testframe.shp', 'frame_bounds': (20.9990, 52.1990, 21.0022, 52.2008), 'batch_size': 8,
           'duplicate_distance': 1.5, 'engine_options': {'weights': w}}
    det = CarDetector(str(tmp_path), cfg)
    assert det.output_dir == os.path.join(str(tmp_path), 'output', 'testframe') and det.model_path.endswith(
        os.path.join('models', 'car_aerial_detection_yolo7_ITCVD_deepness.onnx'))
    out = det.detect(interactive=False, force_restart=True)
    tiles = U.TileGenerator.generate_tiles(cfg['frame_bounds'], 64.0, 0.2)
    assert det.stats['total_tiles'] == len(tiles) > 16
    manual = []
    for s in range(0, len(tiles), 8):
        manual.extend(det.gpu_handler.process_batch(det.tile_handler.fetch_batch(tiles[s:s + 8])))
    ref = det.results_manager.remove_duplicates(det.results_manager.remove_duplicates(manual))      # periodic + final pass, as the loop does
    assert len(manual) > 0 and out == ref
    fc = json.load(open(det.results_manager.output_file))
    assert os.path.basename(det.results_manager.output_file) == "detections_results.geojson"
    assert [(f["geometry"]["coordinates"], f["properties"]["confidence"]) for f in fc["features"]] == [([d['lon'], d['lat']], d['confidence']) for d in out]
    # resume: a checkpoint at tile 16 with the detections of the first 16 tiles continues to the same raw set
    first = []
    for s in range(0, 16, 8):
        first.extend(det.gpu_handler.process_batch(det.tile_handler.fetch_batch(tiles[s:s + 8])))
    det.checkpoint_manager.save_checkpoint(16, first, len(tiles))
    det2 = CarDetector(str(tmp_path), cfg)
    out2 = det2.detect(interactive=False, force_restart=False)
    assert det2.stats['start'] == 16 and len(out2) == len(out)
    assert [d['confidence'] for d in out2] == [d['confidence'] for d in out]
    # the loop's own checkpoints: the saved cursor is the END of the last batch whose detections are in the file, so a
    # resume neither re-runs that batch nor duplicates its detections (duplicate_distance 0: nothing would remove them)
    cfg0 = dict(cfg, duplicate_distance=0, output_prefix="nodup", checkpoint_interval=8)
    full = CarDetector(str(tmp_path), cfg0).detect(interactive=False, force_restart=True)

    class _Stop(Exception):
        pass
    det4 = CarDetector(str(tmp_path), cfg0)
    orig, calls = det4._process_batch, []

    def interrupted(batch_tiles, processed_count, total_tiles):
        if len(calls) == 2:                       # 20 tiles = three batches of 8: stop before the last one
            raise _Stop()
        calls.append(processed_count)
        return orig(batch_tiles, processed_count, total_tiles)
    det4._process_batch = interrupted
    with pytest.raises(_Stop):
        det4.detect(interactive=False, force_restart=True)
    assert det4.stats['checkpoints'] == 2 and json.load(open(det4.checkpoint_manager.state_file))['processed_count'] == 16
    det5 = CarDetector(str(tmp_path), cfg0)
    resumed = det5.detect(interactive=False, force_restart=False)
    assert det5.stats['start'] == 16
    assert sorted(d['confidence'] for d in resumed) == sorted(d['confidence'] for d in full)     # no batch counted twice


# ---- BASELINE size (C2: batch 64 at 640x640): size-independent properties ---------------------------------------------
def test_full_batch_is_permutation_equivariant_and_matches_small_batches():
    """At the benchmark's own size the oracle is too slow to be the checker, so the check is structural: tiles are
    independent, therefore (a) permuting the 64 tiles of a batch permutes the detections and changes nothing else --
    which exercises the M tiles that span several images (8 x 8 x 2 at 40^2, 4 x 4 x 8 at 20^2), the CTA pairs and
    the multi-tile rounds the planner only picks at this size -- and (b) a tile gives bit-identical detections in a
    batch of 64 and in a batch of 4 (different tile shapes, kernels and grid sizes)."""
    from aerial_image_recognition_b200.engine import dets_to_numpy
    g = G.build("yolov8m")
    w = W.make_synthetic_weights(g, 0)
    big = _engine("yolov8m", weights=w, max_batch=64, graph=g)
    base = synth.make_tiles(16, 640, 77)
    idx = (np.arange(64) * 5 + 3) % 16
    tiles = base[idx]
    perm = np.random.default_rng(1).permutation(64)
    a = dets_to_numpy(*big.infer(torch.from_numpy(tiles).cuda(), "identity", conf_thr=0.25, inclusive=False, iou_thr=0.7, max_det=300))
    b = dets_to_numpy(*big.infer(torch.from_numpy(tiles[perm]).cuda(), "identity", conf_thr=0.25, inclusive=False, iou_thr=0.7, max_det=300))
    fields = ("cx", "cy", "w", "h", "conf", "cls", "anchor")
    for k in range(64):
        assert len(a[perm[k]]) == len(b[k]) > 0
        for f in fields:
            assert np.array_equal(a[perm[k]][f], b[k][f]), (k, f)
    # equal tiles inside one batch give equal detections
    for k in range(16, 64):
        j = int(np.nonzero(idx[:16] == idx[k])[0][0])
        assert np.array_equal(a[k]["conf"], a[j]["conf"]) and np.array_equal(a[k]["cx"], a[j]["cx"])
    big.close()
    small = _engine("yolov8m", weights=w, max_batch=4, graph=g)
    c = dets_to_numpy(*small.infer(torch.from_numpy(tiles[:4]).cuda(), "identity", conf_thr=0.25, inclusive=False, iou_thr=0.7, max_det=300))
    for k in range(4):
        for f in fields:
            assert np.array_equal(a[k][f], c[k][f]), (k, f)
    small.close()


# ---- B2D_PREC_FP16: activations and weights stored as fp16 ------------------------------------------------------------
@pytest.mark.parametrize("arch,imgsz,n", [("yolov8m", 320, 2), ("yolov7", 128, 2)])
def test_every_planned_op_matches_torch_fp16(arch, imgsz, n):
    _check_every_op(arch, imgsz, n, precision="fp16")
