"""GPU tests (-m gpu): after the device refuses one of the engine's scratch allocations, the engine's next ordinary call returns
the same bytes as before the refusal.  Each refused request asks for about 2 TB of device memory, several times what a B200
has, so it fails whatever else is resident, and it fails before any kernel reads the caller's pointers: the refusing calls go
through ctypes with small buffers, because the Engine methods would allocate tensors of the refused size."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from aerial_image_recognition_b200 import _lib, graph as G, synth, weights as W

TB = 1 << 40
NMS = dict(conf_thr=0.25, inclusive=False, iou_thr=0.7, max_det=300)


@pytest.fixture(scope="module")
def eng():
    from aerial_image_recognition_b200.engine import Engine
    g = G.build("yolov8m", imgsz=640)
    e = Engine("yolov8m", weights=W.make_synthetic_weights(g, 0), max_batch=64, graph=g)
    yield e
    e.close()


def _refused(rc):
    assert rc == -2
    msg = _lib.load().b2d_last_error().decode()
    assert "cudaMalloc" in msg and "bytes" in msg, msg


def test_candidate_scratch_refusal(eng):
    from aerial_image_recognition_b200.engine import DET_DTYPE, dets_to_numpy
    tiles = torch.from_numpy(synth.make_tiles(4, 640, 3)).cuda()

    def ordinary():
        dets, counts = eng.infer(tiles, "identity", **NMS)                          # b2d_postprocess on the head maps
        rows = eng.decode_rows(4)
        rdets, rcounts = eng.postprocess(4, rows=rows, **NMS)                       # b2d_postprocess_rows
        return [r.tobytes() for r in dets_to_numpy(dets, counts) + dets_to_numpy(rdets, rcounts)]

    before = ordinary()
    assert sum(len(b) for b in before) > 0
    tiles_n, rows_n = 1 << 20, 65536                                               # candidates: tiles_n * rows_n * 32 B = 2 TB
    assert tiles_n * rows_n * DET_DTYPE.itemsize >= TB
    small = torch.zeros(64, dtype=torch.float32, device=eng.device)
    counts = torch.zeros(64, dtype=torch.int32, device=eng.device)
    _refused(eng.lib.b2d_postprocess_rows(eng.h, C.c_void_p(small.data_ptr()), tiles_n, rows_n, 6, 0.25, 0, 0.7, 0, 300,
                                          C.c_void_p(small.data_ptr()), C.c_void_p(counts.data_ptr()), 1, eng.stream))
    assert ordinary() == before
    torch.cuda.synchronize()


def test_host_slot_refusal(eng):
    from aerial_image_recognition_b200.engine import DET_DTYPE, GEO_PARAMS
    n = 6
    tiles = synth.make_tiles(n, 640, 5)
    params = np.zeros((n, GEO_PARAMS))
    for k in range(n):
        params[k, :6] = (21.0 + 0.001 * k, 21.0006 + 0.001 * k, 52.0, 52.0004, 864, 640)

    def ordinary():
        return [r.tobytes() for r in eng.detect_host(tiles, params, **NMS)]

    before = ordinary()
    assert sum(len(b) for b in before) > 0
    cap = 1 << 30                                                                  # each slot's records: max_batch * cap * 32 B = 2 TB
    assert eng.max_batch * cap * DET_DTYPE.itemsize >= TB
    tile = np.zeros((1, 640, 640, 3), np.uint8)
    p = np.zeros((1, GEO_PARAMS))
    out = np.zeros(64, np.uint8)
    counts = np.zeros(1, np.int32)
    _refused(eng.lib.b2d_detect_host(eng.h, C.c_void_p(tile.ctypes.data), 1, 640, 640, 0, 0, 0.25, 0, 0.7, 0, 300, 0,
                                     C.c_void_p(p.ctypes.data), C.c_void_p(out.ctypes.data), C.c_void_p(counts.ctypes.data), cap,
                                     eng.stream))
    assert ordinary() == before
