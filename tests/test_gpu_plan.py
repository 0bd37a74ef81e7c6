"""GPU tests (-m gpu) of what the convolution planner refuses: a layer no tcgen05 kernel can run fails b2d_plan_finalize
with an error, it never runs on another path."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from aerial_image_recognition_b200 import _lib, graph as G


def test_stem_shape_without_a_kernel_fails_plan_finalize():
    """The 4-channel network input is read only by the two TMA-fed stems (3x3, stride 2 or stride 1); a 1x1 conv on it has
    no kernel."""
    from aerial_image_recognition_b200.engine import Engine
    g = G.Graph("stem1x1", nc=1, imgsz=64)
    g.buf("input", 64, 64, 4)
    g.buf("out", 64, 64, 16)
    g.conv("stem", G.Ref("input", 0, 4), G.Ref("out", 0, 16), k=1, s=1)
    g.head = {"kind": "seg", "levels": []}
    rng = np.random.default_rng(0)
    w = {"stem.weight": rng.standard_normal((16, 3, 1, 1), dtype=np.float32), "stem.bias": np.zeros(16, np.float32)}
    with pytest.raises(_lib.B2DError, match="has no tcgen05 kernel"):
        Engine("stem1x1", weights=w, max_batch=2, graph=g)
