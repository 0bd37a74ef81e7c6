"""ctypes binding of ``libb2det.so`` (the C ABI in ``include/b2det.h``).

This is the stub a maintainer of the reference would add (INTEGRATION.md).  The
library is the product: there is no Python or CPU fallback, and loading fails
loudly when the shared object has not been built (``python __graft_entry__.py``
or ``make -C aerial_image_recognition_b200/csrc``).
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_HERE = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ.get("B2D_LIB", _HERE / "libb2det.so"))   # B2D_LIB: A/B-test another build of the same library

c_int, c_float, c_double, c_void_p, c_char_p, c_size_t, c_ll = (
    C.c_int, C.c_float, C.c_double, C.c_void_p, C.c_char_p, C.c_size_t, C.c_longlong)
P = C.POINTER

# name -> (restype, argtypes); must list every symbol include/b2det.h declares
SIGNATURES = {
    "b2d_create": (c_int, [c_int, c_int, P(c_void_p)]),
    "b2d_destroy": (None, [c_void_p]),
    "b2d_last_error": (c_char_p, []),
    "b2d_version": (c_int, []),
    "b2d_device_sm_count": (c_int, [c_void_p]),
    "b2d_set_precision": (c_int, [c_void_p, c_int]),
    "b2d_get_precision": (c_int, [c_void_p]),
    "b2d_plan_buffer": (c_int, [c_void_p, c_int, c_int, c_int, c_int]),
    "b2d_plan_conv": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                              c_void_p, c_void_p, c_int, c_int, c_int]),
    "b2d_plan_dwconv": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "b2d_plan_maxpool": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int]),
    "b2d_plan_upsample2x": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int]),
    "b2d_plan_head_level": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "b2d_plan_finalize": (c_int, [c_void_p]),
    "b2d_buffer_ptr": (c_void_p, [c_void_p, c_int]),
    "b2d_buffer_bytes": (c_size_t, [c_void_p, c_int]),
    "b2d_num_anchors": (c_int, [c_void_p]),
    "b2d_num_kernels_per_forward": (c_int, [c_void_p]),
    "b2d_preprocess": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_ll, c_int, c_int, c_int, c_void_p, c_void_p]),
    "b2d_set_input_f32": (c_int, [c_void_p, c_void_p, c_int, c_void_p]),
    "b2d_forward": (c_int, [c_void_p, c_int, c_void_p]),
    "b2d_decode_rows": (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    "b2d_postprocess": (c_int, [c_void_p, c_int, c_float, c_int, c_float, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p]),
    "b2d_postprocess_rows": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_int, c_float, c_int, c_int,
                                     c_void_p, c_void_p, c_int, c_void_p]),
    "b2d_infer_tiles": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_ll, c_int, c_int, c_float, c_int, c_float, c_int, c_int,
                                c_void_p, c_void_p, c_int, c_void_p]),
    "b2d_detect_host": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float, c_int, c_float, c_int, c_int, c_int,
                                c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "b2d_georef": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "b2d_decode_rows_obb": (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    "b2d_postprocess_obb": (c_int, [c_void_p, c_int, c_float, c_int, c_float, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p]),
    "b2d_georef_obb": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "b2d_mosaic_nms_obb": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_float, c_float, c_void_p, c_void_p]),
    "b2d_dedup": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_double, c_int, c_void_p, c_void_p]),
    "b2d_seam_closure": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_double, c_int, c_void_p, c_void_p]),
    "b2d_utm_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "b2d_cut_windows": (c_int, [c_void_p, c_void_p, c_int, c_int, c_ll, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "b2d_resize_windows": (c_int, [c_void_p, c_void_p, c_int, c_int, c_ll, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p,
                                   c_void_p]),
    "b2d_resize_table": (c_int, [c_int, c_int, c_int, c_void_p, c_void_p, P(c_int)]),
    "b2d_tta_clahe": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_double, c_int, c_int, c_void_p, c_void_p]),
    "b2d_tta_lut": (c_int, [c_void_p, c_void_p, c_int, c_ll, c_void_p, c_int, c_void_p, c_void_p]),
    "b2d_tta_contrast": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_void_p, c_void_p]),
    "b2d_colour_convert": (c_int, [c_void_p, c_void_p, c_ll, c_int, c_void_p, c_void_p]),
    "b2d_set_conf_scale": (c_int, [c_void_p, c_float]),
    "b2d_segment": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "b2d_run_op": (c_int, [c_void_p, c_int, c_int, c_void_p]),
    "b2d_fused_with_next": (c_int, [c_void_p, c_int]),
    "b2d_run_op_fused": (c_int, [c_void_p, c_int, c_int, c_void_p]),
    "b2d_num_ops": (c_int, [c_void_p]),
    "b2d_describe_op": (c_int, [c_void_p, c_int, c_char_p, c_int]),
}

_lib = None


class B2DError(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load the shared library once; raise if it is missing (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    path = str(LIB_PATH)
    if not os.path.exists(path):
        raise B2DError(
            f"{path} not found: build it with `python __graft_entry__.py` (or `make -C "
            f"aerial_image_recognition_b200/csrc`). There is no CPU or PyTorch fallback for this path.")
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str = "", index: bool = False) -> int:
    """Every entry point returns 0 or a negative status; the ``b2d_plan_*`` calls return the index of what they added
    (``index=True``).  Anything else is an error."""
    if rc < 0 or (rc != 0 and not index):
        msg = load().b2d_last_error().decode("utf-8", "replace")
        raise B2DError(f"{what}: {msg}" if what else msg)
    return rc
