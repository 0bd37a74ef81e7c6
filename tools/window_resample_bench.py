"""Kernel time of ``b2d_resize_windows`` (``resize_windows_kernel``) per batch of windows, against its HBM floor.

    python tools/window_resample_bench.py [--win 1200] [--stride 600] [--batch 64] [--iters 50]

The mosaic (default 12 000 x 12 000, 432 MB) is larger than the 126 MB L2, and consecutive timed launches walk different
batches of its windows, so the source bytes come from HBM.  The floor per window is ``w0 * h0 * 3`` bytes read plus
``imgsz^2 * 8`` bytes of 16-bit NHWC4 network input written; the time is CUDA events around ``--iters`` launches into the
engine's input buffer.  Prints one JSON line with the card's name and power limit.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:        # the measurement stands without the label; say so
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--win", type=int, default=1200)
    ap.add_argument("--stride", type=int, default=600)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--size", type=int, default=12000)
    ap.add_argument("--iters", type=int, default=50)
    args = ap.parse_args()

    import torch
    from aerial_image_recognition_b200 import mosaic as M, synth
    from aerial_image_recognition_b200.engine import Engine

    eng = Engine("yolov8m", max_batch=args.batch, seed=0)
    pool = torch.from_numpy(synth.mosaic_block_pool(77)).to(eng.device)
    H = W = args.size
    mosaic = synth.mosaic_band_device(pool, H, W, 0, H, 5)
    wins = M.window_grid(H, W, args.win, args.stride)
    full = wins[(wins[:, 2] == args.win) & (wins[:, 3] == args.win)]          # whole windows: the floor is the same for each batch
    nb = len(full) // args.batch
    assert nb >= 2, "mosaic too small for two batches of whole windows"
    M.check_windows(full, args.win, H, W)
    org = torch.from_numpy(full[:nb * args.batch]).to(eng.device).view(nb, args.batch, 4)
    for b in range(min(nb, 3)):                                                 # warm-up
        eng.resize_windows(mosaic, org[b], args.win, checked=True)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.iters):
        eng.resize_windows(mosaic, org[i % nb], args.win, checked=True)
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / args.iters
    S = eng.imgsz
    floor_bytes = args.batch * (args.win * args.win * 3 + S * S * 8)
    floor_us = floor_bytes / 7.7e12 * 1e6
    print(json.dumps({"kernel": "resize_windows_kernel", "card": card(), "win": args.win, "imgsz": S, "batch": args.batch,
                      "us_per_batch": round(us, 2), "hbm_floor_bytes": floor_bytes, "floor_us_at_7.7TBps": round(floor_us, 2),
                      "achieved_TBps": round(floor_bytes / (us * 1e-6) / 1e12, 3), "share_of_floor": round(floor_us / us, 3),
                      "timing": f"CUDA events over {args.iters} launches, {nb} distinct batches of a {H}x{W} mosaic"}))


if __name__ == "__main__":
    main()
