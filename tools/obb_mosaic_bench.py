"""Oriented-box detection over a synthetic 40k x 40k orthomosaic on one GPU (mosaic.ObbMosaicDetector): prints one JSON line.

    python tools/obb_mosaic_bench.py [--size 40000] [--repeat 2]

Two window grids over the same device-resident mosaic (synth.mosaic_band_device): 640 / 512 (the model input, windows cut), and
Ultralytics' DOTA split, 1024 / 824 (1024 crops, 200 px gap), resampled into the 640 input.  Per grid: windows/s and ms per mosaic
(CUDA events around whole runs: windows -> network -> per-window ProbIoU NMS -> georef -> the mosaic-wide merge -> one read-back),
the merge kernel alone (CUDA events over repeated b2d_mosaic_nms_obb calls on that run's records), and the record counts before
and after the merge.  The GPU name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

GT = (2335637.62, 0.1, 0.0, 6845688.78, 0.0, -0.1)     # 10 cm/px, as tools/mosaic_bench.py


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=40000)
    ap.add_argument("--repeat", type=int, default=2)
    ap.add_argument("--batch", type=int, default=64)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("obb_mosaic_bench.py: no GPU visible; the engine has no CPU fallback")
    from aerial_image_recognition_b200 import mosaic as M, synth
    from aerial_image_recognition_b200.engine import Engine
    from obb_bench import gpu_info

    H = W = args.size
    eng = Engine("yolov8m-obb", max_batch=args.batch, seed=0)
    pool = torch.from_numpy(synth.mosaic_block_pool(77)).to(eng.device)
    band = synth.mosaic_band_device(pool, H, W, 0, H, 5)
    out = {"metric": "yolov8m-obb (nc 15, seeded synthetic weights) over a synthetic orthomosaic: windows -> network -> per-window "
                     "ProbIoU NMS (conf 0.25, IoU 0.7, 300) -> georef -> mosaic-wide ProbIoU fast NMS (conf > 0.4, IoU 0.3)",
           "gpu": gpu_info(0), "size": [H, W], "grids": {}}
    for win, stride in ((640, 512), (1024, 824)):
        det = M.ObbMosaicDetector(eng, GT, win=win, stride=stride)
        res = det.run(band, H, W)                                  # warm-up
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.repeat):
            res = det.run(band, H, W)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / args.repeat
        nwin = len(M.window_grid(H, W, win, stride))
        geo, dets, counts, params = M.run_windows(eng, band, M.window_grid(H, W, win, stride), 0, GT, win, 114, det.nms_conf, det.iou,
                                                  det.max_det)
        eng.mosaic_nms_obb(dets, counts, params, det.conf, det.merge_iou)
        # eligible records outside the merge's bound (short side < 1 px or long / short > 128 in the mosaic frame): each of
        # them is tested against every eligible record
        n, cap = dets.shape[0], dets.shape[1]
        gain = params[:, 10].float()[:, None]
        w, h = dets[..., 2] / gain, dets[..., 3] / gain
        elig = (torch.arange(cap, device=eng.device)[None, :] < counts[:, None]) & (dets[..., 5] > det.conf)
        lo, hi = torch.minimum(w, h), torch.maximum(w, h)
        thin = elig & ~((lo >= 1) & (hi <= 128 * lo))
        reps = 10
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            eng.mosaic_nms_obb(dets, counts, params, det.conf, det.merge_iou)
        e1.record()
        torch.cuda.synchronize()
        merge_ms = e0.elapsed_time(e1) / reps
        out["grids"][f"{win}/{stride}"] = {
            "windows": nwin, "resampled": win != eng.imgsz, "ms_per_mosaic": ms, "windows_per_s": nwin / (ms * 1e-3),
            "merge_kernel_ms": merge_ms, "merge_share": merge_ms / ms, "records_slots": int(dets.shape[0] * dets.shape[1]),
            "records_raw": det.last_raw, "records_after_merge": len(res),
            "records_per_window_nms": int(counts.sum().item()), "records_thin_or_tiny": int(thin.sum().item()),
            "long_side_px_max": float(hi[elig].max().item()) if bool(elig.any()) else 0.0,
            "long_side_px_p99": float(torch.quantile(hi[elig][:1 << 24].float(), 0.99).item()) if bool(elig.any()) else 0.0}
        del geo, dets, counts, params
        torch.cuda.empty_cache()
    out["repeat"] = args.repeat
    out["timing"] = "CUDA events; mosaic resident in HBM; merge kernel timed separately over 10 calls"
    print(json.dumps(out))
    eng.close()


if __name__ == "__main__":
    main()
