"""BASELINE config C4: sliding-window detection over a synthetic H x W orthomosaic (default 40k x 40k,
window 640, stride 512 = 20 % overlap -> 79 x 79 = 6241 windows), window rows sharded across the
ranks, cross-shard seam dedup through the NCCL all-gather of mosaic.MosaicDetector.

    python tools/mosaic_bench.py [--size 40000] [--repeat 2] [--win 640 --stride 512]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P tools/mosaic_bench.py

Every rank materialises only its own band of the mosaic, on the device, from a small pool of
procedural 512-px blocks chosen by a hash of the *global* block coordinates (so the content does
not depend on the sharding); no host traffic on the data path.  Timing: CUDA events around the whole
run (cut windows -> preprocess -> network -> NMS -> georef -> local dedup -> seam exchange -> merge),
max over ranks.  Rank 0 prints one JSON line with windows/s, the number of detections before and after
dedup, the seam records exchanged and an order-independent checksum of the result, which must be
identical for every world size.  ``--win`` / ``--stride`` run another window grid: windows other than
the model input are resampled from the mosaic into the network input (``b2d_resize_windows``), e.g. the reference
notebook's 1200 / 600.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

GT = (2335637.62, 0.1, 0.0, 6845688.78, 0.0, -0.1)     # SURVEY 8d: 10 cm/px, EPSG:3857-style metres


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=40000)
    ap.add_argument("--repeat", type=int, default=2)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--win", type=int, default=640)
    ap.add_argument("--stride", type=int, default=512)
    ap.add_argument("--dump", default="")
    ap.add_argument("--dump-raw", default="", help="debug: save every rank's raw (pre-dedup) detections to <prefix>.rank<r>.npz")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))

    import torch
    import torch.distributed as dist
    from aerial_image_recognition_b200 import mosaic as M, synth
    from aerial_image_recognition_b200.engine import Engine

    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    H = W = args.size
    eng = Engine("yolov8m", max_batch=args.batch, device=local, seed=0)
    pool = torch.from_numpy(synth.mosaic_block_pool(77)).to(eng.device)
    windows, ids, cover = M.shard_windows(H, W, rank, world, args.win, args.stride)
    band = synth.mosaic_band_device(pool, H, W, cover[0], cover[1], 5)
    det = M.MosaicDetector(eng, GT, win=args.win, stride=args.stride, conf=0.4, dedup_thr=1.0)
    det.profile = bool(os.environ.get("B2D_MOSAIC_PROFILE"))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    out = det.run(band, H, W, rank, world, y_offset=cover[0])        # warm-up (also NCCL channel setup)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.repeat):
        out = det.run(band, H, W, rank, world, y_offset=cover[0])
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1) / args.repeat
    # order-independent checksum of this rank's survivors: count, sum of window*65536+slot keys, sums of the coordinates
    key = out["window"].astype(np.int64) * 65536 + out["slot"].astype(np.int64)
    stats = torch.tensor([ms, float(len(out)), float(det.last_raw), float(getattr(det, "last_seam_records", 0) if rank == 0 else 0),
                          float(np.sum(key % 1000003)), float(np.sum(out["x"] - GT[0])), float(np.sum(GT[3] - out["y"]))],
                         dtype=torch.float64, device=eng.device)
    mx = stats.clone()
    if world > 1:
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(stats, op=dist.ReduceOp.SUM)
    if det.profile:
        print(f"rank {rank} dedup phases (ms, summed over {args.repeat + 1} runs): " + ", ".join(f"{k} {v:.1f}" for k, v in det.timings.items()), file=sys.stderr)
    if args.dump_raw:
        x, y, conf, cls, wid, slot, py = det.detect_windows(band, windows, ids, cover[0])
        np.savez(f"{args.dump_raw}.rank{rank}.npz", x=x.cpu().numpy(), y=y.cpu().numpy(), conf=conf.cpu().numpy(), wid=wid.cpu().numpy(),
                 slot=slot.cpu().numpy(), py=py.cpu().numpy())
    if args.dump:
        np.save(f"{args.dump}.rank{rank}.npy", out)
    if rank == 0:
        nwin = len(M.window_grid(H, W, args.win, args.stride))
        print(json.dumps({"workload": f"C4: synthetic {H}x{W} mosaic, window {args.win} stride {args.stride}, {nwin} windows, YOLOv8m (seeded synthetic weights), "
                                      f"conf>0.4, 1 m dedup, row bands over {world} rank(s)",
                          "n_gpus": world, "windows": nwin, "ms_per_mosaic": float(mx[0]), "windows_per_s": nwin / (float(mx[0]) * 1e-3),
                          "detections_raw": int(stats[2]), "detections_after_dedup": int(stats[1]), "seam_records_exchanged": int(stats[3]),
                          "checksum": {"keys_mod": int(stats[4]), "sum_dx_m": float(stats[5]), "sum_dy_m": float(stats[6])},
                          "band_rows_rank0": [int(cover[0]), int(cover[1])], "timing": "CUDA events, max over ranks, mosaic resident in HBM"}))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
