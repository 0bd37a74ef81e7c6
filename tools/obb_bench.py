"""Throughput of the oriented-box model (yolov8m-obb, nc = 15) on one GPU: prints one JSON line.

    python tools/obb_bench.py [--steps K] [--warmup W]

For 640 x 640 at batch 64 and 1024 x 1024 at batch 32 (the published OBB models run at 1024): the settled and the burst
tiles/s of the device-resident step (Engine.infer: preprocess, network, rotated decode, sort, ProbIoU NMS; then georef_obb),
with bench.py's warm-up rule and seeded tiles built like bench.input_batches (four distinct batches, more than the 126 MB L2);
the conv family's TFLOP/s against the sustained peak (bench.conv_roofline); and the post-processing split into decode + compact,
sort and rotated NMS (torch.profiler kernel times), with candidates and kept boxes per tile.  The axis-aligned C2 step
(yolov8m, 640, batch 64) runs in the same process, alternating with each OBB measurement, for context.  The GPU name and power
limit are read in the same call.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402

CONF, IOU, MAX_DET = bench.CONF, bench.IOU, bench.MAX_DET
NPOOL = bench.NPOOL


def gpu_info(dev: int):
    import torch
    out = {"name": torch.cuda.get_device_name(dev)}
    try:
        r = subprocess.run(["nvidia-smi", f"--id={dev}", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30)
        pl, mx = (v.strip() for v in r.stdout.strip().split(","))
        out.update(power_limit_w=float(pl), max_sm_clock_mhz=float(mx))
    except Exception as ex:
        out["power_limit_w"] = f"unread ({str(ex)[:80]})"
    return out


def input_batches(size: int, batch: int):
    """bench.input_batches at another tile size / batch: NPOOL seeded batches drawn from 16 tiles, every other one mirrored."""
    import torch
    from aerial_image_recognition_b200 import synth
    base = synth.make_tiles(16, size, seed=1000)
    out = []
    for b in range(NPOOL):
        idx = (np.arange(batch) * 7 + b * 3) % 16
        h = torch.from_numpy(base[idx]).clone()
        if b % 2:
            h = torch.flip(h, dims=[2]).contiguous()
        out.append(h)
    return out


class Leg:
    def __init__(self, arch, size, batch, nc=None):
        import torch
        from aerial_image_recognition_b200.engine import Engine
        self.arch, self.size, self.batch = arch, size, batch
        self.eng = Engine(arch, max_batch=batch, imgsz=size, nc=nc, seed=0)
        self.pool = [h.to(self.eng.device) for h in input_batches(size, batch)]
        p = np.zeros((batch, 16))
        p[:, :6] = (21.0, 21.00094, 52.2, 52.200575, 864.0, float(size))
        self.params = torch.from_numpy(p).to(self.eng.device)

    def step(self, i):
        e = self.eng
        dets, counts = e.infer(self.pool[i % NPOOL], "identity", False, CONF, False, IOU, 0, MAX_DET)
        return e.georef(dets, counts, self.params, "bounds"), counts

    def settle(self, warmup):
        """bench.py's rule: at least `warmup` steps and windows of 8 steps until three consecutive windows agree within 2 %
        (1 s .. 6 s); returns the first window's ms per step (boost clocks after idle: `burst`)."""
        import torch
        for i in range(2):
            self.step(i)
        torch.cuda.synchronize()
        t, i, prev, stable, burst = time.perf_counter(), 0, None, 0, None
        while True:
            w0, w1 = bench._events()
            w0.record()
            for _ in range(8):
                self.step(i)
                i += 1
            w1.record()
            torch.cuda.synchronize()
            cur = w0.elapsed_time(w1)
            burst = cur / 8 if burst is None else burst
            stable = stable + 1 if prev is not None and abs(cur - prev) <= 0.02 * cur else 0
            prev = cur
            el = time.perf_counter() - t
            if i >= warmup and ((stable >= 3 and el >= 1.0) or el >= 6.0):
                return burst

    def timed(self, steps):
        """Median of three runs of exactly `steps` steps, ms per step."""
        import torch
        runs = []
        for _ in range(3):
            torch.cuda.synchronize()
            e0, e1 = bench._events()
            e0.record()
            for i in range(steps):
                self.step(i)
            e1.record()
            torch.cuda.synchronize()
            runs.append(e0.elapsed_time(e1) / steps)
        return sorted(runs)[1], runs

    def postprocess_split(self, reps=10):
        import torch
        from torch.profiler import ProfilerActivity, profile
        e, n = self.eng, self.batch
        e.preprocess(self.pool[0], "identity")
        e.forward(n)
        rows = e.decode_rows(n)
        cand = float((rows[..., 4] > CONF).sum().item()) / n
        dets, counts = e.postprocess(n, CONF, False, IOU, 0, MAX_DET)
        kept = float(counts.sum().item()) / n
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(reps):
                e.postprocess(n, CONF, False, IOU, 0, MAX_DET)
            torch.cuda.synchronize()
        us = {"decode_compact": 0.0, "sort": 0.0, "rotated_nms": 0.0}
        for ev in prof.key_averages():
            k = ev.key
            t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
            if "obb_head_kernel" in k:
                us["decode_compact"] += t / reps
            elif "sort_keys_kernel" in k:
                us["sort"] += t / reps
            elif "obb_select_kernel" in k:
                us["rotated_nms"] += t / reps
        return {"us_per_batch": us, "batch": n, "candidates_per_tile": cand, "kept_per_tile": kept}

    def close(self):
        self.eng.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=10)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("obb_bench.py: no GPU visible; the engine has no CPU fallback")
    peak_tf, _burst_peak, _hbm, which = bench._peaks()
    out = {"metric": "yolov8m-obb tiles/s (device-resident: preprocess + network + rotated decode + ProbIoU NMS + georef_obb)",
           "gpu": gpu_info(0), "peak_tflops_sustained": peak_tf, "peak_source": which, "legs": {}}
    c2 = Leg("yolov8m", 640, 64)
    c2_runs = []
    for size, batch in ((640, 64), (1024, 32)):
        leg = Leg("yolov8m-obb", size, batch)
        burst = leg.settle(args.warmup)
        ms, runs = leg.timed(args.steps)
        c2.settle(args.warmup)                        # alternate: the axis-aligned C2 step right after, same settled state
        c2_ms, _ = c2.timed(args.steps)
        c2_runs.append(c2_ms)
        roof = bench.conv_roofline(leg.eng, leg.pool, batch)
        tf = roof["flops"] / (roof["tc_ms"] * 1e-3) / 1e12
        out["legs"][f"{size}x{size}_b{batch}"] = {
            "value": batch / (ms * 1e-3), "unit": "tiles/s", "ms_per_step": ms, "ms_per_step_runs": runs,
            "burst": {"value": batch / (burst * 1e-3), "ms_per_step": burst},
            "conv": {"tflops": tf, "frac_of_sustained_peak": tf / peak_tf, "tc_ms": roof["tc_ms"], "fwd_ms": roof["fwd_ms"],
                     "gflop_per_tile": roof["flops"] / batch / 1e9, "launches": roof["launches"]},
            "postprocess": leg.postprocess_split(),
            "c2_v8m_alternating": {"value": 64 / (c2_ms * 1e-3), "ms_per_step": c2_ms}}
        leg.close()
        del leg
        torch.cuda.empty_cache()
    c2.close()
    out["steps"], out["warmup"] = args.steps, args.warmup
    print(json.dumps(out))


if __name__ == "__main__":
    main()
