#!/usr/bin/env python
"""Whole 8K step (480 x 270 macroblocks, COVA_FLAG_CCL_CLUSTER): device-resident windows/s of tensorise -> BlobNet ->
cluster CCL, then per-kernel device time from the library's profiling events (a separate pass: events between kernels
serialise programmatic dependent launches).  Prints one JSON object with the card name and power limit beside the numbers.
STREAMS / FPS / HEAD_BIAS override the shape (default 4 chains x 67 frames = 256 windows)."""
import json, os, subprocess, sys, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cova_b200 import synth, weights
from cova_b200.elements import BlobPipeline


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim, clk = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": plim, "sm_max_clock": clk}
    except Exception as e:  # noqa: BLE001
        return {"gpu": None, "power_limit": None, "error": repr(e)}


h, w = 270, 480
n_streams, fps = int(os.environ.get("STREAMS", 4)), int(os.environ.get("FPS", 67))
hb = float(os.environ.get("HEAD_BIAS", -1.0))
p = BlobPipeline(w, h, weights.to_blob(weights.random_weights(0, head_bias=hb)), n_streams, fps, n_chunks=1, ccl_cluster=True)
p.load_frames(synth.tiled_streams(n_streams, fps, h, w, 1))
n = p.n_windows
for _ in range(3):
    p.run()
p.sync()
steps = 10
t0 = time.perf_counter()
for _ in range(steps):
    p.run()
p.sync()
ms_step = (time.perf_counter() - t0) * 1e3 / steps
p.set_profiling(True)
acc = {}
for _ in range(5):
    p.run(); p.sync()
    for k, v in p.last_timings().items():
        acc.setdefault(k, []).append(v)
p.set_profiling(False)
boxes = p.fetch_boxes_raw()[2]
res = dict(card(), grid=f"{w}x{h} macroblocks", windows=n, head_bias=hb, ms_step=round(ms_step, 4),
           windows_per_s=round(n / ms_step * 1e3, 1), mask_fg=round(float(p.read_mask().mean()), 4),
           boxes_per_window=round(float(((boxes.astype(np.int64) - 8) // 24).mean()), 2),
           kernel_ms={k: round(float(np.median(v[1:])), 4) for k, v in acc.items()})
print(json.dumps(res))
