#!/usr/bin/env python
"""Per-layer timing experiments (development aid): normal / MMA-only / epilogue-only."""
import os, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cova_b200 import _lib, synth, weights
from cova_b200.elements import BlobPipeline

n_streams, fps = int(os.environ.get("STREAMS", 128)), 67
h, w = int(os.environ.get("H", 45)), int(os.environ.get("W", 80))
p = BlobPipeline(w, h, weights.to_blob(weights.random_weights(0, head_bias=-1.0)), n_streams, fps, n_chunks=1)
p.load_frames(synth.tiled_streams(n_streams, fps, h, w, 1))
p.set_profiling(True)
res = {}
import time
VARIANTS = (("normal", 0), ("no_epilogue", 2), ("no_mma", 1), ("neither", 3), ("old_enc", 4), ("no_pdl", 32),
            ("dec_whole", 64))
if os.environ.get("VARIANTS"):          # e.g. VARIANTS="ws3:8,ws3_no_epi:10,ws3_no_mma:9"
    VARIANTS = tuple((v.split(":")[0], int(v.split(":")[1])) for v in os.environ["VARIANTS"].split(","))
steps = {}
for name, flags in VARIANTS:
    # whole step without per-kernel events (events between kernels serialise programmatic dependent launches)
    p.set_profiling(False)
    p.set_debug(flags)
    for _ in range(3):
        p.run()
    p.sync()
    t0 = time.perf_counter()
    for _ in range(10):
        p.run()
    p.sync()
    steps[name] = (time.perf_counter() - t0) * 100.0
    p.set_profiling(True)
    acc = {}
    for _ in range(4):
        p.run(); p.sync()
        for k, v in p.last_timings().items():
            acc.setdefault(k, []).append(v)
    res[name] = {k: float(np.mean(v[1:])) for k, v in acc.items()}
keys = list(dict.fromkeys(k for r in res.values() for k in r))
print(f"{'kernel':16s}" + "".join(f"{n:>14s}" for n in res))
for k in keys:
    print(f"{k:16s}" + "".join(f"{res[n].get(k, 0.0):14.4f}" for n in res))
print(f"{'total':16s}" + "".join(f"{sum(res[n].values()):14.4f}" for n in res), " windows", p.n_windows)
print(f"{'step (no events)':16s}" + "".join(f"{steps[n]:14.4f}" for n in res))
