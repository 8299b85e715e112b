#!/usr/bin/env python
"""Development aid: CCL kernel time on the benchmark's own masks and on the synthetic mask patterns.
8K grids (270 x 480 macroblocks) run the thread-block-cluster kernel (COVA_FLAG_CCL_CLUSTER).  AB=1 adds a forced-band
A/B on 4K masks: the single-CTA kernel against the cluster kernel with k = 2 and 4 bands, alternating, which prices the
seams and the distributed-shared-memory traffic on the same masks."""
import os, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cova_b200 import synth, weights
from cova_b200.elements import BlobPipeline

def time_ccl(p, masks, reps=5):
    p.load_masks(masks)
    p.set_profiling(True)
    ts = []
    for _ in range(reps):
        p.ccl(); p.sync()
        t = p.last_timings()
        ts.append(t.get("ccl_bbox", t.get("ccl_bbox_cluster", float("nan"))))
    p.set_profiling(False)
    boxes = p.fetch_boxes_raw()[2]
    return float(np.median(ts[1:])), float(((boxes.astype(np.int64) - 8) // 24).mean())

CASES = ((45, 80, 128, -1.0), (68, 120, 64, -1.0), (135, 240, 16, -1.0), (135, 240, 16, 0.0),
         (270, 480, 4, -1.0), (270, 480, 4, 0.0))
if os.environ.get("CASES"):             # e.g. CASES=3 -> only the dense 4K case
    CASES = tuple(CASES[int(i)] for i in os.environ["CASES"].split(","))
for (h, w, n_streams, hb) in CASES:
    fps = 67
    p = BlobPipeline(w, h, weights.to_blob(weights.random_weights(0, head_bias=hb)), n_streams, fps, n_chunks=1,
                     ccl_cluster=h * w > 135 * 240)
    n = p.windows_for(n_streams, fps)
    p.load_frames(synth.tiled_streams(n_streams, fps, h, w, 1)); p.run(); p.sync()
    m = p.read_mask()
    ms, nb = time_ccl(p, m)
    print(f"{h}x{w} blobnet masks hb={hb} n={n} {ms*1e3:8.1f} us  {n/ms/1e3:8.2f} M masks/s  boxes/frame {nb:.1f}  fg {m.mean():.3f}")
    if os.environ.get("ONLY_NET"):
        continue
    for name, pat in synth.mask_patterns(h, w, seed=1).items():
        mm = np.broadcast_to(pat, (n,) + pat.shape).copy()
        ms, nb = time_ccl(p, mm)
        print(f"{h}x{w} {name:20s} n={n} {ms*1e3:8.1f} us  {n/ms/1e3:8.2f} M masks/s  boxes/frame {nb:.1f}  fg {pat.mean():.3f}")

if os.environ.get("AB"):
    h, w, n_streams, fps = 135, 240, 16, 67
    blob = weights.to_blob(weights.random_weights(0))
    pipes = {k: BlobPipeline(w, h, blob, n_streams, fps, n_chunks=1, ccl_cluster=k > 0, ccl_bands=k) for k in (0, 2, 4)}
    n = pipes[0].windows_for(n_streams, fps)
    sets = {}
    for hb in (-1.0, 0.0):
        q = BlobPipeline(w, h, weights.to_blob(weights.random_weights(0, head_bias=hb)), n_streams, fps, n_chunks=1)
        q.load_frames(synth.tiled_streams(n_streams, fps, h, w, 1)); q.run(); q.sync()
        sets[f"blobnet hb={hb}"] = q.read_mask()
        del q
    for name, pat in synth.mask_patterns(h, w, seed=1).items():
        sets[name] = np.broadcast_to(pat, (n,) + pat.shape).copy()
    for name, mm in sets.items():
        res = {k: [] for k in pipes}
        for _ in range(3):                       # alternate the kernels
            for k, p in pipes.items():
                res[k].append(time_ccl(p, mm)[0])
        row = "  ".join(f"{'single' if k == 0 else f'k={k}'} {np.median(v)*1e3:8.1f} us" for k, v in res.items())
        print(f"AB {h}x{w} {name:20s} n={n}  {row}")
