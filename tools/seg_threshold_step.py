#!/usr/bin/env python
"""Per-stream segmentation-thresholds (cova_pipeline_set_stream_property_f32) against one threshold for the whole batch:
128 fresh 720p streams x 64 frames per flush on one pipeline, four batches in flight, frames in pinned memory.

Arms, alternated, REPEATS times each:
  (u) uniform     every stream and the pipeline at 0.4: no per-window table, the head compares with one tau
  (t) table       every stream at 0.4, the pipeline at 0.5: the same masks and boxes as (u), through a per-window tau table
                  uploaded with the batch and read by the head; t / u is the cost of the table alone
  (m) mixed       stream s at 0.3 + 0.1 * (s mod 4), through the table; its masks differ, and so do the CCL's work and the
                  bytes of boxes copied back
A timed run submits BATCHES flushes and runs from the first submit to the last collect (boxes copied back); windows/s counts
the windows the batches produced.  Every arm produces the same windows.  Prints one JSON line per arm and repeat and a
summary with the card name and power limit read in the same process.

--profile: instead of the timed runs, the device time of every kernel (cova_pipeline_set_profiling / last_timings) of the
same batch re-run with cova_pipeline_run, PROFILE_RUNS times per arm, alternated; reports the median tc_dec3_head time per
arm.  Run it separately: the timing events sit between the kernels."""
import json, os, subprocess, sys, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cova_b200 import synth, weights
from cova_b200.elements import BlobPipeline, PinnedBuffer

H, W, T = 45, 80, 4
STREAMS, FPS = 128, 64
SEG = "segmentation-threshold"
BATCHES = int(os.environ.get("BATCHES", 32))
REPEATS = int(os.environ.get("REPEATS", 5))
PROFILE_RUNS = int(os.environ.get("PROFILE_RUNS", 20))


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim, clk = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": plim, "sm_max_clock": clk}
    except Exception as e:  # noqa: BLE001
        return {"gpu": None, "power_limit": None, "error": repr(e)}


def set_arm(p, arm, ids):
    p.set_property(SEG, 0.5 if arm == "t" else 0.4)
    p.set_stream_property(SEG, 0.4)
    if arm == "m":
        for k in range(4):
            p.set_stream_property(SEG, 0.3 + 0.1 * k, ids[ids % 4 == k])


def timed(p, frames, ids, n_batches):
    """n_batches submits of the same flush, four in flight.  Returns (seconds, windows)."""
    n = 0
    t0 = time.perf_counter()
    for k in range(n_batches):
        if k >= 4:
            n += int(p.collect(raw=True)[1].size)
        p.submit(frames, stream_ids=ids, cont=False)
    for _ in range(min(4, n_batches)):
        n += int(p.collect(raw=True)[1].size)
    return time.perf_counter() - t0, n


def main():
    profile = "--profile" in sys.argv
    p = BlobPipeline(W, H, weights.to_blob(weights.random_weights(0, head_bias=-1.0)), STREAMS, FPS)
    ids = np.arange(STREAMS, dtype=np.uint32)
    quads = synth.tiled_streams(STREAMS, FPS, H, W, config_idx=7, n_unique=8)
    pm = PinnedBuffer(quads.shape, quads.dtype)
    pm.array[...] = quads
    want = STREAMS * (FPS - T + 1)
    arms = ("u", "t", "m")
    fg = {}
    for arm in arms:                                       # warm-up of every arm
        set_arm(p, arm, ids)
        s, n = timed(p, pm.array, ids, 8)
        assert n == 8 * want, (arm, n, want)
        fg[arm] = round(float(p.read_mask().mean()), 4)
    assert fg["t"] == fg["u"] != fg["m"], fg
    recs = []
    if profile:
        acc = {arm: [] for arm in arms}
        for r in range(PROFILE_RUNS):
            for arm in arms:
                set_arm(p, arm, ids)
                p.submit(pm.array, stream_ids=ids, cont=False)
                p.collect(raw=True)
                p.set_profiling(True)
                p.run()                                    # the same batch again: the slot keeps its tables
                p.sync()
                t = p.last_timings()
                p.set_profiling(False)
                acc[arm].append(t["tc_dec3_head"])
                rec = {"arm": arm, "run": r, "kernel_ms": {k: round(v, 5) for k, v in t.items()}}
                print(json.dumps(rec), flush=True)
        summary = dict(card(), grid=f"{W}x{H} macroblocks", streams=STREAMS, frames=FPS, windows=want,
                       profile_runs=PROFILE_RUNS, mask_fg=fg)
        for arm in arms:
            v = acc[arm]
            summary[arm] = {"tc_dec3_head_ms_median": round(float(np.median(v)), 5), "min": round(min(v), 5),
                            "max": round(max(v), 5)}
        for arm in ("t", "m"):
            summary[f"head_{arm}_over_u"] = round(summary[arm]["tc_dec3_head_ms_median"] /
                                                  summary["u"]["tc_dec3_head_ms_median"], 4)
    else:
        for r in range(REPEATS):
            for arm in arms:
                set_arm(p, arm, ids)
                s, n = timed(p, pm.array, ids, BATCHES)
                rec = {"arm": arm, "repeat": r, "seconds": round(s, 5), "windows": n, "windows_per_s": round(n / s, 1),
                       "flushes": BATCHES}
                print(json.dumps(rec), flush=True)
                recs.append(rec)
        summary = dict(card(), grid=f"{W}x{H} macroblocks", streams=STREAMS, frames=FPS, windows_per_flush=want,
                       flushes=BATCHES, repeats=REPEATS, in_flight=4, mask_fg=fg)
        for arm in arms:
            v = [r["windows_per_s"] for r in recs if r["arm"] == arm]
            summary[arm] = {"median": float(np.median(v)), "min": min(v), "max": max(v),
                            "spread_pct": round(100 * (max(v) - min(v)) / float(np.median(v)), 2)}
        for arm in ("t", "m"):
            summary[f"{arm}_over_u"] = round(summary[arm]["median"] / summary["u"]["median"], 4)
    print(json.dumps(summary))
    p.close()
    pm.close()


if __name__ == "__main__":
    main()
