#!/usr/bin/env python
"""Per-stream gammas (cova_pipeline_set_stream_property) against splitting the streams into one batch per gamma: 128 fresh
720p streams x 64 frames per flush, stream s at gamma 1 + s mod 4, on one pipeline created with gamma 1, four batches in
flight, frames in pinned memory.

Arms, alternated, REPEATS times each:
  (m) mixed   one batch of the 128 streams per flush (submit_host2), each stream with its own gamma
  (s) split   the same streams as four batches of 32, one per gamma, per flush
A timed run submits BATCHES flushes and runs from the first submit to the last collect (boxes copied back); windows/s counts
the windows the batches produced.  Both arms produce the same windows.  Prints one JSON line per arm and repeat and a
summary with the card name and power limit read in the same process."""
import json, os, subprocess, sys, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cova_b200 import synth, weights
from cova_b200.elements import BlobPipeline, PinnedBuffer

H, W, T = 45, 80, 4
STREAMS, FPS, GAMMAS = 128, 64, 4
BATCHES = int(os.environ.get("BATCHES", 32))
REPEATS = int(os.environ.get("REPEATS", 5))


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim, clk = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": plim, "sm_max_clock": clk}
    except Exception as e:  # noqa: BLE001
        return {"gpu": None, "power_limit": None, "error": repr(e)}


def timed(p, jobs):
    """jobs: the submits of all flushes, four in flight.  Returns (seconds, windows)."""
    n = 0
    t0 = time.perf_counter()
    for k, (fr, ids) in enumerate(jobs):
        if k >= 4:
            n += int(p.collect(raw=True)[1].size)
        p.submit(fr, stream_ids=ids, cont=False)
    for _ in range(min(4, len(jobs))):
        n += int(p.collect(raw=True)[1].size)
    return time.perf_counter() - t0, n


def main():
    p = BlobPipeline(W, H, weights.to_blob(weights.random_weights(0, head_bias=-1.0)), STREAMS, FPS, gamma=1)
    ids = np.arange(STREAMS, dtype=np.uint32)
    gamma = 1 + ids % GAMMAS
    for g in range(1, GAMMAS + 1):
        p.set_stream_property("gamma", g, ids[gamma == g])
    quads = synth.tiled_streams(STREAMS, FPS, H, W, config_idx=7, n_unique=8)
    pins, flush = [], {}
    pm = PinnedBuffer(quads.shape, quads.dtype)
    pm.array[...] = quads
    pins.append(pm)
    flush["m"] = [(pm.array, ids)]
    flush["s"] = []
    for g in range(1, GAMMAS + 1):                        # the streams of one gamma, contiguous in their own pinned buffer
        sub = ids[gamma == g]
        pb = PinnedBuffer((sub.size,) + quads.shape[1:], quads.dtype)
        pb.array[...] = quads[sub]
        pins.append(pb)
        flush["s"].append((pb.array, sub))
    want = sum(len(range(T - 1, FPS, int(g))) for g in gamma)
    for arm in flush:                                      # warm-up: every shape of every arm
        s, n = timed(p, flush[arm] * 4)
        assert n == 4 * want, (arm, n, want)
    recs = []
    for r in range(REPEATS):
        for arm in flush:
            s, n = timed(p, flush[arm] * BATCHES)
            rec = {"arm": arm, "repeat": r, "seconds": round(s, 5), "windows": n, "windows_per_s": round(n / s, 1),
                   "flushes": BATCHES, "submits": len(flush[arm]) * BATCHES}
            print(json.dumps(rec), flush=True)
            recs.append(rec)
    summary = dict(card(), grid=f"{W}x{H} macroblocks", streams=STREAMS, frames=FPS, gammas=list(range(1, GAMMAS + 1)),
                   windows_per_flush=want, flushes=BATCHES, repeats=REPEATS, in_flight=4)
    for arm in flush:
        v = [r["windows_per_s"] for r in recs if r["arm"] == arm]
        summary[arm] = {"median": float(np.median(v)), "min": min(v), "max": max(v),
                        "spread_pct": round(100 * (max(v) - min(v)) / float(np.median(v)), 2)}
    summary["mixed_over_split"] = round(summary["m"]["median"] / summary["s"]["median"], 4)
    print(json.dumps(summary))
    p.close()
    for b in pins:
        b.close()


if __name__ == "__main__":
    main()
