#!/usr/bin/env python
"""Continued 720p streams through submit / collect, four batches in flight: what mixing histories and gamma phases in one
batch (COVA_SUBMIT_STAGGERED) costs against lock-step batches and against splitting the mix into lock-step sub-batches.

Every batch is 128 streams x 64 new frames at gamma = 2.  Three arms, alternated, REPEATS times each:
  (a) lock-step    every stream carries 3 frames on the same gamma phase (seen = 3)
  (b) staggered    one batch, streams cycle over seen = 0, 1, 2, 3, 4: histories 0..3 and, at 3, both gamma phases
  (c) split        the mix of (b), one lock-step sub-batch per (history, phase) class: what a caller had to do without
                   the flag (5 submits per 128-stream flush)
A timed run submits BATCHES flushes; every flush uses stream ids of its own, prepared (reset + short feeding batches) before
the clock starts, so that each flush meets exactly the state its arm describes.  The time runs from the first submit to
the last collect (boxes copied back); windows/s counts the windows the batches produced.  Runs with quad input and with
the 2-byte packed input (PACKED=0 / 1 / both).  Prints one JSON line per arm and repeat, then a summary line with the card
name and power limit read in the same process."""
import json, os, subprocess, sys, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cova_b200 import synth, weights
from cova_b200.elements import BlobPipeline, FramePacker, PinnedBuffer

H, W, T, GAMMA = 45, 80, 4, 2
STREAMS, FPS = 128, 64
BATCHES = int(os.environ.get("BATCHES", 32))
REPEATS = int(os.environ.get("REPEATS", 5))
SEEN = [0, 1, 2, 3, 4]                     # class c of the mix: frames seen before the flush


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim, clk = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": plim, "sm_max_clock": clk}
    except Exception as e:  # noqa: BLE001
        return {"gpu": None, "power_limit": None, "error": repr(e)}


def prepare(p, feed, seen_of):
    """Reset every id, then feed seen_of[id] frames to it (one continued batch per distinct count, collected)."""
    p.reset_streams()
    for k in sorted(set(seen_of.values()) - {0}):
        ids = np.array([i for i, v in seen_of.items() if v == k], dtype=np.uint32)
        p.submit(feed[: ids.size, :k], stream_ids=ids, cont=True, staggered=True)
        p.collect(raw=True)


def timed(p, jobs):
    """jobs: (frames, ids) per submit, four in flight.  Returns (seconds, windows)."""
    n = 0
    t0 = time.perf_counter()
    for k, (fr, ids) in enumerate(jobs):
        if k >= 4:
            n += int(p.collect(raw=True)[1].size)
        p.submit(fr, stream_ids=ids, cont=True, staggered=True)
    for _ in range(min(4, len(jobs))):
        n += int(p.collect(raw=True)[1].size)
    return time.perf_counter() - t0, n


def arm_jobs(arm, pin):
    """Per arm: stream id -> frames seen before its flush, and the submits of the timed run."""
    seen_of, jobs = {}, []
    for b in range(BATCHES):
        ids = np.arange(b * STREAMS, (b + 1) * STREAMS, dtype=np.uint32)
        cls = np.arange(STREAMS) % len(SEEN)
        for i, c in zip(ids, cls):
            seen_of[int(i)] = 3 if arm == "a" else SEEN[c]
        if arm in ("a", "b"):
            jobs.append((pin, ids))
        else:
            lo = 0
            for c in range(len(SEEN)):            # contiguous slices of the pinned frames, one per class
                sub = ids[cls == c]
                jobs.append((pin[lo: lo + sub.size], sub))
                lo += sub.size
    return seen_of, jobs


def run(packed):
    max_streams = BATCHES * STREAMS
    # the chunk size a 128-stream pipeline picks (32 chains: ~1024 windows), whatever the id space
    chunks = max_streams // 32
    p = BlobPipeline(W, H, weights.to_blob(weights.random_weights(0, head_bias=-1.0)), max_streams, FPS + T - 1, gamma=GAMMA,
                     n_chunks=chunks, packed_input=packed)
    quads = synth.tiled_streams(STREAMS, FPS, H, W, config_idx=7, n_unique=8)
    src = FramePacker().pack(quads) if packed else quads
    pinb = PinnedBuffer(src.shape, src.dtype)
    pinb.array[...] = src
    pin = pinb.array
    feed = np.repeat(pin[:1, :4], max_streams, axis=0)      # frames of the untimed feeding batches
    out = []
    plans = {arm: arm_jobs(arm, pin) for arm in "abc"}
    for arm in "abc":                             # warm-up: every shape of every arm once
        prepare(p, feed, plans[arm][0])
        timed(p, plans[arm][1][: 4 * (5 if arm == "c" else 1)])
    for r in range(REPEATS):
        for arm in "abc":
            prepare(p, feed, plans[arm][0])
            s, n = timed(p, plans[arm][1])
            rec = {"arm": arm, "packed": packed, "repeat": r, "seconds": round(s, 5), "windows": n,
                   "windows_per_s": round(n / s, 1), "flushes": BATCHES, "submits": len(plans[arm][1])}
            print(json.dumps(rec), flush=True)
            out.append(rec)
    p.close()
    pinb.close()
    return out


def main():
    modes = {"0": [False], "1": [True]}.get(os.environ.get("PACKED", "both"), [False, True])
    recs = [r for m in modes for r in run(m)]
    summary = dict(card(), grid=f"{W}x{H} macroblocks", streams=STREAMS, new_frames=FPS, gamma=GAMMA, flushes=BATCHES,
                   repeats=REPEATS, in_flight=4)
    for m in modes:
        for arm in "abc":
            v = [r["windows_per_s"] for r in recs if r["packed"] == m and r["arm"] == arm]
            w = [r["windows"] // BATCHES for r in recs if r["packed"] == m and r["arm"] == arm]
            summary[f"{'packed' if m else 'quads'}_{arm}"] = {"median": float(np.median(v)), "min": min(v), "max": max(v),
                                                             "spread_pct": round(100 * (max(v) - min(v)) / float(np.median(v)), 2),
                                                             "windows_per_flush": w[0]}
        k = "packed" if m else "quads"
        summary[f"{k}_b_over_a"] = round(summary[f"{k}_b"]["median"] / summary[f"{k}_a"]["median"], 4)
        summary[f"{k}_b_over_c"] = round(summary[f"{k}_b"]["median"] / summary[f"{k}_c"]["median"], 4)
    print(json.dumps(summary))


if __name__ == "__main__":
    main()
