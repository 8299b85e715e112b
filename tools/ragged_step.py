#!/usr/bin/env python
"""Ragged batches (cova_pipeline_submit_ragged) against lock-step batches and against splitting a mix into one batch per
distinct count: 128 fresh 720p chains per flush at gamma = 1, four batches in flight, frames in pinned memory.

Arms, alternated, REPEATS times each:
  (a) lock-step     every chain brings 64 frames (submit_host2)
  (b) ragged        a 25 / 30 fps mix, 53 and 64 frames, chains grouped by count: one batch, two copies per chunk
  (c) split         the mix of (b) as one batch per distinct count (two submits per flush)
  (d) interleaved   the mix of (b) with the counts alternating chain by chain: one copy per chain
  (e) distinct      33 + (s mod 32) frames: every chain's count differs from its neighbours', one copy per chain
A timed run submits BATCHES flushes and runs from the first submit to the last collect (boxes copied back); windows/s
counts the windows the batches produced, H2D bytes the frame bytes crossing PCIe (counted from the shapes).  Then one
profiled run per arm (torch.profiler, CUDA activities, in the same process but apart from the timed runs) gives per flush
the device time of tensorise_frames, enc1_fused and the host-to-device copies, and the number of those copies.  Quads and
the 2-byte packed input (PACKED=0 / 1 / both).  Prints one JSON line per arm and repeat, one per profiled arm, and a
summary with the card name and power limit read in the same process."""
import json, os, subprocess, sys, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cova_b200 import synth, weights
from cova_b200.elements import BlobPipeline, FramePacker, PinnedBuffer

H, W, T, GAMMA = 45, 80, 4, 1
STREAMS, FPS, LOW = 128, 64, 53
BATCHES = int(os.environ.get("BATCHES", 32))
REPEATS = int(os.environ.get("REPEATS", 5))
ARMS = "abcde"


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim, clk = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": plim, "sm_max_clock": clk}
    except Exception as e:  # noqa: BLE001
        return {"gpu": None, "power_limit": None, "error": repr(e)}


def counts_of(arm):
    s = np.arange(STREAMS)
    if arm == "a":
        return np.full(STREAMS, FPS)
    if arm in "bc":
        return np.where(s < STREAMS // 2, LOW, FPS)
    if arm == "d":
        return np.where(s % 2 == 0, LOW, FPS)
    return 33 + s % 32


def arm_jobs(arm, pin):
    """The submits of one flush: (frames, counts or None, stream ids).  pin = [STREAMS * FPS, ...] pinned frames."""
    c = counts_of(arm)
    ids = np.arange(STREAMS, dtype=np.uint32)
    if arm == "a":
        return [(pin[: STREAMS * FPS].reshape(STREAMS, FPS, *pin.shape[1:]), None, ids)]
    if arm == "c":
        jobs, lo = [], 0
        for n in sorted(set(c.tolist())):
            sub = ids[c == n]
            jobs.append((pin[lo: lo + sub.size * n].reshape(sub.size, n, *pin.shape[1:]), None, sub))
            lo += sub.size * n
        return jobs
    return [(pin[: int(c.sum())], c.astype(np.uint32), ids)]


def copies_per_flush(arm, chunk_streams):
    """H2D frame copies the library issues for one flush: one per run of equal counts inside a chunk."""
    n = 0
    for fr, c, ids in arm_jobs(arm, np.zeros((STREAMS * FPS, 1), np.uint8)):
        cc = c if c is not None else np.full(ids.size, fr.shape[1])
        for c0 in range(0, cc.size, chunk_streams):
            part = cc[c0: c0 + chunk_streams]
            n += 1 + int((part[1:] != part[:-1]).sum())
    return n


def timed(p, jobs):
    """jobs: the submits of all flushes, four in flight.  Returns (seconds, windows)."""
    n = 0
    t0 = time.perf_counter()
    for k, (fr, c, ids) in enumerate(jobs):
        if k >= 4:
            n += int(p.collect(raw=True)[1].size)
        p.submit(fr, stream_ids=ids, cont=False, counts=c)
    for _ in range(min(4, len(jobs))):
        n += int(p.collect(raw=True)[1].size)
    return time.perf_counter() - t0, n


def profiled(p, jobs, flushes):
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        timed(p, jobs)
        torch.cuda.synchronize()
    acc = {"tensorise_frames_ms": 0.0, "enc1_fused_ms": 0.0, "h2d_copy_ms": 0.0, "h2d_copies": 0}
    for e in prof.key_averages():
        name = e.key
        us = getattr(e, "device_time_total", None)
        us = e.cuda_time_total if us is None else us
        if "tensorise_frames" in name:
            acc["tensorise_frames_ms"] += us / 1e3
        elif "enc1_fused" in name:
            acc["enc1_fused_ms"] += us / 1e3
        elif "HtoD" in name:                                # frame copies and the small per-batch table uploads
            acc["h2d_copy_ms"] += us / 1e3
            acc["h2d_copies"] += e.count
    return {k: (round(v / flushes, 4) if isinstance(v, float) else round(v / flushes, 2)) for k, v in acc.items()}


def run(packed):
    p = BlobPipeline(W, H, weights.to_blob(weights.random_weights(0, head_bias=-1.0)), STREAMS, FPS, gamma=GAMMA,
                     packed_input=packed)
    chunk_streams = -(-STREAMS // min(16, max(1, STREAMS * (FPS - T + 1) // 1024)))      # the library's automatic chunks
    quads = synth.tiled_streams(STREAMS, FPS, H, W, config_idx=7, n_unique=8).reshape(STREAMS * FPS, H, W, 4)
    src = FramePacker().pack(quads) if packed else quads
    pinb = PinnedBuffer(src.shape, src.dtype)
    pinb.array[...] = src
    pin = pinb.array
    frame_bytes = src[0].nbytes
    flush = {arm: arm_jobs(arm, pin) for arm in ARMS}
    out = []
    for arm in ARMS:                                        # warm-up: every shape of every arm
        timed(p, flush[arm] * 4)
    for r in range(REPEATS):
        for arm in ARMS:
            s, n = timed(p, flush[arm] * BATCHES)
            h2d = int(counts_of(arm).sum()) * frame_bytes * BATCHES
            rec = {"arm": arm, "packed": packed, "repeat": r, "seconds": round(s, 5), "windows": n,
                   "windows_per_s": round(n / s, 1), "h2d_bytes": h2d, "h2d_GB_per_s": round(h2d / s / 1e9, 3),
                   "flushes": BATCHES, "submits": len(flush[arm]) * BATCHES}
            print(json.dumps(rec), flush=True)
            out.append(rec)
    prof = {}
    for arm in ARMS:
        prof[arm] = profiled(p, flush[arm] * 8, 8)
        prof[arm]["copies_counted"] = copies_per_flush(arm, chunk_streams)
        print(json.dumps({"profile": arm, "packed": packed, "per_flush": prof[arm]}), flush=True)
    p.close()
    pinb.close()
    return out, prof, frame_bytes


def main():
    modes = {"0": [False], "1": [True]}.get(os.environ.get("PACKED", "both"), [False, True])
    summary = dict(card(), grid=f"{W}x{H} macroblocks", streams=STREAMS, gamma=GAMMA, flushes=BATCHES, repeats=REPEATS,
                   in_flight=4, arms={a: sorted(set(counts_of(a).tolist()))[:4] for a in ARMS})
    for m in modes:
        recs, prof, fb = run(m)
        k = "packed" if m else "quads"
        for arm in ARMS:
            v = [r["windows_per_s"] for r in recs if r["arm"] == arm]
            g = [r["h2d_GB_per_s"] for r in recs if r["arm"] == arm]
            w = [r["windows"] // BATCHES for r in recs if r["arm"] == arm]
            summary[f"{k}_{arm}"] = {"median": float(np.median(v)), "min": min(v), "max": max(v),
                                     "spread_pct": round(100 * (max(v) - min(v)) / float(np.median(v)), 2),
                                     "windows_per_flush": w[0], "h2d_GB_per_s_median": float(np.median(g)),
                                     "h2d_bytes_per_flush": int(counts_of(arm).sum()) * fb, **prof[arm]}
        for x, y in (("b", "a"), ("b", "c"), ("d", "b"), ("e", "b")):
            summary[f"{k}_{x}_over_{y}"] = round(summary[f"{k}_{x}"]["median"] / summary[f"{k}_{y}"]["median"], 4)
    print(json.dumps(summary))


if __name__ == "__main__":
    main()
