#!/usr/bin/env python
"""End to end on one GPU with sparse input (cova_pipeline_submit_sparse) against the dense input formats.

Workload (bench.py's shapes): CONFIG=c2 128 streams x 67 frames of 720p, c3 64 x 67 of 1080p, c4 16 x 67 of 4K (dense
worst case weights); four batches in flight (submit k+3 before collect k), every host buffer page-locked.  Input
INPUT=synth is synth.tiled_streams; INPUT=real is the committed real-decoder clip (tests/golden/demo_1m_meta.npz, 720p
only), stream s reading frames (s*67 + f) mod 1802.  Four arms, alternated REPEATS times, STEPS batches each:
  quads        4-byte decoder quads, submit_host2
  packed16     2-byte frames packed before the clock starts, submit_host2
  sparse_pre   sparse batches encoded before the clock starts (a producer that writes records), submit_sparse
  sparse_host  cova_packer_pack_sparse on all cores inside the timed region, from the pinned quads, then submit_sparse
Every arm submits with stream ids 0..n-1 (fresh chains), so all four take the same path after the copy stage.
Per arm: frames/s and windows/s (first submit to last collect), H2D bytes per step, host ms per step spent in the submit
call (for the sparse arms it includes the validation walk; sparse minus packed16 estimates it), encoder ms per step.
Then sparse_expand_kernel's device time from torch.profiler (CUDA activities) over PROFILE_STEPS sparse steps, in a
separate pass.  Prints one JSON line per arm and repeat and a summary with the card name and power limit read in the
same process; the boxes of every arm are checked against the quads arm."""
import json, os, subprocess, sys, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cova_b200 import _lib, synth, weights
from cova_b200.elements import BlobPipeline, FramePacker, PinnedBuffer, SparseBatch

CONFIGS = {"c2": (45, 80, 128, -1.0), "c3": (68, 120, 64, -1.0), "c4": (135, 240, 16, 0.0)}
CONFIG = os.environ.get("CONFIG", "c2")
INPUT = os.environ.get("INPUT", "synth")
STEPS = int(os.environ.get("STEPS", 40))
REPEATS = int(os.environ.get("REPEATS", 3))
PROFILE_STEPS = int(os.environ.get("PROFILE_STEPS", 20))
FPS, AHEAD, NBUF = 67, 3, 4
ARMS = ["quads", "packed16", "sparse_pre", "sparse_host"]


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim, clk = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": plim, "sm_max_clock": clk}
    except Exception as e:  # noqa: BLE001
        return {"gpu": None, "power_limit": None, "error": repr(e)}


def inputs(h, w, n):
    if INPUT == "real":
        assert (h, w) == (45, 80), "the real clip is 720p"
        d = np.load(os.path.join(ROOT, "tests", "golden", "demo_1m_meta.npz"))
        clip = np.ascontiguousarray(np.moveaxis(d["planes"], 0, -1))
        idx = (np.arange(n)[:, None] * FPS + np.arange(FPS)[None, :]) % clip.shape[0]
        return clip[idx]
    return synth.tiled_streams(n, FPS, h, w, config_idx=1)


def main():
    h, w, n, head_bias = CONFIGS[CONFIG]
    quads_np = inputs(h, w, n)
    pk = FramePacker()                                       # one thread per online CPU
    ids = np.arange(n, dtype=np.uint32)
    q_pins, p_pins, s_pre, s_out = [], [], [], []
    for i in range(NBUF):                                    # four different batches: rolled stream order
        src = np.roll(quads_np, i, axis=0)
        qp = PinnedBuffer(src.shape)
        qp.array[...] = src
        q_pins.append(qp)
        pp = PinnedBuffer(src.shape[:-1], np.uint16)
        pk.pack(src, out=pp.array)
        p_pins.append(pp)
        b = pk.pack_sparse(src)
        sp = PinnedBuffer(b.data.size)
        sp.array[:] = b.data
        s_pre.append(SparseBatch(sp.array, n, FPS, h, w))
        s_pre[-1].pin = sp
        s_out.append(PinnedBuffer(n * FPS * _lib.sparse_max_frame_bytes(h * w)))
    wblob = weights.to_blob(weights.random_weights(0, head_bias=head_bias))
    pq = BlobPipeline(w, h, wblob, n, FPS, cc_threshold=1)
    pp = BlobPipeline(w, h, wblob, n, FPS, cc_threshold=1, packed_input=True)
    n_frames, n_mb = n * FPS, h * w
    stats = {}

    def frames_for(arm, k):
        if arm == "quads":
            return q_pins[k % NBUF].array
        if arm == "packed16":
            return p_pins[k % NBUF].array
        if arm == "sparse_pre":
            return s_pre[k % NBUF]
        t0 = time.perf_counter()
        b = pk.pack_sparse(q_pins[k % NBUF].array, out=s_out[k % NBUF].array)
        stats["enc"] += time.perf_counter() - t0
        stats["h2d"] += b.data.size
        return b

    def run(arm, steps, check=None):
        p = pq if arm == "quads" else pp
        stats.update(enc=0.0, sub=0.0, h2d=0)
        windows = 0

        def submit(k):
            fr = frames_for(arm, k)
            t0 = time.perf_counter()
            p.submit(fr, stream_ids=ids)
            stats["sub"] += time.perf_counter() - t0

        t0 = time.perf_counter()
        for k in range(min(AHEAD, steps)):
            submit(k)
        for k in range(steps):
            if k + AHEAD < steps:
                submit(k + AHEAD)
            if check is None:
                windows += int(p.collect(raw=True)[1].size)
            else:
                check.append(p.collect())
                windows += len(check[-1])
        s = time.perf_counter() - t0
        return s, windows

    ref = []
    run("quads", NBUF, ref)                                  # warm-up + the reference boxes of the four batches
    same = {}
    for arm in ARMS[1:]:
        got = []
        run(arm, NBUF, got)
        same[arm] = got == ref
    recs = []
    for r in range(REPEATS):
        for arm in ARMS:
            s, nw = run(arm, STEPS)
            h2d = {"quads": n_frames * n_mb * 4, "packed16": n_frames * n_mb * 2,
                   "sparse_pre": int(np.mean([b.data.size for b in s_pre]))}.get(arm, stats["h2d"] / STEPS)
            rec = {"config": CONFIG, "input": INPUT, "arm": arm, "repeat": r, "steps": STEPS, "seconds": round(s, 5),
                   "frames_per_s": round(n_frames * STEPS / s, 1), "windows_per_s": round(nw / s, 1),
                   "h2d_bytes_per_step": int(h2d), "submit_ms_per_step": round(1e3 * stats["sub"] / STEPS, 4),
                   "encoder_ms_per_step": round(1e3 * stats["enc"] / STEPS, 4) if arm == "sparse_host" else None}
            print(json.dumps(rec), flush=True)
            recs.append(rec)

    # sparse_expand_kernel device time: a separate, profiled pass of sparse_pre steps
    kern = {"sparse_expand_kernel_us_per_launch": None}
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile
        launches0 = pp.launch_count()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            run("sparse_pre", PROFILE_STEPS)
            torch.cuda.synchronize()
        ev = [e for e in prof.key_averages() if "sparse_expand_kernel" in e.key]
        if ev:
            dev_us = sum(getattr(e, "device_time_total", 0.0) or getattr(e, "cuda_time_total", 0.0) for e in ev)
            cnt = sum(e.count for e in ev)
            per_step_bytes = n_frames * n_mb * 2 + int(np.mean([b.data.size for b in s_pre]))
            kern = {"sparse_expand_kernel_us_per_launch": round(dev_us / cnt, 3), "sparse_expand_launches": cnt,
                    "sparse_expand_ms_per_step": round(dev_us / 1e3 / PROFILE_STEPS, 4),
                    "sparse_expand_bytes_per_step": per_step_bytes,
                    "sparse_expand_gb_per_s": round(per_step_bytes * PROFILE_STEPS / (dev_us * 1e-6) / 1e9, 1),
                    "pipeline_launches_in_pass": pp.launch_count() - launches0}
    except Exception as e:  # noqa: BLE001
        kern["error"] = repr(e)

    summary = dict(card(), config=CONFIG, input=INPUT, grid=f"{w}x{h} macroblocks", streams=n, frames_per_stream=FPS,
                   in_flight=AHEAD + 1, steps=STEPS, repeats=REPEATS, encoder_threads=None, boxes_identical_to_quads=same, **kern)
    for arm in ARMS:
        v = [r["frames_per_s"] for r in recs if r["arm"] == arm]
        summary[arm] = {"frames_per_s_median": float(np.median(v)), "min": min(v), "max": max(v),
                        "h2d_bytes_per_step": int(np.median([r["h2d_bytes_per_step"] for r in recs if r["arm"] == arm])),
                        "submit_ms_per_step": float(np.median([r["submit_ms_per_step"] for r in recs if r["arm"] == arm]))}
        if arm == "sparse_host":
            summary[arm]["encoder_ms_per_step"] = float(np.median([r["encoder_ms_per_step"] for r in recs if r["arm"] == arm]))
    summary["validation_ms_per_step_est"] = round(summary["sparse_pre"]["submit_ms_per_step"] - summary["packed16"]["submit_ms_per_step"], 4)
    summary["encoder_threads"] = min(os.cpu_count() or 1, 64)     # FramePacker(0): one per online CPU, at most 64
    print(json.dumps(summary), flush=True)


if __name__ == "__main__":
    main()
