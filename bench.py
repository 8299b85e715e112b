#!/usr/bin/env python
"""Benchmark of the blob-detection hot path (tensorise -> BlobNet -> CCL/bbox) on B200.

    python bench.py --gpus N --steps K --warmup W          # this repo's CUDA path
    python bench.py --impl reference ...                     # the CPU path (oracle port) on the host cores
    python bench.py --dump-outputs DIR ...                   # also write the last timed step's boxes as DIR/*.npy

A step = one pass of the whole path over one batch of independent chains of 67 frames (= 64 windows per chain):
    --config c2 (default)  720p,  80x45 macroblocks, 128 chains per GPU = 8192 windows per step
                           (BASELINE.json configs[1] shape per chain, configs[4] chain count per GPU)
    --config c3            1080p, 120x68, 64 chains per GPU = 4096 windows per step (configs[2]: 256 streams over 4 GPUs)
    --config c4            4K,    240x135, 16 chains per GPU = 1024 windows per step, dense worst case (configs[3]:
                           head bias 0 -> about half of the mask is foreground, thousands of components per frame)
    --config c5            = c2 (configs[4]: 1024 concurrent 720p streams over 8 GPUs = 128 chains per GPU; run with --gpus 8)
`value` counts detections (output windows) per second with the frames resident in HBM; `e2e` is the same through
BlobPipeline.submit()/collect() with pinned host frames in and bincode boxes out.  Prints ONE JSON line (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

T = 4
FRAMES_PER_STREAM = 67
# name -> (h_mb, w_mb, chains per GPU, head bias of the random-init weights, description)
CONFIGS = {"c2": (45, 80, 128, -1.0, "synthetic 720p metadata (80x45 MB grid)"),
           "c3": (68, 120, 64, -1.0, "synthetic 1080p metadata (120x68 MB grid)"),
           "c4": (135, 240, 16, 0.0, "synthetic 4K metadata (240x135 MB grid), dense worst case"),
           # BASELINE.json configs[4] (1024 concurrent 720p streams over 8 GPUs) is the c2 workload run with --gpus 8
           "c5": (45, 80, 128, -1.0, "synthetic 720p metadata (80x45 MB grid), 1024 streams over 8 GPUs = 128 per GPU")}
H_MB, W_MB, STREAMS_PER_GPU = CONFIGS["c2"][:3]   # the default workload
METRIC, UNIT = "blob_detection_frames_per_sec", "frames/s"
# kernels of one step in launch order: (name the library reports, bound, BlobNet layer it belongs to)
KERNELS = [("tensorise_frames", "hbm", None), ("tc_enc1_fused", "hbm", "enc1"),
           ("tc_enc1_conv", "tensor", "enc1"), ("enc1_pointwise_tn", "hbm", "enc1"),      # two-kernel fallback of block 1
           ("tc_enc2", "tensor", "enc2"), ("tc_enc3", "tensor", "enc3"), ("tc_enc4", "tensor", "enc4"),
           ("tc_dec0", "tensor", "dec0"), ("tc_dec1", "tensor", "dec1"), ("tc_dec2", "tensor", "dec2"),
           ("tc_dec3_head", "tensor", "dec3_head"), ("ccl_bbox", "hbm", None)]
LAYERS = ["enc1", "enc2", "enc3", "enc4", "dec0", "dec1", "dec2", "dec3_head"]


def layer_flops(h, w):
    """Algorithmic 2*MAC per window of every BlobNet layer (SURVEY.md section 3.4; PointWiseTN is counted with
    its encoder layer, the 1x1 head with dec3), plus the PointWiseTN share of the first block."""
    enc_ch = [(3, 16), (16, 32), (32, 64), (64, 128)]
    dec_ch = [(128, 64), (128, 32), (64, 16), (32, 16)]
    out, sizes = [], []
    hh, ww = h, w
    tn1 = 0
    for i, (ci, co) in enumerate(enc_ch):
        mac = T * hh * ww * 9 * ci * co
        hh, ww = (hh + 1) // 2, (ww + 1) // 2
        tn = co * hh * ww * 2 * T * T
        if i == 0:
            tn1 = 2 * tn
        mac += tn
        sizes.append((hh, ww))
        out.append(2 * mac)
    for i, (ci, co) in enumerate(dec_ch):
        mac = hh * ww * 16 * ci * co
        hh, ww = sizes[2 - i] if i < 3 else (h, w)
        if i == 3:
            mac += h * w * co
        out.append(2 * mac)
    return dict(zip(LAYERS, out)), tn1


def layer_bytes(h, w):
    """ALGORITHMIC HBM bytes per window of every BlobNet layer: each fp16 activation tensor read once and written once
    (encoder: input [Cin,T,H,W], output [Cout,T,H',W'] unless it is the last block, t = 0 skip row [Cout,H',W'];
    decoder: concatenated input, output; head: u8 mask).  Weights (<= 150 KB per layer) are not counted."""
    enc_ch = [(3, 16), (16, 32), (32, 64), (64, 128)]
    dec_ch = [(128, 64), (128, 32), (64, 16), (32, 16)]
    out, sizes = {}, []
    hh, ww = h, w
    for i, (ci, co) in enumerate(enc_ch):
        b_in = ci * T * hh * ww * 2
        hh, ww = (hh + 1) // 2, (ww + 1) // 2
        sizes.append((hh, ww))
        out[LAYERS[i]] = b_in + (co * T * hh * ww * 2 if i < 3 else 0) + co * hh * ww * 2
    for i, (ci, co) in enumerate(dec_ch):
        b_in = ci * hh * ww * 2
        hh, ww = sizes[2 - i] if i < 3 else (h, w)
        out[LAYERS[4 + i]] = b_in + (co * hh * ww * 2 if i < 3 else h * w)
    return out


def kernel_work(h, w, n_boxes):
    """ALGORITHMIC work per window of every kernel: FLOPs for the tensor-bound ones, bytes for the HBM-bound ones
    (SURVEY.md section 8d; DESIGN.md section 3)."""
    fl, tn1 = layer_flops(h, w)
    h1, w1 = (h + 1) // 2, (w + 1) // 2
    fpw = FRAMES_PER_STREAM / (FRAMES_PER_STREAM - T + 1)                      # frames per window of a 67-frame chain
    work = {# every frame read once (4 B per MB) + the per-FRAME fp16 input of the first conv written once (16 B per x pair);
            # SURVEY 8d counts 20*W*H per window for a per-window RGBA stack, which this path never materialises
            "tensorise_frames": fpw * (4 * h * w + 16 * h * ((w + 1) // 2)),
            # fused block 1: one packed input frame read + the window's 4 time planes + the t=0 skip copy written
            "tc_enc1_fused": 16 * h * ((w + 1) // 2) + 16 * h1 * w1 * 2 * (T + 1),
            "tc_enc1_conv": fl["enc1"] - tn1,
            # gather: one new pooled frame read (16 ch fp16) + the window's 4 time planes + the t=0 skip copy written
            "enc1_pointwise_tn": 16 * h1 * w1 * 2 * (1 + T + 1),
            "ccl_bbox": h * w + 24 * n_boxes + 8}
    for name, _, layer in KERNELS:
        if name not in work:
            work[name] = fl[layer]
    return work, fl


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tflops": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "tflops_burst": d["bf16_tflops"], "source": "measured"}
    return {"hbm_gbs": 6650.0, "tflops": 1400.0, "tflops_burst": 1590.0, "source": "fallback"}


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ CPU path
def cpu_path(frames, w, threads):
    """The reference's CPU path restated (oracle port): metapreprocess memcpy stack -> BlobNet fp32 on a CPU
    runtime (torch CPU stands in for ONNX, absent offline) -> threshold -> OpenCV-order CCL + bincode."""
    import torch
    from oracle import blobnet_ref, c_oracle, metapreprocess_ref as mpr
    torch.set_num_threads(threads)
    stacked = np.concatenate([c_oracle.metapreprocess_stream(frames[s], T, 1) for s in range(frames.shape[0])])
    logits = blobnet_ref.blobnet_forward(w, mpr.stacked_to_nchw(stacked, T))
    blobs = c_oracle.bboxcc_batch(blobnet_ref.mask_from_logits(logits), 1)
    return len(blobs)


def time_cpu(w, steps, warmup, h_mb, w_mb, max_streams, target_s=5.0, one_core=True):
    """Bounded sample of the bench workload on the host cores: chains per step sized from a warmed-up probe so that one
    step is about `target_s` seconds of CPU work, never more than the GPU arm's chains per GPU.  Runs exactly `warmup`
    untimed and `steps` timed steps."""
    from cova_b200 import synth
    threads = os.cpu_count() or 1
    fps = FRAMES_PER_STREAM
    probe = synth.tiled_streams(1, fps, h_mb, w_mb, 1)
    n1 = cpu_path(probe, w, threads)                                 # first call pays torch's one-off initialisation
    t0 = time.perf_counter()
    cpu_path(probe, w, threads)
    dt = time.perf_counter() - t0                                    # seconds per chain
    n_streams = int(max(1, min(max_streams, target_s / max(dt, 1e-3))))
    frames = synth.tiled_streams(n_streams, fps, h_mb, w_mb, 1)
    for _ in range(warmup):
        cpu_path(frames, w, threads)
    t0 = time.perf_counter()
    n = 0
    for _ in range(steps):
        n += cpu_path(frames, w, threads)
    dt = time.perf_counter() - t0
    out = {"value": n / dt, "unit": UNIT, "cores": threads, "kind": "port",
           "sample": f"{n_streams} chains x {fps} frames of {w_mb}x{h_mb} MB per step ({n // max(steps, 1)} windows), {steps} steps after "
                     f"{warmup} warm-up, C oracle tensorise/CCL + torch-CPU fp32 BlobNet, {threads} threads"}
    if one_core:
        # one core: the reference runs every chain single-threaded (SURVEY.md section 8d asks for both figures)
        t1 = time.perf_counter()
        n_one = cpu_path(probe, w, 1)
        dt_one = time.perf_counter() - t1
        out["one_core"] = {"value": n_one / dt_one, "unit": UNIT, "cores": 1, "sample": f"1 chain x {fps} frames ({n_one} windows), 1 thread"}
    return out, dt / max(steps, 1) * 1e3, n1


DUMP_BYTES = 64 << 20


def dump_outputs(pipe, out_dir):
    """Writes the boxes of the last step the pipeline ran, as a caller of run() receives them from fetch_boxes_raw(), so
    that two builds can be compared output for output:
        boxes.npy             float32 [n, 5]: left, top, width, height, area of every box, window by window
        boxes_per_window.npy  float64 [w]: how many of those rows belong to each window
        windows.npy           float64 [w]: which windows these are
    All windows, unless that would exceed DUMP_BYTES; then a sample of windows drawn with a fixed seed."""
    blob, offs, lens = pipe.fetch_boxes_raw()
    n_box = (lens.astype(np.int64) - 8) // 24                       # bincode Vec<Bbox>: u64 count, 24 bytes per box
    windows = np.arange(len(lens))
    if int((20 * n_box + 16).sum()) > DUMP_BYTES:
        order = np.random.default_rng(0).permutation(len(lens))
        windows = np.sort(order[np.cumsum(20 * n_box[order] + 16) <= DUMP_BYTES])
    boxes = []
    for i in windows:
        o, k = int(offs[i]), int(n_box[i])
        assert int(blob[o: o + 8].view("<u8")[0]) == k
        boxes.append(blob[o + 8: o + 8 + 24 * k].reshape(k, 24)[:, :20].copy().view("<f4"))   # drop the 4 None tags
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "boxes.npy"), np.concatenate(boxes) if boxes else np.zeros((0, 5), np.float32))
    np.save(os.path.join(out_dir, "boxes_per_window.npy"), n_box[windows].astype(np.float64))
    np.save(os.path.join(out_dir, "windows.npy"), windows.astype(np.float64))


def positive_int(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError("must be at least 1")
    return v


# ------------------------------------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=20, help="timed steps of the device-resident and of each end-to-end loop")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cova_b200", choices=["cova_b200", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--streams", type=int, default=0, help="chains per GPU (default: the config's)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-packed", action="store_true", help="skip the packed-input end-to-end leg")
    ap.add_argument("--chunks", type=int, default=1, help="chunks per batch inside the library (1 = whole-batch kernels)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the boxes of the last timed device-resident step (rank 0) as DIR/*.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "cova_b200" else args.warmup
    h_mb, w_mb, cfg_streams, head_bias, cfg_desc = CONFIGS[args.config]
    args.streams = args.streams or cfg_streams

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    from cova_b200 import weights
    w = weights.random_weights(0, head_bias=head_bias)
    workload = (f"{args.config}: {cfg_desc}, {args.streams} chains x {FRAMES_PER_STREAM} frames "
                f"(64-window batch per chain) per GPU")

    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the CUDA path's boxes; the reference arm keeps none")
        if rank != 0:
            return
        # exactly --steps timed steps after --warmup untimed ones; the per-step sample is sized so that the whole run takes
        # about two minutes of CPU time whatever K and W are
        steps, warmup = max(1, args.steps), max(0, args.warmup)
        cb, ms, _ = time_cpu(w, steps, warmup, h_mb, w_mb, args.streams, target_s=min(6.0, max(0.4, 110.0 / (steps + warmup))), one_core=False)
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload, "note": "CPU path = oracle port (the Rust/GStreamer/TensorRT reference cannot be built here); "
                       "each step is a bounded sample of the workload"},
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: cova_b200 has no CPU fallback (use --impl reference for the CPU path)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from cova_b200 import _lib, shard, synth
    # several ranks on one box: each keeps its pinned frame / box buffers on its GPU's NUMA node (at N = 1 the CPU
    # baseline leg wants every core, and there is no neighbour to share the inter-socket link with)
    numa = shard.bind_rank_to_gpu(local_rank) if world > 1 else None
    from cova_b200.elements import BlobPipeline

    n_streams, fps = args.streams, FRAMES_PER_STREAM
    # stream-sharded: rank r owns chains r, r+world, ... of the global set (weak scaling: n_streams per GPU)
    frames_np = synth.tiled_streams(n_streams, fps, h_mb, w_mb, config_idx=1 + rank)
    # page-locked host frames from the library's own allocator (cova_host_alloc): the library links the CUDA
    # runtime statically, and memory pinned by torch's runtime instance is not seen as pinned by it
    from cova_b200.elements import PinnedBuffer
    AHEAD = 3                                                       # batches submitted ahead of the one being collected
    pins = [PinnedBuffer(frames_np.shape) for _ in range(AHEAD + 1)]
    for i, pb in enumerate(pins):
        pb.array[...] = np.roll(frames_np, i, axis=0)
    pinned = pins[0]
    pipe = BlobPipeline(w_mb, h_mb, weights.to_blob(w), n_streams, fps, cc_threshold=1, device=local_rank,
                        impl=_lib.IMPL_TCGEN05, n_chunks=args.chunks)
    # a real (non-default) stream, shared by torch's events and the library's kernels
    stream = torch.cuda.Stream(device=local_rank)
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    pipe.set_stream(stream.cuda_stream)
    n_windows = pipe.windows_for(n_streams, fps)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing: frames already in HBM
    dev_frames = torch.from_numpy(frames_np).cuda()
    pipe.load_frames(dev_frames.data_ptr(), n_streams, fps)
    for _ in range(args.warmup):
        pipe.run()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = pipe.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(stream)
    for _ in range(args.steps):
        pipe.run()
    ev1.record(stream)
    barrier()
    ms_total = ev0.elapsed_time(ev1)
    launches = pipe.launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(pipe, args.dump_outputs)
    t = torch.tensor([ms_total], device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_region = float(t.item())
    ms_step = ms_region / args.steps
    value = n_windows * world / (ms_step * 1e-3)

    # ---- per-kernel durations, live, CUDA events on the launching stream
    pipe.set_profiling(True)
    acc = {}
    for _ in range(5):
        pipe.run()
        pipe.sync()
        for k, v in pipe.last_timings().items():
            acc.setdefault(k, []).append(v)
    pipe.set_profiling(False)
    kms = {k: float(np.mean(v)) for k, v in acc.items()}

    # ---- end to end: pinned host frames -> boxes on the host, through the public streaming call.  Every step copies
    # its own frames host->device and its boxes device->host inside the timed region; up to four batches are in flight
    # (submit k+3, then collect k), so the copies of one batch overlap the kernels of another and the loop is bound by
    # the slower of PCIe and the kernels, not by one batch's H2D + kernels + D2H latency.
    host_frames = [pb.array for pb in pins]
    pipe.process(host_frames[0], raw=True)
    for hf in host_frames:                                          # warm all four batch slots
        pipe.submit(hf)
    for _ in host_frames:
        pipe.collect(raw=True)
    barrier()
    e2e_steps = args.steps              # as many steps as the device-resident measurement: the pipeline fill is amortised alike
    t0 = time.perf_counter()
    for k in range(min(AHEAD, e2e_steps)):
        pipe.submit(host_frames[k % len(host_frames)])
    d2h = 0
    for k in range(e2e_steps):
        if k + AHEAD < e2e_steps:
            pipe.submit(host_frames[(k + AHEAD) % len(host_frames)])
        blob, offs, lens = pipe.collect(raw=True)
        d2h = pipe.last_blob_len + 16 * n_windows + 16
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps          # wall clock around host-visible completion
    t = torch.tensor([e2e_ms], device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = n_windows * world / (float(t.item()) * 1e-3)

    # ---- the same end-to-end loop through the 2-byte packed input path: the decoder's 4-byte quads are packed on the host
    # (cova_packer_pack, worker threads; INSIDE the timed region) and half the bytes cross PCIe.  Still starts from the
    # reference's own buffers in host memory and ends with the boxes on the host.
    e2e_packed = e2e_prepacked = None
    if not args.no_packed and w_mb % 2 == 0:
        from cova_b200.elements import FramePacker
        lens, offs, blob = lens.copy(), offs.copy(), blob[: int(pipe.last_blob_len)].copy()   # views into the first pipeline's pinned buffers
        del pipe, dev_frames                                        # free the first pipeline's activation buffers
        torch.cuda.empty_cache()
        n_pack = max(1, min(16, (os.cpu_count() or 1) // world))    # the ranks of a node share its cores
        packer = FramePacker(n_pack)
        ppins = [PinnedBuffer(frames_np.shape[:-1], np.uint16) for _ in range(AHEAD + 1)]
        pipe2 = BlobPipeline(w_mb, h_mb, weights.to_blob(w), n_streams, fps, cc_threshold=1, device=local_rank,
                             impl=_lib.IMPL_TCGEN05, n_chunks=args.chunks, packed_input=True)
        pipe2.set_stream(stream.cuda_stream)
        for i in range(len(ppins)):                                 # warm the packer, the four batch slots and the kernels
            packer.pack(host_frames[i], out=ppins[i].array)
            pipe2.submit(ppins[i].array)
        for _ in ppins:
            pipe2.collect(raw=True)
        t0 = time.perf_counter()
        for _ in range(3):
            packer.pack(host_frames[0], out=ppins[0].array)
        pack_ms = (time.perf_counter() - t0) * 1e3 / 3
        barrier()
        t0 = time.perf_counter()
        for k in range(min(AHEAD, e2e_steps)):
            packer.pack(host_frames[k % len(host_frames)], out=ppins[k % len(ppins)].array)
            pipe2.submit(ppins[k % len(ppins)].array)
        for k in range(e2e_steps):
            if k + AHEAD < e2e_steps:
                j = (k + AHEAD) % len(ppins)
                packer.pack(host_frames[j], out=ppins[j].array)
                pipe2.submit(ppins[j].array)
            pblob, poffs, plens = pipe2.collect(raw=True)
        torch.cuda.synchronize()
        p_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
        t = torch.tensor([p_ms], device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        # same boxes as the 4-byte path?  (the order of the windows inside the blob follows the CTAs' arrival order, so compare per window)
        same = bool(np.array_equal(plens, lens)) and all(
            pblob[int(poffs[i]): int(poffs[i] + plens[i])].tobytes() == blob[int(offs[i]): int(offs[i] + lens[i])].tobytes()
            for i in range(0, n_windows, max(1, n_windows // 256)))
        e2e_packed = {"value": n_windows * world / (float(t.item()) * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(ppins[0].array.nbytes),
                      "d2h_bytes_per_step": int(pipe2.last_blob_len + 16 * n_windows + 16), "pack_threads": n_pack,
                      "pack_ms_per_step": round(pack_ms, 3), "boxes_identical_to_quad_path": same}
        # and with frames that ARRIVE packed (a decoder writing the u16 itself: no packer in the loop) - what the format is
        # worth when the host does not have to touch the bytes a second time
        barrier()
        t0 = time.perf_counter()
        for k in range(min(AHEAD, e2e_steps)):
            pipe2.submit(ppins[k % len(ppins)].array)
        for k in range(e2e_steps):
            if k + AHEAD < e2e_steps:
                pipe2.submit(ppins[(k + AHEAD) % len(ppins)].array)
            pipe2.collect(raw=True)
        torch.cuda.synchronize()
        pp_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
        t = torch.tensor([pp_ms], device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_prepacked = {"value": n_windows * world / (float(t.item()) * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(ppins[0].array.nbytes),
                         "d2h_bytes_per_step": e2e_packed["d2h_bytes_per_step"],
                         "path": "packed16 frames already packed in pinned host memory (producer-side packing; NOT the reference's buffer format)"}

    # ---- the drop-in ELEMENT calls (one buffer per call, host memory in and out, as the GStreamer elements make them):
    # slow by construction - a host<->device round trip and a synchronisation per frame - and timed here so that the cost
    # of staying on the per-buffer interface is a number, not a guess
    shims = None
    if rank == 0:
        from cova_b200.elements import BboxCc, MetaPreprocess
        mp, cc = MetaPreprocess(w_mb * 16, h_mb * 16, T, 1, device=local_rank), BboxCc(w_mb, h_mb, 1, device=local_rank)
        one = frames_np[0]
        msk = (np.random.default_rng(0).random((h_mb, w_mb)) < 0.08).astype(np.uint8)
        for f in range(8):
            mp.transform(one[f % one.shape[0]]); cc.transform_ip(msk)
        n_el = 200
        t0 = time.perf_counter()
        for f in range(n_el):
            mp.transform(one[f % one.shape[0]])
        t_mp = (time.perf_counter() - t0) / n_el
        t0 = time.perf_counter()
        for f in range(n_el):
            cc.transform_ip(msk)
        t_cc = (time.perf_counter() - t0) / n_el
        shims = {"metapreprocess_transform_us": round(t_mp * 1e6, 1), "bboxcc_transform_ip_us": round(t_cc * 1e6, 1),
                 "note": "per buffer through the element interface (ctypes call included); the batch path above is the fast one"}
        mp.close(); cc.close()

    if rank == 0:
        pk = peaks()
        # Which tensor peak applies: MEASURED_PEAKS.json holds a burst figure (cuBLAS timed alone, clocks near maximum) and
        # a sustained one (seconds-long loop under the power cap).  The timed region here is steps x ms_step; below two
        # seconds the GPU has not settled at the power-capped clock, so the honest denominator is the BURST peak.  Both
        # fractions are reported for every tensor-bound stage.
        region_s = ms_region * 1e-3
        use_burst = region_s < 2.0
        t_peak = pk["tflops_burst"] if use_burst else pk["tflops"]
        nbox = float(((lens.astype(np.int64) - 8) // 24).mean())
        work, fl = kernel_work(h_mb, w_mb, nbox)
        lbytes = layer_bytes(h_mb, w_mb)
        traffic, traffic_file = {}, None
        for cand in (f"traffic_{'c2' if args.config == 'c5' else args.config}.json", "traffic.json"):
            tpath = os.path.join(ROOT, "profiles", cand)
            if os.path.exists(tpath):
                tj = json.load(open(tpath))
                if tj.get("windows_per_launch") == n_windows and tj.get("grid", [h_mb, w_mb]) == [h_mb, w_mb]:
                    traffic, traffic_file = tj["dram_bytes_per_launch"], cand
                    break
        stages = {}
        for name, bound, layer in KERNELS:
            ms = kms.get(name)
            if not ms:
                continue
            per_s = work[name] * n_windows / (ms * 1e-3)
            st = {"ms": round(ms, 4), "bound": bound, "layer": layer, "traffic": traffic.get(name)}
            if bound == "tensor":
                st.update(achieved=round(per_s / 1e12, 1), unit="TFLOP/s", peak=t_peak, frac=round(per_s / 1e12 / t_peak, 4),
                          frac_burst=round(per_s / 1e12 / pk["tflops_burst"], 4), frac_sustained=round(per_s / 1e12 / pk["tflops"], 4))
                # the same launch against the OTHER roof: algorithmic activation bytes at the measured copy bandwidth.  Where
                # hbm_frac > frac the layer's floor is its HBM time (enc2, dec2), the contraction notwithstanding.
                gbs = lbytes[layer] * n_windows / (ms * 1e-3) / 1e9
                st.update(hbm_achieved=round(gbs, 1), hbm_frac=round(gbs / pk["hbm_gbs"], 4),
                          binding="hbm" if gbs / pk["hbm_gbs"] > st["frac"] else "tensor")
            else:
                st.update(achieved=round(per_s / 1e9, 1), unit="GB/s", peak=pk["hbm_gbs"], frac=round(per_s / 1e9 / pk["hbm_gbs"], 4))
            stages[name] = st
        stages["ccl_bbox"]["boxes_per_frame"] = round(nbox, 2)
        blobnet_ms = sum(stages[n]["ms"] for n, _, layer in KERNELS if layer and n in stages)
        dom = max(stages, key=lambda k: stages[k]["ms"])
        # whole BlobNet two ways: ALGORITHMIC FLOPs (SURVEY 8d: no cross-window reuse, the first conv counted per window) and
        # EXECUTED FLOPs (the fused first block runs its conv once per FRAME: 67 frames serve 64 windows)
        alg = sum(fl.values())
        conv1 = work["tc_enc1_conv"]
        executed = alg - conv1 + conv1 * FRAMES_PER_STREAM / (FRAMES_PER_STREAM - T + 1) / T
        bn_tf = lambda f: f * n_windows / (blobnet_ms * 1e-3) / 1e12   # noqa: E731
        roof = {"bound": stages[dom]["bound"], "kernel": dom, "achieved": stages[dom]["achieved"], "peak": stages[dom]["peak"],
                "unit": stages[dom]["unit"], "frac": stages[dom]["frac"], "traffic": stages[dom]["traffic"],
                "ms_per_launch": stages[dom]["ms"], "share_of_step": round(stages[dom]["ms"] / ms_step, 3),
                "timed_region_s": round(region_s, 4),
                "peak_source": pk["source"] + ((" (BURST bf16: the timed region is shorter than 2 s)" if use_burst else
                                                " (sustained bf16: the timed region is 2 s or longer)") if stages[dom]["bound"] == "tensor"
                                               else " (STREAM-style copy)"),
                "traffic_source": f"profiles/{traffic_file} (ncu --set full of the same workload)" if stages[dom]["traffic"] else None,
                "whole_blobnet_frac": round(bn_tf(alg) / t_peak, 4),
                "whole_blobnet_frac_burst": round(bn_tf(alg) / pk["tflops_burst"], 4),
                "whole_blobnet_frac_sustained": round(bn_tf(alg) / pk["tflops"], 4),
                "whole_blobnet_executed_frac": round(bn_tf(executed) / t_peak, 4),
                "whole_step_frac": round(alg * n_windows / (ms_step * 1e-3) / 1e12 / t_peak, 4)}
        if "frac_burst" in stages[dom]:
            roof.update(frac_burst=stages[dom]["frac_burst"], frac_sustained=stages[dom]["frac_sustained"])
        # `e2e` = the faster of the two public end-to-end paths (both start from the decoder's 4-byte quads in pinned host
        # memory and end with the bincode boxes on the host); `e2e_paths` has both
        e2e_quads = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(pinned.array.size), "d2h_bytes_per_step": int(d2h),
                     "path": "quads: cova_pipeline_submit_host / collect_host on the decoder's 4-byte macroblock quads"}
        e2e_paths = {"quads": e2e_quads}
        e2e_best = e2e_quads
        if e2e_packed:
            e2e_packed["path"] = "packed16: cova_packer_pack (host threads, inside the timed region) + submit_host / collect_host on 2-byte macroblocks"
            e2e_paths["packed16"] = e2e_packed
            e2e_paths["packed16_prepacked"] = e2e_prepacked
            if e2e_packed["value"] > e2e_quads["value"]:
                e2e_best = {k: e2e_packed[k] for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step", "path")}
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            cpu, _, _ = time_cpu(w, 2, 1, h_mb, w_mb, n_streams, target_s=6.0)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16",
            "data": "synthetic",
            "config": {"workload": workload, "grid_mb": [h_mb, w_mb], "windows_per_gpu_per_step": n_windows, "timestep": T, "gamma": 1,
                       "cc_threshold": 1,
                       "l2": "per-step working set (activations, GBs) far exceeds the 126 MB L2; no flush needed",
                       "parallelism": f"chain-sharded x{world}, no collective",
                       "weights": f"random-init (seed 0, head bias {head_bias}), reference architecture",
                       "host_numa": numa},
            "e2e": e2e_best, "e2e_paths": e2e_paths,
            "gpu_launches": int(launches), "roofline": roof, "stages": stages, "element_shims": shims, "cpu_baseline": cpu, "clocks": clocks,
        }
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
