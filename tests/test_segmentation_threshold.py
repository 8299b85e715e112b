"""nvinfer's segmentation-threshold as a property of the batch pipeline: settable per pipeline
(cova_pipeline_set_segmentation_threshold) and per stream (cova_pipeline_set_stream_property_f32), applied in the BlobNet
head's epilogue as `logit > tau`, tau = (float)log((double)t / (1 - (double)t)) (include/cova_b200.h).

The relation tests read back the fp32 logits (COVA_FLAG_KEEP_LOGITS) and check every mask pixel against the tau of its
window's stream; the oracle tests compare with the fp32 reference network; the per-stream tests compare every stream byte
for byte with a one-stream pipeline whose pipeline value is that stream's."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

from cova_b200 import _lib, synth, weights
from cova_b200.elements import BlobPipeline, FramePacker
from oracle import blobnet_ref, c_oracle, metapreprocess_ref as mpr

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
H, W, T = 45, 80, 4
SEG = "segmentation-threshold"
TS = (0.02, 0.3, 0.7, 0.98)
# grid widths whose head layer (dec3 + head, MODE_HEAD) runs each of its tile configurations: every (config, ring depth)
# any supported width selects (test_head_widths_reach_every_head_plan)
HEAD_WIDTHS = (16, 353, 609)
MAX_WIDTH = 736
LOGIT_REL_TOL = 5e-3          # tests/test_gpu_parity.py: device logits against the fp32 oracle, synthetic streams
CLIP_LOGIT_REL_TOL = 2e-2     # tests/test_demo_fixture.py: the same on the real clip
CS = dict(cont=True, staggered=True)


def tau(t):
    """The library's cut-off on the logit for segmentation-threshold t (an fp32 value)."""
    t = float(np.float32(t))
    return np.float32(math.log(t / (1.0 - t)))


def mask_at(logit, t):
    """The oracle's mask (blobnet_ref.mask_from_logits) at segmentation-threshold t."""
    return (logit > tau(t)).astype(np.uint8)


# ----------------------------------------------------------------------------------------------------------- CPU
def _header():
    with open(os.path.join(ROOT, "include", "cova_b200.h")) as f:
        return " ".join(f.read().split())


def test_symbols_are_declared_and_bound():
    hdr = _header()
    assert "int cova_pipeline_set_segmentation_threshold(cova_pipeline *p, float t);" in hdr
    assert ("int cova_pipeline_set_stream_property_f32(cova_pipeline *p, const uint32_t *stream_ids, uint32_t n, "
            "const char *name, float value);") in hdr
    assert ("int cova_pipeline_get_stream_property_f32(const cova_pipeline *p, uint32_t stream_id, const char *name, "
            "float *value);") in hdr
    assert "tau = (float)log((double)t / (1.0 - (double)t))" in hdr
    u32, vp, cp, f32 = ctypes.c_uint32, ctypes.c_void_p, ctypes.c_char_p, ctypes.c_float
    assert _lib.SIGNATURES["cova_pipeline_set_segmentation_threshold"] == (ctypes.c_int, [vp, f32])
    assert _lib.SIGNATURES["cova_pipeline_set_stream_property_f32"] == (ctypes.c_int, [vp, vp, u32, cp, f32])
    assert _lib.SIGNATURES["cova_pipeline_get_stream_property_f32"] == (ctypes.c_int, [vp, u32, cp, ctypes.POINTER(f32)])
    lib = _lib.load()
    for name in ("cova_pipeline_set_segmentation_threshold", "cova_pipeline_set_stream_property_f32",
                 "cova_pipeline_get_stream_property_f32"):
        assert getattr(lib, name).argtypes == _lib.SIGNATURES[name][1]
    v = ctypes.c_float(7.0)
    assert lib.cova_pipeline_set_segmentation_threshold(None, 0.4) == _lib.E_INVAL
    assert lib.cova_pipeline_set_stream_property_f32(None, None, 0, SEG.encode(), 0.4) == _lib.E_INVAL
    assert lib.cova_pipeline_get_stream_property_f32(None, 0, SEG.encode(), ctypes.byref(v)) == _lib.E_INVAL
    assert v.value == 7.0


C_SNIPPET = r"""
#include <stddef.h>
#include <stdint.h>
#include <stdio.h>
#include "cova_b200.h"

int main(void) {
    const uint32_t ids[2] = {0, 3};
    float v = 0.f;
    int a = cova_pipeline_set_segmentation_threshold(NULL, 0.4f);
    int b = cova_pipeline_set_stream_property_f32(NULL, ids, 2, "segmentation-threshold", 0.3f);
    int c = cova_pipeline_get_stream_property_f32(NULL, 1, "segmentation-threshold", &v);
    if (a != COVA_E_INVAL || b != COVA_E_INVAL || c != COVA_E_INVAL || v != 0.f) return 1;
    printf("segmentation threshold ok\n");
    return 0;
}
"""


def test_plain_c_calls_the_declarations(tmp_path):
    _lib.load()                                                      # raises if the library has not been built
    src, exe = tmp_path / "seg.c", str(tmp_path / "seg")
    src.write_text(C_SNIPPET)
    lib_dir = os.path.join(ROOT, "cova_b200")
    r = subprocess.run(["gcc", "-std=c11", "-Wall", "-Wextra", "-Werror", "-I" + os.path.join(ROOT, "include"), str(src),
                        "-L" + lib_dir, "-lcova_b200", "-Wl,-rpath," + lib_dir, "-o", exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "segmentation threshold ok" in r.stdout, (r.stdout, r.stderr)


def test_tau_is_zero_at_one_half_and_strictly_increasing():
    assert tau(0.5) == 0.0 and not np.signbit(tau(0.5))
    ts = np.linspace(1e-3, 1 - 1e-3, 4001, dtype=np.float32)
    taus = np.array([tau(t) for t in ts])
    assert (np.diff(taus) > 0).all()
    assert np.isfinite([tau(np.nextafter(np.float32(0), np.float32(1))), tau(np.nextafter(np.float32(1), np.float32(0)))]).all()


def test_mask_at_one_half_is_the_oracle_mask():
    rng = np.random.default_rng(0)
    z = np.concatenate([rng.normal(0, 3, 4000), [0.0, -0.0, 1e-30, -1e-30]]).astype(np.float32)
    assert (mask_at(z, 0.5) == blobnet_ref.mask_from_logits(z)).all()
    assert (mask_at(z, 0.3) >= mask_at(z, 0.5)).all() and (mask_at(z, 0.3) != mask_at(z, 0.5)).any()


def head_plan(w):
    p = _lib.blobnet_plan(w, 16, 64)[7]
    return p["family"], p["config"], p["n_stage"]


def test_head_widths_reach_every_head_plan():
    every = {head_plan(w) for w in range(16, MAX_WIDTH + 1)}
    assert {head_plan(w) for w in HEAD_WIDTHS} == every and len(every) == len(HEAD_WIDTHS)


# ----------------------------------------------------------------------------------------------------------- GPU
def _wts():
    return weights.to_blob(weights.random_weights(0, head_bias=-1.0))


def pts_of(sid, lo, hi):
    return np.arange(lo, hi, dtype=np.uint64) + np.uint64(sid * 1_000_000)


def submit_ragged(p, frames, ids, pos, counts, **kw):
    fr = np.concatenate([frames[i, pos[i]: pos[i] + c] for i, c in zip(ids, counts)])
    pts = np.concatenate([pts_of(i, pos[i], pos[i] + c) for i, c in zip(ids, counts)])
    p.submit(fr, counts=list(counts), stream_ids=list(ids), pts=pts, **kw)
    for i, c in zip(ids, counts):
        pos[i] += c


def check_relation(mask, logits, taus):
    """Every pixel of window k: mask == (logit > taus[k])."""
    assert mask.shape == logits.shape and len(taus) == mask.shape[0]
    want = logits > np.asarray(taus, dtype=np.float32)[:, None, None]
    assert (mask == want).all(), np.argwhere(mask != want)[:5]


@pytest.mark.gpu
@pytest.mark.parametrize("w", HEAD_WIDTHS)
def test_mask_is_logit_above_tau_on_every_head_plan(w):
    """Pipeline values, then per-stream values mixed in one batch split into three chunks: mask == (logit > tau_w) for every
    pixel, on the tcgen05 head and on the validation head run through run_layer(7, SIMT)."""
    h, n_s, fps = 16, 6, 7
    frames = synth.synth_streams(n_s, fps, h, w, config_idx=200 + w)
    ids = list(range(n_s))
    p = BlobPipeline(w, h, _wts(), n_s, fps, keep_logits=True, n_chunks=3)
    fg = []
    for t in TS:
        p.set_property(SEG, t)
        p.submit(frames, stream_ids=ids)
        p.collect()
        mask, logits = p.read_mask(), p.read_logits()
        check_relation(mask, logits, [tau(t)] * mask.shape[0])
        fg.append(int(mask.sum()))
    assert fg[0] > fg[1] > fg[2] >= fg[3], fg
    mixed = [0.02, 0.3, None, 0.7, 0.98, 0.3]                           # None: follows the pipeline value, 0.5
    v = BlobPipeline(w, h, _wts(), n_s, fps, keep_logits=True, n_chunks=1, validation=True)
    for q in (p, v):
        q.set_property(SEG, 0.5)
        for s, t in enumerate(mixed):
            if t is not None:
                q.set_stream_property(SEG, t, [s])
    want = [np.float32(0.5 if t is None else t) for t in mixed]
    assert [p.get_stream_property(SEG, s) for s in ids] == want
    for q in (p, v):
        q.submit(frames, stream_ids=ids[::-1])                          # chain k is stream n_s - 1 - k
        _, wid, _ = q.collect(meta=True)
        taus = [tau(want[s]) for s in wid.tolist()]
        check_relation(q.read_mask(), q.read_logits(), taus)
    tc_logits = v.read_logits()
    v.run_layer(7, _lib.IMPL_SIMT)
    v.sync()
    simt_logits = v.read_logits()
    assert np.abs(simt_logits - tc_logits).max() <= LOGIT_REL_TOL * np.abs(simt_logits).max()
    check_relation(v.read_mask(), simt_logits, taus)
    v.set_property(SEG, 0.3)                                             # anonymous batch: the pipeline value only
    v.process(frames)
    v.run_layer(7, _lib.IMPL_SIMT)
    v.sync()
    check_relation(v.read_mask(), v.read_logits(), [tau(0.3)] * v.n_windows)


def _clip():
    d = np.load(os.path.join(HERE, "golden", "demo_1m_meta.npz"))
    return np.ascontiguousarray(np.moveaxis(d["planes"][:, 240:252], 0, -1))[None]   # straddles a GoP boundary


def _sigmoid32(z):
    z = z.astype(np.float32)
    return np.float32(1) / (np.float32(1) + np.exp(-z))


@pytest.mark.gpu
@pytest.mark.parametrize("source", ["synthetic", "clip"])
def test_masks_and_boxes_against_the_fp32_oracle(source):
    """720p: a mask pixel may differ from the oracle's fp32 sigmoid(z) > t only where the oracle logit is within the logit
    error bar of tau; the boxes are the C oracle's on the pipeline's own masks.  t = 0.05 makes the masks dense."""
    if source == "synthetic":
        frames, bar = synth.synth_streams(2, 9, H, W, config_idx=210), LOGIT_REL_TOL
    else:
        frames, bar = _clip(), CLIP_LOGIT_REL_TOL
    wts = weights.random_weights(0, head_bias=-1.0)
    p = BlobPipeline(W, H, weights.to_blob(wts), frames.shape[0], frames.shape[1], keep_logits=True, keep_stacked=True)
    stacked = np.concatenate([mpr.tensorise_stream(f, T, 1) for f in frames])
    ref = blobnet_ref.blobnet_forward(wts, mpr.stacked_to_nchw(stacked, T))
    scale = float(np.abs(ref).max())
    dens = {}
    for t in (0.05, 0.3, 0.5, 0.7, 0.95):
        p.set_property(SEG, t)
        boxes = p.process(frames)
        mask = p.read_mask()
        assert (p.read_stacked() == stacked).all()
        assert np.abs(p.read_logits() - ref).max() <= bar * scale
        off = mask != (_sigmoid32(ref) > np.float32(t))
        assert (np.abs(ref[off] - tau(t)) <= bar * scale).all(), (t, np.abs(ref[off] - tau(t)).max())
        assert boxes == c_oracle.bboxcc_batch(mask, 1), t
        dens[t] = float(mask.mean())
    assert dens[0.05] > 0.9 and dens[0.05] > dens[0.3] > dens[0.5] > dens[0.7] >= dens[0.95], dens


_REFS = {}


def reference(frames, t, gamma=1, cc=1, w=W, h=H, **kw):
    """One-stream pipeline with pipeline values (gamma, cc-threshold, segmentation-threshold t) over all of frames:
    (boxes, masks)."""
    n = frames.shape[0]
    key = (gamma, cc, w, h, tuple(sorted(kw.items())))
    if key not in _REFS or _REFS[key].max_fps < n:
        _REFS[key] = BlobPipeline(w, h, _wts(), 1, max(n, 32), gamma=gamma, cc_threshold=cc, **kw)
    p = _REFS[key]
    p.set_property(SEG, t)
    boxes = p.process(frames[None])
    return boxes, p.read_mask()


def per_stream(ids, wid, *arrays):
    return {s: [[a[k] for k in np.flatnonzero(wid == s)] for a in arrays] for s in ids}


MIX8 = [0.1, None, 0.3, 0.6, None, 0.8, 0.95, 0.04]                  # None: never set, follows the pipeline value


def set_mix(p, mix, pipeline_value):
    p.set_property(SEG, pipeline_value)
    for s, t in enumerate(mix):
        if t is not None:
            p.set_stream_property(SEG, t, [s])
    return [np.float32(pipeline_value if t is None else t) for t in mix]


@pytest.mark.gpu
@pytest.mark.parametrize("chunks", [1, 3])
def test_per_stream_mix_equals_one_stream_pipelines(chunks):
    """Eight streams, six with their own threshold and two never set: fresh, continued, staggered and ragged batches; every
    stream's boxes and masks equal a one-stream pipeline's with that pipeline value over the uncut stream."""
    frames = synth.synth_streams(8, 40, H, W, config_idx=220)
    p = BlobPipeline(W, H, _wts(), 8, 16, n_chunks=chunks)
    ts = set_mix(p, MIX8, 0.4)
    assert [p.get_stream_property(SEG, s) for s in range(8)] == ts
    schedule = [(list(range(8)), [9] * 8, {}),                                       # fresh, lock-step
                (list(range(8)), [6] * 8, dict(cont=True)),                          # continued, lock-step
                ([5, 0, 3, 7, 1], [4, 11, 2, 9, 13], CS),                            # staggered, ragged
                ([2, 4, 6, 1, 0, 7, 3, 5], [12, 5, 9, 3, 7, 10, 1, 8], CS)]
    pos, got = [0] * 8, [[[], []] for _ in range(8)]
    for ids, counts, kw in schedule:
        submit_ragged(p, frames, ids, pos, counts, **kw)
        boxes, wid, _ = p.collect(meta=True)
        for s, (b, m) in per_stream(ids, wid, boxes, p.read_mask()).items():
            got[s][0] += b
            got[s][1] += m
    for s in range(8):
        rb, rm = reference(frames[s, : pos[s]], ts[s])
        assert got[s][0] == rb, s
        assert len(got[s][1]) == len(rm) and (np.stack(got[s][1]) == rm).all(), s
    assert sum(m.sum() for m in got[7][1]) > sum(m.sum() for m in got[0][1]) > sum(m.sum() for m in got[6][1])


@pytest.mark.gpu
def test_one_batch_mixing_gamma_cc_threshold_and_segmentation_threshold():
    props = [(1, 1, 0.5), (2, 30, 0.2), (3, 1, 0.85), (2, 5, None), (1, 30, 0.1)]  # (gamma, cc-threshold, seg)
    frames = synth.synth_streams(5, 14, H, W, config_idx=230)
    p = BlobPipeline(W, H, _wts(), 5, 14, gamma=1, cc_threshold=1, n_chunks=2)
    p.set_property(SEG, 0.6)
    for s, (g, c, t) in enumerate(props):
        p.set_stream_property("gamma", g, [s])
        p.set_stream_property("cc-threshold", c, [s])
        if t is not None:
            p.set_stream_property(SEG, t, [s])
    ids = [4, 2, 0, 1, 3]
    p.submit(frames[ids], stream_ids=ids)                               # chain k carries stream ids[k]
    boxes, wid, _ = p.collect(meta=True)
    got = per_stream(range(5), wid, boxes, p.read_mask())
    for s, (g, c, t) in enumerate(props):
        rb, rm = reference(frames[s], 0.6 if t is None else t, gamma=g, cc=c)
        assert got[s][0] == rb and (np.stack(got[s][1]) == rm).all(), s


@pytest.mark.gpu
@pytest.mark.parametrize("cluster", [False, True])
@pytest.mark.parametrize("mode", ["quads", "packed", "sparse"])
def test_defaults_are_byte_identical(mode, cluster):
    """An untouched pipeline, one with the pipeline value and every stream value set to 0.5, and one whose pipeline value is
    0.3 with every stream set to 0.5 (the per-window table, all zero): the same boxes, masks and logits, byte for byte."""
    frames = synth.synth_streams(4, 30, H, W, config_idx=240)
    pk = FramePacker(2)
    src = frames if mode == "quads" else pk.pack(frames)
    kw = dict(ccl_cluster=True, ccl_bands=3) if cluster else {}
    pipes = [BlobPipeline(W, H, _wts(), 4, 16, keep_logits=True, packed_input=mode != "quads", n_chunks=2, **kw)
             for _ in range(3)]
    pipes[1].set_property(SEG, 0.5)
    pipes[1].set_stream_property(SEG, 0.5)
    pipes[2].set_property(SEG, 0.3)
    pipes[2].set_stream_property(SEG, 0.5)
    assert [pipes[2].get_stream_property(SEG, s) for s in range(4)] == [0.5] * 4
    schedule = [([0, 1, 2, 3], [10, 7, 12, 4], {}), ([3, 1, 0, 2], [9, 12, 3, 8], CS)]
    runs = []
    for p in pipes:
        pos, res = [0] * 4, []
        for ids, counts, fl in schedule:
            if mode == "sparse":
                fr = np.concatenate([frames[i, pos[i]: pos[i] + c] for i, c in zip(ids, counts)])
                p.submit(pk.pack_sparse(fr, counts=counts), stream_ids=ids, cont=bool(fl), staggered=bool(fl))
                for i, c in zip(ids, counts):
                    pos[i] += c
            else:
                submit_ragged(p, src, ids, pos, counts, **fl)
            boxes, wid, _ = p.collect(meta=True)
            res.append((boxes, wid.copy(), p.read_mask(), p.read_logits()))
        runs.append(res)
    for other in runs[1:]:
        for a, b in zip(runs[0], other):
            assert a[0] == b[0] and len(a[0]) > 0
            for x, y in zip(a[1:], b[1:]):
                assert x.shape == y.shape and x.tobytes() == y.tobytes()
    if mode != "sparse":                                                 # the anonymous path of the 0.5 pipeline
        outs = []
        for p in pipes[:2]:
            outs.append((p.process(src[:, :9]), p.read_mask(), p.read_logits()))
        assert outs[0][0] == outs[1][0]
        assert outs[0][1].tobytes() == outs[1][1].tobytes() and outs[0][2].tobytes() == outs[1][2].tobytes()


@pytest.mark.gpu
def test_four_batches_in_flight_and_slot_reuse():
    """Seven batches of one shape, four in flight, values changed between the submits: every batch uses the values at its
    submit.  Batches 4-6 reuse the slots of batches 0-2 with the same chain shape; batch 5's slot held a table that differs
    from its own in the thresholds only."""
    frames = synth.synth_streams(4, 56, H, W, config_idx=250)
    p = BlobPipeline(W, H, _wts(), 4, 8)
    # before batch b: (pipeline value or None, {stream: value})
    changes = [(0.5, {}), (None, {1: 0.2}), (0.3, {}), (None, {1: 0.3}), (None, {0: 0.9}), (None, {1: 0.2, 2: 0.6}),
               (0.7, {3: 0.1})]
    effective, got = [], []
    for b, (pv, sv) in enumerate(changes):
        if pv is not None:
            p.set_property(SEG, pv)
        for s, t in sv.items():
            p.set_stream_property(SEG, t, [s])
        effective.append([p.get_stream_property(SEG, s) for s in range(4)])
        if b >= 4:                                                       # four in flight: the oldest frees its slot
            boxes, wid, _ = p.collect(meta=True)
            got.append((boxes, wid.copy()))
        p.submit(np.ascontiguousarray(frames[:, 8 * b: 8 * b + 8]), stream_ids=[0, 1, 2, 3])
    for _ in range(4):
        boxes, wid, _ = p.collect(meta=True)
        got.append((boxes, wid.copy()))
    assert effective[3] == [np.float32(0.3)] * 4
    assert effective[6] == [np.float32(v) for v in (0.9, 0.2, 0.6, 0.1)]
    for b, (boxes, wid) in enumerate(got):
        for s, (bs,) in per_stream(range(4), wid, boxes).items():
            assert bs == reference(frames[s, 8 * b: 8 * b + 8], effective[b][s])[0], (b, s)


@pytest.mark.gpu
def test_anonymous_and_stage_wise_calls_use_the_pipeline_value():
    frames = synth.synth_streams(4, 24, H, W, config_idx=260)
    fr = np.ascontiguousarray(frames[:, :8])
    p = BlobPipeline(W, H, _wts(), 4, 8, keep_logits=True)
    plain = BlobPipeline(W, H, _wts(), 4, 8, keep_logits=True)
    p.set_stream_property(SEG, 0.9)                                      # every stream
    p.set_property(SEG, 0.2)
    plain.set_property(SEG, 0.2)
    assert [p.get_stream_property(SEG, s) for s in range(4)] == [np.float32(0.9)] * 4
    want = plain.process(fr)
    want_mask = plain.read_mask()
    assert p.process(fr) == want and (p.read_mask() == want_mask).all()   # process_host
    check_relation(p.read_mask(), p.read_logits(), [tau(0.2)] * p.n_windows)
    p.submit(fr)                                                         # submit_host
    assert p.collect() == want and (p.read_mask() == want_mask).all()
    p.load_frames(fr)                                                    # stage-wise
    p.run()
    assert p.fetch_boxes() == want and (p.read_mask() == want_mask).all()
    p.load_frames(fr)                                                    # read when blobnet is called
    p.tensorise()
    p.set_property(SEG, 0.7)
    p.blobnet()
    p.ccl()
    boxes = p.fetch_boxes()
    mask = p.read_mask()
    check_relation(mask, p.read_logits(), [tau(0.7)] * p.n_windows)
    assert boxes == c_oracle.bboxcc_batch(mask, 1) and mask.sum() < want_mask.sum()
    # the pipeline value moves the streams never set and leaves the others; values survive reset_streams
    q = BlobPipeline(W, H, _wts(), 4, 16)
    q.set_stream_property(SEG, 0.8, [3, 1])
    q.set_property(SEG, 0.35)
    eff = [np.float32(v) for v in (0.35, 0.8, 0.35, 0.8)]
    assert [q.get_stream_property(SEG, s) for s in range(4)] == eff
    pos = [0] * 4
    submit_ragged(q, frames, [0, 1, 2, 3], pos, [8, 8, 8, 8])
    q.collect()
    q.reset_streams([1])
    q.reset_streams()
    assert [q.get_stream_property(SEG, s) for s in range(4)] == eff
    pos = [0] * 4
    submit_ragged(q, frames, [2, 1, 0, 3], pos, [12, 12, 12, 12], **CS)   # every stream restarts: a fresh window
    boxes, wid, _ = q.collect(meta=True)
    for s, (bs, ms) in per_stream(range(4), wid, boxes, q.read_mask()).items():
        rb, rm = reference(frames[s, :12], eff[s])
        assert bs == rb and (np.stack(ms) == rm).all(), s


@pytest.mark.gpu
@pytest.mark.parametrize("res", ["1080p", "4K", "8K"])
def test_mixed_batch_at_large_grids(res):
    w, h, kw = {"1080p": (120, 68, {}), "4K": (240, 135, {}), "8K": (480, 270, dict(ccl_cluster=True))}[res]
    mix = [0.15, None, 0.7]
    frames = synth.synth_streams(3, 6, h, w, config_idx=270)
    p = BlobPipeline(w, h, _wts(), 3, 6, n_chunks=2, **kw)
    ts = set_mix(p, mix, 0.45)
    ids = [2, 0, 1]
    p.submit(frames[ids], stream_ids=ids)                               # chain k carries stream ids[k]
    boxes, wid, _ = p.collect(meta=True)
    got = per_stream(range(3), wid, boxes, p.read_mask())
    dens = []
    for s in range(3):
        rb, rm = reference(frames[s], ts[s], w=w, h=h, **kw)
        assert got[s][0] == rb and (np.stack(got[s][1]) == rm).all(), s
        dens.append(float(rm.mean()))
    assert dens[0] > dens[1] > dens[2], dens


def _ptr(a):
    return ctypes.c_void_p(a.ctypes.data)


@pytest.mark.gpu
def test_refusals_change_nothing():
    p = BlobPipeline(W, H, _wts(), 4, 8, gamma=2, cc_threshold=1)
    L, h = p._L, p._h
    p.set_stream_property(SEG, 0.25, [2])
    p.set_property(SEG, 0.4)

    def state():
        return ([(p.get_stream_property("gamma", s), p.get_stream_property("cc-threshold", s),
                  p.get_stream_property(SEG, s)) for s in range(4)])

    before = state()
    assert [x[2] for x in before] == [np.float32(v) for v in (0.4, 0.4, 0.25, 0.4)]
    bad = np.array([0, 4], dtype=np.uint32)
    ok = np.array([1, 3], dtype=np.uint32)
    seg = SEG.encode()
    f, u = ctypes.c_float(9.0), ctypes.c_uint32(99)
    refused = [lambda: L.cova_pipeline_set_segmentation_threshold(None, 0.3)]
    for t in (0.0, 1.0, -0.5, 1.5, float("nan"), float("inf"), float("-inf")):
        refused += [lambda t=t: L.cova_pipeline_set_segmentation_threshold(h, t),
                    lambda t=t: L.cova_pipeline_set_stream_property_f32(h, _ptr(ok), 2, seg, t),
                    lambda t=t: L.cova_pipeline_set_stream_property_f32(h, None, 0, seg, t)]
    refused += [
        lambda: L.cova_pipeline_set_stream_property_f32(None, None, 0, seg, 0.3),          # null handle
        lambda: L.cova_pipeline_set_stream_property_f32(h, None, 0, None, 0.3),            # null name
        lambda: L.cova_pipeline_set_stream_property_f32(h, None, 0, b"segmentation_threshold", 0.3),
        lambda: L.cova_pipeline_set_stream_property_f32(h, _ptr(bad), 2, seg, 0.3),       # an id >= max_streams last
        lambda: L.cova_pipeline_set_stream_property_f32(h, _ptr(ok), 2, b"gamma", 4.0),    # u32 names
        lambda: L.cova_pipeline_set_stream_property_f32(h, _ptr(ok), 2, b"cc-threshold", 4.0),
        lambda: L.cova_pipeline_set_stream_property(h, _ptr(ok), 2, seg, 0),               # the float name, u32 call
        lambda: L.cova_pipeline_set_stream_property(h, None, 0, seg, 1),
        lambda: L.cova_pipeline_get_stream_property_f32(h, 4, seg, ctypes.byref(f)),
        lambda: L.cova_pipeline_get_stream_property_f32(h, 0, b"gamma", ctypes.byref(f)),
        lambda: L.cova_pipeline_get_stream_property_f32(h, 0, b"cc-threshold", ctypes.byref(f)),
        lambda: L.cova_pipeline_get_stream_property_f32(h, 0, None, ctypes.byref(f)),
        lambda: L.cova_pipeline_get_stream_property_f32(h, 0, seg, None),
        lambda: L.cova_pipeline_get_stream_property_f32(None, 0, seg, ctypes.byref(f)),
        lambda: L.cova_pipeline_get_stream_property(h, 0, seg, ctypes.byref(u)),
    ]
    for k, call in enumerate(refused):
        assert call() == _lib.E_INVAL, k
        assert state() == before, k
    assert f.value == 9.0 and u.value == 99
    with pytest.raises(KeyError):
        p.set_property("segmentation_threshold", 0.3)
    # the edges of the open interval are accepted
    lo, hi = np.nextafter(np.float32(0), np.float32(1)), np.nextafter(np.float32(1), np.float32(0))
    p.set_stream_property(SEG, float(lo), [0])
    p.set_stream_property(SEG, float(hi), [1])
    assert p.get_stream_property(SEG, 0) == lo and p.get_stream_property(SEG, 1) == hi
