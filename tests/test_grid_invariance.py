"""Every hot-path kernel gives the same bytes at any grid size (cova_pipeline_set_sm_limit).

The tcgen05 BlobNet layers are persistent kernels: CTA c walks tile groups c, c + n_cta, ... and carries state from one
group to the next (operand-ring slot and parity, TMEM accumulator slot, epilogue warp group, dec0 / dec1 half-tile
barriers); enc1_fused_kernel cuts its work into whole items and one evenly split sequence of left-over steps (plan_enc1),
differently for every CTA count.  Which CTA runs a tile decides nothing about its arithmetic, so every output must be
byte-identical whatever grid the kernel is launched with.  At the SM count of a B200 and the small shapes the layer
tests can afford, most CTAs run a single tile group and none of that carried state is exercised; capped at one SM, each
CTA walks every group of its layer.

The CPU tests check the plans at capped SM counts; the GPU tests compare outputs byte for byte across caps (layer by
layer on identical input, block 1's partition on fresh, staggered and ragged batches, and the whole path), and check
every window of the benchmark's shapes against the fp32 validation kernels with a per-window bar."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from cova_b200 import _lib, synth, weights
from cova_b200.elements import BlobPipeline, FramePacker
from test_tile_plans import CASES, DEBUGS, FLOOR, NAMES, _last_groups, _layer_output, _plan, _positions, _weights

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
B200_SMS = 148
CAPS = (1, 2, 3, 7, 37)                       # SM caps of the layer tests; 0 = the device's count
# the layer-by-layer cases: every reachable plan (CASES), whole-tile dec0 / dec1 accumulators (debug bit 6) at three ring
# depths, and the grids of the existing layer-by-layer parity tests
LAYER_CASES = CASES + [(200, 17, 64), (400, 17, 64), (700, 17, 64), (80, 45, 0), (120, 68, 0), (47, 33, 0)]
ENC1_GRID = (120, 68)                         # 9 tile pairs per frame: odd, so that 2 and 5 CTAs leave items over
ENC1_CHAINS = 17                              # 153 items: whole items and left-over items at 2, 5 and 148 CTAs
PER_WINDOW_TOL = 4e-3                         # the activation bar of tests/test_gpu_parity.py, applied per window
# tile groups every CTA of every layer walks at one SM: more than the 8 TMEM accumulator slots a layer has at most, so
# that slots, epilogue warp groups and ring stages (at most 4 deep) all come round again
MIN_GROUPS = 9


def _nsplit(layer):
    return 2 if layer == 4 else 1             # dec0 runs its two N-halves on separate CTAs


def groups_per_cta(layer, plan):
    """The most tile groups (block 1: frame steps) one CTA of the plan walks."""
    per_half = plan["ctas"] // _nsplit(layer)
    return -(-plan["n_groups"] // per_half)


def _always_whole(layer, w, h, plan):
    """A window's positions fill whole tile groups of the layer (enc2 at 700 macroblocks: 4224 = 11 x 384): no window
    count leaves its last group partial."""
    s, tn = _positions(layer, h, w, 1)
    return (s * tn) % (plan["tps"] * plan["tile"]) == 0


def layer_windows(w, h, dbg):
    """The smallest window count at which the last tile group of every layer is partial (where a window count can make
    it so) and, capped at one SM, every CTA of every layer walks at least MIN_GROUPS groups."""
    for n in range(2, 1025):
        plans = _plan(w, h, n, dbg)
        if not all(partial or _always_whole(layer, w, h, plans[layer])
                   for layer, (partial, _) in _last_groups(h, w, n, plans).items()):
            continue
        if all(groups_per_cta(layer, p) >= MIN_GROUPS for layer, p in enumerate(_plan(w, h, n, dbg, 1))):
            return n
    raise AssertionError((w, h, dbg))


def _header():
    with open(os.path.join(ROOT, "include", "cova_b200.h")) as f:
        return " ".join(f.read().split())


# ----------------------------------------------------------------------------------------------------------------- CPU
def test_cases_are_the_tile_plan_cases():
    assert CASES == [(16, 17, 0), (736, 17, 0), (16, 16, 4), (121, 16, 4), (253, 18, 4), (309, 16, 4), (509, 19, 4),
                     (625, 16, 4), (16, 20, 8), (161, 20, 8), (253, 17, 8), (599, 18, 8), (625, 16, 8)]
    assert DEBUGS == (0, 4, 8)


def test_symbol_is_declared_exported_and_bound():
    hdr = _header()
    assert "int cova_pipeline_set_sm_limit(cova_pipeline *p, int n_sms);" in hdr
    assert hdr.index("int cova_pipeline_set_sm_limit(") > hdr.index("int cova_pipeline_set_debug(")
    assert "Results do not depend on it" in hdr
    assert _lib.SIGNATURES["cova_pipeline_set_sm_limit"] == (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int])
    lib = _lib.load()
    assert lib.cova_pipeline_set_sm_limit.argtypes == [ctypes.c_void_p, ctypes.c_int]
    for n in (0, 1, -1):
        assert lib.cova_pipeline_set_sm_limit(None, n) == _lib.E_INVAL
    assert b"null handle" in lib.cova_last_error()
    assert hasattr(BlobPipeline, "set_sm_limit")


C_SNIPPET = r"""
#include <stddef.h>
#include <stdio.h>
#include "cova_b200.h"

int main(void) {
    if (cova_pipeline_set_sm_limit(NULL, 1) != COVA_E_INVAL || cova_pipeline_set_sm_limit(NULL, 0) != COVA_E_INVAL) return 1;
    printf("sm limit ok\n");
    return 0;
}
"""


def test_plain_c_calls_the_declaration(tmp_path):
    _lib.load()                                                      # raises if the library has not been built
    src, exe = tmp_path / "sm_limit.c", str(tmp_path / "sm_limit")
    src.write_text(C_SNIPPET)
    lib_dir = os.path.join(ROOT, "cova_b200")
    r = subprocess.run(["gcc", "-std=c11", "-Wall", "-Wextra", "-Werror", "-I" + os.path.join(ROOT, "include"), str(src),
                        "-L" + lib_dir, "-lcova_b200", "-Wl,-rpath," + lib_dir, "-o", exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "sm limit ok" in r.stdout, (r.stdout, r.stderr)


@pytest.mark.parametrize("w,h", sorted({(w, h) for w, h, _ in CASES}))
def test_plans_at_capped_sm_counts(w, h):
    """At 1, 2, 3, 7 and 37 SMs every layer keeps the (family, config, tps, n_stage) it picks at 148; only the CTA count
    changes, to min(n_sms / nsplit, n_groups) * nsplit (block 1: min(n_sms, frame steps))."""
    for dbg in DEBUGS:
        try:
            _plan(w, h, 64, dbg)
        except _lib.CovaError as e:                                   # a debug route without a plan at this width
            assert e.code == _lib.E_UNSUPPORTED
            with pytest.raises(_lib.CovaError):
                _plan(w, h, 64, dbg, 1)
            continue
        for n in sorted({layer_windows(w, h, dbg), 3, 4096}):
            base = _plan(w, h, n, dbg)
            for n_sms in CAPS:
                capped = _plan(w, h, n, dbg, n_sms)
                for layer, (a, b) in enumerate(zip(base, capped)):
                    key = ("family", "config", "tps", "tile", "n_stage", "n_groups")
                    assert {k: a[k] for k in key} == {k: b[k] for k in key}, (w, h, dbg, n, n_sms, NAMES[layer])
                    if layer == 0:
                        want = max(1, min(n_sms, b["n_groups"]))
                    else:
                        want = max(1, min(n_sms // _nsplit(layer), b["n_groups"])) * _nsplit(layer)
                    assert b["ctas"] == want, (w, h, dbg, n, n_sms, NAMES[layer])


@pytest.mark.parametrize("w,h,dbg", LAYER_CASES)
def test_one_sm_walks_every_layer_through_several_groups(w, h, dbg):
    """The coverage claim of the layer-by-layer GPU test: at its window count every layer's last group is partial and, at
    one SM, every layer has more tile groups than CTAs - each CTA carries its ring, TMEM and barrier state across groups."""
    n = layer_windows(w, h, dbg)
    for layer, p in enumerate(_plan(w, h, n, dbg, 1)):
        assert p["n_groups"] > p["ctas"] // _nsplit(layer) and groups_per_cta(layer, p) >= MIN_GROUPS, (NAMES[layer], p)


def enc1_items(w, h, n_chains):
    s, _ = _positions(0, h, w, 1)
    return n_chains * -(-s // 256)                                   # (chain, tile pair) items of block 1


def test_enc1_partition_has_whole_and_left_over_items():
    """The block-1 GPU test's shape: at 2, 5 and 148 CTAs the partition hands out whole items and cuts left-over ones."""
    n_items = enc1_items(*ENC1_GRID, ENC1_CHAINS)
    assert n_items == 153
    for ctas in (2, 5, B200_SMS):
        assert n_items >= ctas and n_items % ctas, ctas


# ----------------------------------------------------------------------------------------------------------------- GPU
def _n_sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _same(a, b, what):
    assert a.shape == b.shape and a.dtype == b.dtype, what
    if a.tobytes() != b.tobytes():
        bad = np.argwhere(a != b)
        raise AssertionError(f"{what}: {len(bad)} elements differ, first at {bad[:4].tolist()}, windows {np.unique(bad[:, 0])[:16].tolist()}")


def _outputs(p, layer):
    """Everything a tcgen05 layer writes: its output and, for blocks 1-3, the decoder input that holds its t = 0 skip."""
    out = [_layer_output(p, layer)]
    if layer < 3:
        out.append(p.read_activation(7 - layer))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,dbg", LAYER_CASES)
def test_layers_are_byte_identical_at_every_grid(w, h, dbg):
    """Each tcgen05 layer on identical input at the device's SM count and capped at 1, 2, 3, 7 and 37 SMs: outputs
    byte-identical, and the plan launched is the one cova_blobnet_plan gives for that count.  Before every launch the
    validation kernel rewrites the layer's outputs, so a tile a capped grid leaves unwritten cannot keep the value of the
    launch before it."""
    n_dev, n = _n_sms(), layer_windows(w, h, dbg)
    frames = synth.synth_streams(1, n + 3, h, w, config_idx=w % 7)
    p = BlobPipeline(w, h, weights.to_blob(_weights(w + h + dbg)), 1, n + 3, impl=_lib.IMPL_SIMT, keep_logits=True)
    p.set_debug(dbg)
    p.load_frames(frames)
    p.run()
    for layer in range(8):
        ref = None
        for cap in (0,) + CAPS:
            p.run_layer(layer, _lib.IMPL_SIMT)
            p.set_sm_limit(cap)
            p.run_layer(layer, _lib.IMPL_TCGEN05)
            assert p.last_plan()[layer] == _plan(w, h, n, dbg, cap or n_dev)[layer], (NAMES[layer], cap)
            got = _outputs(p, layer)
            if ref is None:
                ref = got
            else:
                for k, (a, b) in enumerate(zip(ref, got)):
                    _same(b, a, f"{NAMES[layer]} output {k} at {cap} SMs")
        p.set_sm_limit(0)                                              # the next layer reads the default grid's output


def _submit(p, frames, ids, pos, counts, **kw):
    fr = np.concatenate([frames[i, pos[i]: pos[i] + c] for i, c in zip(ids, counts)])
    pts = np.concatenate([np.arange(pos[i], pos[i] + c, dtype=np.uint64) + np.uint64(i * 1_000_000)
                          for i, c in zip(ids, counts)])
    p.submit(fr, counts=list(counts), stream_ids=list(ids), pts=pts, **kw)
    for i, c in zip(ids, counts):
        pos[i] += c


@pytest.mark.gpu
@pytest.mark.parametrize("gamma", [1, 2, 3])
def test_enc1_partition_is_grid_independent(gamma):
    """Block 1 at 1, 2 and 5 CTAs against the device's count, on a fresh lock-step batch (equal chain ends), a continued
    staggered ragged batch and a fresh ragged batch (the chain-table path of the partition): X1, the decoder input with
    block 1's t = 0 skip, and the logits byte-identical.  Each pipeline's previous batch differs, so a step a partition
    skips keeps a different value."""
    w, h = ENC1_GRID
    ns = ENC1_CHAINS
    frames = synth.synth_streams(ns, 40, h, w, config_idx=gamma)
    blob = weights.to_blob(_weights(11 + gamma))
    pipes = {cap: BlobPipeline(w, h, blob, ns, 16, gamma=gamma, keep_logits=True) for cap in (0, 1, 2, 5)}
    for cap, p in pipes.items():
        p.set_sm_limit(cap)
    rng = np.random.default_rng(gamma)
    ids = list(range(ns))
    schedule = [([9] * ns, {}),                                                   # fresh, equal ends
                (list(rng.integers(1, 13, ns)), dict(cont=True, staggered=True)),  # continued, staggered, ragged
                (list(rng.integers(4, 14, ns)), {})]                               # fresh, ragged
    pos = {cap: [0] * ns for cap in pipes}
    for b, (counts, kw) in enumerate(schedule):
        outs = {}
        for cap, p in pipes.items():
            _submit(p, frames, ids, pos[cap], counts, **kw)
            boxes, wid, pts = p.collect(meta=True)
            assert p.n_windows > 0
            outs[cap] = [p.read_activation(1), p.read_activation(7), p.read_logits(), wid.copy(), pts.copy()]
            assert p.last_plan()[0]["ctas"] == (cap or _n_sms()), cap
        for cap in (1, 2, 5):
            for k, (a, c) in enumerate(zip(outs[0], outs[cap])):
                _same(c, a, f"batch {b} output {k} at {cap} CTAs")


WH = (80, 45)


def _whole_path_pipes(caps, **kw):
    """One pipeline per cap: six streams of at most 16 frames per batch on the 720p grid."""
    w, h = WH
    blob = weights.to_blob(_weights(5, head_bias=-0.5))
    pipes = []
    for cap in caps:
        p = BlobPipeline(w, h, blob, 6, 16, keep_logits=True, **kw)
        p.set_sm_limit(cap)
        pipes.append(p)
    return pipes


def _compare_runs(runs, what):
    for cap, run in runs[1:]:
        assert len(run) == len(runs[0][1])
        for b, (x, y) in enumerate(zip(runs[0][1], run)):
            assert x[0] == y[0], f"{what}: boxes of batch {b} at {cap} SMs"
            for k, (a, c) in enumerate(zip(x[1:], y[1:])):
                _same(c, a, f"{what}: batch {b} array {k} at {cap} SMs")


@pytest.mark.gpu
def test_whole_path_is_byte_identical_at_every_grid():
    """process(), a continued schedule of staggered ragged batches over three chunks with per-stream gamma, cc-threshold and
    segmentation-threshold and four batches in flight, packed16 and sparse input: boxes, masks, logits, window stream ids
    and PTS at 1 and 7 SMs equal the device's count, byte for byte."""
    w, h = WH
    frames = synth.synth_streams(6, 80, h, w, config_idx=31)
    caps = (0, 1, 7)

    runs = []                                                          # process(): fresh chains, three chunks
    for cap, p in zip(caps, _whole_path_pipes(caps, n_chunks=3)):
        boxes = p.process(np.ascontiguousarray(frames[:, :16]))
        runs.append((cap, [(boxes, p.read_mask(), p.read_logits())]))
        assert p.last_plan()[1]["ctas"] == min(cap or _n_sms(), p.last_plan()[1]["n_groups"])
    _compare_runs(runs, "process")

    props = [(1, 1, 0.5), (2, 30, 0.2), (3, 1, 0.85), (2, 5, None), (1, 30, 0.1), (3, 2, 0.6)]   # gamma, cc, seg
    schedule = [([0, 1, 2, 3, 4, 5], [9, 9, 9, 9, 9, 9]), ([3, 1, 0, 5, 2, 4], [4, 11, 2, 9, 13, 6]),
                ([5, 0, 3, 2, 4, 1], [12, 5, 9, 3, 7, 10]), ([1, 2, 4, 0, 3, 5], [1, 8, 13, 6, 2, 12]),
                ([2, 5, 1, 4, 0, 3], [7, 3, 10, 12, 5, 1]), ([0, 3, 4, 1, 5, 2], [13, 9, 1, 4, 11, 7])]
    runs = []
    for cap, p in zip(caps, _whole_path_pipes(caps, n_chunks=3)):
        p.set_property("segmentation-threshold", 0.4)
        for s, (g, c, t) in enumerate(props):
            p.set_stream_property("gamma", g, [s])
            p.set_stream_property("cc-threshold", c, [s])
            if t is not None:
                p.set_stream_property("segmentation-threshold", t, [s])
        pos, res = [0] * 6, []
        for b, (ids, counts) in enumerate(schedule):
            if b >= 4:                                                 # four in flight: the oldest frees its slot
                boxes, wid, pts = p.collect(meta=True)
                res.append((boxes, wid.copy(), pts.copy()))
            _submit(p, frames, ids, pos, counts, cont=b > 0, staggered=b > 0)
        for _ in range(4):
            boxes, wid, pts = p.collect(meta=True)
            res.append((boxes, wid.copy(), pts.copy()))
        res.append(([], p.read_mask(), p.read_logits()))             # the last batch's masks and logits
        runs.append((cap, res))
    assert sum(len(r[0]) for r in runs[0][1]) > 100
    _compare_runs(runs, "in flight")

    pk = FramePacker(2)
    for mode in ("packed", "sparse"):
        runs = []
        for cap, p in zip(caps, _whole_path_pipes(caps, packed_input=True, n_chunks=2)):
            pos, res = [0] * 6, []
            for b, (ids, counts) in enumerate(schedule[:3]):
                if mode == "sparse":
                    fr = np.concatenate([frames[i, pos[i]: pos[i] + c] for i, c in zip(ids, counts)])
                    p.submit(pk.pack_sparse(fr, counts=counts), stream_ids=ids, cont=b > 0, staggered=b > 0)
                    for i, c in zip(ids, counts):
                        pos[i] += c
                else:
                    _submit(p, pk.pack(frames), ids, pos, counts, cont=b > 0, staggered=b > 0)
                boxes, wid, pts = p.collect(meta=True)
                res.append((boxes, wid.copy(), pts.copy(), p.read_mask(), p.read_logits()))
            runs.append((cap, res))
        _compare_runs(runs, mode)


@pytest.mark.gpu
def test_cap_changes_between_batches_on_reused_slots():
    """Seven synchronous batches (slots 0-3, then reused) on one pipeline whose cap moves between them - 1, 7, the
    device's, 3, ... - against a pipeline at the device's count: the same boxes, masks, logits, ids and PTS."""
    w, h = WH
    frames = synth.synth_streams(6, 80, h, w, config_idx=41)
    ref, moved = _whole_path_pipes((0, 0), n_chunks=2)
    caps = [1, 7, 0, 3, 37, 1, 2]
    pos = {id(p): [0] * 6 for p in (ref, moved)}
    for b, cap in enumerate(caps):
        moved.set_sm_limit(cap)
        ids = list(np.random.default_rng(b).permutation(6))
        counts = [int(c) for c in np.random.default_rng(100 + b).integers(1, 12, 6)]
        outs = []
        for p in (ref, moved):
            _submit(p, frames, ids, pos[id(p)], counts, cont=b > 0, staggered=b > 0)
            boxes, wid, pts = p.collect(meta=True)
            outs.append((boxes, wid.copy(), pts.copy(), p.read_mask(), p.read_logits()))
        assert moved.last_plan()[3]["ctas"] == min(cap or _n_sms(), ref.last_plan()[3]["n_groups"])
        assert outs[0][0] == outs[1][0], b
        for k, (a, c) in enumerate(zip(outs[0][1:], outs[1][1:])):
            _same(c, a, f"batch {b} array {k} at {cap} SMs")


@pytest.mark.gpu
def test_refusals_change_nothing():
    """A negative cap, one above the device's count, a null handle and a call while a batch is in flight are refused with
    COVA_E_INVAL; the pipeline then launches the grids of its last accepted cap and gives the same results."""
    w, h = WH
    n_dev = _n_sms()
    frames = synth.synth_streams(2, 12, h, w, config_idx=51)
    ref, p = _whole_path_pipes((0, 7))
    L = _lib.load()
    want = ref.process(frames)
    for bad in (-1, n_dev + 1, 1 << 30):
        assert L.cova_pipeline_set_sm_limit(p._h, bad) == _lib.E_INVAL
    assert L.cova_pipeline_set_sm_limit(None, 1) == _lib.E_INVAL
    assert p.process(frames) == want and (p.read_mask() == ref.read_mask()).all()
    assert p.last_plan()[1]["ctas"] == 7
    p.submit(frames)
    assert L.cova_pipeline_set_sm_limit(p._h, 1) == _lib.E_INVAL
    assert b"in flight" in L.cova_last_error()
    assert p.collect() == want and p.last_plan()[1]["ctas"] == 7
    p.set_sm_limit(n_dev)                                              # the device's count itself is accepted
    assert p.process(frames) == want and p.last_plan() == ref.last_plan()


def _per_window(got, ref):
    """Per window: max |got - ref| over the window's largest |ref|, with the fp16 floor (tests/test_tile_plans.py)."""
    n = ref.shape[0]
    err = np.abs(got.reshape(n, -1).astype(np.float64) - ref.reshape(n, -1)).max(1)
    bar = PER_WINDOW_TOL * np.abs(ref.reshape(n, -1)).max(1) + FLOOR
    return err / bar


@pytest.mark.gpu
def test_every_window_of_a_bench_chunk_layer_by_layer():
    """One chunk of the c2 workload (16 chains x 67 frames of 720p, 1024 windows, hundreds to thousands of tile groups per
    layer): each tcgen05 layer against the fp32 validation kernel on identical input, every window within 4e-3 of its own
    largest |ref| - an error confined to a quiet window cannot hide behind the batch's largest value."""
    w, h, n_chains, fps = 80, 45, 16, 67
    frames = synth.tiled_streams(n_chains, fps, h, w, config_idx=1)
    p = BlobPipeline(w, h, weights.to_blob(_weights(0)), n_chains, fps, impl=_lib.IMPL_SIMT, keep_logits=True)
    p.load_frames(frames)
    assert p.n_windows == 1024
    p.run()
    simt = {layer: _layer_output(p, layer) for layer in range(8)}
    plans = _plan(w, h, 1024, 0, _n_sms())
    for layer in range(8):
        p.run_layer(layer, _lib.IMPL_TCGEN05)
        if layer:                                                       # block 1's steps count the chunk's 16 x 67 frames
            assert p.last_plan()[layer] == plans[layer]
        ratio = _per_window(_layer_output(p, layer), simt[layer])
        worst = int(ratio.argmax())
        assert ratio.max() <= 1.0, (NAMES[layer], plans[layer], "window", worst, float(ratio[worst]))
        p.run_layer(layer, _lib.IMPL_SIMT)                              # the next layer's input: the validation kernel's
    assert max(groups_per_cta(layer, pl) for layer, pl in enumerate(plans)) > 10


@pytest.mark.gpu
def test_every_window_of_the_c5_batch_logits():
    """The c5 batch per GPU (128 chains x 67 frames of 720p, 8192 windows in 8 chunks): tcgen05 logits of every window
    within 4e-3 of that window's largest |logit| of the validation pipeline; a mask pixel differs only where the
    reference logit lies within that bar of the threshold."""
    w, h, n_chains, fps = 80, 45, 128, 67
    frames = synth.tiled_streams(n_chains, fps, h, w, config_idx=1)
    blob = weights.to_blob(_weights(0))
    out = []
    for impl in (_lib.IMPL_TCGEN05, _lib.IMPL_SIMT):
        p = BlobPipeline(w, h, blob, n_chains, fps, impl=impl, keep_logits=True)
        p.process(frames, raw=True)
        assert p.n_windows == 8192
        out.append((p.read_logits(), p.read_mask()))
        p.close()
    (got, got_mask), (ref, ref_mask) = out
    ratio = _per_window(got, ref)
    assert ratio.max() <= 1.0, (int(ratio.argmax()), float(ratio.max()))
    bar = (PER_WINDOW_TOL * np.abs(ref.reshape(len(ref), -1)).max(1) + FLOOR)[:, None, None]
    flipped = got_mask != ref_mask
    assert (np.abs(ref) <= bar)[flipped].all()
    assert (ref_mask == (ref > 0)).all()
