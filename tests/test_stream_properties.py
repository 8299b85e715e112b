"""Per-stream element properties of a batch pipeline (cova_pipeline_set_stream_property / _get_stream_property): every
stream of a pipeline has its own `gamma` (metapreprocess) and `cc-threshold` (bboxcc), settable between batches like the
properties of the elements each stream replaces.

Every stream is compared byte for byte with a reference: a one-stream pipeline created with the stream's gamma, the
element restatement (MetaPreprocessRef) with its gamma changed at the same frame boundaries, or the bboxcc element with
the stream's threshold on the very masks the batch produced."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from cova_b200 import _lib, synth, weights
from cova_b200.elements import FLOW_OK, BboxCc, BlobPipeline, FramePacker
from oracle import metapreprocess_ref as mpr

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
H, W, T = 45, 80, 4
ACT_REL_TOL = 4e-3
CS = dict(cont=True, staggered=True)


# ----------------------------------------------------------------------------------------------------------- CPU
def _header():
    with open(os.path.join(ROOT, "include", "cova_b200.h")) as f:
        return " ".join(f.read().split())


def test_stream_property_symbols_are_declared_and_bound():
    hdr = _header()
    assert ("int cova_pipeline_set_stream_property(cova_pipeline *p, const uint32_t *stream_ids, uint32_t n, const char *name, "
            "uint32_t value);") in hdr
    assert ("int cova_pipeline_get_stream_property(const cova_pipeline *p, uint32_t stream_id, const char *name, "
            "uint32_t *value);") in hdr
    u32, vp, cp = ctypes.c_uint32, ctypes.c_void_p, ctypes.c_char_p
    assert _lib.SIGNATURES["cova_pipeline_set_stream_property"] == (ctypes.c_int, [vp, vp, u32, cp, u32])
    assert _lib.SIGNATURES["cova_pipeline_get_stream_property"] == (ctypes.c_int, [vp, u32, cp, ctypes.POINTER(u32)])
    lib = _lib.load()
    for name in ("cova_pipeline_set_stream_property", "cova_pipeline_get_stream_property"):
        assert getattr(lib, name).argtypes == _lib.SIGNATURES[name][1]
    v = ctypes.c_uint32(7)
    assert lib.cova_pipeline_set_stream_property(None, None, 0, b"gamma", 2) == _lib.E_INVAL
    assert lib.cova_pipeline_get_stream_property(None, 0, b"gamma", ctypes.byref(v)) == _lib.E_INVAL
    assert v.value == 7


C_SNIPPET = r"""
#include <stddef.h>
#include <stdint.h>
#include <stdio.h>
#include "cova_b200.h"

int main(void) {
    const uint32_t ids[2] = {0, 3};
    uint32_t v = 0;
    int a = cova_pipeline_set_stream_property(NULL, ids, 2, "gamma", 2);
    int b = cova_pipeline_set_stream_property(NULL, NULL, 0, "cc-threshold", 30);
    int c = cova_pipeline_get_stream_property(NULL, 1, "cc-threshold", &v);
    if (a != COVA_E_INVAL || b != COVA_E_INVAL || c != COVA_E_INVAL || v != 0) return 1;
    printf("stream properties ok\n");
    return 0;
}
"""


def test_plain_c_calls_both_declarations(tmp_path):
    _lib.load()                                                      # raises if the library has not been built
    src, exe = tmp_path / "props.c", str(tmp_path / "props")
    src.write_text(C_SNIPPET)
    lib_dir = os.path.join(ROOT, "cova_b200")
    r = subprocess.run(["gcc", "-std=c11", "-Wall", "-Wextra", "-Werror", "-I" + os.path.join(ROOT, "include"), str(src),
                        "-L" + lib_dir, "-lcova_b200", "-Wl,-rpath," + lib_dir, "-o", exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "stream properties ok" in r.stdout, (r.stdout, r.stderr)


def element_windows(frames, gamma0, changes=None):
    """MetaPreprocessRef over one stream, with el.gamma = changes[f] set before frame f: [(newest frame, stacked)]."""
    el = mpr.MetaPreprocessRef(W * 16, H * 16, T, gamma0)
    out = []
    for f in range(frames.shape[0]):
        if changes and f in changes:
            el.gamma = changes[f]
        rc, o = el.transform(frames[f])
        if rc == FLOW_OK:
            out.append((f, np.frombuffer(o, dtype=np.uint8).reshape(T * H, W, 4)))
    return out


def test_element_windows_restates_the_closed_form():
    fr = np.zeros((40, H, W, 4), dtype=np.uint8)
    fr[:, 0, 0, 0] = np.arange(40)
    for g in (1, 2, 3, 5):
        assert [f for f, _ in element_windows(fr, g)] == mpr.window_newest_indices(40, T, g)
    # gamma 5 -> 2 at frame 10, in the middle of a countdown: the change shows after the window at frame 13
    assert [f for f, _ in element_windows(fr, 5, {10: 2})] == [3, 8, 13, 15, 17, 19, 21, 23, 25, 27, 29, 31, 33, 35, 37, 39]


# ----------------------------------------------------------------------------------------------------------- GPU
def _wts():
    return weights.to_blob(weights.random_weights(0, head_bias=-1.0))


_REFS = {}


def reference(frames, gamma, mode="quads"):
    """A one-stream pipeline created with `gamma`, over all of `frames`: (boxes, masks, stacked or None, newest indices)."""
    n = frames.shape[0]
    key = (gamma, mode)
    if key not in _REFS or _REFS[key].max_fps < n:
        _REFS[key] = BlobPipeline(W, H, _wts(), 1, max(n, 64), gamma=gamma, keep_stacked=mode == "quads",
                                  packed_input=mode != "quads")
    p = _REFS[key]
    boxes = p.process(frames[None])
    return boxes, p.read_mask(), p.read_stacked() if mode == "quads" else None, mpr.window_newest_indices(n, T, gamma)


def pts_of(sid, lo, hi):
    return np.arange(lo, hi, dtype=np.uint64) + np.uint64(sid * 1_000_000)


def per_stream(ids, wid, *arrays):
    """{stream id: [its windows of every array]} of one collected batch, in window order."""
    return {s: [[a[k] for k in np.flatnonzero(wid == s)] for a in arrays] for s in ids}


def submit_ragged(p, frames, ids, pos, counts, **kw):
    fr = np.concatenate([frames[i, pos[i]: pos[i] + c] for i, c in zip(ids, counts)])
    pts = np.concatenate([pts_of(i, pos[i], pos[i] + c) for i, c in zip(ids, counts)])
    p.submit(fr, counts=list(counts), stream_ids=list(ids), pts=pts, **kw)
    for i, c in zip(ids, counts):
        pos[i] += c


@pytest.mark.gpu
@pytest.mark.parametrize("chunks", [1, 3])
@pytest.mark.parametrize("ragged", [False, True])
def test_fresh_batch_mixing_gammas(ragged, chunks):
    """Eight fresh streams of gammas 1, 2, 3, 5 (twice) in one batch: each equals a one-stream pipeline created with its
    gamma - boxes, masks, stacked windows, window stream ids and PTS."""
    gammas = [1, 2, 3, 5, 5, 3, 2, 1]
    counts = [16, 9, 16, 13, 4, 16, 7, 11] if ragged else [16] * 8
    frames = synth.synth_streams(8, 16, H, W, config_idx=110)
    p = BlobPipeline(W, H, _wts(), 8, 16, gamma=1, keep_stacked=True, n_chunks=chunks)
    for g in set(gammas):
        p.set_stream_property("gamma", g, [s for s in range(8) if gammas[s] == g])
    assert [p.get_stream_property("gamma", s) for s in range(8)] == gammas
    if ragged:
        submit_ragged(p, frames, range(8), [0] * 8, counts)
    else:
        p.submit(frames, stream_ids=list(range(8)), pts=np.stack([pts_of(s, 0, 16) for s in range(8)]))
    boxes, wid, wpts = p.collect(meta=True)
    got = per_stream(range(8), wid, boxes, p.read_mask(), p.read_stacked(), wpts)
    assert (np.diff(wid.astype(np.int64)) >= 0).all()                                  # stream-major
    for s in range(8):
        rb, rm, rs, newest = reference(frames[s, : counts[s]], gammas[s])
        b, m, st, pt = got[s]
        assert b == rb, s
        assert len(m) == len(rm) and (len(m) == 0 or ((np.stack(m) == rm).all() and (np.stack(st) == rs).all())), s
        assert [int(v) for v in pt] == [int(v) for v in pts_of(s, 0, counts[s])[newest]], s
    assert p.windows_for(8, 16) == 8 * len(mpr.window_newest_indices(16, T, 1))     # counts at the creation gamma


def check_stream(sid, frames, got, gamma0, changes):
    """got = [(boxes, mask, stacked, pts)] of one stream over its whole life: the element with its gamma changed at the same
    frame boundaries decides which frames emit and their stacked bytes; the gamma-1 run of the whole stream gives the masks
    and boxes of those newest frames."""
    want = element_windows(frames, gamma0, changes)
    newest = [f for f, _ in want]
    assert [g[3] for g in got] == [int(v) for v in pts_of(sid, 0, frames.shape[0])[newest]], sid
    for (f, st), g in zip(want, got):
        if g[2] is not None:
            assert (g[2] == st).all(), (sid, f)
    rb, rm, _, _ = reference(frames, 1)
    assert [g[0] for g in got] == [rb[f - (T - 1)] for f in newest], sid
    if got and got[0][1] is not None:
        assert (np.stack([g[1] for g in got]) == rm[[f - (T - 1) for f in newest]]).all(), sid
    return len(got)


@pytest.mark.gpu
@pytest.mark.parametrize("chunks", [1, 2])
def test_gamma_changed_mid_stream(chunks):
    """Four continued streams, staggered, gamma changed between batches: at seams where the countdown is 0 and where it is
    in the middle (the element keeps counting down the old gamma and takes the new one after its next window)."""
    n_ids, n_frames = 4, 64
    frames = synth.synth_streams(n_ids, n_frames, H, W, config_idx=120)
    p = BlobPipeline(W, H, _wts(), n_ids, 16, gamma=1, keep_stacked=True, n_chunks=chunks)
    # (ids, counts, {stream: gamma set before the batch})
    schedule = [([0, 1, 2, 3], [9, 6, 11, 5], {0: 5, 1: 2, 2: 3}),
                ([0, 1, 2, 3], [3, 7, 2, 8], {0: 2, 2: 1, 3: 4}),
                ([1, 3, 0], [9, 4, 6], {1: 5, 3: 1}),
                ([2, 0, 3, 1], [12, 5, 10, 1], {0: 3, 1: 1, 2: 5}),
                ([0, 1, 2, 3], [7, 12, 9, 11], {0: 1, 2: 2, 3: 3})]
    pos, changes, got = [0] * n_ids, [dict() for _ in range(n_ids)], [[] for _ in range(n_ids)]
    mid = 0
    ref_els = [mpr.MetaPreprocessRef(W * 16, H * 16, T, 1) for _ in range(n_ids)]   # countdowns at the seams
    for ids, counts, sets in schedule:
        for s, g in sets.items():
            p.set_stream_property("gamma", g, [s])
            changes[s][pos[s]] = g
            mid += ref_els[s].gamma_idx != 0
            ref_els[s].gamma = g
        for s, c in zip(ids, counts):
            for f in range(pos[s], pos[s] + c):
                ref_els[s].transform(frames[s, f])
        submit_ragged(p, frames, ids, pos, counts, **CS)
        boxes, wid, wpts = p.collect(meta=True)
        for s, (b, m, st, pt) in per_stream(ids, wid, boxes, p.read_mask(), p.read_stacked(), wpts).items():
            got[s] += list(zip(b, m, st, [int(v) for v in pt]))
    assert mid >= 2                                                      # some seams fall inside a countdown
    total = sum(check_stream(s, frames[s, : pos[s]], got[s], 1, changes[s]) for s in range(n_ids))
    assert total > 0


@pytest.mark.gpu
@pytest.mark.parametrize("cluster", [False, True])
def test_cc_threshold_per_stream(cluster):
    """Five streams of the same frames with thresholds 0, 1, 3, 30 and 2^31 + 5 (negative as i32): the boxes of every window
    are the bboxcc element's with that threshold on that window's mask.  cluster: the cluster CCL with three bands."""
    thr = [0, 1, 3, 30, 2**31 + 5]
    one = synth.synth_streams(1, 14, H, W, config_idx=130)
    frames = np.repeat(one, 5, axis=0)
    kw = dict(ccl_cluster=True, ccl_bands=3) if cluster else {}
    p = BlobPipeline(W, H, _wts(), 5, 14, cc_threshold=1, n_chunks=2, **kw)
    for s, t in enumerate(thr):
        p.set_stream_property("cc-threshold", t, [s])
    assert [p.get_stream_property("cc-threshold", s) for s in range(5)] == thr
    p.submit(frames, stream_ids=[4, 3, 2, 1, 0])                         # chain s is stream 4 - s
    boxes, wid, _ = p.collect(meta=True)
    masks = p.read_mask()
    els = {t: BboxCc(W, H, t) for t in thr}
    for k, s in enumerate(wid.tolist()):
        assert boxes[k] == els[thr[s]].transform_ip(masks[k]), (k, s)
    n = {s: [len(boxes[k]) for k in np.flatnonzero(wid == s)] for s in range(5)}
    assert n[0] == n[4] and sum(n[0]) > sum(n[3])                        # the thresholds do differ


@pytest.mark.gpu
def test_isolation_defaults_and_reset():
    """Streams never set give what a pipeline without stream properties gives; set_cc_threshold moves only them; properties
    survive reset_streams; get_stream_property reports the effective values."""
    frames = synth.synth_streams(4, 40, H, W, config_idx=140)
    plain = BlobPipeline(W, H, _wts(), 4, 16, gamma=2, cc_threshold=1, keep_stacked=True, n_chunks=2)
    p = BlobPipeline(W, H, _wts(), 4, 16, gamma=2, cc_threshold=1, keep_stacked=True, n_chunks=2)
    p.set_stream_property("gamma", 3, [1, 3])
    p.set_stream_property("cc-threshold", 30, [3, 1])
    assert [p.get_stream_property("gamma", s) for s in range(4)] == [2, 3, 2, 3]
    assert [p.get_stream_property("cc-threshold", s) for s in range(4)] == [1, 30, 1, 30]
    pos_a, pos_b = [0] * 4, [0] * 4
    schedule = [([0, 1, 2, 3], [8, 8, 8, 8], False), ([2, 1, 0], [5, 9, 6], True), ([3, 0, 2], [7, 3, 12], True)]
    for b, (ids, counts, cont) in enumerate(schedule):
        if b == 2:
            for q in (plain, p):
                q.set_property("cc-threshold", 7)
            assert [p.get_stream_property("cc-threshold", s) for s in range(4)] == [7, 30, 7, 30]
        res = []
        for q, pos in ((plain, pos_a), (p, pos_b)):
            submit_ragged(q, frames, ids, pos, counts, cont=cont, staggered=cont)
            boxes, wid, wpts = q.collect(meta=True)
            res.append(per_stream(ids, wid, boxes, q.read_mask(), q.read_stacked(), wpts))
        for s in ids:
            if s in (0, 2):                                              # never set: exactly the plain pipeline
                a, c = res[0][s], res[1][s]
                assert a[0] == c[0] and len(a[1]) == len(c[1]), (b, s)
                for x, y in zip(a[1:], c[1:]):
                    assert all((u == v).all() for u, v in zip(x, y)), (b, s)
            else:                                                        # own threshold on the masks it produced
                el = BboxCc(W, H, 30)
                assert res[1][s][0] == [el.transform_ip(m) for m in res[1][s][1]], (b, s)
    p.reset_streams([1])
    p.reset_streams()
    assert [p.get_stream_property("gamma", s) for s in range(4)] == [2, 3, 2, 3]
    assert [p.get_stream_property("cc-threshold", s) for s in range(4)] == [7, 30, 7, 30]
    submit_ragged(p, frames, [1, 0], [0, 0], [16, 16], cont=True, staggered=True)   # a reset stream starts afresh
    boxes, wid, wpts = p.collect(meta=True)
    got = per_stream([0, 1], wid, boxes, p.read_stacked(), wpts)
    for s, g in ((0, 2), (1, 3)):
        rb, _, rs, newest = reference(frames[s, :16], g)
        assert len(got[s][1]) == len(rs) and all((x == y).all() for x, y in zip(got[s][1], rs)), s
        assert [int(v) for v in got[s][2]] == [int(v) for v in pts_of(s, 0, 16)[newest]], s


@pytest.mark.gpu
def test_four_batches_in_flight_keep_their_values():
    """Four batches queued before the first collect, properties changed between the submits: every batch reflects the
    values at its submit, exactly as when each is collected before the next submit."""
    frames = synth.synth_streams(4, 60, H, W, config_idx=150)
    sets = [({0: 2, 2: 3}, {1: 30}), ({0: 1, 3: 5}, {0: 3, 1: 0}), ({1: 4}, {2: 2**31 + 5}), ({0: 3, 2: 1}, {1: 30, 3: 3})]
    batches = [([0, 1, 2, 3], [9, 5, 12, 7]), ([2, 0, 3], [4, 11, 6]), ([0, 1, 2, 3], [8, 8, 3, 10]), ([3, 1, 0], [12, 2, 5])]
    runs = []
    for in_flight in (False, True):
        p = BlobPipeline(W, H, _wts(), 4, 16, gamma=1, cc_threshold=1)
        pos, out = [0] * 4, []
        for (gs, ts), (ids, counts) in zip(sets, batches):
            for s, g in gs.items():
                p.set_stream_property("gamma", g, [s])
            for s, t in ts.items():
                p.set_stream_property("cc-threshold", t, [s])
            submit_ragged(p, frames, ids, pos, counts, **CS)
            if not in_flight:
                out.append(p.collect(meta=True))
        if in_flight:
            with pytest.raises(_lib.CovaError):
                p.set_stream_property("gamma", 0, [0])                       # refused, with four batches in flight
            out = [p.collect(meta=True) for _ in batches]
        runs.append([(b, w.copy(), t.copy()) for b, w, t in out])
    for a, b in zip(*runs):
        assert a[0] == b[0] and (a[1] == b[1]).all() and (a[2] == b[2]).all()
    # which frames emitted: the element with the same gamma changes
    pos, changes, got = [0] * 4, [dict() for _ in range(4)], [[] for _ in range(4)]
    for (gs, _), (ids, counts), (_, wid, wpts) in zip(sets, batches, runs[1]):
        for s, g in gs.items():
            changes[s][pos[s]] = g
        for s, c in zip(ids, counts):
            pos[s] += c
        for s in ids:
            got[s] += [int(v) for v in wpts[wid == s]]
    for s in range(4):
        want = [f for f, _ in element_windows(frames[s, : pos[s]], 1, changes[s])]
        assert got[s] == [int(v) for v in pts_of(s, 0, pos[s])[want]], s


@pytest.mark.gpu
def test_packed_and_sparse_inputs_equal_dense_with_mixed_properties():
    frames = synth.synth_streams(4, 30, H, W, config_idx=160)
    pk = FramePacker(2)
    packed = pk.pack(frames)
    schedule = [([0, 1, 2, 3], [10, 7, 12, 4]), ([3, 1, 0, 2], [9, 12, 3, 8])]
    runs = []
    for mode in ("quads", "packed", "sparse"):
        p = BlobPipeline(W, H, _wts(), 4, 16, gamma=1, cc_threshold=1, packed_input=mode != "quads", n_chunks=2)
        p.set_stream_property("gamma", 2, [1])
        p.set_stream_property("gamma", 3, [2, 3])
        p.set_stream_property("cc-threshold", 30, [0, 2])
        pos, res = [0] * 4, []
        for ids, counts in schedule:
            if mode == "sparse":
                fr = np.concatenate([frames[i, pos[i]: pos[i] + c] for i, c in zip(ids, counts)])
                pts = np.concatenate([pts_of(i, pos[i], pos[i] + c) for i, c in zip(ids, counts)])
                p.submit(pk.pack_sparse(fr, counts=counts), stream_ids=ids, pts=pts, **CS)
                for i, c in zip(ids, counts):
                    pos[i] += c
            else:
                submit_ragged(p, frames if mode == "quads" else packed, ids, pos, counts, **CS)
            boxes, wid, wpts = p.collect(meta=True)
            res.append((boxes, wid.copy(), wpts.copy(), p.read_mask()))
        runs.append(res)
    for other in runs[1:]:
        for a, b in zip(runs[0], other):
            assert a[0] == b[0] and len(a[0]) > 0
            for x, y in zip(a[1:], b[1:]):
                assert x.shape == y.shape and (x == y).all()


@pytest.mark.gpu
def test_block1_paths_agree_on_a_mixed_gamma_batch():
    """One staggered batch, one chunk, gammas 1, 2, 3, 5 with histories 0, 1, 3, 3 and different countdowns: the BlobNet
    input equals the element's windows, and the fused first block agrees with the fp32 validation kernel."""
    gammas, pre, counts = [1, 2, 3, 5], [0, 1, 5, 6], [11, 9, 12, 10]
    frames = synth.synth_streams(4, 20, H, W, config_idx=170)
    outs = []
    for impl in (_lib.IMPL_TCGEN05, _lib.IMPL_SIMT):
        p = BlobPipeline(W, H, _wts(), 4, 16, gamma=1, n_chunks=1, impl=impl)
        for s, g in enumerate(gammas):
            p.set_stream_property("gamma", g, [s])
            if pre[s]:
                p.submit(frames[s: s + 1, : pre[s]], stream_ids=[s], cont=True, staggered=True)
                p.collect()
        fr = np.concatenate([frames[s, pre[s]: pre[s] + counts[s]] for s in range(4)])
        p.submit(fr, counts=counts, stream_ids=[0, 1, 2, 3], cont=True, staggered=True)
        _, wid, _ = p.collect(meta=True)
        outs.append((wid, p.read_activation(0), p.read_activation(1)))
    want = []
    for s in range(4):
        st = mpr.tensorise_stream(frames[s, : pre[s] + counts[s]], T, gammas[s])
        k = int((outs[0][0] == s).sum())
        assert k == len(st) - len(mpr.tensorise_stream(frames[s, : pre[s]], T, gammas[s])) and k > 0
        want.append(st[len(st) - k:])
    x = np.clip(mpr.stacked_to_nchw(np.concatenate(want), T), 0, 6)
    for wid, a0, _ in outs:
        assert (wid == outs[0][0]).all()
        assert a0.shape == x.shape and (a0 == x).all()
    fused, simt = outs[0][2], outs[1][2]
    assert np.abs(fused - simt).max() <= ACT_REL_TOL * np.abs(simt).max()


@pytest.mark.gpu
def test_refusals_change_nothing():
    frames = synth.synth_streams(4, 20, H, W, config_idx=180)
    p = BlobPipeline(W, H, _wts(), 4, 16, gamma=2, cc_threshold=1)
    L, h = p._L, p._h
    ids = np.array([0, 4], dtype=np.uint32)
    ok = np.array([1, 2], dtype=np.uint32)
    v = ctypes.c_uint32(99)

    def state():
        return [(p.get_stream_property("gamma", s), p.get_stream_property("cc-threshold", s)) for s in range(4)]

    def nothing_in_flight():
        ln = ctypes.c_size_t()
        assert L.cova_pipeline_collect_host(h, None, 0, ctypes.byref(ln), None, None, None) == _lib.E_INVAL

    p.set_stream_property("cc-threshold", 3, [2])
    before = state()
    refused = [
        lambda: L.cova_pipeline_set_stream_property(h, None, 0, None, 3),                      # null name
        lambda: L.cova_pipeline_set_stream_property(h, None, 0, b"gama", 3),                   # unknown name
        lambda: L.cova_pipeline_set_stream_property(h, None, 0, b"cc_threshold", 3),
        lambda: L.cova_pipeline_set_stream_property(h, _lib_ptr(ok), 2, b"gamma", 0),          # gamma 0
        lambda: L.cova_pipeline_set_stream_property(h, _lib_ptr(ok), 2, b"gamma", 1),          # below the creation gamma
        lambda: L.cova_pipeline_set_stream_property(h, _lib_ptr(ids), 2, b"gamma", 3),         # an id >= max_streams ...
        lambda: L.cova_pipeline_set_stream_property(h, _lib_ptr(ids), 2, b"cc-threshold", 9),  # ... after a valid one
        lambda: L.cova_pipeline_get_stream_property(h, 4, b"gamma", ctypes.byref(v)),
        lambda: L.cova_pipeline_get_stream_property(h, 0, b"gama", ctypes.byref(v)),
        lambda: L.cova_pipeline_get_stream_property(h, 0, None, ctypes.byref(v)),
        lambda: L.cova_pipeline_get_stream_property(h, 0, b"gamma", None),
    ]
    for k, call in enumerate(refused):
        assert call() == _lib.E_INVAL, k
        assert state() == before, k
    assert v.value == 99
    nothing_in_flight()
    # the lock-step rule: streams 0 and 1 share history (3) and countdown (1) after 8 fresh frames at gamma 2 ...
    pos = [0] * 4
    submit_ragged(p, frames, [0, 1, 2, 3], pos, [8, 8, 8, 7])
    p.collect()
    assert [x[0] for x in state()] == [2, 2, 2, 2]
    p.set_stream_property("gamma", 4, [1])                                                     # ... but not the gamma
    with pytest.raises(_lib.CovaError):
        p.submit(frames[:2, 8:12], stream_ids=[0, 1], cont=True)
    nothing_in_flight()
    with pytest.raises(_lib.CovaError):                                  # streams 2 and 3: same gamma, other countdowns
        p.submit(frames[2:4, 8:12], stream_ids=[2, 3], cont=True)
    nothing_in_flight()
    # a fresh batch may mix gammas without STAGGERED; the next valid continued batches yield the right windows
    p.submit(frames[:2, :8], stream_ids=[0, 1], pts=np.stack([pts_of(s, 0, 8) for s in (0, 1)]))
    _, wid, wpts = p.collect(meta=True)
    assert [int(x) for x in wpts] == [int(x) for x in pts_of(0, 0, 8)[[3, 5, 7]]] + [int(x) for x in pts_of(1, 0, 8)[[3, 7]]]
    pos = [8, 8, 8, 7]
    submit_ragged(p, frames, [0, 1, 2, 3], pos, [6, 6, 5, 6], **CS)
    _, wid, wpts = p.collect(meta=True)
    for s, g in enumerate([2, 4, 2, 2]):                                 # stream 1 restarted at gamma 4
        want = [f for f, _ in element_windows(frames[s, : pos[s]], g)]
        want = [f for f in want if f >= pos[s] - [6, 6, 5, 6][s]]
        assert [int(x) for x in wpts[wid == s]] == [int(x) for x in pts_of(s, 0, pos[s])[want]], s


def _lib_ptr(a):
    return ctypes.c_void_p(a.ctypes.data)
