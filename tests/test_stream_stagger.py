"""Staggered continued batches (COVA_SUBMIT_STAGGERED): streams with different histories and gamma phases share one batch.

Every stream of such a batch must yield exactly the windows its uncut sequence yields - boxes, masks, stacked RGBA windows,
window stream ids and PTS byte for byte - whatever the other streams of the batch carry.  The reference for a stream is one
process() call over all frames it received since it (re)started."""
import ctypes
import os
import re

import numpy as np
import pytest

from cova_b200 import _lib, synth, weights
from cova_b200.elements import FLOW_OK, BlobPipeline, FramePacker, MetaPreprocess
from oracle import metapreprocess_ref as mpr

HERE = os.path.dirname(os.path.abspath(__file__))
H, W, T = 45, 80, 4
ACT_REL_TOL = 4e-3


def test_header_define_matches_the_binding():
    with open(os.path.join(HERE, "..", "include", "cova_b200.h")) as f:
        m = re.search(r"#define COVA_SUBMIT_STAGGERED (\d+)u", f.read())
    assert m and int(m.group(1)) == _lib.SUBMIT_STAGGERED == 2
    assert _lib.SUBMIT_STAGGERED & _lib.SUBMIT_CONTINUE == 0


def _wts():
    return weights.to_blob(weights.random_weights(0, head_bias=-1.0))


class Streams:
    """Feeds stream ids through staggered continued batches and records, per life of a stream (from its start or its last
    reset), the frames it was fed and the windows the batches returned for it."""

    def __init__(self, p, gamma, n_ids, n_frames, config_idx, packed=False, inspect=True, stacked=True):
        # inspect: also compare masks (and with stacked, the stacked windows) - only valid with one batch in flight
        self.p, self.gamma, self.inspect, self.stacked = p, gamma, inspect, stacked
        self.quads = synth.synth_streams(n_ids, n_frames, H, W, config_idx=config_idx)
        self.frames = FramePacker(2).pack(self.quads) if packed else self.quads
        self.pos = [0] * n_ids                     # next frame of every id
        self.start = [0] * n_ids                   # first frame of the id's current life
        self.got = [[] for _ in range(n_ids)]
        self.lives = []                            # (id, first frame, end frame, windows)
        self.pending = []

    def pts(self, sid, lo, hi):
        return np.arange(lo, hi, dtype=np.uint64) + np.uint64(sid * 1_000_000)

    def submit(self, ids, fps, staggered=True):
        ids = [int(i) for i in ids]
        fr = np.stack([self.frames[i, self.pos[i]: self.pos[i] + fps] for i in ids])
        pts = np.stack([self.pts(i, self.pos[i], self.pos[i] + fps) for i in ids])
        self.p.submit(fr, stream_ids=ids, pts=pts, cont=True, staggered=staggered)
        for i in ids:
            self.pos[i] += fps
        self.pending.append((fr, ids))

    def collect(self):
        fr, ids = self.pending.pop(0)
        boxes, wid, wpts = self.p.collect(meta=True)
        mask = self.p.read_mask() if self.inspect else None
        stacked = self.p.read_stacked() if self.inspect and self.stacked else None
        assert set(wid.tolist()) <= set(ids)
        assert (np.diff([ids.index(int(i)) for i in wid]) >= 0).all()      # stream-major
        for k, sid in enumerate(wid.tolist()):
            self.got[sid].append((boxes[k], None if mask is None else mask[k], None if stacked is None else stacked[k], int(wpts[k])))
        return boxes, wid, wpts

    def step(self, ids, fps, staggered=True):
        self.submit(ids, fps, staggered)
        return self.collect()

    def reset(self, ids):
        self.p.reset_streams(ids)
        for i in ids:
            self._close(int(i))

    def _close(self, i):
        self.lives.append((i, self.start[i], self.pos[i], self.got[i]))
        self.start[i], self.got[i] = self.pos[i], []

    def check(self, ref):
        """Every life equals the uncut run of its frames through `ref` (a one-stream pipeline)."""
        for i in range(len(self.pos)):
            self._close(i)
        for sid, lo, hi, got in self.lives:
            n = hi - lo
            if n == 0:
                assert got == []
                continue
            want = ref.process(self.frames[sid, lo:hi][None])
            assert len(got) == len(want) == len(mpr.window_newest_indices(n, T, self.gamma)), (sid, lo, hi)
            assert [g[0] for g in got] == want, (sid, lo, hi)
            want_pts = [int(v) for v in self.pts(sid, lo, hi)[mpr.window_newest_indices(n, T, self.gamma)]]
            assert [g[3] for g in got] == want_pts, (sid, lo, hi)
            if want and got[0][1] is not None:
                assert (np.stack([g[1] for g in got]) == ref.read_mask()).all(), (sid, lo, hi)
            if want and got[0][2] is not None:
                assert (np.stack([g[2] for g in got]) == ref.read_stacked()).all(), (sid, lo, hi)


def _pipe(gamma, max_streams, max_fps, keep_stacked=True, **kw):
    return BlobPipeline(W, H, _wts(), max_streams, max_fps, gamma=gamma, keep_stacked=keep_stacked, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("gamma", [1, 2, 3])
def test_three_streams_with_different_histories_and_phases_share_a_batch(gamma):
    """Streams carrying 0, 2 and 3 frames, the last one on another gamma phase, run in one staggered batch and two more
    after it; each equals its uncut run, and its window count is what one metapreprocess element per stream emits."""
    p = _pipe(gamma, 3, 16)
    st = Streams(p, gamma, 3, 40, config_idx=21)
    st.step([1], 2)                                # stream 1: 2 frames of history
    st.step([2], 3)                                # stream 2: 3 frames of history ...
    st.step([2], 1)                                # ... after one more frame (one window out): gamma phase 1 for gamma > 1
    assert st.pos == [0, 2, 4]
    for fps in (9, 7, 12):
        boxes, wid, _ = st.step([0, 1, 2], fps)
        counts = [int((wid == s).sum()) for s in range(3)]
        for s in range(3):                         # windows whose newest frame is among this batch's frames
            before = len(mpr.window_newest_indices(st.pos[s] - fps, T, gamma))
            assert counts[s] == len(mpr.window_newest_indices(st.pos[s], T, gamma)) - before, (fps, s, counts)
    el = [MetaPreprocess(W * 16, H * 16, T, gamma) for _ in range(3)]
    for s in range(3):
        outs = [o for f in range(st.pos[s]) for rc, o in [el[s].transform(st.quads[s, f])] if rc == FLOW_OK]
        assert len(outs) == len(st.got[s])
        assert all(o == g[2].tobytes() for o, g in zip(outs, st.got[s]))
    st.check(_pipe(gamma, 1, 40))


@pytest.mark.gpu
@pytest.mark.parametrize("gamma", [1, 2, 3])
@pytest.mark.parametrize("packed", [False, True])
def test_seeded_join_leave_schedule_in_chunks(gamma, packed):
    """12 stream ids over 8 staggered batches: random subsets join and leave, random frames per batch, some resets; three
    chunks per batch put chunk boundaries between chains of different window counts."""
    rng = np.random.default_rng(100 * gamma + packed)
    p = _pipe(gamma, 12, 12, keep_stacked=not packed, n_chunks=3, packed_input=packed)
    st = Streams(p, gamma, 12, 8 * 9, config_idx=22 + gamma, packed=packed, stacked=not packed)
    for b in range(8):
        ids = rng.permutation(12)[: int(rng.integers(1, 13))]
        st.step(ids, int(rng.integers(1, 10)))
        if b in (2, 5):
            st.reset(rng.permutation(12)[:3])
    st.check(_pipe(gamma, 1, 8 * 9, keep_stacked=not packed, packed_input=packed))


@pytest.mark.gpu
def test_four_staggered_batches_in_flight():
    """Four batches of different history / phase mixes queued before the first collect: each slot has its own window
    tables, and a stream that appears in several queued batches continues across them."""
    gamma = 2
    p = _pipe(gamma, 8, 16, keep_stacked=False)
    st = Streams(p, gamma, 8, 48, config_idx=30, inspect=False)
    for ids, fps in (([1, 7], 1), ([2, 6], 2), ([3], 5), ([4], 6), ([6], 1)):
        st.step(ids, fps)                          # seen: 0:0 1:1 2:2 3:5 4:6 5:0 6:3 7:1
    assert st.pos == [0, 1, 2, 5, 6, 0, 3, 1]
    batches = [([0, 1, 2, 3], 5), ([4, 5, 6, 0], 6), ([7, 1, 4], 3), ([2, 5, 7, 6, 3], 8)]
    for ids, fps in batches:
        st.submit(ids, fps)
    with pytest.raises(_lib.CovaError):
        st.submit([0], 1)                          # a fifth batch does not fit (and changes nothing)
    for _ in batches:
        st.collect()
    st.check(_pipe(gamma, 1, 48, keep_stacked=False))


@pytest.mark.gpu
def test_block1_paths_agree_on_a_staggered_batch():
    """One staggered batch, one chunk: the BlobNet input equals the element's windows, and the first block's output from
    the fused kernel agrees with the fp32 validation kernel."""
    gamma = 2
    frames = synth.synth_streams(4, 20, H, W, config_idx=40)
    pre = [0, 1, 3, 4]                             # frames fed before the batch: histories 0, 1, 3, 3 on two phases
    outs = []
    for impl in (_lib.IMPL_TCGEN05, _lib.IMPL_SIMT):
        p = BlobPipeline(W, H, _wts(), 4, 16, gamma=gamma, n_chunks=1, impl=impl)
        for s, n in enumerate(pre):
            if n:
                p.submit(frames[s: s + 1, :n], stream_ids=[s], cont=True, staggered=True)
                p.collect()
        p.submit(np.stack([frames[s, pre[s]: pre[s] + 11] for s in range(4)]), stream_ids=[0, 1, 2, 3], cont=True, staggered=True)
        _, wid, _ = p.collect(meta=True)
        outs.append((wid, p.read_activation(0), p.read_activation(1)))
    want = []
    for s in range(4):
        st = mpr.tensorise_stream(frames[s, : pre[s] + 11], T, gamma)
        want.append(st[len(st) - int((outs[0][0] == s).sum()):])
    x = np.clip(mpr.stacked_to_nchw(np.concatenate(want), T), 0, 6)
    for wid, a0, _ in outs:
        assert (wid == outs[0][0]).all()
        assert a0.shape == x.shape and (a0 == x).all()
    fused, simt = (o[2] for o in outs)
    assert np.abs(fused - simt).max() <= ACT_REL_TOL * np.abs(simt).max()


@pytest.mark.gpu
@pytest.mark.parametrize("gamma", [1, 2])
def test_lock_step_batches_are_unaffected_by_the_flag(gamma):
    frames = synth.synth_streams(3, 21, H, W, config_idx=50)
    got = []
    for staggered in (False, True):
        p = _pipe(gamma, 3, 16)
        p.submit(frames[:, :5], stream_ids=[2, 0, 1], cont=True)
        p.collect()
        res = []
        for lo, n in ((5, 7), (12, 9)):
            p.submit(frames[:, lo: lo + n], stream_ids=[2, 0, 1], pts=np.arange(3 * n, dtype=np.uint64).reshape(3, n),
                     cont=True, staggered=staggered)
            boxes, wid, wpts = p.collect(meta=True)
            res.append((boxes, wid.copy(), wpts.copy(), p.read_mask(), p.read_stacked()))
        got.append(res)
    for a, b in zip(*got):
        assert a[0] == b[0] and len(a[0]) > 0
        for x, y in zip(a[1:], b[1:]):
            assert x.shape == y.shape and (x == y).all()


@pytest.mark.gpu
def test_staggered_submit_rules():
    frames = synth.synth_streams(2, 12, H, W, config_idx=51)
    p = BlobPipeline(W, H, _wts(), 4, 12)
    L = p._L
    ids = np.array([0, 1], dtype=np.uint32)

    def raw(fr, flags, sid=ids):
        a = np.ascontiguousarray(fr)
        return L.cova_pipeline_submit_host2(p._h, ctypes.c_void_p(a.ctypes.data), a.shape[0], a.shape[1],
                                            ctypes.c_void_p(sid.ctypes.data), None, flags)

    assert raw(frames[:, :4], _lib.SUBMIT_STAGGERED) == _lib.E_INVAL              # STAGGERED without CONTINUE
    assert raw(frames[:, :4], 4) == _lib.E_INVAL                                   # unknown bit
    assert raw(frames[:, :4], _lib.SUBMIT_CONTINUE | 8) == _lib.E_INVAL
    with pytest.raises(_lib.CovaError) as e:
        p.submit(frames[:, :4], stream_ids=[0, 1], cont=False, staggered=True)
    assert e.value.code == _lib.E_INVAL
    p.submit(frames[:1, :5], stream_ids=[3], cont=True, staggered=True)            # stream 3: 3 frames of history
    p.collect()
    for fps, ok in ((9, True), (10, False)):                                      # 9 + 3 carried fit 12, 10 + 3 do not
        fr = frames[:, :fps]
        if ok:
            p.submit(fr, stream_ids=[0, 3], cont=True, staggered=True)
            assert len(p.collect()) == (fps - 3) + fps
        else:
            with pytest.raises(_lib.CovaError) as e:
                p.submit(fr, stream_ids=[0, 3], cont=True, staggered=True)
            assert e.value.code == _lib.E_INVAL
    with pytest.raises(_lib.CovaError) as e:
        p.submit(frames[:, :4], stream_ids=[1, 1], cont=True, staggered=True)     # duplicate id
    assert e.value.code == _lib.E_INVAL
    with pytest.raises(_lib.CovaError) as e:                                       # the lock-step rule stays without the flag
        p.submit(frames[:, :4], stream_ids=[2, 3], cont=True)
    assert e.value.code == _lib.E_INVAL
