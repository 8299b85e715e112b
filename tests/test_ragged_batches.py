"""Ragged batches (cova_pipeline_submit_ragged, cova_pipeline_submit_sparse_ragged): the streams of one batch bring different
numbers of new frames - GoP shards of different lengths, live flushes with a different frame count per camera.

Every stream of such a batch must yield exactly the windows its uncut sequence yields - boxes, masks, stacked RGBA windows,
window stream ids and PTS byte for byte - whatever the other streams of the batch bring.  The reference for a stream is one
process() call over all frames it received since it (re)started, on a one-stream pipeline.  With equal counts the ragged
calls are byte-identical to submit_host2 / submit_sparse."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from cova_b200 import _lib, synth, weights
from cova_b200.elements import FLOW_OK, BlobPipeline, FramePacker, MetaPreprocess
from oracle import metapreprocess_ref as mpr
from oracle import sparse_ref

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
H, W, T = 45, 80, 4
ACT_REL_TOL = 4e-3
GRIDS = {"720p": (45, 80), "1080p": (68, 120), "4K": (135, 240)}


# ----------------------------------------------------------------------------------------------------------- CPU
def _header():
    with open(os.path.join(ROOT, "include", "cova_b200.h")) as f:
        return f.read()


def test_ragged_symbols_are_declared_exported_and_bound():
    hdr = " ".join(_header().split())
    assert ("int cova_pipeline_submit_ragged(cova_pipeline *p, const uint8_t *frames, uint32_t n_streams, const uint32_t "
            "*n_frames, const uint32_t *stream_ids, const uint64_t *pts, uint32_t flags);") in hdr
    assert ("int cova_pipeline_submit_sparse_ragged(cova_pipeline *p, const uint8_t *data, size_t data_len, uint32_t n_streams, "
            "const uint32_t *n_frames, const uint32_t *stream_ids, const uint64_t *pts, uint32_t flags);") in hdr
    u32, vp, sz = ctypes.c_uint32, ctypes.c_void_p, ctypes.c_size_t
    assert _lib.SIGNATURES["cova_pipeline_submit_ragged"] == (ctypes.c_int, [vp, vp, u32, vp, vp, vp, u32])
    assert _lib.SIGNATURES["cova_pipeline_submit_sparse_ragged"] == (ctypes.c_int, [vp, vp, sz, u32, vp, vp, vp, u32])
    lib = _lib.load()
    for name in ("cova_pipeline_submit_ragged", "cova_pipeline_submit_sparse_ragged"):
        assert getattr(lib, name).argtypes == _lib.SIGNATURES[name][1]
    # no handle: refused before anything else, as every entry point does
    n = (ctypes.c_uint32 * 2)(3, 4)
    assert lib.cova_pipeline_submit_ragged(None, b"x", 2, n, None, None, 0) == _lib.E_INVAL
    assert lib.cova_pipeline_submit_sparse_ragged(None, b"x", 1, 2, n, None, None, 0) == _lib.E_INVAL


C_SNIPPET = r"""
#include <stddef.h>
#include <stdint.h>
#include <stdio.h>
#include "cova_b200.h"

int main(void) {
    const uint8_t frames[4] = {0, 0, 0, 0};
    const uint32_t n_frames[2] = {3, 5}, ids[2] = {0, 1};
    const uint64_t pts[8] = {0, 1, 2, 3, 4, 5, 6, 7};
    int a = cova_pipeline_submit_ragged(NULL, frames, 2, n_frames, ids, pts, COVA_SUBMIT_CONTINUE | COVA_SUBMIT_STAGGERED);
    int b = cova_pipeline_submit_sparse_ragged(NULL, frames, sizeof(frames), 2, n_frames, ids, pts, 0);
    if (a != COVA_E_INVAL || b != COVA_E_INVAL) return 1;
    printf("ragged ok\n");
    return 0;
}
"""


def test_plain_c_calls_both_declarations(tmp_path):
    _lib.load()                                                      # raises if the library has not been built
    src, exe = tmp_path / "ragged.c", str(tmp_path / "ragged")
    src.write_text(C_SNIPPET)
    lib_dir = os.path.join(ROOT, "cova_b200")
    r = subprocess.run(["gcc", "-std=c11", "-Wall", "-Wextra", "-Werror", "-I" + os.path.join(ROOT, "include"), str(src),
                        "-L" + lib_dir, "-lcova_b200", "-Wl,-rpath," + lib_dir, "-o", exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "ragged ok" in r.stdout, (r.stdout, r.stderr)


def test_pack_sparse_with_counts_is_the_reference_encoding():
    counts = np.array([3, 1, 7, 4], dtype=np.uint32)
    quads = synth.synth_streams(1, int(counts.sum()), H, W, config_idx=60)[0]
    pk = FramePacker(3)
    b = pk.pack_sparse(quads, counts=counts)
    assert b.n_streams == 4 and (b.counts == counts).all()
    assert b.data.tobytes() == sparse_ref.encode(pk.pack(quads))
    whole = pk.pack_sparse(quads[None])                              # the same frames as one stream: the same bytes
    assert whole.data.tobytes() == b.data.tobytes()


# ----------------------------------------------------------------------------------------------------------- GPU
def _wts():
    return weights.to_blob(weights.random_weights(0, head_bias=-1.0))


class Streams:
    """Feeds stream ids through ragged batches and records, per life of a stream (from its start, its last reset or its
    last fresh restart), the frames it was fed and the windows the batches returned for it.  mode: "quads", "packed"
    (dense packed16) or "sparse" (pack_sparse(counts=) of the same frames)."""

    def __init__(self, p, gamma, n_ids, n_frames, config_idx, mode="quads", inspect=True):
        # inspect: also compare masks (and for quads the stacked windows) - only valid with one batch in flight
        self.p, self.gamma, self.mode, self.inspect = p, gamma, mode, inspect
        self.quads = synth.synth_streams(n_ids, n_frames, H, W, config_idx=config_idx)
        self.packer = FramePacker(2)
        self.frames = self.quads if mode == "quads" else self.packer.pack(self.quads)
        self.pos = [0] * n_ids
        self.start = [0] * n_ids
        self.got = [[] for _ in range(n_ids)]
        self.lives = []
        self.pending = []

    def pts(self, sid, lo, hi):
        return np.arange(lo, hi, dtype=np.uint64) + np.uint64(sid * 1_000_000)

    def submit(self, ids, counts, cont=True, staggered=True):
        ids, counts = [int(i) for i in ids], [int(c) for c in counts]
        if not cont:
            for i in ids:
                self._close(i)
        src = self.quads if self.mode == "sparse" else self.frames
        fr = np.concatenate([src[i, self.pos[i]: self.pos[i] + c] for i, c in zip(ids, counts)])
        pts = np.concatenate([self.pts(i, self.pos[i], self.pos[i] + c) for i, c in zip(ids, counts)])
        if self.mode == "sparse":
            self.p.submit(self.packer.pack_sparse(fr, counts=counts), stream_ids=ids, pts=pts, cont=cont, staggered=staggered)
        else:
            self.p.submit(fr, counts=counts, stream_ids=ids, pts=pts, cont=cont, staggered=staggered)
        for i, c in zip(ids, counts):
            self.pos[i] += c
        self.pending.append(ids)

    def collect(self):
        ids = self.pending.pop(0)
        boxes, wid, wpts = self.p.collect(meta=True)
        mask = self.p.read_mask() if self.inspect else None
        stacked = self.p.read_stacked() if self.inspect and self.mode == "quads" else None
        assert set(wid.tolist()) <= set(ids)
        assert (np.diff([ids.index(int(i)) for i in wid]) >= 0).all()      # stream-major
        for k, sid in enumerate(wid.tolist()):
            self.got[sid].append((boxes[k], None if mask is None else mask[k], None if stacked is None else stacked[k], int(wpts[k])))
        return boxes, wid, wpts

    def step(self, ids, counts, cont=True, staggered=True):
        self.submit(ids, counts, cont, staggered)
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
        n_windows = 0
        for sid, lo, hi, got in self.lives:
            n = hi - lo
            if n == 0:
                assert got == []
                continue
            want = ref.process(self.frames[sid, lo:hi][None])
            newest = mpr.window_newest_indices(n, T, self.gamma)
            assert len(got) == len(want) == len(newest), (sid, lo, hi)
            assert [g[0] for g in got] == want, (sid, lo, hi)
            assert [g[3] for g in got] == [int(v) for v in self.pts(sid, lo, hi)[newest]], (sid, lo, hi)
            if want and got[0][1] is not None:
                assert (np.stack([g[1] for g in got]) == ref.read_mask()).all(), (sid, lo, hi)
            if want and got[0][2] is not None:
                assert (np.stack([g[2] for g in got]) == ref.read_stacked()).all(), (sid, lo, hi)
            n_windows += len(got)
        return n_windows


def _pipe(gamma, max_streams, max_fps, mode="quads", keep_stacked=True, **kw):
    return BlobPipeline(W, H, _wts(), max_streams, max_fps, gamma=gamma, keep_stacked=keep_stacked and mode == "quads",
                        packed_input=mode != "quads", **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("chunks", [1, 3])
@pytest.mark.parametrize("mode", ["quads", "packed"])
@pytest.mark.parametrize("gamma", [1, 2, 3])
def test_fresh_chains_of_different_lengths(gamma, mode, chunks):
    """GoP shards: ten fresh chains of 1 .. max_frames_per_stream frames in one batch - shorter than a window, exactly one
    window's worth, the full pipeline length - with chunk borders (three chunks: chains 0-3, 4-7, 8-9) between chains of
    different lengths."""
    counts = [16, 3, 4, 9, 1, 16, 7, 5, 12, 2]
    p = _pipe(gamma, 10, 16, mode, n_chunks=chunks)
    st = Streams(p, gamma, 10, 16, config_idx=61 + gamma, mode=mode)
    boxes, wid, _ = st.step(range(10), counts, cont=False, staggered=False)
    assert [int((wid == s).sum()) for s in range(10)] == [len(mpr.window_newest_indices(c, T, gamma)) for c in counts]
    if chunks == 1:                                                      # block 1 walks the frames that exist
        assert p.last_plan()[0]["n_groups"] % sum(counts) == 0
    if mode == "quads" and chunks == 1:                                  # the element shim agrees window for window
        for s in (0, 3, 8):
            el = MetaPreprocess(W * 16, H * 16, T, gamma)
            outs = [o for f in range(counts[s]) for rc, o in [el.transform(st.quads[s, f])] if rc == FLOW_OK]
            assert len(outs) == len(st.got[s]) and all(o == g[2].tobytes() for o, g in zip(outs, st.got[s]))
    st.check(_pipe(gamma, 1, 16, mode))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["quads", "packed", "sparse"])
@pytest.mark.parametrize("gamma", [1, 3])
def test_seeded_continue_stagger_reset_schedule(gamma, mode):
    """12 stream ids over 9 batches in three chunks: random subsets, a random count per stream and batch, staggered
    continues, fresh restarts and resets.  Every life of every id equals its uncut run."""
    rng = np.random.default_rng(200 + 10 * gamma + len(mode))
    p = _pipe(gamma, 12, 12, mode, n_chunks=3)
    st = Streams(p, gamma, 12, 9 * 9, config_idx=70 + gamma, mode=mode)
    for b in range(9):
        ids = rng.permutation(12)[: int(rng.integers(1, 13))]
        counts = rng.integers(1, 10, size=ids.size)
        if b == 4:
            st.step(ids, counts, cont=False, staggered=False)             # these ids restart with an empty window
        else:
            st.step(ids, counts)
        if b in (2, 6):
            st.reset(rng.permutation(12)[:3])
    assert st.check(_pipe(gamma, 1, 9 * 9, mode)) > 0


@pytest.mark.gpu
@pytest.mark.parametrize("sparse", [False, True])
def test_equal_counts_are_byte_identical_to_the_uniform_calls(sparse):
    """The ragged calls with n_frames[s] = fps for every s give what submit_host2 / submit_sparse give: boxes, masks, window
    ids and PTS, over a fresh, a staggered continued and a lock-step continued batch."""
    gamma = 2
    quads = synth.synth_streams(4, 30, H, W, config_idx=80)
    pk = FramePacker(2)
    frames = pk.pack(quads) if sparse else quads
    # fresh; lock-step continued; staggered continued (same histories, other gamma phases), twice
    schedule = [([0, 1, 2, 3], 5, False), ([1, 3], 3, True), ([0, 1, 2, 3], 9, True), ([2, 0, 1, 3], 7, True)]
    runs = []
    for ragged in (False, True):
        p = _pipe(gamma, 4, 12, "sparse" if sparse else "quads", n_chunks=2)
        res = []
        seen = [0] * 4
        for ids, fps, cont in schedule:
            fr = np.stack([frames[i, seen[i]: seen[i] + fps] for i in ids])
            pts = np.stack([np.arange(fps, dtype=np.uint64) + np.uint64(1000 * i + seen[i]) for i in ids])
            for i in ids:
                seen[i] += fps
            kw = dict(stream_ids=ids, cont=cont, staggered=cont and len(ids) == 4)
            if sparse:
                q = np.stack([quads[i, seen[i] - fps: seen[i]] for i in ids])
                b = pk.pack_sparse(q.reshape(-1, H, W, 4), counts=[fps] * len(ids)) if ragged else pk.pack_sparse(q)
                p.submit(b, pts=pts.reshape(-1) if ragged else pts, **kw)
            elif ragged:
                p.submit(fr.reshape(-1, H, W, 4), counts=[fps] * len(ids), pts=pts.reshape(-1), **kw)
            else:
                p.submit(fr, pts=pts, **kw)
            boxes, wid, wpts = p.collect(meta=True)
            res.append((boxes, wid.copy(), wpts.copy(), p.read_mask()))
        runs.append(res)
    for a, b in zip(*runs):
        assert a[0] == b[0]
        for x, y in zip(a[1:], b[1:]):
            assert x.shape == y.shape and (x == y).all()
    assert sum(len(r[0]) for r in runs[0]) > 0


@pytest.mark.gpu
@pytest.mark.parametrize("grid", ["720p", "1080p", "4K"])
def test_sparse_ragged_equals_dense_ragged_packed16(grid):
    h, w = GRIDS[grid]
    plan = [([0, 1, 2, 3], [5, 9, 2, 7]), ([2, 0, 3], [8, 1, 4])] if grid != "4K" else [([0, 1], [3, 6])]
    quads = synth.synth_streams(4, 12, h, w, config_idx=90)
    pk = FramePacker(4)
    packed = pk.pack(quads)
    runs = []
    for sparse in (False, True):
        p = BlobPipeline(w, h, _wts(), 4, 12, gamma=1, packed_input=True, n_chunks=2)
        pos, res = [0] * 4, []
        for ids, counts in plan:
            src = quads if sparse else packed
            fr = np.concatenate([src[i, pos[i]: pos[i] + c] for i, c in zip(ids, counts)])
            pts = np.concatenate([np.arange(pos[i], pos[i] + c, dtype=np.uint64) + np.uint64(100 * i) for i, c in zip(ids, counts)])
            for i, c in zip(ids, counts):
                pos[i] += c
            if sparse:
                p.submit(pk.pack_sparse(fr, counts=counts), stream_ids=ids, pts=pts, cont=True, staggered=True)
            else:
                p.submit(fr, counts=counts, stream_ids=ids, pts=pts, cont=True, staggered=True)
            boxes, wid, wpts = p.collect(meta=True)
            res.append((boxes, wid.copy(), wpts.copy(), p.read_mask()))
        runs.append(res)
    for a, b in zip(*runs):
        assert a[0] == b[0] and len(a[0]) > 0
        for x, y in zip(a[1:], b[1:]):
            assert x.shape == y.shape and (x == y).all()


@pytest.mark.gpu
def test_four_ragged_batches_in_flight_and_a_reused_slot():
    """Four ragged batches of different shapes queued before the first collect, twice.  The fifth batch lands in the first
    one's slot with the same ids, the same (fresh) phases and the same stride but other counts: its chain table must be
    uploaded again, not kept."""
    gamma = 2
    p = _pipe(gamma, 8, 12, keep_stacked=False)
    st = Streams(p, gamma, 8, 60, config_idx=95, inspect=False)
    rounds = [
        [([0, 1, 2], [5, 9, 3], False), ([3, 4], [2, 8], False), ([5, 6, 7], [7, 1, 4], False), ([0, 3], [4, 6], True)],
        [([0, 1, 2], [9, 3, 5], False), ([4, 5, 6, 7], [3, 3, 2, 9], True), ([1, 3], [6, 1], True), ([2, 6], [1, 8], True)],
    ]
    for batches in rounds:
        for ids, counts, cont in batches:
            st.submit(ids, counts, cont=cont, staggered=cont)
        with pytest.raises(_lib.CovaError):
            st.submit([7], [1])                                            # a fifth batch does not fit (and changes nothing)
        for _ in batches:
            st.collect()
    assert st.check(_pipe(gamma, 1, 60, keep_stacked=False)) > 0


@pytest.mark.gpu
def test_block1_paths_agree_on_a_ragged_batch():
    """One staggered ragged batch, one chunk.  Histories 0, 1, 3, 3 and counts 11, 6, 9, 2 give chain ends 14, 9, 12, 5 (two
    not a multiple of the 4-frame ring); with 4 chains x tile pairs < 148 CTAs every item is split and the pieces cross
    from one chain's items to the next one's.  The BlobNet input equals the element's windows, and the fused first block
    agrees with the fp32 validation kernel."""
    gamma = 2
    frames = synth.synth_streams(4, 20, H, W, config_idx=97)
    pre, counts = [0, 1, 3, 4], [11, 6, 9, 2]
    outs = []
    for impl in (_lib.IMPL_TCGEN05, _lib.IMPL_SIMT):
        p = BlobPipeline(W, H, _wts(), 4, 16, gamma=gamma, n_chunks=1, impl=impl)
        for s, n in enumerate(pre):
            if n:
                p.submit(frames[s: s + 1, :n], stream_ids=[s], cont=True, staggered=True)
                p.collect()
        fr = np.concatenate([frames[s, pre[s]: pre[s] + counts[s]] for s in range(4)])
        p.submit(fr, counts=counts, stream_ids=[0, 1, 2, 3], cont=True, staggered=True)
        _, wid, _ = p.collect(meta=True)
        outs.append((wid, p.read_activation(0), p.read_activation(1), p.last_plan()[0]))
    plan = outs[0][3]
    lead = 3
    assert plan["n_groups"] % sum(lead + c for c in counts) == 0 and plan["n_groups"] // sum(lead + c for c in counts) < 148 // 4
    want = []
    for s in range(4):
        st = mpr.tensorise_stream(frames[s, : pre[s] + counts[s]], T, gamma)
        k = int((outs[0][0] == s).sum())
        assert k == len(st) - len(mpr.tensorise_stream(frames[s, : pre[s]], T, gamma))
        want.append(st[len(st) - k:])
    x = np.clip(mpr.stacked_to_nchw(np.concatenate(want), T), 0, 6)
    for wid, a0, _, _ in outs:
        assert (wid == outs[0][0]).all()
        assert a0.shape == x.shape and (a0 == x).all()
    fused, simt = outs[0][2], outs[1][2]
    assert np.abs(fused - simt).max() <= ACT_REL_TOL * np.abs(simt).max()


@pytest.mark.gpu
def test_ragged_refusals_leave_nothing_in_flight():
    quads = synth.synth_streams(3, 12, H, W, config_idx=99)
    p = BlobPipeline(W, H, _wts(), 4, 10, packed_input=True)
    pk = FramePacker(2)
    packed = pk.pack(quads)
    L = p._L
    p._ensure_out(p._worst_case_cap(40))
    keep = []                                                            # host buffers stay alive until their collect
    u32 = lambda *v: np.array(v, dtype=np.uint32)                       # noqa: E731

    def dense(counts, ids=None, flags=0, null_counts=False):
        c = u32(*counts)
        fr = np.ascontiguousarray(np.concatenate([packed[s, : n] for s, n in enumerate(counts)]) if sum(counts) else packed[0, :1])
        i = None if ids is None else u32(*ids)
        keep.append(fr)
        return L.cova_pipeline_submit_ragged(p._h, ctypes.c_void_p(fr.ctypes.data), len(counts),
                                             None if null_counts else ctypes.c_void_p(c.ctypes.data),
                                             None if i is None else ctypes.c_void_p(i.ctypes.data), None, flags)

    def sparse(counts, extra=0, flags=0, null_counts=False):
        c = u32(*counts)
        b = pk.pack_sparse(np.concatenate([quads[s, : n] for s, n in enumerate(counts)]), counts=counts)
        d = np.concatenate([b.data, np.zeros(max(extra, 0), np.uint8)])[: b.data.size + extra]
        d = np.ascontiguousarray(d)
        keep.append(d)
        return L.cova_pipeline_submit_sparse_ragged(p._h, ctypes.c_void_p(d.ctypes.data), d.size, len(counts),
                                                    None if null_counts else ctypes.c_void_p(c.ctypes.data), None, None, flags)

    def nothing_in_flight():
        ln = ctypes.c_size_t()
        assert L.cova_pipeline_collect_host(p._h, None, 0, ctypes.byref(ln), None, None, None) == _lib.E_INVAL

    CS = _lib.SUBMIT_CONTINUE | _lib.SUBMIT_STAGGERED
    refused = [
        lambda: dense([3, 4], null_counts=True),                          # n_frames NULL
        lambda: sparse([3, 4], null_counts=True),
        lambda: dense([3, 0, 2]),                                         # a zero count
        lambda: sparse([0, 2]),
        lambda: dense([11, 2]),                                           # more than max_frames_per_stream
        lambda: dense([2, 2], flags=8),                                   # unknown flag
        lambda: dense([2, 2], flags=_lib.SUBMIT_STAGGERED),               # STAGGERED without CONTINUE
        lambda: dense([2, 2], ids=[1, 1]),                                # duplicate id
        lambda: dense([2, 2], ids=[0, 4]),                                # id out of range
        lambda: sparse([3, 4], extra=4),                                  # bytes past the last record
        lambda: sparse([3, 4], extra=-4),                                 # the last record cut short
        lambda: dense([0] * 5),                                           # more streams than max_streams
    ]
    for k, call in enumerate(refused):
        assert call() == _lib.E_INVAL, k
        nothing_in_flight()
    assert dense([1], ids=[2], flags=CS) == _lib.OK                       # stream 2: 1 frame of history ...
    p.collect()
    assert dense([3], ids=[3], flags=CS) == _lib.OK                       # ... stream 3: 3 frames of history
    p.collect()
    assert dense([7, 7], ids=[0, 3], flags=CS) == _lib.OK                 # lead 3 + 7 fits 10
    p.collect()
    for call in (lambda: dense([2, 8], ids=[0, 3], flags=CS),             # lead 3 + 8 does not
                 lambda: dense([2, 3], ids=[2, 0], flags=_lib.SUBMIT_CONTINUE)):   # lock-step rule without STAGGERED
        assert call() == _lib.E_INVAL
        nothing_in_flight()
    # the lock-step rule compares histories and phases, not counts; and a valid batch still runs
    assert dense([2, 5], ids=[0, 3], flags=_lib.SUBMIT_CONTINUE) == _lib.OK
    boxes = p.collect()
    assert len(boxes) == 2 + 5
    assert sparse([4, 2, 6]) == _lib.OK
    assert len(p.collect()) == 1 + 0 + 3
