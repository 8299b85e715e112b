"""Sparse input (cova_packer_pack_sparse, cova_pipeline_submit_sparse): frames as a per-frame background plus the macroblocks
that differ from it, expanded into the packed16 frame pool on the device.

CPU: the C++ encoder is byte-identical to the NumPy reference (oracle/sparse_ref.py) at any thread count, decodes back to
cova_packer_pack's output, and reports its size exactly.  GPU: a sparse submit gives the same bytes as a dense packed16
submit of the same frames - boxes, masks, logits, BlobNet input, window stream ids and PTS - and a malformed batch is
refused before any device call without disturbing the handle."""
import ctypes
import os
import re

import numpy as np
import pytest

from cova_b200 import _lib, synth, weights
from cova_b200.elements import BlobPipeline, FramePacker, PinnedBuffer, SparseBatch
from oracle import sparse_ref

HERE = os.path.dirname(os.path.abspath(__file__))
T = 4
GRIDS = {"720p": (45, 80), "1080p": (68, 120), "4K": (135, 240)}


def _clip():
    d = np.load(os.path.join(HERE, "golden", "demo_1m_meta.npz"))
    return np.ascontiguousarray(np.moveaxis(d["planes"], 0, -1))          # [1802, 45, 80, 4]


def _wts():
    return weights.to_blob(weights.random_weights(0, head_bias=-1.0))


# ----------------------------------------------------------------------------------------------------------- CPU
def _random_quads(rng, n, h, w):
    q = rng.integers(0, 256, size=(n, h, w, 4), dtype=np.uint8)          # values above 6 and garbage in byte 3
    q[..., :3] = np.where(rng.random((n, h, w, 3)) < 0.8, 0, q[..., :3])   # mostly background, as in real clips
    return q


def _inputs():
    rng = np.random.default_rng(7)
    cases = {}
    for h, w in ((45, 80), (68, 120)):                                  # n_mb = 3600 (not a multiple of 32), 8160 (one)
        cases[f"random_{h}x{w}"] = _random_quads(rng, 9, h, w)
        cases[f"one_frame_{h}x{w}"] = _random_quads(rng, 1, h, w)
    bg = np.zeros((3, 45, 80, 4), np.uint8)
    bg[..., 3] = 200                                                     # stale byte only: every frame all background
    cases["all_background"] = bg
    distinct = np.zeros((2, 8, 64, 4), np.uint8)                         # 512 values, each once: the mode is 0 (smallest)
    v = np.arange(512).reshape(8, 64)
    distinct[..., 0], distinct[..., 1], distinct[..., 2] = v & 7, (v >> 3) & 7, v >> 6
    distinct = np.minimum(distinct, 6)                                   # clip keeps it valid input; values repeat as 6s
    cases["all_distinct"] = np.ascontiguousarray(np.concatenate([distinct, np.stack([np.roll(distinct[0], 5, axis=1)])]))
    iframe = np.zeros((2, 45, 80, 4), np.uint8)
    iframe[..., 0] = 6                                                   # I-frames: every macroblock weight 6
    iframe[1, ..., 1:3] = rng.integers(0, 9, size=(45, 80, 2))
    cases["iframes"] = iframe
    tie = np.zeros((2, 16, 16, 4), np.uint8)                              # two values, 128 macroblocks each: smaller wins
    tie[0, :8, :, 0] = 5
    tie[1, :8, :, 1] = 1
    tie[1, 8:, :, 0] = 2
    cases["mode_ties"] = tie
    cases["many_frames"] = synth.tiled_streams(4, 40, 45, 80, config_idx=3).reshape(-1, 45, 80, 4)
    clip = _clip()
    cases["real_clip"] = clip[np.r_[0:60, 240:300, 1740:1802]]           # includes the IDR frames 0, 250
    for name, (h, w) in GRIDS.items():
        cases[f"synth_{name}"] = synth.synth_streams(2, 4, h, w, config_idx=5).reshape(-1, h, w, 4)
    return cases


INPUTS = _inputs()


@pytest.mark.parametrize("threads", [1, 3, 16])
@pytest.mark.parametrize("name", sorted(INPUTS))
def test_encoder_is_byte_identical_to_the_reference(name, threads):
    q = INPUTS[name]
    pk = FramePacker(threads)
    b = pk.pack_sparse(q[None])
    want = sparse_ref.encode(FramePacker(1).pack(q))
    assert b.data.tobytes() == want
    assert (b.n_streams, b.frames_per_stream, b.h_mb, b.w_mb) == (1, q.shape[0], q.shape[1], q.shape[2])


@pytest.mark.parametrize("name", sorted(INPUTS))
def test_decode_of_encode_is_the_packed16_frames(name):
    q = INPUTS[name]
    pk = FramePacker(4)
    b = pk.pack_sparse(q[None])
    got = sparse_ref.decode(b.data.tobytes(), q.shape[0], q.shape[1] * q.shape[2])
    assert (got == pk.pack(q).reshape(q.shape[0], -1)).all()


def test_mode_tie_goes_to_the_smallest_value():
    b = FramePacker(1).pack_sparse(INPUTS["mode_ties"][None]).data
    first = np.frombuffer(b[:8].tobytes(), "<u4")
    assert first[0] == 0 and first[1] == 128                             # values 0 and 5 tie at 128 each


def test_too_small_reports_the_exact_size():
    q = INPUTS["random_45x80"]
    pk = FramePacker(3)
    lib = _lib.load()
    need = ctypes.c_size_t()
    out = np.zeros(16, np.uint8)
    rc = lib.cova_packer_pack_sparse(pk._h, ctypes.c_void_p(q.ctypes.data), q.shape[0], 80, 45, ctypes.c_void_p(out.ctypes.data),
                                     out.size, ctypes.byref(need))
    assert rc == _lib.E_TOOSMALL and (out == 0).all()
    want = len(sparse_ref.encode(FramePacker(1).pack(q)))
    assert need.value == want <= q.shape[0] * _lib.sparse_max_frame_bytes(3600)
    out = np.zeros(want, np.uint8)                                      # exactly enough
    b = pk.pack_sparse(q[None], out=out)
    assert b.data.size == want and b.data.tobytes() == sparse_ref.encode(FramePacker(1).pack(q))
    with pytest.raises(_lib.CovaError) as e:
        pk.pack_sparse(q[None], out=np.zeros(want - 4, np.uint8))
    assert e.value.code == _lib.E_TOOSMALL


def test_worst_case_size_is_the_header_macro():
    for name in ("all_distinct", "iframes", "random_68x120"):
        q = INPUTS[name]
        n_mb = q.shape[1] * q.shape[2]
        assert FramePacker(2).pack_sparse(q[None]).data.size <= q.shape[0] * _lib.sparse_max_frame_bytes(n_mb)
    assert sparse_ref.record_bytes(3600, 3600) == _lib.sparse_max_frame_bytes(3600) == 8 + 4 * 113 + 4 * 1800


def test_header_macro_matches_its_python_mirror():
    hdr = open(os.path.join(HERE, "..", "include", "cova_b200.h")).read()
    m = re.search(r"#define\s+COVA_SPARSE_MAX_FRAME_BYTES\(n_mb\)\s*\\?\s*\n?\s*(\(.*?\))\s*/\*", hdr, re.S)
    assert m, "COVA_SPARSE_MAX_FRAME_BYTES"
    expr = re.sub(r"\(size_t\)", "", m.group(1)).replace("u", "").replace("/", "//")
    for n_mb in (1, 31, 32, 33, 3600, 8160, 32400, 129600):
        assert eval(expr, {"n_mb": n_mb}) == _lib.sparse_max_frame_bytes(n_mb), n_mb
    assert "cova_packer_pack_sparse" in _lib.SIGNATURES and "cova_pipeline_submit_sparse" in _lib.SIGNATURES


# ----------------------------------------------------------------------------------------------------------- GPU
def _pair(h, w, max_streams, max_fps, gamma=1, **kw):
    return [BlobPipeline(w, h, _wts(), max_streams, max_fps, gamma=gamma, packed_input=True, keep_logits=True, **kw)
            for _ in range(2)]


def _same_run(dense, sparse, q, pk, ids=None, pts=None, cont=False, staggered=False, activation=False):
    """submit the quads as dense packed16 to one pipeline and as a sparse batch to the other; compare every output"""
    packed = pk.pack(q)
    b = pk.pack_sparse(q)
    res = []
    for p, frames in ((dense, packed), (sparse, b)):
        p.submit(frames, stream_ids=ids if ids is not None else list(range(q.shape[0])), pts=pts, cont=cont, staggered=staggered)
        boxes, wid, wpts = p.collect(meta=True)
        res.append((boxes, wid.copy(), wpts.copy(), p.read_mask(), p.read_logits(),
                    p.read_activation(0) if activation else None))
    (b0, i0, t0, m0, l0, a0), (b1, i1, t1, m1, l1, a1) = res
    assert b0 == b1 and (i0 == i1).all() and (t0 == t1).all()
    assert m0.shape == m1.shape and (m0 == m1).all()
    assert l0.tobytes() == l1.tobytes()
    if activation:
        assert a0.shape == a1.shape and (a0 == a1).all()
    return b0


@pytest.mark.gpu
@pytest.mark.parametrize("grid", sorted(GRIDS))
@pytest.mark.parametrize("gamma", [1, 2, 3])
def test_sparse_equals_dense_packed16(grid, gamma):
    h, w = GRIDS[grid]
    n_streams, fps = (3, 9) if grid != "4K" else (2, 7)
    q = synth.synth_streams(n_streams, fps, h, w, config_idx=60 + gamma)
    pk = FramePacker(4)
    dense, sparse = _pair(h, w, n_streams, fps, gamma, n_chunks=1)
    boxes = _same_run(dense, sparse, q, pk, activation=True)             # one chunk: the BlobNet input too
    assert len(boxes) == n_streams * ((fps - T) // gamma + 1)
    dense, sparse = _pair(h, w, n_streams, fps, gamma, n_chunks=3)       # chunk boundaries between chains
    _same_run(dense, sparse, q, pk)


@pytest.mark.gpu
def test_sparse_equals_dense_packed16_at_8k():
    """480x270 macroblocks: 4,050 bitmap words per record, so the kernel's scan runs over four tiles."""
    h, w = 270, 480
    q = synth.synth_streams(1, 5, h, w, config_idx=70)
    dense, sparse = _pair(h, w, 1, 5, n_chunks=1, ccl_cluster=True)
    _same_run(dense, sparse, q, FramePacker(4), activation=True)


@pytest.mark.gpu
def test_real_clip_through_sparse_gives_the_quad_path_boxes():
    clip = _clip()[:400]
    quads = BlobPipeline(80, 45, _wts(), 4, 100, cc_threshold=30)
    sp = BlobPipeline(80, 45, _wts(), 4, 100, cc_threshold=30, packed_input=True)
    want = quads.process(clip.reshape(4, 100, 45, 80, 4))
    sp.submit(FramePacker(4).pack_sparse(clip.reshape(4, 100, 45, 80, 4)), stream_ids=[0, 1, 2, 3])
    assert sp.collect() == want and len(want) == 4 * 97


@pytest.mark.gpu
@pytest.mark.parametrize("gamma", [1, 2, 3])
def test_seeded_continue_stagger_join_leave_reset_schedule(gamma):
    """12 stream ids, 8 continued staggered batches of random subsets and lengths, two rounds of resets, three chunks: the
    sparse handle yields exactly the windows, PTS and stream ids of the dense packed16 handle."""
    rng = np.random.default_rng(200 + gamma)
    h, w = 45, 80
    quads = synth.synth_streams(12, 8 * 9, h, w, config_idx=80 + gamma)
    pk = FramePacker(4)
    dense, sparse = _pair(h, w, 12, 12, gamma, n_chunks=3)
    pos = [0] * 12
    total = 0
    for b in range(8):
        ids = [int(i) for i in rng.permutation(12)[: int(rng.integers(1, 13))]]
        fps = int(rng.integers(1, 10))
        q = np.stack([quads[i, pos[i]: pos[i] + fps] for i in ids])
        pts = np.stack([np.arange(pos[i], pos[i] + fps, dtype=np.uint64) + np.uint64(i * 1000) for i in ids])
        total += len(_same_run(dense, sparse, q, pk, ids=ids, pts=pts, cont=True, staggered=True))
        for i in ids:
            pos[i] += fps
        if b in (2, 5):
            r = rng.permutation(12)[:3]
            dense.reset_streams(r)
            sparse.reset_streams(r)
    assert total > 0


@pytest.mark.gpu
def test_four_batches_in_flight_alternating_dense_and_sparse():
    h, w = 45, 80
    pk = FramePacker(4)
    ref = BlobPipeline(w, h, _wts(), 6, 12, packed_input=True)
    p = BlobPipeline(w, h, _wts(), 6, 12, packed_input=True, n_chunks=2)
    shapes = [(6, 12), (2, 5), (5, 9), (1, 4)]
    batches = [synth.synth_streams(n, f, h, w, config_idx=90 + i) for i, (n, f) in enumerate(shapes)]
    pins = []
    for i, q in enumerate(batches):
        if i % 2:
            b = pk.pack_sparse(q)
            pin = PinnedBuffer(b.data.size)
            pin.array[:] = b.data
            pins.append(pin)
            p.submit(SparseBatch(pin.array, b.n_streams, b.frames_per_stream, h, w), stream_ids=list(range(q.shape[0])))
        else:
            p.submit(pk.pack(q))
    for q in batches:
        assert p.collect() == ref.process(pk.pack(q))


def _malformed_cases(good, n_mb, n_frames):
    """One batch per rule of the format, each breaking exactly that rule in an otherwise valid batch.  The record patched is
    the first with at least two differing macroblocks (a first frame can be all background, count 0)."""
    nw = (n_mb + 31) // 32
    off = [0]
    for _ in range(n_frames):
        off.append(off[-1] + sparse_ref.record_bytes(n_mb, int(np.frombuffer(good[off[-1] + 4: off[-1] + 8].tobytes(), "<u4")[0])))
    assert off[-1] == good.size
    j = next(f for f in range(n_frames) if int(np.frombuffer(good[off[f] + 4: off[f] + 8].tobytes(), "<u4")[0]) >= 2)
    r0, r1 = off[j], off[j + 1]
    bg, count = (int(x) for x in np.frombuffer(good[r0: r0 + 8].tobytes(), "<u4"))

    def patched(a, offset, value, dtype="<u4"):
        a = a.copy()
        a[r0 + offset: r0 + offset + np.dtype(dtype).itemsize] = np.frombuffer(np.array([value], dtype).tobytes(), np.uint8)
        return a

    word = lambda k: int(np.frombuffer(good[r0 + 8 + 4 * k: r0 + 12 + 4 * k].tobytes(), "<u4")[0])
    cases = {
        "reserved background bits": patched(good, 0, bg | (1 << 9)),
        "count above popcount": patched(good, 4, count + 1),
        "count below popcount": patched(good, 4, count - 1),
        "bit past n_mb": patched(good, 8 + 4 * (nw - 1), word(nw - 1) | (1 << 31)),   # 3600 % 32 = 16: bits 16..31 of the last word
        "truncated": good[:-4],
        "trailing bytes": np.concatenate([good, np.zeros(4, np.uint8)]),
        "too few records": good[:off[1]],
    }
    if count % 2:
        cases["nonzero padding"] = patched(good, r1 - r0 - 2, 1, "<u2")
    else:           # an odd count of the same record size: clear one set bit, count - 1, and a non-zero last u16
        k = next(k for k in range(nw) if word(k))
        a = patched(good, 8 + 4 * k, word(k) & (word(k) - 1))
        a = patched(a, 4, count - 1)
        cases["nonzero padding"] = patched(a, r1 - r0 - 2, 1, "<u2")
    return cases


def test_every_malformed_case_breaks_the_format():
    """CPU check of the cases the GPU test submits: the reference decoder rejects each of them, and accepts the batch."""
    h, w = 45, 80
    pk = FramePacker(2)
    q = synth.synth_streams(2, 6, h, w, config_idx=95)
    good = pk.pack_sparse(q).data.copy()
    assert (sparse_ref.decode(good.tobytes(), 12, h * w) == pk.pack(q).reshape(12, -1)).all()
    cases = _malformed_cases(good, h * w, 12)
    assert len(cases) == 8
    for name, data in cases.items():
        with pytest.raises((AssertionError, ValueError, IndexError)):
            sparse_ref.decode(data.tobytes(), 12, h * w)


@pytest.mark.gpu
def test_malformed_batches_are_refused_and_the_handle_recovers():
    h, w = 45, 80
    pk = FramePacker(2)
    q = synth.synth_streams(2, 6, h, w, config_idx=95)
    good = pk.pack_sparse(q).data.copy()
    ref = BlobPipeline(w, h, _wts(), 2, 6, packed_input=True).process(pk.pack(q))
    p = BlobPipeline(w, h, _wts(), 2, 6, packed_input=True)
    L = p._L

    def submit(data, n_streams=2, fps=6):
        a = np.ascontiguousarray(data, dtype=np.uint8)
        return L.cova_pipeline_submit_sparse(p._h, ctypes.c_void_p(a.ctypes.data), a.size, n_streams, fps, None, None, 0)

    for name, data in _malformed_cases(good, h * w, 12).items():
        assert submit(data) == _lib.E_INVAL, name
        assert b"sparse" in L.cova_last_error(), name
        p.submit(SparseBatch(good, 2, 6, h, w), stream_ids=[0, 1])        # nothing was left in flight: this one works
        assert p.collect() == ref, name
    quads = BlobPipeline(w, h, _wts(), 2, 6)
    rc = quads._L.cova_pipeline_submit_sparse(quads._h, ctypes.c_void_p(good.ctypes.data), good.size, 2, 6, None, None, 0)
    assert rc == _lib.E_INVAL                                             # a quads pipeline refuses sparse input
    assert quads.process(q) == ref
