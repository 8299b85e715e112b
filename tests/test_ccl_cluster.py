"""COVA_FLAG_CCL_CLUSTER: the thread-block-cluster CCL for masks that do not fit one CTA's shared memory (8K video).
Host-side flag handling runs anywhere; everything else is marked gpu."""
import ctypes
import os
import re
import threading

import numpy as np
import pytest

from cova_b200 import _lib, synth, weights
from cova_b200.elements import BboxCc, BlobPipeline, deserialize_vec
from oracle import bboxcc_ref, blobnet_ref, c_oracle, metapreprocess_ref as mpr

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))
LOGIT_REL_TOL, MAX_FLIP = 5e-3, 1e-3          # the bars of test_gpu_parity.py
W8, H8 = 480, 270                             # 8K video in macroblocks
SEAM_ROWS = (68, 136, 204)                    # first pixel row of bands 1..3 at 8K (4 bands of 34 block rows)


# ----------------------------------------------------------------------------------------- host side (no device needed)
def test_header_cluster_flags_match_python():
    hdr = open(os.path.join(ROOT, "include", "cova_b200.h")).read()
    m = re.search(r"#define\s+COVA_FLAG_CCL_CLUSTER\s+(0x[0-9a-fA-F]+)u", hdr)
    assert m and int(m.group(1), 16) == _lib.FLAG_CCL_CLUSTER == 0x800
    m = re.search(r"#define\s+COVA_FLAG_CCL_BANDS\(k\)\s+\(\(\(uint32_t\)\(k\)\s*&\s*(0x[0-9a-fA-F]+)u\)\s*<<\s*(\d+)\)", hdr)
    assert m, "COVA_FLAG_CCL_BANDS"
    mask, shift = int(m.group(1), 16), int(m.group(2))
    for k in range(2, 9):
        assert _lib.flag_ccl_bands(k) == (k & mask) << shift
    assert "cova_bboxcc_new2" in hdr and "cova_bboxcc_new2" in _lib.SIGNATURES


def _n_devices():
    n = ctypes.c_int()
    _lib.load().cova_device_count(ctypes.byref(n))
    return n.value


BAD = [_lib.flag_ccl_bands(4),                                   # BANDS without CLUSTER
       _lib.FLAG_CCL_CLUSTER | _lib.flag_ccl_bands(1),           # k = 1
       _lib.FLAG_CCL_CLUSTER | _lib.flag_ccl_bands(9),           # k > 8
       _lib.FLAG_CCL_CLUSTER | _lib.flag_ccl_bands(15),
       _lib.FLAG_CCL_CLUSTER | 0x1000,                           # unknown bits
       _lib.FLAG_CCL_CLUSTER | 0x10000000]
GOOD = [0, _lib.FLAG_CCL_CLUSTER, _lib.FLAG_CCL_CLUSTER | _lib.flag_ccl_bands(2), _lib.FLAG_CCL_CLUSTER | _lib.flag_ccl_bands(8)]


def test_invalid_cluster_flags_are_refused_before_any_device_call():
    lib = _lib.load()
    blob = weights.to_blob(weights.random_weights(0))
    buf = ctypes.create_string_buffer(blob, len(blob))
    dev = _n_devices() > 0

    def pipeline(w, h, flags):
        hd = ctypes.c_void_p()
        rc = lib.cova_pipeline_new(ctypes.byref(hd), 0, w, h, 4, 1, 1, 8, ctypes.cast(buf, ctypes.c_void_p), len(blob), 1, flags)
        if hd.value:
            lib.cova_pipeline_free(hd)
        return rc

    def bboxcc(w, h, flags):
        hd = ctypes.c_void_p()
        rc = lib.cova_bboxcc_new2(ctypes.byref(hd), 0, w, h, 1, flags)
        if hd.value:
            lib.cova_bboxcc_free(hd)
        return rc

    for flags in BAD:
        assert pipeline(80, 45, flags) == _lib.E_INVAL, hex(flags)
        assert bboxcc(80, 45, flags) == _lib.E_INVAL, hex(flags)
    # k > ceil(H/2): 16 macroblock rows are 8 block rows (the pipeline's smallest grid), 5 pixel rows are 3
    assert pipeline(16, 16, _lib.FLAG_CCL_CLUSTER | _lib.flag_ccl_bands(8)) != _lib.E_INVAL
    assert pipeline(20, 17, _lib.FLAG_CCL_CLUSTER | _lib.flag_ccl_bands(8)) != _lib.E_INVAL
    assert bboxcc(7, 5, _lib.FLAG_CCL_CLUSTER | _lib.flag_ccl_bands(4)) == _lib.E_INVAL
    assert bboxcc(7, 5, _lib.FLAG_CCL_CLUSTER | _lib.flag_ccl_bands(3)) != _lib.E_INVAL
    assert bboxcc(7, 2, _lib.FLAG_CCL_CLUSTER | _lib.flag_ccl_bands(2)) == _lib.E_INVAL
    # the valid combinations get as far as the device
    want = _lib.OK if dev else _lib.E_NODEVICE
    for flags in GOOD:
        assert pipeline(80, 45, flags) == want, hex(flags)
        assert bboxcc(80, 45, flags) == want, hex(flags)


# ----------------------------------------------------------------------------------------- device
def _golden():
    g = np.load(os.path.join(HERE, "golden", "ccl_golden.npz"))
    return g, [m.split(",") for m in g["meta"]]


G, META = _golden()


def _check_element(el, m, thresholds=(1,), tag=""):
    """labels, stats and bincode of one mask against the C oracle"""
    h, w = m.shape
    n, labels, stats = el.labels(m)
    n2, l2, s2 = c_oracle.ccl(m)
    assert n == n2 and (labels == l2).all(), tag
    if n > 1:
        assert (stats[1:] == s2[1:]).all(), tag
    for thr in thresholds:
        el.set_property("cc-threshold", thr)
        assert el.transform_ip(m) == c_oracle.bboxcc(m, thr), (tag, thr)


@pytest.mark.gpu
@pytest.mark.parametrize("i", range(len(META)))
def test_forced_bands_match_the_opencv_golden(i):
    """Every OpenCV golden case through the cluster kernel with bands of one to a few rows: seams everywhere, and the
    label order across them must still be OpenCV's."""
    h, w, name, n = META[i]
    h, w, n = int(h), int(w), int(n)
    raw = G[f"raw_{i}"]
    m = raw.reshape(h, w) if raw.size else np.unpackbits(G[f"mask_{i}"])[: h * w].reshape(h, w)
    labels, stats = G[f"labels_{i}"].astype(np.int32), G[f"stats_{i}"]
    nby = (h + 1) // 2
    if nby < 2:
        pytest.skip("one block row: no band to split")
    for k in sorted({2, min(8, nby)}):
        el = BboxCc(w, h, 1, cluster=True, bands=k)
        n2, l2, s2 = el.labels(m)
        assert n2 == n and (l2 == labels).all(), (name, k)
        if n > 1:
            assert (s2[1:] == stats).all(), (name, k)
        for thr in (0, 1, 3, 30):
            el.set_property("cc-threshold", thr)
            want = bboxcc_ref.serialize_vec([bboxcc_ref.bbox_new(*stats[j, :4]) for j in range(n - 1) if stats[j, 4] >= thr])
            assert el.transform_ip(m) == want, (name, k, thr)
        el.close()


@pytest.mark.gpu
def test_forced_bands_on_random_grids_equal_the_oracle_and_the_single_cta_kernel():
    rng = np.random.default_rng(23)
    shapes = [(3, 200), (4, 1), (5, 7), (129, 130), (135, 240), (150, 150), (33, 47), (34, 48)]
    shapes += [(int(rng.integers(3, 151)), int(rng.integers(1, 151))) for _ in range(32)]
    for h, w in shapes:
        nby = (h + 1) // 2
        k = int(rng.integers(2, min(8, nby) + 1))
        m = (rng.random((h, w)) < rng.uniform(0.05, 0.9)).astype(np.uint8)
        el, one = BboxCc(w, h, 1, cluster=True, bands=k), BboxCc(w, h, 1)
        _check_element(el, m, (1, 5), (h, w, k))
        n, labels, stats = el.labels(m)
        n1, l1, s1 = one.labels(m)
        assert n == n1 and (labels == l1).all() and (stats == s1).all(), (h, w, k)
        for thr in (1, 5):
            el.set_property("cc-threshold", thr); one.set_property("cc-threshold", thr)
            assert el.transform_ip(m) == one.transform_ip(m), (h, w, k, thr)
        el.close(); one.close()


def _seam_cases(h, w):
    cases = {}
    m = np.zeros((h, w), np.uint8)
    for s, y in enumerate(SEAM_ROWS):                  # diagonal pairs straddling every seam, both directions, both parities
        for x in (0, 1, 2, 3, 100 + s, 101 + s, w - 3):
            m[y - 1, x] = 1; m[y, x + 1] = 1           # the upper pixel is north-west of the lower one
        for x in (20, 21, 200 + s, 201 + s, w - 2):
            m[y - 1, x + 1] = 1; m[y, x] = 1           # north-east
    cases["diagonals"] = m
    m = np.zeros((h, w), np.uint8)
    m[:, 100] = 1; m[:, w - 1] = 1; m[:, 0] = 1
    cases["vertical_lines"] = m
    m = np.zeros((h, w), np.uint8)
    m[0, 300] = 1; m[0:h - 20, 301] = 1                 # first block in band 0, the bulk in band 3
    m[h - 60: h, 250: 420] = 1
    m[h - 40: h - 30, 260: 280] = 0
    cases["first_block_in_band0"] = m
    m = np.zeros((h, w), np.uint8)
    m[h - 1, :] = 1; m[h - 1, ::7] = 0; m[h - 2, 3] = 1
    m[::3, 5] = 1
    cases["last_row"] = m
    m = np.zeros((h, w), np.uint8)
    m[::2, ::2] = 1                                     # isolated pixels: the most components, many per seam
    cases["dots"] = m
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("h,w", [(H8, W8), (H8 - 1, W8 - 1)])
def test_native_8k_element_against_the_oracle(h, w):
    """The 8K grid picks 4 bands by itself; every synthetic mask family and hand-made seam cases (an odd last pixel row
    in the 269-row grid) give the oracle's labels, statistics and boxes."""
    el = BboxCc(w, h, 1, cluster=True)
    cases = dict(synth.mask_patterns(h, w, seed=3))
    cases.update(_seam_cases(h, w))
    for name, m in cases.items():
        _check_element(el, np.ascontiguousarray(m, dtype=np.uint8), (1, 30), name)
    el.close()


@pytest.mark.gpu
def test_ccl_cluster_dense_mask_stress_8k():
    """Bernoulli masks around the percolation threshold at 8K: the CAS links and compressions now race across CTAs of a
    cluster as well; several hundred masks, twice, against the C oracle."""
    n = 320
    rng = np.random.default_rng(8)
    dens = rng.uniform(0.3, 0.8, n).astype(np.float32)
    masks = (rng.random((n, H8, W8), dtype=np.float32) < dens[:, None, None]).astype(np.uint8)
    p = BlobPipeline(W8, H8, weights.to_blob(weights.random_weights(0)), 8, 4 + n // 8, cc_threshold=1, ccl_cluster=True)
    want = c_oracle.bboxcc_batch(masks, 1)
    p.set_profiling(True)
    for _ in range(2):
        p.load_masks(masks)
        p.ccl()
        got = p.fetch_boxes()
        bad = [i for i in range(n) if got[i] != want[i]]
        assert not bad, (len(bad), bad[:5], float(dens[bad[0]]))
    assert "ccl_bbox_cluster" in p.last_timings()


@pytest.mark.gpu
@pytest.mark.parametrize("head_bias", [-0.5, 0.0])
def test_whole_path_at_8k(head_bias):
    """tensorise -> BlobNet (tcgen05; enc2-enc4 with a one-stage ring at this size) -> cluster CCL at 480x270: boxes
    bit-exact for the device mask, logits within the fp16 bars of the fp32 oracle on a window."""
    wts = weights.random_weights(1, head_bias=head_bias)
    frames = synth.synth_streams(1, 5, H8, W8, config_idx=3)
    p = BlobPipeline(W8, H8, weights.to_blob(wts), 1, 5, keep_logits=True, keep_stacked=True, ccl_cluster=True)
    blobs = p.process(frames)
    mask, logits = p.read_mask(), p.read_logits()
    assert len(blobs) == 2
    assert blobs == c_oracle.bboxcc_batch(mask, 1)
    assert max(len(deserialize_vec(b)) for b in blobs) >= 1
    stacked = p.read_stacked()[:1]
    assert (stacked == mpr.tensorise_stream(frames[0], 4, 1)[:1]).all()
    ref = blobnet_ref.blobnet_forward(wts, mpr.stacked_to_nchw(stacked, 4))
    scale = float(np.abs(ref).max())
    assert float(np.abs(logits[:1] - ref).max()) <= LOGIT_REL_TOL * scale
    assert float(((logits[:1] > 0) != (ref > 0)).mean()) <= MAX_FLIP


@pytest.mark.gpu
def test_tcgen05_layers_match_validation_kernels_at_8k():
    """Every tcgen05 layer against the fp32 validation kernels on identical inputs at 480x270, where enc2-enc4 run with
    a one-stage operand ring that the smaller grids never use."""
    wts = weights.random_weights(11, head_bias=-1.0)
    frames = synth.synth_streams(1, 4, H8, W8, config_idx=2)
    p = BlobPipeline(W8, H8, weights.to_blob(wts), 1, 4, impl=_lib.IMPL_SIMT, keep_logits=True, ccl_cluster=True)
    p.load_frames(frames)
    p.run()
    ref_act = {layer: p.read_activation(layer) for layer in range(8)}
    ref_logits = p.read_logits()
    for layer in range(8):
        p.run_layer(layer, _lib.IMPL_TCGEN05)
        if layer < 7:
            a = p.read_activation(layer + 1)
            assert np.abs(a - ref_act[layer + 1]).max() <= 4e-3 * np.abs(ref_act[layer + 1]).max(), layer
            p.run_layer(layer, _lib.IMPL_SIMT)
        else:
            assert np.abs(p.read_logits() - ref_logits).max() <= 4e-3 * np.abs(ref_logits).max()


@pytest.mark.gpu
def test_streaming_and_chunks_at_8k():
    wts = weights.random_weights(0, head_bias=-0.5)
    blob = weights.to_blob(wts)
    batches = [synth.synth_streams(2, 5, H8, W8, config_idx=50 + i) for i in range(3)]
    one = BlobPipeline(W8, H8, blob, 2, 5, n_chunks=1, ccl_cluster=True)
    two = BlobPipeline(W8, H8, blob, 2, 5, n_chunks=2, ccl_cluster=True)
    want = [one.process(b) for b in batches]
    assert [two.process(b) for b in batches] == want
    for p in (one, two):
        got = []
        p.submit(batches[0])
        for k in range(len(batches)):
            if k + 1 < len(batches):
                p.submit(batches[k + 1])
            got.append(p.collect())
        assert got == want


@pytest.mark.gpu
def test_grids_that_fit_one_cta_keep_the_single_cta_kernel():
    wts = weights.random_weights(0, head_bias=-1.0)
    frames = synth.synth_streams(2, 8, 45, 80, config_idx=4)
    a = BlobPipeline(80, 45, weights.to_blob(wts), 2, 8)
    b = BlobPipeline(80, 45, weights.to_blob(wts), 2, 8, ccl_cluster=True)
    want = a.process(frames)
    b.set_profiling(True)
    assert b.process(frames) == want
    b.load_frames(frames); b.run(); b.sync()
    names = b.last_timings()
    assert "ccl_bbox" in names and "ccl_bbox_cluster" not in names
    # forced bands on the same grid: the cluster kernel, the same bytes
    c = BlobPipeline(80, 45, weights.to_blob(wts), 2, 8, ccl_cluster=True, ccl_bands=3)
    c.set_profiling(True)
    assert c.process(frames) == want
    c.load_frames(frames); c.run(); c.sync()
    assert "ccl_bbox_cluster" in c.last_timings()


@pytest.mark.gpu
def test_single_cta_and_cluster_handles_on_two_threads():
    """A 4K single-CTA element and an 8K cluster element, each on its own thread: both kernels set their shared-memory
    attribute on every launch, always to the same value, so concurrent use cannot take it away from the other."""
    rng = np.random.default_rng(4)
    cfg = [(135, 240, False), (H8, W8, True)]
    els, masks, want = [], [], []
    for h, w, cl in cfg:
        els.append(BboxCc(w, h, 1, cluster=cl))
        ms = [(rng.random((h, w)) < d).astype(np.uint8) for d in (0.2, 0.45, 0.6)]
        masks.append(ms)
        want.append([c_oracle.bboxcc(m, 1) for m in ms])
    errors = []

    def worker(i):
        try:
            for r in range(12):
                j = r % 3
                assert els[i].transform_ip(masks[i][j]) == want[i][j]
        except Exception as e:  # noqa: BLE001
            errors.append((i, repr(e)))

    ts = [threading.Thread(target=worker, args=(i,)) for i in range(2)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errors, errors
