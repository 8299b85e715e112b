"""Every launch plan the tcgen05 BlobNet layers can pick, against an fp64 restatement with a per-element error bound.

Each layer picks its plan (kernel family, tile configuration, operand-ring depth) on the host from a candidate list, by what
fits shared memory for the grid WIDTH (cova_abi.cu, plan_layer).  cova_blobnet_plan reports that choice without a device.
The CPU tests below pin known plans, sweep the widths for reachability and the maximum width, and check that CASES (the
GPU cases) reach every plan any width can select.  The GPU tests run each case layer by layer against the fp32 validation
kernels and an fp64 restatement, and the whole path against the oracles.

Per-element bound of a layer output (u = 2^-11, the unit round-off of fp16):
    |got - ref| <= c * u * mag + u * |ref| + FLOOR
ref is the layer in fp64 on the device's own fp16 input; mag is the same layer on |x| with the magnitudes of the weights
the kernel rounds to fp16 and without bias, shift and ReLU: |s| * (|W| * |x|) max-pooled, then PointWiseTN on |tn_w| plus
the residual (encoder); |s| * (|W| * relu(x)) (decoder); |W . head_w| * relu(x) (folded head).  It bounds how an error
of the products propagates: max-pooling, ReLU and the max of PointWiseTN are 1-Lipschitz, BatchNorm scales it by |s|.
Derivation of c from the kernels' rounding points:
    1      the weights are rounded to fp16 once (x / 6 and BatchNorm stay out of the encoder weights, the head is folded
           in double): each product w * x, x an exact fp16 value, is off by at most u * |w x|
    1      the fused block-1 kernel rounds the pooled activation to fp16 before PointWiseTN (blobnet_enc1.cuh): at most
           u * |y| <= u * mag_pool, carried through PointWiseTN like mag
    1/4    fp32 accumulation of at most K = 9 * 64 (block 4) or 4 * 128 (dec0) products plus ~16 fp32 epilogue operations:
           (K + 16) * 2^-24 = (K + 16) / 8192 * u < 0.08 u per unit of mag, rounded up with margin
    c = 9/4.  The u * |ref| term is the final rounding of the output to fp16; FLOOR covers fp16 subnormals and the fp32
           round-off of bias, BatchNorm shift and PointWiseTN where the output cancels to nearly zero.
The fp32 validation kernels have fp32 weights and no intermediate fp16 rounding: only the accumulation item remains, so
their outputs must meet c = 1/4."""
import ctypes
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from cova_b200 import _lib, synth, weights
from cova_b200.elements import BlobPipeline
from oracle import blobnet_ref, c_oracle, metapreprocess_ref as mpr

U = 2.0 ** -11
C_KERNEL = 9 / 4
C_SIMT = 1 / 4
FLOOR = 2.0 ** -16
ACT_REL_TOL, LOGIT_REL_TOL, MAX_FLIP = 4e-3, 5e-3, 1e-3      # the bars of tests/test_gpu_parity.py
MAX_WIDTH = 736                                               # include/cova_b200.h: block 4 runs out of shared memory first
DEBUGS = (0, 4, 8)                                            # default; bit 2: positions-as-M blocks 2 and 4; bit 3: weights-stationary block 3
NAMES = ("enc1", "enc2", "enc3", "enc4", "dec0", "dec1", "dec2", "dec3+head")
ENC_COUT, DEC_COUT = (16, 32, 64, 128), (64, 32, 16, 16)
# length of every candidate list of cova_abi.cu: (layer, family) -> entries
CANDIDATES = {(0, _lib.PLAN_ENC1): 1, (1, _lib.PLAN_WS): 3, (2, _lib.PLAN_WS): 2, (3, _lib.PLAN_WS): 2,
              (1, _lib.PLAN_POS): 3, (2, _lib.PLAN_POS): 2, (3, _lib.PLAN_POS): 1,
              (4, _lib.PLAN_POS): 1, (5, _lib.PLAN_POS): 1, (6, _lib.PLAN_POS): 2, (7, _lib.PLAN_POS): 3}
# GPU cases (w_mb, h_mb, debug): together they select every (layer, family, config, n_stage) that any width selects
# (test_cases_cover_every_reachable_plan).  Heights 16..20: height does not change a plan, short grids keep the oracle cheap.
CASES = [(16, 17, 0), (736, 17, 0), (16, 16, 4), (121, 16, 4), (253, 18, 4), (309, 16, 4), (509, 19, 4), (625, 16, 4),
         (16, 20, 8), (161, 20, 8), (253, 17, 8), (599, 18, 8), (625, 16, 8)]
ERRLOG = os.environ.get("COVA_PARITY_LOG")


def _log(line):
    if ERRLOG:
        with open(ERRLOG, "a") as f:
            f.write(line + "\n")


def _plan(w, h, n, dbg=0, n_sms=148):
    return _lib.blobnet_plan(w, h, n, dbg, n_sms)


def _key(plan):
    return plan["family"], plan["config"], plan["n_stage"]


def _sweep(dbg, hi=MAX_WIDTH + 16):
    """width -> plans (None where a layer has no plan)."""
    out = {}
    for w in range(16, hi + 1):
        try:
            out[w] = _plan(w, 16, 64, dbg)
        except _lib.CovaError as e:
            assert e.code == _lib.E_UNSUPPORTED
            out[w] = None
    return out


_SWEEPS = {}


def sweeps():
    if not _SWEEPS:
        _SWEEPS.update({dbg: _sweep(dbg) for dbg in DEBUGS})
    return _SWEEPS


def reachable():
    return {(layer, *_key(p)) for s in sweeps().values() for plans in s.values() if plans for layer, p in enumerate(plans)}


# ----------------------------------------------------------------------------------------------------------------- CPU
def test_known_plans():
    """720p, 1080p, 4K and 8K: (family, config, n_stage) per layer.  At 8K blocks 2-4 run a one-stage ring."""
    E1, WS, POS = _lib.PLAN_ENC1, _lib.PLAN_WS, _lib.PLAN_POS
    want = {
        80: [(E1, 0, 8), (WS, 0, 2), (POS, 0, 2), (WS, 0, 2), (POS, 0, 4), (POS, 0, 4), (POS, 0, 3), (POS, 0, 2)],
        120: [(E1, 0, 8), (WS, 0, 2), (POS, 0, 2), (WS, 0, 2), (POS, 0, 4), (POS, 0, 4), (POS, 0, 3), (POS, 0, 2)],
        240: [(E1, 0, 8), (WS, 1, 2), (POS, 1, 2), (WS, 1, 2), (POS, 0, 4), (POS, 0, 4), (POS, 0, 3), (POS, 0, 2)],
        480: [(E1, 0, 8), (WS, 0, 1), (POS, 1, 1), (WS, 0, 1), (POS, 0, 4), (POS, 0, 3), (POS, 0, 2), (POS, 1, 2)],
    }
    for w, h in ((80, 45), (120, 68), (240, 135), (480, 270)):
        plans = _plan(w, h, 1024)
        assert [_key(p) for p in plans] == want[w], w
        assert [_key(p) for p in _plan(w, 16, 3)] == want[w], w           # height and window count do not matter
        assert plans[1]["tps"] == (3 if w <= 156 else 2 if w <= 252 else 3) and plans[1]["tile"] == 192
        assert plans[0]["tps"] == 2 and plans[0]["tile"] == 128
        for layer, p in enumerate(plans):
            assert 1 <= p["ctas"] <= 148 and p["n_groups"] >= 1, (w, layer, p)


def test_query_arguments_and_ctas():
    plans = _plan(80, 45, 8192, n_sms=148)
    assert all(p["ctas"] == min(148 // (2 if layer == 4 else 1), p["n_groups"]) * (2 if layer == 4 else 1)
               for layer, p in enumerate(plans[1:], 1))
    assert [p["ctas"] for p in _plan(80, 45, 8192, n_sms=7)] == [7, 7, 7, 7, 6, 7, 7, 7]
    lib = _lib.load()
    out = (_lib.LayerPlan * 8)()
    assert lib.cova_blobnet_plan(80, 45, 0, 0, 148, out) == _lib.E_INVAL
    assert lib.cova_blobnet_plan(80, 45, 8, 0, 0, out) == _lib.E_INVAL
    assert lib.cova_blobnet_plan(15, 45, 8, 0, 148, out) == _lib.E_UNSUPPORTED
    assert lib.cova_blobnet_plan(MAX_WIDTH + 1, 16, 8, 0, 148, out) == _lib.E_UNSUPPORTED
    assert b"enc4" in lib.cova_last_error()
    assert [p.family != 0 for p in out] == [True] * 3 + [False] * 5           # filled up to the layer without a plan


def test_every_candidate_is_reachable_and_the_width_limit():
    s = sweeps()
    assert all(s[0][w] is not None for w in range(16, MAX_WIDTH + 1))
    assert all(s[0][w] is None for w in range(MAX_WIDTH + 1, MAX_WIDTH + 17))
    seen = {}
    for layer, fam, cfg, _ in reachable():
        seen.setdefault((layer, fam), set()).add(cfg)
    assert {k: len(v) for k, v in seen.items()} == CANDIDATES
    assert all(v == set(range(CANDIDATES[k])) for k, v in seen.items())
    # creation refuses the width no plan fits, before it looks for a device; the limit itself passes that check
    blob = weights.to_blob(weights.random_weights(0))
    lib = _lib.load()
    h = ctypes.c_void_p()
    buf = ctypes.create_string_buffer(blob, len(blob))
    for w, ok in ((MAX_WIDTH + 1, False), (MAX_WIDTH + 100, False), (MAX_WIDTH, True)):
        rc = lib.cova_pipeline_new(ctypes.byref(h), 0, w, 16, 4, 1, 1, 8, buf, len(blob), 1, 0)
        if ok:
            assert rc != _lib.E_UNSUPPORTED, lib.cova_last_error()
            if rc == _lib.OK:
                lib.cova_pipeline_free(h)
        else:
            assert rc == _lib.E_UNSUPPORTED and (w > MAX_WIDTH + 1 or b"enc4" in lib.cova_last_error()), w


def test_cases_cover_every_reachable_plan():
    covered = {(layer, *_key(p)) for w, h, dbg in CASES for layer, p in enumerate(_plan(w, h, 8, dbg))}
    missing = sorted(reachable() - covered)
    assert not missing, "plans no GPU case runs (layer, family, config, n_stage): " + ", ".join(
        f"{NAMES[m[0]]} {m[1:]}" for m in missing)
    assert all(16 <= h <= 20 for _, h, _ in CASES) and any(h % 2 for _, h, _ in CASES)
    for w, h, dbg in CASES:                                   # a window count with a partial last tile group in every layer
        choose_windows(w, h, dbg, 148)


# fp64 restatement of one layer ------------------------------------------------------------------------------------------
def _w64(wts):
    return {k: v.astype(np.float64) for k, v in wts.items()}


def _scale(w, prefix):
    return torch.from_numpy(w[f"{prefix}.bn_gamma"] / np.sqrt(w[f"{prefix}.bn_var"] + blobnet_ref.BN_EPS))


def _crop(y, target):
    ct, cb = blobnet_ref._crop_amounts(y.shape[-2], target[0])
    cl, cr = blobnet_ref._crop_amounts(y.shape[-1], target[1])
    return y[..., ct: y.shape[-2] - cb, cl: y.shape[-1] - cr]


def restate(w, layer, x, target=None):
    """(ref, mag) of `layer` (0..3 encoder blocks, 4..6 dec0..dec2, 7 dec3 + head) in float64 on its input x
    [N, C, T, H, W] as the device holds it.  Outputs as the device stores them: blocks 1-3 all four frames, block 4 frame 0,
    decoder blocks after their ReLU, the head as logits [N, H, W].  target: (H, W) of a decoder output."""
    x = torch.as_tensor(x, dtype=torch.float64)
    if layer < 4:
        i = layer
        n, c, t, h, wd = x.shape
        cw = torch.from_numpy(w[f"enc{i}.conv_w"]) / (6.0 if i == 0 else 1.0)   # block 1's input is clip(x, 0, 6)
        y = x.permute(0, 2, 1, 3, 4).reshape(n * t, c, h, wd)
        ref = blobnet_ref._bn(torch.relu(F.conv2d(y, cw, torch.from_numpy(w[f"enc{i}.conv_b"]), padding=1)), w, f"enc{i}")
        mag = F.conv2d(y.abs(), cw.abs(), padding=1) * _scale(w, f"enc{i}").abs().view(1, -1, 1, 1)
        out = []
        for v in (ref, mag):
            v = F.pad(F.max_pool2d(v, 2), (wd % 2, 0, h % 2, 0))              # zero column left / row on top when odd
            out.append(v.reshape(n, t, *v.shape[1:]).permute(0, 2, 1, 3, 4))
        ref = blobnet_ref._pointwise_tn(out[0], w[f"enc{i}.tn_w1"], w[f"enc{i}.tn_w2"])
        mt = out[1].permute(0, 1, 3, 4, 2)
        mag = out[1] + ((mt @ torch.from_numpy(np.abs(w[f"enc{i}.tn_w1"]))) @ torch.from_numpy(np.abs(w[f"enc{i}.tn_w2"]))).permute(0, 1, 4, 2, 3)
        return (ref[:, :, :1], mag[:, :, :1]) if i == 3 else (ref, mag)
    i = layer - 4
    xr = torch.relu(x[:, :, 0])
    cw = torch.from_numpy(w[f"dec{i}.convt_w"])
    ref = _crop(F.conv_transpose2d(xr, cw, torch.from_numpy(w[f"dec{i}.convt_b"]), stride=2), target)
    if i < 3:
        mag = _crop(F.conv_transpose2d(xr, cw.abs(), stride=2), target) * _scale(w, f"dec{i}").abs().view(1, -1, 1, 1)
        return torch.relu(blobnet_ref._bn(ref, w, f"dec{i}"))[:, :, None], mag[:, :, None]
    hw = torch.from_numpy(w["head_w"]).view(1, -1, 1, 1)
    fold = (cw * hw).sum(1, keepdim=True)
    mag = _crop(F.conv_transpose2d(xr, fold.abs(), stride=2), target)[:, 0]
    return (ref * hw).sum(1) + float(w["head_b"][0]), mag


def bound_ratio(got, ref, mag, c):
    """max over elements of |got - ref| / (c u mag + u |ref| + FLOOR): <= 1 passes."""
    got = np.asarray(got, np.float64)
    ref, mag = np.asarray(ref, np.float64), np.asarray(mag, np.float64)
    assert got.shape == ref.shape == mag.shape, (got.shape, ref.shape, mag.shape)
    return float((np.abs(got - ref) / (c * U * mag + U * np.abs(ref) + FLOOR)).max())


@pytest.mark.parametrize("h,w", [(19, 121), (20, 16), (17, 37)])
def test_restatement_matches_the_oracle_layer_by_layer(h, w):
    """The per-layer fp64 restatement, fed the fp32 oracle's own intermediates, gives the oracle's next intermediate (odd
    extents: zero pad on top / left, crops)."""
    wts = weights.random_weights(9, head_bias=-1.0)
    for i in range(4):
        wts[f"enc{i}.bn_gamma"][::3] *= -1
    frames = synth.synth_streams(1, 6, h, w, config_idx=5)
    x = mpr.stacked_to_nchw(mpr.tensorise_stream(frames[0], 4, 1), 4)
    logit, inter = blobnet_ref.blobnet_forward(wts, x, return_intermediates=True)
    acts = [np.clip(x, 0, 6), inter["enc0"], inter["enc1"], inter["enc2"], inter["enc3"][:, :, :1]]
    acts += [np.maximum(inter[f"dec{i}"], 0)[:, :, None] for i in range(3)]
    w64 = _w64(wts)
    for layer in range(8):
        want = logit if layer == 7 else acts[layer + 1][:, : DEC_COUT[layer - 4]] if layer >= 4 else acts[layer + 1]
        target = (h, w) if layer == 7 else want.shape[-2:]
        ref, mag = (t.numpy() for t in restate(w64, layer, acts[layer], target))
        assert ref.shape == want.shape == mag.shape, NAMES[layer]
        assert np.abs(ref - want).max() <= 1e-5 * (np.abs(want).max() + mag.max()), NAMES[layer]
        assert (mag >= 0).all() and (mag > 0).any()


def test_per_element_bound_flags_what_the_global_bar_misses():
    """A reference output with one small element perturbed by 8 u of its magnitude bound: the per-element check flags it,
    the global bar (4e-3 of the largest |y|) does not.  Host data only."""
    w = _w64(weights.random_weights(4, head_bias=-1.0))
    rng = np.random.default_rng(0)

    def sparse(shape):                                        # post-ReLU activations, mostly zero
        return np.maximum(rng.normal(0, 1, shape), 0) * (rng.random(shape) < 0.1)
    cases = [(1, sparse((2, 16, 4, 12, 20)), None), (5, sparse((2, 128, 1, 6, 10)), (11, 19))]
    for layer, x, target in cases:
        ref, mag = (t.numpy() for t in restate(w, layer, x, target))
        assert bound_ratio(ref, ref, mag, C_KERNEL) == 0.0
        # fp16 rounding of the output alone stays inside the bound
        assert bound_ratio(ref.astype(np.float16), ref, mag, C_KERNEL) <= 1.0
        delta = 8 * U * mag
        ok = (delta < ACT_REL_TOL * np.abs(ref).max()) & (np.abs(ref) < 5 * mag) & (mag > 1e-2)
        assert ok.any(), layer
        k = np.flatnonzero(ok.ravel())[np.argmin(np.abs(ref).ravel()[ok.ravel()])]
        bad = ref.copy().ravel()
        bad[k] += delta.ravel()[k]
        bad = bad.reshape(ref.shape)
        assert np.abs(bad - ref).max() <= ACT_REL_TOL * np.abs(ref).max()          # the global bar passes it
        assert bound_ratio(bad, ref, mag, C_KERNEL) > 1.0, layer                   # the per-element bound does not


# ----------------------------------------------------------------------------------------------------------------- GPU
def _n_sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _extents(h, w):
    sizes = [(h, w)]
    for _ in range(4):
        sizes.append(((sizes[-1][0] + 1) // 2, (sizes[-1][1] + 1) // 2))
    return sizes


def _positions(layer, h, w, n):
    """(positions per window, Tn) of the input planes of `layer` (common.cuh, make_geom); block 1: per frame."""
    sizes = _extents(h, w)
    ih, iw = sizes[layer] if layer < 4 else sizes[8 - layer]
    s = ((ih + 1) // 2 + 1) * ((iw + 1) // 2 + 1)
    return s, (4 if 1 <= layer <= 3 else 1)


def _last_groups(h, w, n, plans):
    """per layer: is the last tile group partial, and the window its first position belongs to (layers 1..7)."""
    out = {}
    for layer in range(1, 8):
        p = plans[layer]
        s, tn = _positions(layer, h, w, n)
        span = p["tps"] * p["tile"]
        out[layer] = ((n * s * tn) % span != 0, min(n - 1, (p["n_groups"] - 1) * span // (s * tn)))
    return out


def choose_windows(w, h, dbg, n_sms, cap_mb=400_000):
    """The window count for a case: the last tile group of every layer partial, then as many layers as possible with more
    tile groups than CTAs (ring slots reused), within a budget of cap_mb macroblocks; the smallest such count."""
    best = None
    for n in range(2, max(3, min(256, cap_mb // (w * h))) + 1):
        plans = _plan(w, h, n, dbg, n_sms)
        lg = _last_groups(h, w, n, plans)
        if not all(partial for partial, _ in lg.values()):
            continue
        score = sum(plans[layer]["n_groups"] > plans[layer]["ctas"] for layer in range(8))
        if best is None or score > best[0]:
            best = (score, n)
    assert best is not None, (w, h, dbg)
    return best[1]


def _weights(seed, head_bias=-1.0):
    wts = weights.random_weights(seed, head_bias=head_bias)
    for i in range(4):                                        # negative BatchNorm scales: min-pool / negated-weight paths
        wts[f"enc{i}.bn_gamma"][::3] = -wts[f"enc{i}.bn_gamma"][::3]
    return wts


def _layer_output(p, layer):
    if layer < 3:
        return p.read_activation(layer + 1)
    if layer == 3:
        return p.read_activation(4)
    if layer < 7:
        return p.read_activation(layer + 1)[:, : DEC_COUT[layer - 4]]
    return p.read_logits()


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,dbg", CASES)
def test_layer_plans_against_fp64_restatement(w, h, dbg):
    """Each tcgen05 layer on the validation kernels' input: every window within the existing bar of the fp32 validation
    kernel, sampled windows (first, last, those holding a layer's last partial tile group) within the per-element fp64
    bound, and the plan it launched is the one cova_blobnet_plan reports."""
    n_sms = _n_sms()
    n = choose_windows(w, h, dbg, n_sms)
    plans = _plan(w, h, n, dbg, n_sms)
    sample = sorted({0, n - 1} | {win for _, win in _last_groups(h, w, n, plans).values()})
    wts = _weights(w + h + dbg)
    w64 = _w64(wts)
    frames = synth.synth_streams(1, n + 3, h, w, config_idx=w % 7)
    p = BlobPipeline(w, h, weights.to_blob(wts), 1, n + 3, impl=_lib.IMPL_SIMT, keep_logits=True)
    p.set_debug(dbg)
    p.load_frames(frames)
    p.run()
    act = {layer: p.read_activation(layer) for layer in range(8)}
    act[8] = p.read_logits()
    targets = {4: act[5].shape[-2:], 5: act[6].shape[-2:], 6: act[7].shape[-2:], 7: (h, w)}
    worst = {}
    for layer in range(8):
        p.run_layer(layer, _lib.IMPL_TCGEN05)
        got = _layer_output(p, layer)
        simt = act[8] if layer == 7 else (act[layer + 1][:, : DEC_COUT[layer - 4]] if layer >= 4 else act[layer + 1])
        assert got.shape == simt.shape
        assert np.abs(got - simt).max() <= ACT_REL_TOL * np.abs(simt).max(), (NAMES[layer], "vs validation kernel")
        if layer < 3:                                         # the t = 0 skip inside the decoder input is the same value
            skip = p.read_activation(7 - layer)[:, DEC_COUT[2 - layer]:, 0]
            assert (skip == got[:, :, 0]).all(), NAMES[layer]
        ref, mag = (t.numpy() for t in restate(w64, layer, act[layer][sample], targets.get(layer)))
        worst[layer] = bound_ratio(got[sample], ref, mag, C_KERNEL)
        simt_ratio = bound_ratio(simt[sample], ref, mag, C_SIMT)
        _log(f"tile_plans {w}x{h} dbg={dbg} n={n} {NAMES[layer]} plan={plans[layer]} ratio={worst[layer]:.3g} simt_ratio={simt_ratio:.3g}")
        assert simt_ratio <= 1.0, (NAMES[layer], "the restatement disagrees with the fp32 validation kernel", simt_ratio)
        assert worst[layer] <= 1.0, (NAMES[layer], plans[layer], worst[layer])
        if layer < 7:
            p.run_layer(layer, _lib.IMPL_SIMT)
    assert p.last_plan() == plans


@pytest.mark.gpu
@pytest.mark.parametrize("w,h", sorted({(w, h) for w, h, _ in CASES}))
def test_whole_path_at_default_debug(w, h):
    """process() at the covering widths (the widest supported grid included): logits of every window within the bars of the
    fp32 oracle, boxes bit-exact against the C oracle for the device mask (up to 368 blocks per row).  The flip bar is a
    fraction, so at least 4096 pixels are compared; and a pixel may only flip where the oracle's logit lies within the
    logit error bar of zero - a flip is that error crossing the threshold, nothing else."""
    n_sms, n = _n_sms(), max(8, -(-4096 // (w * h)))
    wts = _weights(2 * w + h, head_bias=0.0)
    frames = synth.synth_streams(1, n + 3, h, w, config_idx=h)
    p = BlobPipeline(w, h, weights.to_blob(wts), 1, n + 3, keep_logits=True)
    boxes = p.process(frames)
    assert len(boxes) == n and p.last_plan() == _plan(w, h, n, 0, n_sms)
    logits, mask = p.read_logits(), p.read_mask()
    ref = blobnet_ref.blobnet_forward(wts, mpr.stacked_to_nchw(mpr.tensorise_stream(frames[0], 4, 1), 4))
    scale = float(np.abs(ref).max())
    err = float(np.abs(logits - ref).max())
    flipped = (logits > 0) != (ref > 0)
    _log(f"whole_path {w}x{h} n={n} logit_err_rel={err / scale:.3g} flips={int(flipped.sum())}/{flipped.size}")
    assert err <= LOGIT_REL_TOL * scale
    assert float(flipped.mean()) <= MAX_FLIP
    assert (np.abs(ref[flipped]) <= LOGIT_REL_TOL * scale).all()
    assert (mask == (logits > 0)).all()
    assert boxes == c_oracle.bboxcc_batch(mask, 1)


@pytest.mark.gpu
@pytest.mark.parametrize("w", [200, 400, 700])
def test_whole_tile_decoder_accumulators_are_bit_identical(w):
    """Debug bit 6 (whole-tile dec0 / dec1 accumulators instead of two half-tiles) at widths of three different dec0 / dec1
    ring depths: dec0 / dec1 outputs and logits byte-identical to the default."""
    h, n = 17, 12
    depths = [(pl[4]["n_stage"], pl[5]["n_stage"]) for pl in [_plan(w, h, n)]]
    assert depths[0] == {200: (4, 4), 400: (4, 3), 700: (3, 2)}[w]
    wts = _weights(w)
    frames = synth.synth_streams(1, n + 3, h, w, config_idx=3)
    p = BlobPipeline(w, h, weights.to_blob(wts), 1, n + 3, keep_logits=True)
    out = []
    for dbg in (0, 64):
        p.set_debug(dbg)
        p.process(frames)
        out.append((p.read_activation(5), p.read_activation(6), p.read_logits()))
    for a, b in zip(*out):
        assert a.tobytes() == b.tobytes()


@pytest.mark.gpu
def test_width_limit_and_debug_routes_without_a_plan():
    """One macroblock past the widest supported grid is refused at creation; a debug route with no plan at the pipeline's
    width (positions-as-M block 2 beyond 688 macroblocks) is refused by the run call before any BlobNet layer launches."""
    blob = weights.to_blob(weights.random_weights(0, head_bias=-1.0))
    for impl in (_lib.IMPL_TCGEN05, _lib.IMPL_SIMT):
        with pytest.raises(_lib.CovaError) as e:
            BlobPipeline(MAX_WIDTH + 1, 16, blob, 1, 5, impl=impl)
        assert e.value.code == _lib.E_UNSUPPORTED
    w = 700
    with pytest.raises(_lib.CovaError) as e:
        _plan(w, 16, 2, 4)
    assert e.value.code == _lib.E_UNSUPPORTED
    p = BlobPipeline(w, 16, blob, 1, 5)
    frames = synth.synth_streams(1, 5, 16, w, config_idx=1)
    p.set_debug(4)
    p.load_frames(frames)
    p.tensorise()
    before = p.launch_count()
    for call in (p.blobnet, p.run):
        with pytest.raises(_lib.CovaError) as e:
            call()
        assert e.value.code == _lib.E_UNSUPPORTED
    assert p.launch_count() - before <= 1                      # run() re-tensorises; no BlobNet layer was launched
    assert all(pl["family"] == 0 for pl in p.last_plan())
    p.set_debug(0)
    assert len(p.process(frames)) == 2
