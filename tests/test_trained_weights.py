"""BlobNet on weights with trained statistics (weights.trained_like_weights): every layer, window and channel against an
fp64 restatement on the weights the device multiplies by, with a per-element bound derived from the kernels' rounding
points.

Trained BatchNorm normalises channels whose raw scales differ by decades: one layer holds channels of maximum 1e-3 next to
ones of 45, dead channels (bias -1e3) whose output is the BatchNorm shift alone, shifts of tens.  A bar relative to a
tensor's largest value cannot see a small channel zeroed, read with a neighbour's scale or shift, or its shift rounded to
fp16; the bound below is per element, and its only absolute term is half the fp16 subnormal spacing.

The restatement is test_tile_plans.restate, fed the DEVICE IMAGE of the weights (device_weights): the fp16 operands the
tensor cores multiply (block 1: fp16(fp32(W) / 6), other layers fp16(W), the head folded into dec3 in double and rounded
to fp32 then fp16) and the fp32 epilogue constants the host folds (scale s = gamma / sqrtf(var + 1e-3f), encoder shift
beta - mean s, decoder offset (b - mean) s + beta, head constant head_b + sum head_w b).  The weight rounding of
test_tile_plans (its c = 1 term) is then gone.  Per-element bound of a tcgen05 layer output (u = 2^-11, fp16's unit
round-off):
    |got - ref| <= C_ACC u mag  +  [block 1: u (mag + E)]  +  u |ref|  +  C_CONST E  +  ABS
  mag    test_tile_plans.restate's magnitude: |s| (|W| * |x|) pooled and carried through PointWiseTN on |tn_w| (encoder),
         |s| (|W| * relu(x)) (decoder), |fold| * relu(x) (head); no bias, shift or ReLU.
  E      the per-channel epilogue constant, as a magnitude: k = |s| max(b, 0) + |shift| carried through PointWiseTN on
         |tn_w| like mag (encoder: relu(c + b) <= |c| + max(b, 0), so the pooled BatchNorm value is at most mag_pool + k);
         |offset| (decoder); 0 (head: its constant is added once, an error inside u |ref|).
  C_ACC = 1/4  fp32 accumulation of at most K = 576 products (block 4) and ~16 fp32 epilogue operations on them:
         (K + 16) 2^-24 < 0.08 u per unit of mag (as test_tile_plans), rounded up with margin.
  u (mag + E)  block 1 rounds its pooled activation (|y| <= mag_pool + k) to fp16 before PointWiseTN (blobnet_enc1.cuh).
  u |ref|      the output's rounding to fp16.
  C_CONST = 2^-20  the fp32 operations that touch the constant: bias add and BatchNorm FMA (2) and the eight FMAs of
         PointWiseTN (8) each round at 2^-24 of a value bounded by mag + E: 10 2^-24 < 16 2^-24.  Rounding a shift or
         offset to fp16 moves an output by up to 2^-12 |shift| = 256 2^-20 |shift|: it stands out wherever mag and |ref|
         are small next to the shift.
  ABS = 2^-25  half the fp16 subnormal spacing (u |ref| vanishes there).
The fp32 validation (SIMT) kernels multiply fp32 weights, apply BatchNorm from gamma / var / mean in fp32 and run dec3 and
then the head unfolded, accumulating the bias with the products; their reference is the restatement on the fp32 weights,
their head magnitude sum |W| |head_w| (not |fold|), and their bound C_SIMT u (mag + E_simt) + u |ref| + ABS with
E_simt = |s| (|b| + |mean|) + |beta| (encoder: through PointWiseTN), |s| (|b| + |mean|) + |beta| (decoder),
|head_b| + sum |head_w| |b| (head), C_SIMT = 1/4 as in test_tile_plans.

The whole path is also held against the fp32 oracle with the global bars of tests/test_gpu_parity.py, but not with the
4e-3 per-window bar: with these weights fp16 storage alone moves a window's logits by up to ~4e-3 of its scale (CPU
emulation of the device's rounding points over the windows below), so that bar would fail without a fault."""
import ctypes
import functools
import os

import numpy as np
import pytest

from cova_b200 import _lib, synth, weights
from cova_b200.elements import BlobPipeline
from oracle import blobnet_ref, metapreprocess_ref as mpr
from test_tile_plans import (ACT_REL_TOL, C_KERNEL, C_SIMT, CASES, DEC_COUT, FLOOR, LOGIT_REL_TOL, MAX_FLIP, NAMES, U,
                             _layer_output, _log, _n_sms, _w64, bound_ratio, choose_windows, restate)

C_ACC, C_CONST, ABS = 1 / 4, 2.0 ** -20, 2.0 ** -25
HERE = os.path.dirname(os.path.abspath(__file__))
SEEDS = (0, 1, 2, 3)
FAMILIES = [("calibrated", s) for s in SEEDS] + [("extremes", 0)]
ENC_COUT = (16, 32, 64, 128)


@functools.lru_cache(None)
def clip():
    d = np.load(os.path.join(HERE, "golden", "demo_1m_meta.npz"))
    return np.ascontiguousarray(np.moveaxis(d["planes"], 0, -1))          # [1802, 45, 80, 4], GoPs start every 250


@functools.lru_cache(None)
def calib_x():
    """Real-clip frames 0-40 and one synthetic stream, as BlobNet input."""
    real = mpr.tensorise_stream(clip()[0:41], 4, 1)
    syn = mpr.tensorise_stream(synth.synth_streams(1, 20, 45, 80, config_idx=1)[0], 4, 1)
    return mpr.stacked_to_nchw(np.concatenate([real, syn]), 4).astype(np.float32)


@functools.lru_cache(None)
def trained(family, seed):
    return weights.trained_like_weights(seed, family, calib_x())


def _f16(a):
    return np.asarray(a, np.float32).astype(np.float16).astype(np.float64)


def _scale32(w, p):
    return w[f"{p}.bn_gamma"] / np.sqrt(w[f"{p}.bn_var"] + np.float32(1e-3))   # float32 throughout, as weights_pack.cuh


def device_weights(w):
    """fp64 weight dict whose restatement is what the tcgen05 kernels compute: fp16 operands, fp32 folded constants.
    BatchNorm is re-expressed with var = 1 - 1e-3 (var + eps = 1 exactly in fp64), mean 0, gamma = s and beta = the
    folded shift / offset; dec3 + head as one output channel holding the fold, head_b the folded constant."""
    d = _w64(w)
    d["enc0.conv_w"] = _f16(w["enc0.conv_w"] / np.float32(6.0)) * 6.0           # restate divides by 6 again: exact
    for i in range(1, 4):
        d[f"enc{i}.conv_w"] = _f16(w[f"enc{i}.conv_w"])
    for i in range(4):
        p = f"enc{i}"
        s = _scale32(w, p)
        d[f"{p}.bn_gamma"], d[f"{p}.bn_beta"] = s.astype(np.float64), (w[f"{p}.bn_beta"] - w[f"{p}.bn_mean"] * s).astype(np.float64)
        d[f"{p}.bn_mean"], d[f"{p}.bn_var"] = np.zeros_like(d[f"{p}.bn_mean"]), np.full_like(d[f"{p}.bn_var"], 1.0 - 1e-3)
    for i in range(3):
        p = f"dec{i}"
        s = _scale32(w, p)
        d[f"{p}.convt_w"] = _f16(w[f"{p}.convt_w"])
        d[f"{p}.bn_gamma"] = s.astype(np.float64)
        d[f"{p}.bn_beta"] = ((w[f"{p}.convt_b"] - w[f"{p}.bn_mean"]) * s + w[f"{p}.bn_beta"]).astype(np.float64)
        d[f"{p}.convt_b"] = np.zeros_like(d[f"{p}.convt_b"])
        d[f"{p}.bn_mean"], d[f"{p}.bn_var"] = np.zeros_like(d[f"{p}.bn_mean"]), np.full_like(d[f"{p}.bn_var"], 1.0 - 1e-3)
    hw = w["head_w"].astype(np.float64)
    fold = np.einsum("ickl,c->ikl", w["dec3.convt_w"].astype(np.float64), hw)
    d["dec3.convt_w"] = np.zeros_like(d["dec3.convt_w"])
    d["dec3.convt_w"][:, 0] = _f16(fold.astype(np.float32))
    d["dec3.convt_b"] = np.zeros_like(d["dec3.convt_b"])
    d["head_w"] = np.eye(len(hw))[0]
    d["head_b"] = np.array([np.float32(float(w["head_b"][0]) + float(hw @ w["dec3.convt_b"].astype(np.float64)))], np.float64)
    return d


def _tn_carry(k, w, i):
    """Per-channel constant k carried through PointWiseTN on |tn_w| (as restate's mag): [1, C, T, 1, 1]."""
    a = np.abs(w[f"enc{i}.tn_w1"]).sum(0) @ np.abs(w[f"enc{i}.tn_w2"])            # [T_out]
    e = k[None, :, None, None, None] * (1.0 + a)[None, None, :, None, None]
    return e[:, :, :1] if i == 3 else e


def const_term(w, layer):
    """E of the tcgen05 bound (module docstring), broadcastable to the layer's output."""
    if layer < 4:
        s = _scale32(w, f"enc{layer}").astype(np.float64)
        shift = (w[f"enc{layer}.bn_beta"] - w[f"enc{layer}.bn_mean"] * _scale32(w, f"enc{layer}")).astype(np.float64)
        return _tn_carry(np.abs(s) * np.maximum(w[f"enc{layer}.conv_b"], 0) + np.abs(shift), w, layer)
    if layer < 7:
        p = f"dec{layer - 4}"
        s = _scale32(w, p)
        return np.abs((w[f"{p}.convt_b"] - w[f"{p}.bn_mean"]) * s + w[f"{p}.bn_beta"]).astype(np.float64)[None, :, None, None, None]
    return np.zeros((1, 1, 1))


def const_term_simt(w, layer):
    if layer == 7:
        return np.full((1, 1, 1), abs(float(w["head_b"][0])) + float(np.abs(w["head_w"]) @ np.abs(w["dec3.convt_b"])))
    p = f"enc{layer}" if layer < 4 else f"dec{layer - 4}"
    b = w[f"{p}.conv_b"] if layer < 4 else w[f"{p}.convt_b"]
    s = np.abs(_scale32(w, p)).astype(np.float64)
    k = s * (np.abs(b) + np.abs(w[f"{p}.bn_mean"])) + np.abs(w[f"{p}.bn_beta"])
    return _tn_carry(k, w, layer) if layer < 4 else k[None, :, None, None, None]


def ratios(got, ref, mag, extra, layer):
    """|got - ref| / bound per element (tcgen05 bound; extra = E)."""
    got, ref, mag = (np.asarray(a, np.float64) for a in (got, ref, mag))
    assert got.shape == ref.shape == mag.shape, (got.shape, ref.shape, mag.shape)
    b = C_ACC * U * mag + U * np.abs(ref) + C_CONST * extra + ABS
    if layer == 0:
        b = b + U * (mag + extra)
    return np.abs(got - ref) / b


def ratios_simt(got, ref, mag, extra):
    got, ref, mag = (np.asarray(a, np.float64) for a in (got, ref, mag))
    return np.abs(got - ref) / (C_SIMT * U * (mag + extra) + U * np.abs(ref) + ABS)


def restate_simt(w64, layer, x, target):
    """(ref, mag) for the validation kernels: fp32 weights; the head unfolded (mag on sum |W| |head_w|)."""
    ref, mag = restate(w64, layer, x, target)
    if layer == 7:
        wa = dict(w64, **{"dec3.convt_w": np.abs(w64["dec3.convt_w"]), "head_w": np.abs(w64["head_w"])})
        _, mag = restate(wa, layer, x, target)
    return ref, mag


def per_channel(r):
    """worst ratio per channel of a layer output ([N, C, T, H, W]) or of the logits ([N, H, W]: one channel)."""
    r = np.asarray(r)
    return r.reshape(1, -1).max(1) if r.ndim == 3 else r.max(axis=(0, 2, 3, 4))


def _report(tag, layer, r):
    pc = per_channel(r)
    worst = int(np.argmax(pc))
    _log(f"{tag} {NAMES[layer]} worst={pc.max():.3g} (channel {worst}) per_channel=" + ",".join(f"{v:.2g}" for v in pc))
    return float(pc.max())


# ----------------------------------------------------------------------------------------------------------------- CPU
def _forward_stats(w, frames):
    x = mpr.stacked_to_nchw(mpr.tensorise_stream(frames, 4, 1), 4)
    logit, inter = blobnet_ref.blobnet_forward(w, x, return_intermediates=True)
    spans = {}
    for k, v in inter.items():
        m = np.abs(v).max(axis=tuple(a for a in range(v.ndim) if a != 1))
        spans[k] = float(m.max() / m[m > 0].min())
    return logit, spans


@pytest.mark.parametrize("family,seed", FAMILIES)
def test_generator_keeps_the_weights_trained_like(family, seed):
    """The generator must stay wild: per-channel maxima over >= 3 decades in some layer, dead channels whose calibrated
    statistics are zero, the intended signs of the BatchNorm scales, foreground between 5% and 20% on clip frames it was
    not calibrated on.  And it is deterministic."""
    w = trained(family, seed)
    assert all(np.isfinite(v).all() for v in w.values())
    again = weights.trained_like_weights(seed, family, calib_x())
    assert all((again[k] == w[k]).all() for k in w)
    logit, spans = _forward_stats(w, clip()[200:260])
    assert max(spans.values()) >= 1e3, spans
    # dead channels (bias -1e3): never positive on the calibration input, so their calibrated mean and variance are 0
    dead = [(w[f"enc{i}.conv_b"] == weights.DEAD_BIAS) & (w[f"enc{i}.bn_mean"] == 0) & (w[f"enc{i}.bn_var"] == 0)
            for i in range(4)]
    assert sum(int(d.sum()) for d in dead) >= 5
    assert 0.05 <= float((logit > 0).mean()) <= 0.20
    nonneg = [bool((w[f"enc{i}.bn_gamma"] >= 0).all()) for i in range(4)]
    s = [np.abs(_scale32(w, f"enc{i}")) for i in range(4)]
    if family == "calibrated":
        assert nonneg == [False] * 4
        assert min(a[a > 0].min() for a in s) < 0.01 and max(a.max() for a in s) > 10
        return
    g = [w[f"enc{i}.bn_gamma"] for i in range(4)]
    assert nonneg == [False, True, False, False]                   # bn_nonneg takes both values
    assert (g[0] < 0).any() and (g[0] > 0).any()
    assert g[1][5] == 0 and not np.signbit(g[1][5]) and g[1][6] == 0 and np.signbit(g[1][6])
    assert (np.flatnonzero(g[2] < 0) == [ENC_COUT[2] - 1]).all()
    assert (g[3] < 0).all()
    assert (w["enc0.tn_w1"] == 0).all() and (w["enc0.tn_w2"] == 0).all() and np.abs(w["enc2.tn_w1"]).max() > 2
    assert (w["enc1.conv_w"][:, 3] == 0).all() and (w["dec1.convt_w"][7] == 0).all() and (w["enc2.conv_w"][:, :, 0, 2] == 0).all()
    x = mpr.stacked_to_nchw(mpr.tensorise_stream(clip()[200:220], 4, 1), 4)
    _, inter = blobnet_ref.blobnet_forward(w, x, return_intermediates=True)
    big, tiny = np.abs(inter["enc1"][:, 11]).max(), np.abs(inter["enc1"][:, 10]).max()
    assert 2.0 ** 13 <= big < 65504 and 0 < tiny < 2.0 ** -14                    # ~2^14, and fp16-subnormal outputs
    fold = np.einsum("ickl,c->ikl", w["dec3.convt_w"].astype(np.float64), w["head_w"].astype(np.float64))
    tot = np.einsum("ickl,c->ikl", np.abs(w["dec3.convt_w"]).astype(np.float64), np.abs(w["head_w"]).astype(np.float64))
    assert (np.abs(fold) < 1e-3 * tot).sum() >= 16                              # the head fold cancels for some taps


@functools.lru_cache(None)
def _host_case(family, seed, layer):
    """(device image, x, ref, mag) of one layer on the fp16-rounded oracle intermediates of clip frames 200-215."""
    w = trained(family, seed)
    x = mpr.stacked_to_nchw(mpr.tensorise_stream(clip()[200:216], 4, 1), 4)
    logit, inter = blobnet_ref.blobnet_forward(w, x, return_intermediates=True)
    acts = [np.clip(x, 0, 6), inter["enc0"], inter["enc1"], inter["enc2"], inter["enc3"][:, :, :1]]
    acts += [np.maximum(inter[f"dec{i}"], 0)[:, :, None] for i in range(3)]
    xin = _f16(acts[layer])
    target = (45, 80) if layer == 7 else (acts[layer + 1].shape[-2:] if layer >= 4 else None)
    dw = device_weights(w)
    ref, mag = (t.numpy() for t in restate(dw, layer, xin, target))
    return w, dw, xin, target, ref, mag


def _old_bound_passes(bad, ref, w, xin, layer, target):
    _, mag_old = (t.numpy() for t in restate(_w64(w), layer, xin, target))
    return bound_ratio(bad, ref, mag_old, C_KERNEL) <= 1.0


def test_bound_flags_what_the_global_bar_and_the_old_floor_miss():
    """Host data only, calibrated seed 0.  (1) In blocks 2-4, one element of the smallest live channel in which such an
    element exists, moved by 1% of its value; (2) every BatchNorm shift / offset of a layer rounded to fp16 in the device
    image (what a half-precision epilogue constant would do).  The 4e-3 global bar and the bound of test_tile_plans (its
    2^-16 floor) pass all of them; the bound flags (1) in every block and (2) in some layer.  The exact outputs and their
    fp16 roundings stay inside it."""
    flagged = {}
    for layer in range(7):
        w, dw, xin, target, ref, mag = _host_case("calibrated", 0, layer)
        e = np.broadcast_to(const_term(w, layer), ref.shape)
        assert ratios(ref, ref, mag, e, layer).max() == 0.0
        assert ratios(_f16(ref), ref, mag, e, layer).max() <= 1.0, NAMES[layer]
        _, mag_old = (t.numpy() for t in restate(_w64(w), layer, xin, target))
        if 1 <= layer <= 3:
            new = ratios(ref * 1.01, ref, mag, e, layer) > 1.0
            old_ok = 0.01 * np.abs(ref) <= C_KERNEL * U * mag_old + U * np.abs(ref) + FLOOR
            cand = new & old_ok & (w[f"enc{layer}.conv_b"] != weights.DEAD_BIAS)[None, :, None, None, None]
            cmax = np.where(cand.any(axis=(0, 2, 3, 4)), np.abs(ref).max(axis=(0, 2, 3, 4)), np.inf)
            c = int(np.argmin(cmax))
            assert np.isfinite(cmax[c]), NAMES[layer]
            k = np.unravel_index(np.argmax(cand[:, c]), cand[:, c].shape)
            idx = (k[0], c) + tuple(k[1:])
            bad = ref.copy()
            bad[idx] *= 1.01
            assert np.abs(bad - ref).max() <= ACT_REL_TOL * np.abs(ref).max()
            assert bound_ratio(bad, ref, mag_old, C_KERNEL) <= 1.0
            assert ratios(bad, ref, mag, e, layer).max() > 1.0
        p = f"enc{layer}" if layer < 4 else f"dec{layer - 4}"
        dw16 = dict(dw, **{f"{p}.bn_beta": _f16(dw[f"{p}.bn_beta"])})
        bad, _ = (t.numpy() for t in restate(dw16, layer, xin, target))
        assert np.abs(bad - ref).max() <= ACT_REL_TOL * np.abs(ref).max()
        assert bound_ratio(bad, ref, mag_old, C_KERNEL) <= 1.0
        flagged[NAMES[layer]] = float(ratios(bad, ref, mag, e, layer).max())
    assert max(flagged.values()) > 1.0, flagged


@pytest.mark.parametrize("family,seed", [("calibrated", 1), ("extremes", 0)])
def test_device_image_restatement_against_the_oracle(family, seed):
    """The restatement on the device image, fed the fp32 oracle's intermediates rounded to fp16, stays within the
    fp64 oracle's output of each layer up to the weight roundings it models: within test_tile_plans' bound (c = 9/4)
    of the exact-weight restatement.  And the SIMT reference is the exact-weight restatement itself."""
    for layer in range(8):
        w, dw, xin, target, ref, mag = _host_case(family, seed, layer)
        ref64, mag64 = (t.numpy() for t in restate(_w64(w), layer, xin, target))
        r = bound_ratio(ref, ref64, np.maximum(mag64, mag), C_KERNEL)
        assert r <= 1.0, (NAMES[layer], r)


# refusals --------------------------------------------------------------------------------------------------------------
def _new(wts, impl=_lib.IMPL_TCGEN05):
    blob = weights.to_blob(wts)
    lib = _lib.load()
    h = ctypes.c_void_p()
    buf = ctypes.create_string_buffer(blob, len(blob))
    rc = lib.cova_pipeline_new(ctypes.byref(h), 0, 80, 45, 4, 1, 1, 8, buf, len(blob), 1, impl)
    if rc == _lib.OK:
        lib.cova_pipeline_free(h)
    return rc, lib.cova_last_error().decode()


def test_weights_the_kernels_cannot_represent_are_refused_before_device_use():
    """NaN-free containers that would give NaN / Inf outputs: COVA_E_WEIGHTS naming the tensor, with or without a GPU.
    The largest representable values next to each limit pass that check."""
    base = trained("calibrated", 0)

    def edit(name, idx, v):
        w = {k: v2.copy() for k, v2 in base.items()}
        w[name][idx] = v
        return w
    bad = [
        (edit("enc2.bn_var", 3, -0.5), "enc2.bn_var"),
        (edit("dec1.bn_var", 0, -2e-3), "dec1.bn_var"),
        (edit("enc1.bn_gamma", 0, 3e38), "enc1.bn_gamma"),
        (edit("dec0.bn_gamma", 5, -3e38), "dec0.bn_gamma"),
        (edit("enc3.bn_mean", 2, 3e38), "enc3.bn_mean"),
        (edit("enc0.conv_w", (1, 0, 1, 1), 6 * 65520.0), "enc0.conv_w"),
        (edit("enc2.conv_w", (0, 0, 0, 0), -65520.0), "enc2.conv_w"),
        (edit("dec2.convt_w", (0, 0, 0, 0), 1e5), "dec2.convt_w"),
        (edit("head_w", 0, 1e5 / max(float(np.abs(base["dec3.convt_w"][:, 0]).max()), 1e-3)), "head_w"),
    ]
    for w, name in bad:
        rc, msg = _new(w)
        assert rc == _lib.E_WEIGHTS and name in msg, (name, rc, msg)
    ok = [edit("enc0.conv_w", (1, 0, 1, 1), 6 * 65504.0), edit("enc2.conv_w", (0, 0, 0, 0), 65504.0),
          edit("enc2.bn_var", 3, 0.0), edit("enc2.bn_gamma", 3, -0.0)]
    for w in ok:
        rc, msg = _new(w)
        assert rc != _lib.E_WEIGHTS, msg


# ----------------------------------------------------------------------------------------------------------------- GPU
PROD = slice(200, 520)               # 320 frames of the clip: 317 windows at 80x45, across the GoP edge at frame 250


def _acts(p):
    act = {layer: p.read_activation(layer) for layer in range(8)}
    act[8] = p.read_logits()
    return act


def _targets(act, h, w):
    return {4: act[5].shape[-2:], 5: act[6].shape[-2:], 6: act[7].shape[-2:], 7: (h, w)}


def _check_layers(tag, p, w, act, h, wd, windows=None):
    """Every tcgen05 layer output of p against the restatement of its own device input (windows: all, or a sample)."""
    dw = device_weights(w)
    sel = slice(None) if windows is None else windows
    targets = _targets(act, h, wd)
    worst = {}
    for layer in range(8):
        got = _layer_output(p, layer)[sel]
        assert np.isfinite(got).all(), (tag, NAMES[layer])
        ref, mag = (t.numpy() for t in restate(dw, layer, act[layer][sel], targets.get(layer)))
        worst[layer] = _report(tag, layer, ratios(got, ref, mag, const_term(w, layer), layer))
    return worst


@pytest.mark.gpu
@pytest.mark.parametrize("family,seed", FAMILIES)
def test_production_path_every_layer_window_and_channel(family, seed):
    """process() on clip frames 200-519 (317 windows, one chunk): every layer's tcgen05 output within the bound of the
    restatement on that layer's own device input, every activation finite, the mask exactly logit > 0.  For the
    calibrated family also the whole path against the fp32 oracle: logits within the global bar, flips rare and only
    where the oracle's logit lies within the bar of zero."""
    w = trained(family, seed)
    frames = clip()[PROD]
    p = BlobPipeline(80, 45, weights.to_blob(w), 1, len(frames), keep_logits=True, n_chunks=1)
    boxes = p.process(frames[None])
    assert len(boxes) == 317
    act = _acts(p)
    assert all(np.isfinite(a).all() for a in act.values())
    assert (p.read_mask() == (act[8] > 0)).all()
    worst = _check_layers(f"production {family} seed={seed}", p, w, act, 45, 80)
    _log(f"production {family} seed={seed} worst per layer: " + " ".join(f"{NAMES[k]}={v:.3g}" for k, v in worst.items()))
    bad = {NAMES[k]: v for k, v in worst.items() if not v <= 1.0}
    assert not bad, bad
    if family != "calibrated":
        return
    ref = blobnet_ref.blobnet_forward(w, mpr.stacked_to_nchw(mpr.tensorise_stream(frames, 4, 1), 4))
    logits = act[8]
    scale = float(np.abs(ref).max())
    err = np.abs(logits - ref)
    per_window = err.max(axis=(1, 2)) / np.abs(ref).max(axis=(1, 2))
    flipped = (logits > 0) != (ref > 0)
    _log(f"production {family} seed={seed} vs fp32 oracle: global={err.max() / scale:.3g} "
         f"per_window_max={per_window.max():.3g} flips={int(flipped.sum())}/{flipped.size} "
         f"flip_max_abs_ref_rel={float(np.abs(ref[flipped]).max() / scale) if flipped.any() else 0:.3g}")
    assert err.max() <= LOGIT_REL_TOL * scale
    assert float(flipped.mean()) <= MAX_FLIP
    assert (np.abs(ref[flipped]) <= LOGIT_REL_TOL * scale).all()


@pytest.mark.gpu
@pytest.mark.parametrize("family", ["calibrated", "extremes"])
@pytest.mark.parametrize("w,h,dbg", CASES)
def test_every_tile_plan_every_window(w, h, dbg, family):
    """test_tile_plans' cases (every layer, family, configuration and ring depth) with the same window counts: each
    tcgen05 layer on the validation kernels' input within the bound on every window, the validation kernels within
    theirs."""
    n_sms = _n_sms()
    n = choose_windows(w, h, dbg, n_sms)
    seed = CASES.index((w, h, dbg)) % len(SEEDS) if family == "calibrated" else 0
    wts = trained(family, seed)
    w64, dw = _w64(wts), device_weights(wts)
    frames = synth.synth_streams(1, n + 3, h, w, config_idx=w % 7)
    p = BlobPipeline(w, h, weights.to_blob(wts), 1, n + 3, impl=_lib.IMPL_SIMT, keep_logits=True)
    p.set_debug(dbg)
    p.load_frames(frames)
    p.run()
    act = _acts(p)
    targets = _targets(act, h, w)
    tag = f"tile_plans {family} seed={seed} {w}x{h} dbg={dbg} n={n}"
    for layer in range(8):
        simt = act[8] if layer == 7 else (act[layer + 1][:, : DEC_COUT[layer - 4]] if layer >= 4 else act[layer + 1])
        ref, mag = restate_simt(w64, layer, act[layer], targets.get(layer))
        rs = float(ratios_simt(simt, ref, mag, const_term_simt(wts, layer)).max())
        p.run_layer(layer, _lib.IMPL_TCGEN05)
        got = _layer_output(p, layer)
        assert np.isfinite(got).all(), NAMES[layer]
        ref, mag = (t.numpy() for t in restate(dw, layer, act[layer], targets.get(layer)))
        r = _report(tag, layer, ratios(got, ref, mag, const_term(wts, layer), layer))
        _log(f"{tag} {NAMES[layer]} simt_ratio={rs:.3g}")
        assert rs <= 1.0, (NAMES[layer], "the validation kernel is outside its bound", rs)
        assert r <= 1.0, (NAMES[layer], r)
        if layer < 7:
            p.run_layer(layer, _lib.IMPL_SIMT)


@pytest.mark.gpu
@pytest.mark.parametrize("w,h", [(120, 68), (240, 135)])
def test_larger_grids_sampled_windows(w, h):
    """1080p and 4K grids, synthetic streams, calibrated seed 0: first, middle and last window of every layer within
    the bound, the mask exactly logit > 0."""
    wts = trained("calibrated", 0)
    n_frames = 12
    frames = synth.synth_streams(1, n_frames, h, w, config_idx=2)
    p = BlobPipeline(w, h, weights.to_blob(wts), 1, n_frames, keep_logits=True, n_chunks=1)
    p.process(frames)
    act = _acts(p)
    n = act[8].shape[0]
    assert n == n_frames - 3 and (p.read_mask() == (act[8] > 0)).all()
    worst = _check_layers(f"grid {w}x{h}", p, wts, act, h, w, windows=[0, n // 2, n - 1])
    bad = {NAMES[k]: v for k, v in worst.items() if not v <= 1.0}
    assert not bad, bad
