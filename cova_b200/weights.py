"""BlobNet weight container ("CVBN" v1) and the seeded synthetic initialiser.

No trained weights ship with the reference (model/tf_model/.placeholder, README.md:198 points at a
Google-Drive link), so benchmarks and tests use random-init weights of the reference architecture
(utils/train-blobnet.py:57-69): He-normal conv kernels (encoder.py:41, decoder.py:20), BatchNorm
statistics drawn so that gamma can be exercised on both sides of 1, final bias tuned by the caller.

Container layout (little endian), parsed by csrc/weights_pack.cuh and by the oracle:
    u32 magic 'CVBN' (0x4E425643), u32 version = 1, u32 timestep = 4, u32 reserved = 0, then fp32
    tensors in torch layouts, in this order:
      for e in 0..3 (Cin,Cout = 3->16->32->64->128):
          conv_w[Cout][Cin][3][3], conv_b[Cout], bn_gamma, bn_beta, bn_mean, bn_var [Cout],
          tn_w1[4][4], tn_w2[4][4]            (Conv1D over T as [T_in][T_out])
      for d in 0..3 (Cin,Cout = 128->64, 128->32, 64->16, 32->16):
          convt_w[Cin][Cout][4][4], convt_b[Cout], and for d < 3: bn_gamma, bn_beta, bn_mean, bn_var
      head_w[16], head_b[1]
"""
from __future__ import annotations

import struct

import numpy as np

MAGIC = 0x4E425643
VERSION = 1
T = 4
ENC_CH = [(3, 16), (16, 32), (32, 64), (64, 128)]
DEC_CH = [(128, 64), (128, 32), (64, 16), (32, 16)]


def schema():
    s = []
    for i, (ci, co) in enumerate(ENC_CH):
        s += [(f"enc{i}.conv_w", (co, ci, 3, 3)), (f"enc{i}.conv_b", (co,)),
              (f"enc{i}.bn_gamma", (co,)), (f"enc{i}.bn_beta", (co,)),
              (f"enc{i}.bn_mean", (co,)), (f"enc{i}.bn_var", (co,)),
              (f"enc{i}.tn_w1", (T, T)), (f"enc{i}.tn_w2", (T, T))]
    for i, (ci, co) in enumerate(DEC_CH):
        s += [(f"dec{i}.convt_w", (ci, co, 4, 4)), (f"dec{i}.convt_b", (co,))]
        if i < 3:
            s += [(f"dec{i}.bn_gamma", (co,)), (f"dec{i}.bn_beta", (co,)),
                  (f"dec{i}.bn_mean", (co,)), (f"dec{i}.bn_var", (co,))]
    s += [("head_w", (DEC_CH[-1][1],)), ("head_b", (1,))]
    return s


def n_params() -> int:
    return sum(int(np.prod(shape)) for _, shape in schema())


def random_weights(seed: int = 0, head_bias: float = 0.0) -> dict[str, np.ndarray]:
    """SURVEY.md section 8d: He-normal kernels, BN gamma~U(0.5,1.5), small beta/mean, var~U(0.5,1.5)."""
    rng = np.random.default_rng(seed)
    w = {}
    for name, shape in schema():
        kind = name.split(".")[-1]
        if kind == "conv_w":
            fan_in = shape[1] * shape[2] * shape[3]
            v = rng.normal(0.0, np.sqrt(2.0 / fan_in), shape)
        elif kind == "convt_w":
            # Keras he_normal on a Conv3DTranspose kernel (kd,kh,kw,Cout,Cin): fan_in = kh*kw*Cout
            fan_in = shape[1] * shape[2] * shape[3]
            v = rng.normal(0.0, np.sqrt(2.0 / fan_in), shape)
        elif kind in ("conv_b", "convt_b", "bn_beta", "bn_mean"):
            v = rng.normal(0.0, 0.05, shape)
        elif kind in ("bn_gamma", "bn_var"):
            v = rng.uniform(0.5, 1.5, shape)
        elif kind in ("tn_w1", "tn_w2"):
            v = rng.normal(0.0, 0.5, shape)          # glorot-ish for a 4x4 matrix, both signs
        elif name == "head_w":
            v = rng.normal(0.0, np.sqrt(2.0 / shape[0]), shape)
        elif name == "head_b":
            v = np.full(shape, head_bias)
        else:
            raise AssertionError(name)
        w[name] = np.ascontiguousarray(v, dtype=np.float32)
    return w


DEAD_BIAS = -1e3


def trained_like_weights(seed: int, family: str, calib_x: np.ndarray) -> dict[str, np.ndarray]:
    """Weights with the statistics training leaves, for tests: per-channel scales over decades, dead channels, BatchNorm
    statistics measured on real activations.  Deterministic in (seed, family, calib_x).

    calib_x: BlobNet input [N, 3, T, H, W] (raw metadata bytes, as oracle.blobnet_ref.blobnet_forward takes it).  Layer by
    layer, in float64 with the oracle's helpers, each layer's BatchNorm statistics are the per-channel mean and variance of
    the tensor its BatchNorm sees on calib_x (encoder: the post-ReLU conv output; decoder: the cropped transposed-conv
    output), given the layers before it already final.
      calibrated  conv weights He-normal x a per-output-channel gain 2^U(-6, 4) (encoder) / 2^U(-4, 3) (decoder), bias
                  N(0, 0.1) x gain, about 10% of the channels dead (bias -1e3); |gamma| = 2^U(-6, 1), 25% negative;
                  beta N(0, 0.3); head_b = -(90th percentile of the logits): about 10% foreground.
      extremes    calibrated plus edits aimed at value-dependent code paths: pruned input channels (enc2, dec1), a zero
                  tap (enc3); BatchNorm scales mixed in block 1, all >= 0 in block 2 with gamma = +0 and -0 in two
                  channels and two channels of fp16-subnormal outputs (|gamma| ~ 2^-12 and 2^-15, beta 0) and one driven
                  to ~2^14, only channel Cout-1 negative in block 3, all negative in block 4; PointWiseTN zero in block
                  1 and |w| up to 3 in block 3; dec3 + head folds that cancel to ~1e-7 of sum |W| |head_w| for the taps
                  of four input channels."""
    import torch
    import torch.nn.functional as F

    from oracle import blobnet_ref as ref

    assert family in ("calibrated", "extremes"), family
    ext = family == "extremes"
    rng = np.random.default_rng([seed, 1 if ext else 0])
    w64 = {}

    def t(name):
        return torch.from_numpy(w64[name])

    def conv_params(prefix, wname, bname, shape, fan_in, cout_axis, lo, hi):
        gain = 2.0 ** rng.uniform(lo, hi, shape[cout_axis])
        gshape = [1] * len(shape)
        gshape[cout_axis] = -1
        w64[wname] = rng.normal(0.0, np.sqrt(2.0 / fan_in), shape) * gain.reshape(gshape)
        b = rng.normal(0.0, 0.1, shape[cout_axis]) * gain
        b[rng.random(b.shape) < 0.1] = DEAD_BIAS
        w64[bname] = b

    def bn_params(prefix, y, dims):
        co = y.shape[1]
        w64[f"{prefix}.bn_mean"] = y.mean(dims).numpy()
        w64[f"{prefix}.bn_var"] = y.var(dims, correction=0).numpy()
        w64[f"{prefix}.bn_gamma"] = 2.0 ** rng.uniform(-6, 1, co) * np.where(rng.random(co) < 0.25, -1.0, 1.0)
        w64[f"{prefix}.bn_beta"] = rng.normal(0.0, 0.3, co)

    def round32():                                            # what the container will hold
        for k, v in w64.items():
            w64[k] = np.asarray(v, np.float32).astype(np.float64)

    with torch.no_grad():
        x = torch.clamp(torch.as_tensor(calib_x, dtype=torch.float64), 0.0, 6.0) / 6.0
        skips = []
        for i, (ci, co) in enumerate(ENC_CH):
            p = f"enc{i}"
            conv_params(p, f"{p}.conv_w", f"{p}.conv_b", (co, ci, 3, 3), ci * 9, 0, -6, 4)
            w64[f"{p}.tn_w1"] = rng.normal(0.0, 0.5, (T, T))
            w64[f"{p}.tn_w2"] = rng.normal(0.0, 0.5, (T, T))
            if ext and i == 1:
                w64[f"{p}.conv_w"][:, 3] = 0.0                     # pruned input channel
            if ext and i == 2:
                w64[f"{p}.conv_w"][:, :, 0, 2] = 0.0               # one tap (dy = -1, dx = +1) zero
            if ext and i == 0:
                w64[f"{p}.tn_w1"][:] = 0.0
                w64[f"{p}.tn_w2"][:] = 0.0
            if ext and i == 2:
                w64[f"{p}.tn_w1"] = rng.uniform(-3.0, 3.0, (T, T))
                w64[f"{p}.tn_w2"] = rng.uniform(-3.0, 3.0, (T, T))
            round32()
            n, c, tt, h, wd = x.shape
            y = x.permute(0, 2, 1, 3, 4).reshape(n * tt, c, h, wd)
            y = torch.relu(F.conv2d(y, t(f"{p}.conv_w"), t(f"{p}.conv_b"), padding=1))
            bn_params(p, y, (0, 2, 3))
            g = w64[f"{p}.bn_gamma"]
            if ext and i == 1:                                     # all >= 0, with +0, -0 and fp16-subnormal outputs
                g[:] = np.abs(g)
                g[5], g[6] = 0.0, -0.0
                g[9], g[10] = 2.0 ** -12, 2.0 ** -15
                w64[f"{p}.bn_beta"][[9, 10]] = 0.0
                w64[f"{p}.bn_mean"][[9, 10]] = 0.0
            if ext and i == 2:
                g[:] = np.abs(g)
                g[co - 1] = -g[co - 1]
            if ext and i == 3:
                g[:] = -np.abs(g)
            round32()

            def block(y):
                yb = F.max_pool2d(ref._bn(y, w64, p), 2)
                yb = F.pad(yb, (wd % 2, 0, h % 2, 0))
                yb = yb.reshape(n, tt, *yb.shape[1:]).permute(0, 2, 1, 3, 4)
                return ref._pointwise_tn(yb, w64[f"{p}.tn_w1"], w64[f"{p}.tn_w2"])
            out = block(y)
            if ext and i == 1:                                     # channel 11 to ~2^14 (BN, pool and TN are 1-homogeneous)
                w64[f"{p}.bn_beta"][11] = 0.0
                w64[f"{p}.bn_mean"][11] = 0.0
                g = w64[f"{p}.bn_gamma"]
                g[11] = abs(g[11]) * 2.0 ** 14 / max(float(out[:, 11].abs().max()), 1e-30)
                g[11] = abs(g[11]) if np.isfinite(g[11]) else 1.0
                round32()
                out = block(y)
            x = out
            skips.append(x[:, :, 0])
        x = skips[3]
        H, W = calib_x.shape[-2:]
        targets = [skips[2].shape[-2:], skips[1].shape[-2:], skips[0].shape[-2:], (H, W)]
        for i, (ci, co) in enumerate(DEC_CH):
            p = f"dec{i}"
            conv_params(p, f"{p}.convt_w", f"{p}.convt_b", (ci, co, 4, 4), co * 16, 1, -4, 3)
            if ext and i == 1:
                w64[f"{p}.convt_w"][7] = 0.0                      # pruned input channel
            if ext and i == 3:                                     # head folds that cancel for the taps of inputs 0..3
                hw = rng.normal(0.0, np.sqrt(2.0 / co), co)
                k = int(np.argmax(np.abs(hw)))
                cw = w64[f"{p}.convt_w"]
                others = [j for j in range(co) if j != k]
                for c_in in range(4):
                    cw[c_in, k] = -np.tensordot(hw[others], cw[c_in, others], axes=(0, 0)) / hw[k]
                w64["head_w"] = hw
            round32()
            y = F.conv_transpose2d(torch.relu(x), t(f"{p}.convt_w"), t(f"{p}.convt_b"), stride=2)
            ct, cb = ref._crop_amounts(y.shape[-2], targets[i][0])
            cl, cr = ref._crop_amounts(y.shape[-1], targets[i][1])
            y = y[:, :, ct: y.shape[-2] - cb, cl: y.shape[-1] - cr]
            if i < 3:
                bn_params(p, y, (0, 2, 3))
                round32()
                x = torch.cat([ref._bn(y, w64, p), skips[2 - i]], dim=1)
            else:
                x = y
        if "head_w" not in w64:
            w64["head_w"] = rng.normal(0.0, np.sqrt(2.0 / DEC_CH[-1][1]), DEC_CH[-1][1])
        round32()
        logit = (x * t("head_w").view(1, -1, 1, 1)).sum(1)
        w64["head_b"] = np.array([-np.percentile(logit.numpy(), 90)])
    out = {name: np.ascontiguousarray(w64[name], dtype=np.float32) for name, _ in schema()}
    assert set(out) == set(w64)
    return out


def to_blob(w: dict[str, np.ndarray]) -> bytes:
    out = bytearray(struct.pack("<IIII", MAGIC, VERSION, T, 0))
    for name, shape in schema():
        a = np.ascontiguousarray(w[name], dtype="<f4")
        if a.shape != tuple(shape):
            raise ValueError(f"{name}: shape {a.shape} != {shape}")
        out += a.tobytes()
    return bytes(out)


def from_blob(blob: bytes) -> dict[str, np.ndarray]:
    magic, version, t, _ = struct.unpack_from("<IIII", blob, 0)
    if magic != MAGIC or version != VERSION or t != T:
        raise ValueError("not a CVBN v1 weight blob")
    off = 16
    w = {}
    for name, shape in schema():
        n = int(np.prod(shape))
        w[name] = np.frombuffer(blob, dtype="<f4", count=n, offset=off).reshape(shape).copy()
        off += 4 * n
    if off != len(blob):
        raise ValueError("blob length mismatch")
    return w
