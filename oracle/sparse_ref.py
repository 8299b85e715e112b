"""Plain NumPy reference of the sparse input format (include/cova_b200.h, COVA_SPARSE_MAX_FRAME_BYTES), written from the
format's definition: one record per frame, little-endian, 4-byte aligned,

    u32 background        bits 0-8 a packed16 value, bits 9-31 zero
    u32 count             macroblocks whose value is not the background
    u32 bitmap[ceil(n_mb / 32)]   bit i % 32 of word i / 32 set = macroblock i differs; bits >= n_mb zero
    u16 values[count]     the differing values in raster order, zero-padded to a multiple of 4 bytes

The canonical encoding takes the most frequent value of the frame as background (ties: the smallest) and zero padding."""
from __future__ import annotations

import numpy as np


def record_bytes(n_mb: int, count: int) -> int:
    return 8 + 4 * ((n_mb + 31) // 32) + 4 * ((count + 1) // 2)


def encode_frame(v: np.ndarray) -> bytes:
    v = np.asarray(v, dtype=np.uint16).reshape(-1)
    n_mb = v.size
    hist = np.bincount(v, minlength=512)
    bg = int(np.argmax(hist))                    # argmax returns the first (smallest) of equal maxima
    diff = v != bg
    vals = v[diff]
    bits = np.zeros(((n_mb + 31) // 32) * 32, dtype=np.uint8)
    bits[:n_mb] = diff
    words = np.packbits(bits.reshape(-1, 32)[:, ::-1], axis=1).view(">u4").reshape(-1).astype("<u4")
    if vals.size % 2:
        vals = np.concatenate([vals, np.zeros(1, dtype=np.uint16)])
    out = np.array([bg, int(diff.sum())], dtype="<u4").tobytes() + words.tobytes() + vals.astype("<u2").tobytes()
    assert len(out) == record_bytes(n_mb, int(diff.sum()))
    return out


def encode(packed: np.ndarray) -> bytes:
    """packed16 frames [F, h, w] (or [..., h, w]) -> the batch of their records, in order."""
    p = np.asarray(packed, dtype=np.uint16)
    p = p.reshape(-1, p.shape[-2] * p.shape[-1])
    return b"".join(encode_frame(f) for f in p)


def decode(data: bytes, n_frames: int, n_mb: int) -> np.ndarray:
    """A batch of n_frames records -> packed16 u16 [n_frames, n_mb].  Checks every rule of the format (AssertionError)."""
    buf = np.frombuffer(data, dtype=np.uint8)
    nw = (n_mb + 31) // 32
    out = np.empty((n_frames, n_mb), dtype=np.uint16)
    pos = 0
    for f in range(n_frames):
        bg, count = (int(x) for x in buf[pos: pos + 8].view("<u4"))
        assert bg < 512, "reserved background bits"
        words = buf[pos + 8: pos + 8 + 4 * nw].view("<u4")
        bits = np.unpackbits(words.astype(">u4").view(np.uint8).reshape(-1, 4), axis=1).reshape(-1, 32)[:, ::-1].reshape(-1)
        assert not bits[n_mb:].any(), "bit at or past n_mb"
        diff = bits[:n_mb].astype(bool)
        assert int(diff.sum()) == count, "count != popcount(bitmap)"
        size = record_bytes(n_mb, count)
        vals = buf[pos + 8 + 4 * nw: pos + size].view("<u2")
        assert vals[count:].size == count % 2 and not vals[count:].any(), "padding"
        row = np.full(n_mb, bg, dtype=np.uint16)
        row[diff] = vals[:count]
        out[f] = row
        pos += size
    assert pos == len(buf), "data length is not the sum of the record sizes"
    return out
