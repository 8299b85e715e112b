"""Demux + gopsplit in front of the path (SURVEY section 8f row f4): host C++ behind the C ABI against the Python
restatements in oracle/demux_ref.py, pinned on the moov box of the reference's own demo clip
(tests/golden/demo_1m_moov.bin, tools/make_moov_fixture.py).  Host-only code: no GPU needed."""
import os
import struct

import numpy as np
import pytest

from cova_b200 import _lib, shard
from oracle import demux_ref

HERE = os.path.dirname(os.path.abspath(__file__))
MOOV = open(os.path.join(HERE, "golden", "demo_1m_moov.bin"), "rb").read()
META = np.load(os.path.join(HERE, "golden", "demo_1m_meta.npz"))


def demo_clip_with_synthetic_media(seed=0):
    """The demo clip as a whole MP4 file: its own ftyp and moov boxes around an mdat whose samples sit at the offsets and
    have the sizes the clip's sample table gives.  The media bytes are synthetic: each sample is a run of 4-byte
    length-prefixed NAL units (an optional SEI, then one to three IDR or non-IDR slices, first_mb_in_slice = 0 only
    on the first) with random non-zero bodies, so that no start code appears inside a NAL unit, as in a real stream."""
    samples, _ = demux_ref.mp4_video_samples(MOOV)
    ftyp_size = struct.unpack_from(">I", MOOV)[0]
    assert samples[0][0] == ftyp_size + 16                   # the clip has an 8-byte free box, then the mdat header
    rng = np.random.default_rng(seed)
    mdat = bytearray()
    for off, size, key, _dts, _pts in samples:
        assert off == samples[0][0] + len(mdat)
        n_slices = int(rng.integers(1, 4)) if size >= 64 else 1
        kinds = ([6] if size >= 64 and rng.random() < 0.2 else []) + [5 if key else 1] * n_slices
        cuts = np.sort(rng.choice(np.arange(1, size - 12 * len(kinds)), len(kinds) - 1, replace=False)) if len(kinds) > 1 else []
        bodies = np.diff(np.r_[0, cuts, size - 12 * len(kinds)]) + 8   # every NAL body at least 8 bytes
        for i, (typ, n) in enumerate(zip(kinds, bodies)):
            body = rng.integers(1, 256, int(n), dtype=np.uint8)
            body[0] = (0x60 if typ == 5 else 0x40 if typ == 1 else 0) | typ
            if typ in (1, 5):                                  # ue(first_mb_in_slice): '1' = 0, '01..' > 0
                body[1] = 0x80 | body[1] if kinds.index(typ) == i else max(1, body[1] & 0x7F)
            mdat += struct.pack(">I", int(n)) + body.tobytes()
        assert len(mdat) == off + size - samples[0][0]
    return (MOOV[:ftyp_size] + struct.pack(">I4s", 8, b"free") + struct.pack(">I4s", 8 + len(mdat), b"mdat") + bytes(mdat)
            + MOOV[ftyp_size:])


def test_mp4_sample_table_on_the_demo_clip():
    samples, info = shard.demux_mp4(MOOV)
    ref, ref_info = demux_ref.mp4_video_samples(MOOV)
    assert samples == ref and info == ref_info
    assert len(samples) == 1802 and (info["width"], info["height"]) == (1280, 720) and info["nal_length_size"] == 4
    keys = [i for i, s in enumerate(samples) if s[2]]
    assert keys == list(range(0, 1802, 250))
    # the sync samples are exactly the frames the patched decoder reports as all-intra (fixture f1)
    assert keys == np.nonzero(META["key"])[0].tolist()
    offs = [s[0] for s in samples]
    assert offs == sorted(offs) and all(a + s[1] <= b for a, s, b in zip(offs, samples, offs[1:]))
    dts = [s[3] for s in samples]
    assert all(b > a for a, b in zip(dts, dts[1:]))
    # same frame spacing as the PTS the decoder dumped (30 fps)
    assert len(set(np.diff(dts))) == 1 and abs(info["timescale"] / (dts[1] - dts[0]) - 30.0) < 0.1


def test_demo_clip_sharded_like_gopsplit():
    samples, _ = shard.demux_mp4(MOOV)
    key = [s[2] for s in samples]
    for pads in (1, 2, 3, 4, 8, 16):
        got = shard.gopsplit_ranges(key, pads)
        assert got == demux_ref.gopsplit_ranges(key, pads)
        assert got == [shard.frames_of_shard(key, pads, p) for p in range(pads)]
    assert shard.gopsplit_ranges(key, 4) == [(0, 500), (500, 1000), (1000, 1500), (1500, 1802)]
    assert shard.gopsplit_ranges(key, 16)[:9] == [(250 * i, min(250 * (i + 1), 1802)) for i in range(8)] + [(0, 0)]


@pytest.mark.parametrize("seed", range(6))
def test_gopsplit_ranges_random_streams(seed):
    rng = np.random.default_rng(seed)
    n = int(rng.integers(1, 400))
    key = (rng.random(n) < rng.choice([0.02, 0.1, 0.5])).tolist()
    if seed % 2 == 0:
        key[0] = True          # odd seeds start with delta frames: they form a GoP of their own
    for pads in (1, 2, 3, 5, 8, 64):
        got = shard.gopsplit_ranges(key, pads)
        assert got == demux_ref.gopsplit_ranges(key, pads)
        assert got == [shard.frames_of_shard(key, pads, p) for p in range(pads)]
        covered = sorted(f for a, b in got for f in range(a, b))
        assert covered == list(range(n)), "every frame goes to exactly one pad"
    with pytest.raises(_lib.CovaError):
        shard.gopsplit_ranges(key, 0)


def nal(typ, payload=b"", first_mb_zero=True, long_sc=False):
    body = bytes([0x60 | typ])
    if typ in (1, 5):
        body += bytes([0x80 if first_mb_zero else 0x40]) + payload   # ue(first_mb_in_slice): '1' = 0, '010' = 1
    else:
        body += payload
    return (b"\x00\x00\x00\x01" if long_sc else b"\x00\x00\x01") + body


def test_annexb_access_units_synthetic():
    s = b"".join([
        nal(9, b"\x10", long_sc=True), nal(7, b"\x42\x00\x1f", long_sc=True), nal(8, b"\xce"), nal(5, b"\xaa\xbb"),     # IDR
        nal(5, b"\xcc", first_mb_zero=False),                                                                   # 2nd slice, same frame
        nal(9, b"\x30", long_sc=True), nal(1, b"\x11\x22\x33"),                                                  # P frame after AUD
        nal(1, b"\x44"),                                                                                        # P frame, no AUD
        nal(6, b"\x05\x01"), nal(1, b"\x55"),                                                                   # SEI starts a unit
        nal(7, b"\x42", long_sc=True), nal(8, b"\xce"), nal(5, b"\x66"),                                         # second IDR
    ])
    got = shard.demux_annexb(s)
    assert got == demux_ref.annexb_frames(s)
    assert [k for _, _, k in got] == [True, False, False, False, True]
    assert got[0][0] == 0 and sum(sz for _, sz, _ in got) == len(s)
    assert all(a + sz == b for (a, sz, _), (b, _, _) in zip(got, got[1:]))
    assert shard.demux_annexb(b"") == [] and shard.demux_annexb(b"\x00\x00\x01\x67\x42") == []   # parameter sets only


def test_annexb_scan_recovers_the_demo_clip_layout():
    """AVCC samples of the demo clip (its sample table, synthetic media bytes) rewritten as an Annex-B stream (length
    prefixes -> start codes): the scanner must find the same 1802 frames and the same 8 key frames the MP4 tables list."""
    d = demo_clip_with_synthetic_media()
    samples, info = shard.demux_mp4(d)
    assert (samples, info) == demux_ref.mp4_video_samples(d)
    stream, starts = bytearray(), []
    for off, size, _key, _dts, _pts in samples:
        starts.append(len(stream))
        p = off
        while p < off + size:
            (n,) = struct.unpack_from(">I", d, p)
            stream += b"\x00\x00\x00\x01" + d[p + 4: p + 4 + n]
            p += 4 + n
        assert p == off + size
    got = shard.demux_annexb(bytes(stream))
    assert got == demux_ref.annexb_frames(bytes(stream))
    assert [g[0] for g in got] == starts
    assert [g[2] for g in got] == [s[2] for s in samples]


def test_malformed_mp4_never_reads_out_of_bounds_or_aborts():
    """The parser is driven by file contents: an oversized avc1 sample-entry size, stco / co64 / stsc bodies shorter than
    their headers, a 4-billion-entry fixed-size stsz and random corruption must all come back as an error code (or a
    valid table) - run in a child process so that a crash is a test failure, not the end of the session."""
    import subprocess
    import sys
    script = r'''
import sys, struct
import numpy as np
sys.path.insert(0, %r)
from cova_b200 import _lib, shard
moov = bytearray(open(%r, "rb").read())
def attempt(buf):
    try:
        shard.demux_mp4(bytes(buf))
    except _lib.CovaError as e:
        assert e.code in (_lib.E_INVAL, _lib.E_UNSUPPORTED, _lib.E_NOMEM), e.code
def box(tag):
    i = bytes(moov).find(tag)
    assert i >= 4
    return i - 4
# (1) avc1 sample entry claiming to be 4 GB / 0 bytes long
i = box(b"stsd") + 16
for v in (0xFFFFFFF0, 0, 40):
    m = bytearray(moov); m[i:i + 4] = struct.pack(">I", v); attempt(m)
# (2) stco / stsc / stsz truncated to less than their fixed header, (3) absurd counts
for tag in (b"stco", b"stsc", b"stsz", b"stts", b"ctts", b"stss"):
    i = box(tag)
    for sz in (8, 10, 12, 15):
        m = bytearray(moov); m[i:i + 4] = struct.pack(">I", sz); attempt(m)
    m = bytearray(moov); m[i + 12:i + 16] = b"\xff\xff\xff\xff"; attempt(m)
    m = bytearray(moov); m[i + 16:i + 20] = b"\xff\xff\xff\xff"; attempt(m)
i = box(b"stsz")
m = bytearray(moov); m[i + 12:i + 16] = struct.pack(">I", 1000); m[i + 16:i + 20] = b"\xff\xff\xff\xf0"; attempt(m)   # fixed size, 4e9 samples
# (4) random corruption and truncation
rng = np.random.default_rng(0)
for _ in range(300):
    m = bytearray(moov)
    for _ in range(int(rng.integers(1, 8))):
        m[int(rng.integers(0, len(m)))] = int(rng.integers(0, 256))
    attempt(m[: int(rng.integers(16, len(m) + 1))] if rng.random() < 0.3 else m)
print("ok")
''' % (os.path.dirname(HERE), os.path.join(HERE, "golden", "demo_1m_moov.bin"))
    r = subprocess.run([sys.executable, "-c", script], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), (r.returncode, r.stdout[-300:], r.stderr[-800:])
