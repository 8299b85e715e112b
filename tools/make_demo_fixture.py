#!/usr/bin/env python
"""Generates tests/golden/demo_1m_meta.npz (SURVEY §8 f1): the per-macroblock metadata the reference's patched
avdec_h264 produces for its own demo clip (`demo/1m.mp4`, config C1 of BASELINE.json).

Runs only where /root/reference exists (the build container).  Steps:
  1. configure the reference's patched FFmpeg OUT OF TREE into oracle/_ref/ffmpeg-build (git-ignored; nothing is
     written into /root/reference, no reference source is copied) with only the H.264 decoder/parser and the mov demuxer;
  2. compile tools/dump_h264_meta.c against the static libs;
  3. dump every frame's first (W/16)*(H/16)*4 bytes of plane 0 and store them LZMA-compressed (save_fixture).

The fixture holds the frames of the clip in decode-output order, the key-frame flags (GoP boundaries for the
gopsplit-style sharding, gstgopsplit.cpp:712-723) and the PTS values.
"""
import hashlib
import io
import os
import subprocess
import sys
import zipfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference"
FF_SRC = os.path.join(REF, "third_parties", "FFmpeg")
BUILD = os.path.join(ROOT, "oracle", "_ref", "ffmpeg-build")
TOOL = os.path.join(ROOT, "oracle", "_ref", "dump_h264_meta")
OUT = os.path.join(ROOT, "tests", "golden", "demo_1m_meta.npz")
CONFIGURE = ["--disable-x86asm", "--disable-inline-asm", "--disable-everything", "--disable-programs", "--disable-doc",
             "--disable-avdevice", "--disable-avfilter", "--disable-swscale", "--disable-swresample", "--disable-postproc",
             "--disable-network", "--disable-autodetect", "--enable-decoder=h264", "--enable-parser=h264",
             "--enable-demuxer=mov", "--enable-protocol=file", "--enable-static", "--disable-shared"]


def run(cmd, **kw):
    print("+", " ".join(cmd), flush=True)
    subprocess.run(cmd, check=True, **kw)


def build_tool():
    os.makedirs(BUILD, exist_ok=True)
    if not os.path.exists(os.path.join(BUILD, "libavcodec", "libavcodec.a")):
        run([os.path.join(FF_SRC, "configure")] + CONFIGURE, cwd=BUILD)
        run(["make", "-j", str(os.cpu_count() or 4)], cwd=BUILD, stdout=subprocess.DEVNULL)
    libs = [os.path.join(BUILD, d, f"lib{d[3:]}.a") for d in ("libavformat", "libavcodec", "libavutil")]
    run(["gcc", "-O2", "-o", TOOL, os.path.join(ROOT, "tools", "dump_h264_meta.c"), "-I", FF_SRC, "-I", BUILD] + libs
        + ["-lm", "-lpthread", "-lz"])


def save_fixture(path, frames, key, pts, md5):
    """An .npz that np.load reads as usual, with its members LZMA-compressed and the frames stored byte-plane first
    (`planes`: [4, F, H, W]): the four bytes of a macroblock vary independently, and split into planes the clip packs into
    well under 1 MB, about a third of what deflate makes of the interleaved frames."""
    arrays = dict(planes=np.ascontiguousarray(np.moveaxis(frames, -1, 0)), key=key, pts=pts, md5=np.array(md5),
                  source=np.array("demo/1m.mp4"))
    with zipfile.ZipFile(path, "w", compression=zipfile.ZIP_LZMA) as z:
        for name, a in arrays.items():
            buf = io.BytesIO()
            np.lib.format.write_array(buf, a, allow_pickle=False)
            z.writestr(name + ".npy", buf.getvalue())


def main():
    if not os.path.isdir(FF_SRC):
        sys.exit("the reference tree is not present; the committed fixture is the only copy on this machine")
    build_tool()
    raw = os.path.join(ROOT, "oracle", "_ref", "demo_1m_meta.bin")
    run([TOOL, os.path.join(REF, "demo", "1m.mp4"), raw])
    buf = np.fromfile(raw, dtype=np.uint8)
    n, w_mb, h_mb, _ = buf[:16].view(np.int32)
    sz = int(n) * int(w_mb) * int(h_mb) * 4
    frames = buf[16:16 + sz].reshape(n, h_mb, w_mb, 4)
    key = buf[16 + sz:16 + sz + n].copy()
    pts = buf[16 + sz + n:16 + sz + n + 8 * n].copy().view(np.int64)
    md5 = hashlib.md5(frames.tobytes()).hexdigest()
    save_fixture(OUT, frames, key, pts, md5)
    hist = np.bincount(frames[..., 0].ravel(), minlength=8)
    print(f"{n} frames of {w_mb}x{h_mb}, md5 {md5}, {int(key.sum())} key frames, "
          f"mb_weight histogram {(hist / hist.sum()).round(4).tolist()}, byte3 max {int(frames[..., 3].max())}, "
          f"fixture {os.path.getsize(OUT) / 1e6:.2f} MB")
    if "--keep" not in sys.argv:          # the snapshot sent to the GPU box should not carry 60 MB of objects
        import shutil
        os.remove(raw)
        shutil.rmtree(BUILD, ignore_errors=True)


if __name__ == "__main__":
    main()
