"""Host-side mirror of the reference's element interface for the blob-detection path.

The reference host language is Rust (GStreamer elements in cova-rs/gst-plugins); there is no Rust
toolchain in this image, so the layer above the C ABI is Python, keeping the reference's element names,
property names, caps arithmetic and flow results:

  MetaPreprocess   <- cova-rs/gst-plugins/src/metapreprocess/imp.rs  (properties timestep, gamma)
  BboxCc           <- cova-rs/gst-plugins/src/bboxcc/imp.rs          (property cc-threshold, default 30)
  SortTracker      <- cova-rs/gst-plugins/src/sorttracker/imp.rs     (properties iou-threshold, maxage, minhits;
                      host C++ behind the same C ABI, fed with the boxes the GPU path returns)
  CovaSelect       <- cova-rs/gst-plugins/src/cova/imp.rs            (frame selection: which encoded frames still
                      need a pixel decode; properties sort-iou, sort-maxage, sort-minhits, port, infer-i, alpha, beta)
  BlobPipeline     <- the chain metapreprocess ! nvvideoconvert ! nvstreammux ! nvinfer(BlobNet) !
                      nvstreamdemux ! maskcopy ! bboxcc of pipeline/cova/pipeline.py:101-250, batched
                      over many chains, with only the bincode boxes returning to the host.

All compute happens in libcova_b200.so (CUDA, sm_100a); nothing here has a CPU fallback.
"""
from __future__ import annotations

import ctypes
import struct
from dataclasses import dataclass

import numpy as np

from . import _lib
from ._lib import CovaError, check

FLOW_OK = _lib.OK
FLOW_DROPPED = _lib.DROPPED          # gst_base::BASE_TRANSFORM_FLOW_DROPPED
DEFAULT_TIMESTEP = 1                 # metapreprocess/imp.rs:20
DEFAULT_GAMMA = 1                    # metapreprocess/imp.rs:21
DEFAULT_CC_THRESHOLD = 30            # bboxcc/imp.rs:16


def _ptr(a: np.ndarray):
    return ctypes.c_void_p(a.ctypes.data)


class PinnedBuffer:
    """Page-locked host memory (cova_host_alloc) viewed as a numpy array; lets process() overlap copies."""

    def __init__(self, shape, dtype=np.uint8):
        self.shape, self.dtype = tuple(int(v) for v in np.atleast_1d(shape)), np.dtype(dtype)
        self.nbytes = max(1, int(np.prod(self.shape)) * self.dtype.itemsize)
        self._p = ctypes.c_void_p()
        check(_lib.load().cova_host_alloc(ctypes.byref(self._p), self.nbytes))
        buf = (ctypes.c_uint8 * self.nbytes).from_address(self._p.value)
        self.array = np.frombuffer(buf, dtype=self.dtype, count=int(np.prod(self.shape))).reshape(self.shape)

    def close(self):
        if self._p:
            self.array = None
            _lib.load().cova_host_free(self._p)
            self._p = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


@dataclass
class SparseBatch:
    """A batch in the sparse input format (include/cova_b200.h, COVA_SPARSE_MAX_FRAME_BYTES): the records of
    n_streams x frames_per_stream frames, stream-major.  `data` is u8 and exactly the batch's bytes (it may be a view of
    a PinnedBuffer array).  BlobPipeline(packed_input=True).submit() takes it like a dense frames array."""
    data: np.ndarray
    n_streams: int
    frames_per_stream: int
    h_mb: int
    w_mb: int


class FramePacker:
    """Host packer for BlobPipeline(packed_input=True): decoder quads [.., h, w, 4] u8 -> [.., h, w] u16
    (cova_packer_pack: min(b, 6) of bytes 0-2 in 3 bits each; worker threads live as long as the packer), or -> a
    SparseBatch (pack_sparse)."""

    def __init__(self, n_threads: int = 0):
        self._h = ctypes.c_void_p()
        check(_lib.load().cova_packer_new(ctypes.byref(self._h), n_threads))

    def pack(self, quads: np.ndarray, out: np.ndarray | None = None) -> np.ndarray:
        a = np.ascontiguousarray(quads, dtype=np.uint8)
        assert a.shape[-1] == 4, a.shape
        if out is None:
            out = np.empty(a.shape[:-1], dtype=np.uint16)
        assert out.dtype == np.uint16 and out.size == a.size // 4 and out.flags.c_contiguous
        check(_lib.load().cova_packer_pack(self._h, _ptr(a), _ptr(out), out.size))
        return out

    def pack_sparse(self, quads: np.ndarray, out: np.ndarray | None = None) -> SparseBatch:
        """quads [n_streams, frames, h, w, 4] u8 -> SparseBatch (cova_packer_pack_sparse).  `out`: a u8 array to encode
        into (e.g. PinnedBuffer(...).array); data is then a view of its first bytes.  Raises CovaError(E_TOOSMALL) when
        it is too small."""
        a = np.ascontiguousarray(quads, dtype=np.uint8)
        assert a.ndim == 5 and a.shape[-1] == 4, a.shape
        n_streams, fps, h_mb, w_mb = a.shape[:4]
        n_frames = n_streams * fps
        if out is None:
            out = np.empty(n_frames * _lib.sparse_max_frame_bytes(h_mb * w_mb), dtype=np.uint8)
        assert out.dtype == np.uint8 and out.flags.c_contiguous
        ln = ctypes.c_size_t()
        check(_lib.load().cova_packer_pack_sparse(self._h, _ptr(a), n_frames, w_mb, h_mb, _ptr(out), out.size, ctypes.byref(ln)))
        return SparseBatch(out.reshape(-1)[: ln.value], n_streams, fps, h_mb, w_mb)

    def close(self):
        if self._h:
            _lib.load().cova_packer_free(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MetaPreprocess:
    """`metapreprocess` element: one instance == one stream == one sliding window."""

    ELEMENT_NAME = "metapreprocess"

    def __init__(self, width: int, height: int, timestep: int = DEFAULT_TIMESTEP, gamma: int = DEFAULT_GAMMA,
                 device: int = 0):
        self._h = ctypes.c_void_p()
        check(_lib.load().cova_metapreprocess_new(ctypes.byref(self._h), device, width, height, timestep, gamma))
        self.timestep, self._gamma = timestep, gamma
        w, h, sz = ctypes.c_uint32(), ctypes.c_uint32(), ctypes.c_size_t()
        check(_lib.load().cova_metapreprocess_out_caps(self._h, ctypes.byref(w), ctypes.byref(h), ctypes.byref(sz)))
        self.out_width, self.out_height, self.out_size = w.value, h.value, sz.value
        self.size_per_buf = self.out_size // timestep

    # GObject-style property access with the reference's property names
    def set_property(self, name: str, value: int):
        if name == "gamma":
            check(_lib.load().cova_metapreprocess_set_gamma(self._h, value))
            self._gamma = value
        elif name == "timestep":
            raise CovaError(_lib.E_INVAL, "timestep is only mutable in READY state: create a new element")
        else:
            raise KeyError(name)

    def get_property(self, name: str) -> int:
        return {"gamma": self._gamma, "timestep": self.timestep}[name]

    def transform_caps(self) -> dict:
        """src caps for I420 sink caps of this size (imp.rs:247-286)."""
        return {"format": "RGBA", "width": self.out_width, "height": self.out_height}

    def transform(self, inbuf) -> tuple[int, bytes | None]:
        a = np.frombuffer(inbuf, dtype=np.uint8) if not isinstance(inbuf, np.ndarray) else np.ascontiguousarray(inbuf).reshape(-1)
        out = np.empty(self.out_size, dtype=np.uint8)
        rc = check(_lib.load().cova_metapreprocess_transform(self._h, _ptr(a), a.size, _ptr(out), out.size))
        return (FLOW_OK, out.tobytes()) if rc == FLOW_OK else (FLOW_DROPPED, None)

    def close(self):
        if self._h:
            _lib.load().cova_metapreprocess_free(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class BboxCc:
    """`bboxcc` element: mask buffer in, bincode(Vec<Bbox>) out (in place in the reference)."""

    ELEMENT_NAME = "bboxcc"

    def __init__(self, width: int, height: int, cc_threshold: int = DEFAULT_CC_THRESHOLD, device: int = 0,
                 cluster: bool = False, bands: int = 0):
        # cluster=True: grids beyond one CTA's shared memory (8K) run the thread-block-cluster CCL instead of being
        # refused; bands=k forces that kernel with k bands on any grid (COVA_FLAG_CCL_CLUSTER / COVA_FLAG_CCL_BANDS)
        self._h = ctypes.c_void_p()
        flags = (_lib.FLAG_CCL_CLUSTER if cluster else 0) | (_lib.flag_ccl_bands(bands) if bands else 0)
        check(_lib.load().cova_bboxcc_new2(ctypes.byref(self._h), device, width, height, cc_threshold, flags))
        self.width, self.height = width, height
        self._cap = _lib.load().cova_bboxcc_max_out_size(self._h)

    def set_property(self, name: str, value: int):
        if name != "cc-threshold":
            raise KeyError(name)
        check(_lib.load().cova_bboxcc_set_cc_threshold(self._h, value))

    def get_property(self, name: str) -> int:
        if name != "cc-threshold":
            raise KeyError(name)
        v = ctypes.c_uint32()
        check(_lib.load().cova_bboxcc_get_cc_threshold(self._h, ctypes.byref(v)))
        return v.value

    def transform_ip(self, buf) -> bytes:
        a = np.frombuffer(buf, dtype=np.uint8) if not isinstance(buf, np.ndarray) else np.ascontiguousarray(buf, dtype=np.uint8).reshape(-1)
        out = np.empty(self._cap, dtype=np.uint8)
        n = ctypes.c_size_t()
        check(_lib.load().cova_bboxcc_transform_ip(self._h, _ptr(a), a.size, _ptr(out), out.size, ctypes.byref(n)))
        return out[: n.value].tobytes()

    def labels(self, mask: np.ndarray):
        """What cv::connectedComponentsWithStats returns for this mask (parity helper)."""
        a = np.ascontiguousarray(mask, dtype=np.uint8).reshape(-1)
        labels = np.empty(self.height * self.width, dtype=np.int32)
        nb = ((self.height + 1) // 2) * ((self.width + 1) // 2)
        stats = np.zeros((nb + 1, 5), dtype=np.int32)
        n = ctypes.c_int32()
        check(_lib.load().cova_bboxcc_labels(self._h, _ptr(a), a.size, _ptr(labels), _ptr(stats), ctypes.byref(n)))
        return n.value, labels.reshape(self.height, self.width), stats[: n.value]

    def close(self):
        if self._h:
            _lib.load().cova_bboxcc_free(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def deserialize_vec(buf: bytes) -> list[tuple]:
    """Bbox::deserialize_vec (cova-rs/bbox/src/bbox.rs:88-90) for boxes whose Options are all None."""
    (n,) = struct.unpack_from("<Q", buf, 0)
    out, off = [], 8
    for _ in range(n):
        left, top, w, h, area = struct.unpack_from("<5f", buf, off)
        if buf[off + 20: off + 24] != b"\0\0\0\0":
            raise ValueError("unexpected Some(..) in a bboxcc box")
        out.append((left, top, w, h, area))
        off += 24
    if off != len(buf):
        raise ValueError("trailing bytes after Vec<Bbox>")
    return out


def deserialize_vec_full(buf: bytes) -> list[tuple]:
    """Bbox::deserialize_vec for boxes that may carry Some(track_id / timestamp / class_id / confidence):
    (left, top, width, height, area, track_id, timestamp, class_id, confidence), None where absent."""
    (n,) = struct.unpack_from("<Q", buf, 0)
    out, off = [], 8
    for _ in range(n):
        vals = list(struct.unpack_from("<5f", buf, off))
        off += 20
        for fmt, size in (("<Q", 8), ("<Q", 8), ("<I", 4), ("<f", 4)):
            tag = buf[off]
            off += 1
            if tag > 1:
                raise ValueError("bad Option tag")
            vals.append(struct.unpack_from(fmt, buf, off)[0] if tag else None)
            off += size if tag else 0
        out.append(tuple(vals))
    if off != len(buf):
        raise ValueError("trailing bytes after Vec<Bbox>")
    return out


class SortTracker:
    """`sorttracker` element: per-frame bincode(Vec<Bbox>) in, bincode of the histories of the tracks that died on
    this frame out; `eos()` is the extra buffer pushed on EOS (sorttracker/imp.rs:238-287)."""

    ELEMENT_NAME = "sorttracker"
    OUT_SIZE = 1 << 21  # transform_size(): constant 2 MiB (imp.rs:322-332)

    def __init__(self, **props):
        self._h = ctypes.c_void_p()
        check(_lib.load().cova_sorttracker_new(ctypes.byref(self._h)))
        self._out = np.empty(self.OUT_SIZE, dtype=np.uint8)
        for k, v in props.items():
            self.set_property(k.replace("_", "-"), v)

    def set_property(self, name: str, value):
        if name not in ("iou-threshold", "maxage", "minhits"):
            raise KeyError(name)
        check(_lib.load().cova_sorttracker_set_property(self._h, name.encode(), float(value)))

    def get_property(self, name: str):
        if name not in ("iou-threshold", "maxage", "minhits"):
            raise KeyError(name)
        v = ctypes.c_double()
        check(_lib.load().cova_sorttracker_get_property(self._h, name.encode(), ctypes.byref(v)))
        return v.value if name == "iou-threshold" else int(v.value)

    def set_caps(self, width: int, height: int):
        check(_lib.load().cova_sorttracker_set_caps(self._h, width, height))

    def _call(self, fn, *args) -> bytes:
        n = ctypes.c_size_t()
        rc = fn(self._h, *args, _ptr(self._out), self._out.size, ctypes.byref(n))
        if rc == _lib.E_TOOSMALL and fn is _lib.load().cova_sorttracker_eos:
            self._out = np.empty(n.value, dtype=np.uint8)
            rc = fn(self._h, *args, _ptr(self._out), self._out.size, ctypes.byref(n))
        check(rc)
        return self._out[: n.value].tobytes()

    def transform(self, buf: bytes, pts_ns: int) -> bytes:
        a = np.frombuffer(buf, dtype=np.uint8)
        return self._call(_lib.load().cova_sorttracker_transform, _ptr(a), a.size, pts_ns)

    def eos(self) -> bytes:
        return self._call(_lib.load().cova_sorttracker_eos)

    def n_tracks(self) -> tuple[int, int]:
        t, a = ctypes.c_uint32(), ctypes.c_uint32()
        check(_lib.load().cova_sorttracker_n_tracks(self._h, ctypes.byref(t), ctypes.byref(a)))
        return t.value, a.value

    def close(self):
        if self._h:
            _lib.load().cova_sorttracker_free(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class CovaSelect:
    """`cova` element: `sink_enc(id, pts, flags)` for every encoded frame, `sink_mask(boxes, pts)` for every box
    blob; both return / accumulate the buffer lists the element would push downstream as tuples
    (id, pts, flags, list index)."""

    ELEMENT_NAME = "cova"
    FLAG_DELTA_UNIT, FLAG_DISCONT, FLAG_DROPPABLE = 1, 2, 4
    EMPTY_LIST = 2**64 - 1

    def __init__(self, **props):
        self._h = ctypes.c_void_p()
        check(_lib.load().cova_select_new(ctypes.byref(self._h)))
        self._out = (_lib.PushedBuffer * 4096)()
        for k, v in props.items():
            self.set_property(k.replace("_", "-"), v)

    def set_property(self, name: str, value):
        check(_lib.load().cova_select_set_property(self._h, name.encode(), float(value)))

    def get_property(self, name: str):
        v = ctypes.c_double()
        check(_lib.load().cova_select_get_property(self._h, name.encode(), ctypes.byref(v)))
        return v.value if name == "sort-iou" else (bool(v.value) if name in ("infer-i", "debug") else int(v.value))

    def sink_enc(self, buf_id: int, pts_ns: int, flags: int):
        check(_lib.load().cova_select_sink_enc(self._h, buf_id, pts_ns, flags))

    def _pushed(self, rc: int, n) -> list[tuple]:
        if rc == _lib.E_TOOSMALL:
            self._out = (_lib.PushedBuffer * n.value)()
            rc = _lib.load().cova_select_take_pushed(self._h, self._out, len(self._out), ctypes.byref(n))
        check(rc)
        return [(b.id, b.pts_ns, b.flags, b.list) for b in self._out[: n.value]]

    def sink_mask(self, boxes: bytes, pts_ns: int) -> list[tuple]:
        a = np.frombuffer(boxes, dtype=np.uint8)
        n = ctypes.c_size_t()
        rc = _lib.load().cova_select_sink_mask(self._h, _ptr(a), a.size, pts_ns, self._out, len(self._out), ctypes.byref(n))
        return self._pushed(rc, n)

    def eos(self, pad: int):
        """pad 0 = sink_enc, 1 = sink_mask; None until both pads have seen EOS."""
        n = ctypes.c_size_t()
        rc = _lib.load().cova_select_eos(self._h, pad, self._out, len(self._out), ctypes.byref(n))
        out = self._pushed(rc, n)
        return None if rc == _lib.DROPPED else out

    def take_wire(self) -> bytes:
        n = ctypes.c_size_t()
        lib = _lib.load()
        rc = lib.cova_select_take_wire(self._h, None, 0, ctypes.byref(n))
        if rc == _lib.OK:
            return b""
        buf = np.empty(n.value, dtype=np.uint8)
        check(lib.cova_select_take_wire(self._h, _ptr(buf), buf.size, ctypes.byref(n)))
        return buf.tobytes()

    def close(self):
        if self._h:
            _lib.load().cova_select_free(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class BlobPipeline:
    """Fused batch path on one GPU.  `process(frames)` is the call a user makes: host frames in
    ([n_streams, frames_per_stream, h_mb, w_mb, 4] u8), per-window bincode blobs out."""

    def __init__(self, w_mb: int, h_mb: int, weights_blob: bytes, max_streams: int, max_frames_per_stream: int,
                 timestep: int = 4, gamma: int = 1, cc_threshold: int = 1, device: int = 0,
                 impl: int = _lib.IMPL_TCGEN05, keep_logits: bool = False, keep_stacked: bool = False, n_chunks: int = 0,
                 validation: bool = False, packed_input: bool = False, ccl_cluster: bool = False, ccl_bands: int = 0):
        # validation=True (or impl=IMPL_SIMT) binds this handle to libcova_b200_val.so, the build that also holds the
        # fp32 validation kernels; the product library refuses IMPL_SIMT
        self._L = _lib.load_validation() if (validation or impl == _lib.IMPL_SIMT) else _lib.load()
        self._h = ctypes.c_void_p()
        flags = impl | (_lib.FLAG_KEEP_LOGITS if keep_logits else 0) | (_lib.FLAG_KEEP_STACKED if keep_stacked else 0)
        flags |= (n_chunks & 0xff) << 16
        flags |= _lib.FLAG_INPUT_PACKED16 if packed_input else 0
        # ccl_cluster / ccl_bands: as BboxCc's cluster / bands
        flags |= (_lib.FLAG_CCL_CLUSTER if ccl_cluster else 0) | (_lib.flag_ccl_bands(ccl_bands) if ccl_bands else 0)
        # packed_input: every frames argument is [n_streams, frames, h_mb, w_mb] u16 (FramePacker) instead of [.., 4] u8
        self.packed_input = packed_input
        self._wbuf = ctypes.create_string_buffer(weights_blob, len(weights_blob))
        self._check(self._L.cova_pipeline_new(ctypes.byref(self._h), device, w_mb, h_mb, timestep, gamma, max_streams,
                                            max_frames_per_stream, ctypes.cast(self._wbuf, ctypes.c_void_p),
                                            len(weights_blob), cc_threshold, flags))
        self.w_mb, self.h_mb, self.timestep, self.gamma = w_mb, h_mb, timestep, gamma
        self.max_streams, self.max_fps = max_streams, max_frames_per_stream
        self.n_windows = 0
        self._blob = None

    def _check(self, rc: int) -> int:
        return check(rc, self._L)

    # ---- configuration
    def set_property(self, name: str, value: int):
        if name != "cc-threshold":
            raise KeyError(name)
        self._check(self._L.cova_pipeline_set_cc_threshold(self._h, value))

    def set_stream(self, cuda_stream: int | None):
        self._check(self._L.cova_pipeline_set_stream(self._h, ctypes.c_void_p(cuda_stream or 0)))

    def windows_for(self, n_streams: int, frames_per_stream: int) -> int:
        n = ctypes.c_uint32()
        self._check(self._L.cova_pipeline_n_windows(self._h, n_streams, frames_per_stream, ctypes.byref(n)))
        return n.value

    def _frames(self, frames) -> np.ndarray:
        if self.packed_input:
            a = np.ascontiguousarray(frames, dtype=np.uint16)
            assert a.shape[2:] == (self.h_mb, self.w_mb), a.shape
        else:
            a = np.ascontiguousarray(frames, dtype=np.uint8)
            assert a.shape[2:] == (self.h_mb, self.w_mb, 4), a.shape
        return a

    # ---- stages
    def load_frames(self, frames, n_streams: int | None = None, frames_per_stream: int | None = None):
        """frames: numpy array (host; u8 quads, or u16 with packed_input) or an int device pointer (then the two counts
        are required)."""
        if isinstance(frames, np.ndarray):
            a = self._frames(frames)
            n_streams, frames_per_stream = a.shape[0], a.shape[1]
            self._keep = a
            self._check(self._L.cova_pipeline_load_frames(self._h, _ptr(a), n_streams, frames_per_stream, 0))
        else:
            self._check(self._L.cova_pipeline_load_frames(self._h, ctypes.c_void_p(int(frames)), n_streams, frames_per_stream, 1))
        self.n_windows = self.windows_for(n_streams, frames_per_stream)

    def load_masks(self, masks, n: int | None = None):
        if isinstance(masks, np.ndarray):
            a = np.ascontiguousarray(masks, dtype=np.uint8)
            n = a.shape[0]
            self._keep = a
            self._check(self._L.cova_pipeline_load_masks(self._h, _ptr(a), n, 0))
        else:
            self._check(self._L.cova_pipeline_load_masks(self._h, ctypes.c_void_p(int(masks)), n, 1))
        self.n_windows = n

    def tensorise(self):
        self._check(self._L.cova_pipeline_tensorise(self._h))

    def blobnet(self):
        self._check(self._L.cova_pipeline_blobnet(self._h))

    def run_layer(self, layer: int, impl: int):
        self._check(self._L.cova_pipeline_run_layer(self._h, layer, impl))

    def ccl(self):
        self._check(self._L.cova_pipeline_ccl(self._h))

    def run(self):
        self._check(self._L.cova_pipeline_run(self._h))

    def sync(self):
        self._check(self._L.cova_pipeline_sync(self._h))

    def fetch_boxes_raw(self, blob_cap: int | None = None):
        """(blob, offsets, lens): window i's bincode(Vec<Bbox>) is blob[offsets[i] : offsets[i] + lens[i]].
        The arrays are reused by the next call.  `blob_cap` bounds the host arena (default: worst case)."""
        n = self.n_windows
        cap = blob_cap or n * (8 + 24 * ((self.h_mb + 1) // 2) * ((self.w_mb + 1) // 2))
        self._ensure_out(cap)
        ln = ctypes.c_size_t()
        self._check(self._L.cova_pipeline_fetch_boxes(self._h, _ptr(self._blob), self._blob.size, ctypes.byref(ln),
                                                    _ptr(self._offs), _ptr(self._lens)))
        self.last_blob_len = ln.value
        return self._blob, self._offs[:n], self._lens[:n]

    def _ensure_out(self, cap: int):
        if self._blob is None or self._blob.size < cap:
            nw = max(self.max_streams * self.max_fps, 1)
            self._pin = [[PinnedBuffer(max(cap, 8)), PinnedBuffer(nw, np.uint64), PinnedBuffer(nw, np.uint64)] for _ in range(2)]
            self._blob, self._offs, self._lens = (b.array for b in self._pin[0])

    def _worst_case_cap(self, n_windows: int) -> int:
        return n_windows * (8 + 24 * ((self.h_mb + 1) // 2) * ((self.w_mb + 1) // 2))

    # ---- asynchronous streaming form: at most four batches in flight
    def submit(self, frames: np.ndarray, blob_cap: int | None = None, stream_ids=None, pts=None, cont: bool | None = None,
               staggered: bool = False):
        """Enqueue one batch (copies + kernels) and return immediately.  `frames` should live in page-locked
        memory (PinnedBuffer) and must stay untouched until the matching collect().

        With `stream_ids` / `pts` / `cont` the batch goes through cova_pipeline_submit_host2: chain s belongs to stream
        stream_ids[s] (default 0, 1, ...), `pts[s, f]` is echoed per window by collect(meta=True), and cont=True continues
        the streams from their previous batch (carried timestep-1 frames + gamma phase) like one long-lived metapreprocess
        element would.  staggered=True (with cont=True) lets those streams differ in history and gamma phase: each continues
        from its own state, so chains may yield different numbers of windows (collect(meta=True) maps them to streams).

        `frames` may be a SparseBatch (packed_input pipelines): it goes through cova_pipeline_submit_sparse with the same
        stream semantics as cova_pipeline_submit_host2."""
        if isinstance(frames, SparseBatch):
            self._submit_sparse(frames, blob_cap, stream_ids, pts, cont, staggered)
            return
        a = self._frames(frames)
        if stream_ids is None and pts is None and cont is None and not staggered:
            self._ensure_out(blob_cap or self._worst_case_cap(self.windows_for(a.shape[0], a.shape[1])))
            self._check(self._L.cova_pipeline_submit_host(self._h, _ptr(a), a.shape[0], a.shape[1]))
        else:
            # a continued chain can emit one window per new frame
            self._ensure_out(blob_cap or self._worst_case_cap(a.shape[0] * a.shape[1]))
            ids = None if stream_ids is None else np.ascontiguousarray(stream_ids, dtype=np.uint32)
            p = None if pts is None else np.ascontiguousarray(pts, dtype=np.uint64)
            assert ids is None or ids.shape == (a.shape[0],)
            assert p is None or p.shape == a.shape[:2]
            self._check(self._L.cova_pipeline_submit_host2(self._h, _ptr(a), a.shape[0], a.shape[1], None if ids is None else _ptr(ids),
                                                         None if p is None else _ptr(p),
                                                         (_lib.SUBMIT_CONTINUE if cont else 0) | (_lib.SUBMIT_STAGGERED if staggered else 0)))
        self._inflight = getattr(self, "_inflight", []) + [a]

    def _submit_sparse(self, b: SparseBatch, blob_cap, stream_ids, pts, cont, staggered):
        assert (b.h_mb, b.w_mb) == (self.h_mb, self.w_mb), (b.h_mb, b.w_mb)
        d = b.data
        assert d.dtype == np.uint8 and d.ndim == 1 and d.flags.c_contiguous
        self._ensure_out(blob_cap or self._worst_case_cap(b.n_streams * b.frames_per_stream))
        ids = None if stream_ids is None else np.ascontiguousarray(stream_ids, dtype=np.uint32)
        p = None if pts is None else np.ascontiguousarray(pts, dtype=np.uint64)
        assert ids is None or ids.shape == (b.n_streams,)
        assert p is None or p.shape == (b.n_streams, b.frames_per_stream)
        self._check(self._L.cova_pipeline_submit_sparse(self._h, _ptr(d), d.size, b.n_streams, b.frames_per_stream,
                                                        None if ids is None else _ptr(ids), None if p is None else _ptr(p),
                                                        (_lib.SUBMIT_CONTINUE if cont else 0) | (_lib.SUBMIT_STAGGERED if staggered else 0)))
        self._inflight = getattr(self, "_inflight", []) + [d]

    def reset_streams(self, stream_ids=None):
        if stream_ids is None:
            self._check(self._L.cova_pipeline_reset_streams(self._h, None, 0))
        else:
            ids = np.ascontiguousarray(stream_ids, dtype=np.uint32)
            self._check(self._L.cova_pipeline_reset_streams(self._h, _ptr(ids), ids.size))

    def collect(self, raw: bool = False, meta: bool = False):
        """Wait for the oldest submitted batch; same return value as process().  meta=True (batches submitted with
        stream_ids / pts): returns (result, window_stream_ids, window_pts) through cova_pipeline_collect_host2."""
        k = getattr(self, "_collect_idx", 0)
        self._collect_idx = k ^ 1
        blob, offs, lens = (b.array for b in self._pin[k])
        ln, nw = ctypes.c_size_t(), ctypes.c_uint32()
        if meta:
            wid, wpts = np.zeros(offs.size, dtype=np.uint32), np.zeros(offs.size, dtype=np.uint64)
            rc = self._L.cova_pipeline_collect_host2(self._h, _ptr(blob), blob.size, ctypes.byref(ln), _ptr(offs), _ptr(lens),
                                                         ctypes.byref(nw), _ptr(wid), _ptr(wpts))
        else:
            rc = self._L.cova_pipeline_collect_host(self._h, _ptr(blob), blob.size, ctypes.byref(ln), _ptr(offs), _ptr(lens),
                                                        ctypes.byref(nw))
        if getattr(self, "_inflight", None):
            self._inflight.pop(0)
        self._check(rc)
        self.n_windows, self.last_blob_len = nw.value, ln.value
        n = nw.value
        res = (blob, offs[:n], lens[:n]) if raw else [blob[int(o): int(o) + int(l)].tobytes() for o, l in zip(offs[:n], lens[:n])]
        return (res, wid[:n], wpts[:n]) if meta else res

    def fetch_boxes(self) -> list[bytes]:
        blob, offs, lens = self.fetch_boxes_raw()
        return [blob[int(o): int(o) + int(l)].tobytes() for o, l in zip(offs, lens)]

    def process(self, frames: np.ndarray, raw: bool = False, blob_cap: int | None = None):
        """Host frames -> per-window bincode(Vec<Bbox>) blobs (stream-major, time-minor): a list of bytes,
        or with raw=True the (blob, offsets, lens) arrays without per-window Python objects."""
        a = self._frames(frames)
        n_streams, fps = a.shape[0], a.shape[1]
        n = self.windows_for(n_streams, fps)
        self._ensure_out(blob_cap or self._worst_case_cap(n))
        self._collect_idx = 0
        ln, nw = ctypes.c_size_t(), ctypes.c_uint32()
        self._check(self._L.cova_pipeline_process_host(self._h, _ptr(a), n_streams, fps, _ptr(self._blob), self._blob.size,
                                                     ctypes.byref(ln), _ptr(self._offs), _ptr(self._lens), ctypes.byref(nw)))
        self.n_windows, self.last_blob_len = nw.value, ln.value
        if raw:
            return self._blob, self._offs[:n], self._lens[:n]
        return [self._blob[int(o): int(o) + int(l)].tobytes() for o, l in zip(self._offs[:n], self._lens[:n])]

    # ---- inspection (parity tests)
    def read_stacked(self) -> np.ndarray:
        out = np.empty((self.n_windows, self.timestep * self.h_mb, self.w_mb, 4), dtype=np.uint8)
        self._check(self._L.cova_pipeline_read_stacked(self._h, _ptr(out), out.size))
        return out

    def read_mask(self) -> np.ndarray:
        out = np.empty((self.n_windows, self.h_mb, self.w_mb), dtype=np.uint8)
        self._check(self._L.cova_pipeline_read_mask(self._h, _ptr(out), out.size))
        return out

    def read_logits(self) -> np.ndarray:
        out = np.empty((self.n_windows, self.h_mb, self.w_mb), dtype=np.float32)
        self._check(self._L.cova_pipeline_read_logits(self._h, _ptr(out), out.size))
        return out

    def read_activation(self, layer: int) -> np.ndarray:
        cap = self.n_windows * 128 * 4 * self.h_mb * self.w_mb
        out = np.empty(cap, dtype=np.float32)
        shape = (ctypes.c_uint32 * 5)()
        self._check(self._L.cova_pipeline_read_activation(self._h, layer, _ptr(out), out.size, shape))
        shp = tuple(int(v) for v in shape)
        return out[: int(np.prod(shp))].reshape(shp).copy()

    def set_debug(self, flags: int):
        self._check(self._L.cova_pipeline_set_debug(self._h, flags))

    def last_plan(self) -> list[dict]:
        """cova_pipeline_last_plan: per layer the launch plan of its last tcgen05 launch (family 0: not launched yet)."""
        out = (_lib.LayerPlan * _lib.N_LAYERS)()
        self._check(self._L.cova_pipeline_last_plan(self._h, out))
        return [p.as_dict() for p in out]

    def launch_count(self) -> int:
        c = ctypes.c_uint64()
        self._check(self._L.cova_pipeline_launch_count(self._h, ctypes.byref(c)))
        return c.value

    def set_profiling(self, enable: bool):
        self._check(self._L.cova_pipeline_set_profiling(self._h, int(enable)))

    def last_timings(self) -> dict[str, float]:
        names = ctypes.create_string_buffer(1024)
        ms = (ctypes.c_float * 64)()
        n = ctypes.c_uint32(64)
        self._check(self._L.cova_pipeline_last_timings(self._h, names, 1024, ms, ctypes.byref(n)))
        keys = names.value.decode().split(";") if names.value else []
        return {k: float(ms[i]) for i, k in enumerate(keys)}

    def close(self):
        if self._h:
            self._L.cova_pipeline_free(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
