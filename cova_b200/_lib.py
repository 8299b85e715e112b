"""ctypes binding of libcova_b200.so (include/cova_b200.h).  Fails loudly if the library is missing:
there is no Python / CPU fallback for any of the entry points."""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libcova_b200.so")
SO_VAL_PATH = os.path.join(_HERE, "libcova_b200_val.so")   # product sources + the validation kernels (tests only)

OK, DROPPED = 0, 1
E_INVAL, E_CUDA, E_NOMEM, E_TOOSMALL, E_WEIGHTS, E_UNSUPPORTED, E_NODEVICE, E_NUMERIC, E_STATE = -1, -2, -3, -4, -5, -6, -7, -8, -9
IMPL_TCGEN05, IMPL_SIMT = 0, 1
FLAG_KEEP_LOGITS, FLAG_KEEP_STACKED, FLAG_INPUT_PACKED16 = 0x100, 0x200, 0x400
FLAG_CCL_CLUSTER = 0x800


def flag_ccl_bands(k: int) -> int:
    """COVA_FLAG_CCL_BANDS(k): force the cluster CCL with k bands (k = 2..8; needs FLAG_CCL_CLUSTER)."""
    return (k & 0xF) << 24


SUBMIT_CONTINUE = 1
SUBMIT_STAGGERED = 2       # with SUBMIT_CONTINUE: the continued streams of a batch may differ in history and gamma phase


def sparse_max_frame_bytes(n_mb: int) -> int:
    """COVA_SPARSE_MAX_FRAME_BYTES(n_mb): the size of a sparse record in which every macroblock differs."""
    return 8 + 4 * ((n_mb + 31) // 32) + 4 * ((n_mb + 1) // 2)


class CovaError(RuntimeError):
    def __init__(self, code: int, detail: str):
        super().__init__(f"cova_b200 error {code}: {detail}")
        self.code = code


_u8p = ctypes.POINTER(ctypes.c_uint8)
_i32p = ctypes.POINTER(ctypes.c_int32)
_u32p = ctypes.POINTER(ctypes.c_uint32)
_u64p = ctypes.POINTER(ctypes.c_uint64)
_f32p = ctypes.POINTER(ctypes.c_float)
_szp = ctypes.POINTER(ctypes.c_size_t)
_vp = ctypes.c_void_p
_vpp = ctypes.POINTER(ctypes.c_void_p)

# name -> (restype, argtypes); every symbol include/cova_b200.h declares
SIGNATURES = {
    "cova_version": (ctypes.c_char_p, []),
    "cova_strerror": (ctypes.c_char_p, [ctypes.c_int]),
    "cova_last_error": (ctypes.c_char_p, []),
    "cova_device_count": (ctypes.c_int, [ctypes.POINTER(ctypes.c_int)]),
    "cova_host_alloc": (ctypes.c_int, [_vpp, ctypes.c_size_t]),
    "cova_bind_host_to_device": (ctypes.c_int, [ctypes.c_int, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)]),
    "cova_host_free": (None, [_vp]),
    "cova_metapreprocess_new": (ctypes.c_int, [_vpp, ctypes.c_int, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32]),
    "cova_metapreprocess_free": (None, [_vp]),
    "cova_metapreprocess_set_gamma": (ctypes.c_int, [_vp, ctypes.c_uint32]),
    "cova_metapreprocess_out_caps": (ctypes.c_int, [_vp, _u32p, _u32p, _szp]),
    "cova_metapreprocess_transform": (ctypes.c_int, [_vp, _vp, ctypes.c_size_t, _vp, ctypes.c_size_t]),
    "cova_bboxcc_new": (ctypes.c_int, [_vpp, ctypes.c_int, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32]),
    "cova_bboxcc_new2": (ctypes.c_int, [_vpp, ctypes.c_int, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32]),
    "cova_bboxcc_free": (None, [_vp]),
    "cova_bboxcc_set_cc_threshold": (ctypes.c_int, [_vp, ctypes.c_uint32]),
    "cova_bboxcc_get_cc_threshold": (ctypes.c_int, [_vp, _u32p]),
    "cova_bboxcc_max_out_size": (ctypes.c_size_t, [_vp]),
    "cova_bboxcc_transform_ip": (ctypes.c_int, [_vp, _vp, ctypes.c_size_t, _vp, ctypes.c_size_t, _szp]),
    "cova_bboxcc_labels": (ctypes.c_int, [_vp, _vp, ctypes.c_size_t, _vp, _vp, _i32p]),
    "cova_pipeline_new": (ctypes.c_int, [_vpp, ctypes.c_int, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32,
                                        ctypes.c_uint32, ctypes.c_uint32, _vp, ctypes.c_size_t, ctypes.c_uint32, ctypes.c_uint32]),
    "cova_pipeline_free": (None, [_vp]),
    "cova_pipeline_set_cc_threshold": (ctypes.c_int, [_vp, ctypes.c_uint32]),
    "cova_pipeline_set_segmentation_threshold": (ctypes.c_int, [_vp, ctypes.c_float]),
    "cova_pipeline_set_stream": (ctypes.c_int, [_vp, _vp]),
    "cova_pipeline_n_windows": (ctypes.c_int, [_vp, ctypes.c_uint32, ctypes.c_uint32, _u32p]),
    "cova_pipeline_load_frames": (ctypes.c_int, [_vp, _vp, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_int]),
    "cova_pipeline_tensorise": (ctypes.c_int, [_vp]),
    "cova_pipeline_blobnet": (ctypes.c_int, [_vp]),
    "cova_pipeline_ccl": (ctypes.c_int, [_vp]),
    "cova_pipeline_run": (ctypes.c_int, [_vp]),
    "cova_pipeline_sync": (ctypes.c_int, [_vp]),
    "cova_pipeline_fetch_boxes": (ctypes.c_int, [_vp, _vp, ctypes.c_size_t, _szp, _vp, _vp]),
    "cova_pipeline_process_host": (ctypes.c_int, [_vp, _vp, ctypes.c_uint32, ctypes.c_uint32, _vp, ctypes.c_size_t, _szp, _vp, _vp, _u32p]),
    "cova_pipeline_submit_host": (ctypes.c_int, [_vp, _vp, ctypes.c_uint32, ctypes.c_uint32]),
    "cova_pipeline_collect_host": (ctypes.c_int, [_vp, _vp, ctypes.c_size_t, _szp, _vp, _vp, _u32p]),
    "cova_pipeline_submit_host2": (ctypes.c_int, [_vp, _vp, ctypes.c_uint32, ctypes.c_uint32, _vp, _vp, ctypes.c_uint32]),
    "cova_pipeline_collect_host2": (ctypes.c_int, [_vp, _vp, ctypes.c_size_t, _szp, _vp, _vp, _u32p, _vp, _vp]),
    "cova_pipeline_reset_streams": (ctypes.c_int, [_vp, _vp, ctypes.c_uint32]),
    "cova_pipeline_set_stream_property": (ctypes.c_int, [_vp, _vp, ctypes.c_uint32, ctypes.c_char_p, ctypes.c_uint32]),
    "cova_pipeline_get_stream_property": (ctypes.c_int, [_vp, ctypes.c_uint32, ctypes.c_char_p, _u32p]),
    "cova_pipeline_set_stream_property_f32": (ctypes.c_int, [_vp, _vp, ctypes.c_uint32, ctypes.c_char_p, ctypes.c_float]),
    "cova_pipeline_get_stream_property_f32": (ctypes.c_int, [_vp, ctypes.c_uint32, ctypes.c_char_p, _f32p]),
    "cova_packer_new": (ctypes.c_int, [_vpp, ctypes.c_uint32]),
    "cova_packer_free": (None, [_vp]),
    "cova_packer_pack": (ctypes.c_int, [_vp, _vp, _vp, ctypes.c_size_t]),
    "cova_packer_pack_sparse": (ctypes.c_int, [_vp, _vp, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32, _vp, ctypes.c_size_t, _szp]),
    "cova_pipeline_submit_sparse": (ctypes.c_int, [_vp, _vp, ctypes.c_size_t, ctypes.c_uint32, ctypes.c_uint32, _vp, _vp, ctypes.c_uint32]),
    "cova_pipeline_submit_ragged": (ctypes.c_int, [_vp, _vp, ctypes.c_uint32, _vp, _vp, _vp, ctypes.c_uint32]),
    "cova_pipeline_submit_sparse_ragged": (ctypes.c_int, [_vp, _vp, ctypes.c_size_t, ctypes.c_uint32, _vp, _vp, _vp, ctypes.c_uint32]),
    "cova_pipeline_load_masks": (ctypes.c_int, [_vp, _vp, ctypes.c_uint32, ctypes.c_int]),
    "cova_pipeline_read_stacked": (ctypes.c_int, [_vp, _vp, ctypes.c_size_t]),
    "cova_pipeline_read_mask": (ctypes.c_int, [_vp, _vp, ctypes.c_size_t]),
    "cova_pipeline_read_logits": (ctypes.c_int, [_vp, _vp, ctypes.c_size_t]),
    "cova_pipeline_read_activation": (ctypes.c_int, [_vp, ctypes.c_int, _vp, ctypes.c_size_t, _u32p]),
    "cova_pipeline_run_layer": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_uint32]),
    "cova_pipeline_set_debug": (ctypes.c_int, [_vp, ctypes.c_int]),
    "cova_pipeline_set_sm_limit": (ctypes.c_int, [_vp, ctypes.c_int]),
    "cova_blobnet_plan": (ctypes.c_int, [ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_int, ctypes.c_int, _vp]),
    "cova_pipeline_last_plan": (ctypes.c_int, [_vp, _vp]),
    "cova_pipeline_launch_count": (ctypes.c_int, [_vp, _u64p]),
    "cova_pipeline_set_profiling": (ctypes.c_int, [_vp, ctypes.c_int]),
    "cova_pipeline_last_timings": (ctypes.c_int, [_vp, ctypes.c_char_p, ctypes.c_size_t, _f32p, _u32p]),
    "cova_sorttracker_new": (ctypes.c_int, [_vpp]),
    "cova_sorttracker_free": (None, [_vp]),
    "cova_sorttracker_set_property": (ctypes.c_int, [_vp, ctypes.c_char_p, ctypes.c_double]),
    "cova_sorttracker_get_property": (ctypes.c_int, [_vp, ctypes.c_char_p, ctypes.POINTER(ctypes.c_double)]),
    "cova_sorttracker_set_caps": (ctypes.c_int, [_vp, ctypes.c_int32, ctypes.c_int32]),
    "cova_sorttracker_transform": (ctypes.c_int, [_vp, _vp, ctypes.c_size_t, ctypes.c_uint64, _vp, ctypes.c_size_t, _szp]),
    "cova_sorttracker_eos": (ctypes.c_int, [_vp, _vp, ctypes.c_size_t, _szp]),
    "cova_sorttracker_n_tracks": (ctypes.c_int, [_vp, _u32p, _u32p]),
    "cova_sort_linear_assignment": (ctypes.c_int, [_vp, ctypes.c_uint32, ctypes.c_uint32, _vp, _u32p]),
    "cova_sort_iou_matrix": (ctypes.c_int, [_vp, ctypes.c_uint32, _vp, ctypes.c_uint32, _vp]),
    "cova_sort_match_dets": (ctypes.c_int, [_vp, _vp, ctypes.c_uint32, _vp, ctypes.c_uint32, ctypes.c_float, _vp, _u32p]),
}



PLAN_ENC1, PLAN_POS, PLAN_WS = 1, 2, 3
N_LAYERS = 8


class LayerPlan(ctypes.Structure):
    """cova_layer_plan"""
    _fields_ = [(k, ctypes.c_int32) for k in ("family", "config", "tps", "tile", "n_stage", "n_groups", "ctas")]

    def as_dict(self) -> dict:
        return {k: getattr(self, k) for k, _ in self._fields_}


def blobnet_plan(w_mb: int, h_mb: int, windows: int, debug: int = 0, n_sms: int = 148) -> list[dict]:
    """cova_blobnet_plan: per layer the launch plan the library would pick (host arithmetic, no device).  Raises CovaError
    (E_UNSUPPORTED) when a layer has no plan."""
    lib = load()
    out = (LayerPlan * N_LAYERS)()
    check(lib.cova_blobnet_plan(w_mb, h_mb, windows, debug, n_sms, out), lib)
    return [p.as_dict() for p in out]


class PushedBuffer(ctypes.Structure):
    """cova_pushed_buffer"""
    _fields_ = [("id", ctypes.c_uint64), ("pts_ns", ctypes.c_uint64), ("flags", ctypes.c_uint32), ("list", ctypes.c_uint32)]


class Sample(ctypes.Structure):
    """cova_sample"""
    _fields_ = [("offset", ctypes.c_uint64), ("size", ctypes.c_uint32), ("flags", ctypes.c_uint32),
                ("dts", ctypes.c_uint64), ("pts", ctypes.c_uint64)]


class Mp4Info(ctypes.Structure):
    """cova_mp4_info"""
    _fields_ = [("timescale", ctypes.c_uint32), ("width", ctypes.c_uint32), ("height", ctypes.c_uint32),
                ("nal_length_size", ctypes.c_uint32)]


SIGNATURES.update({
    "cova_demux_mp4_samples": (ctypes.c_int, [_vp, ctypes.c_size_t, _vp, ctypes.c_size_t, _szp, _vp]),
    "cova_demux_annexb_frames": (ctypes.c_int, [_vp, ctypes.c_size_t, _vp, ctypes.c_size_t, _szp]),
    "cova_gopsplit_ranges": (ctypes.c_int, [_vp, ctypes.c_size_t, ctypes.c_uint32, _vp, _vp]),
    "cova_select_new": (ctypes.c_int, [_vpp]),
    "cova_select_free": (None, [_vp]),
    "cova_select_set_property": (ctypes.c_int, [_vp, ctypes.c_char_p, ctypes.c_double]),
    "cova_select_get_property": (ctypes.c_int, [_vp, ctypes.c_char_p, ctypes.POINTER(ctypes.c_double)]),
    "cova_select_sink_enc": (ctypes.c_int, [_vp, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint32]),
    "cova_select_sink_mask": (ctypes.c_int, [_vp, _vp, ctypes.c_size_t, ctypes.c_uint64, _vp, ctypes.c_size_t, _szp]),
    "cova_select_eos": (ctypes.c_int, [_vp, ctypes.c_int, _vp, ctypes.c_size_t, _szp]),
    "cova_select_take_pushed": (ctypes.c_int, [_vp, _vp, ctypes.c_size_t, _szp]),
    "cova_select_take_wire": (ctypes.c_int, [_vp, _vp, ctypes.c_size_t, _szp]),
})

_lib = None
_lib_val = None


def _open(path: str) -> ctypes.CDLL:
    if not os.path.exists(path):
        raise ImportError(f"{path} is missing: run `python -m cova_b200.build` (nvcc, sm_100a). "
                          "cova_b200 has no CPU fallback.")
    lib = ctypes.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib


def load() -> ctypes.CDLL:
    """Load the shared library (built in-tree by cova_b200/build.py).  Raises if it is absent."""
    global _lib
    if _lib is None:
        _lib = _open(SO_PATH)
    return _lib


def load_validation() -> ctypes.CDLL:
    """The validation build (product + COVA_IMPL_SIMT kernels): only the layer-by-layer parity tests ask for it."""
    global _lib_val
    if _lib_val is None:
        _lib_val = _open(SO_VAL_PATH)
    return _lib_val


def check(rc: int, lib: ctypes.CDLL | None = None) -> int:
    if rc < 0:
        raise CovaError(rc, (lib or load()).cova_last_error().decode(errors="replace"))
    return rc
