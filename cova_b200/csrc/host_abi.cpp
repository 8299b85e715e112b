// C ABI of the host-side components that sit directly behind the GPU path (include/cova_b200.h, "sorttracker").
// No CUDA in this translation unit.
#include <stdio.h>

#include <new>

#include "../../include/cova_b200.h"
#include "cova_select.hpp"
#include "frame_packer.hpp"
#include "gop_demux.hpp"
#include "sort_tracker.hpp"

namespace cova {
extern thread_local char g_err[512];
}
static int fail(int code, const char *msg) {
    snprintf(cova::g_err, sizeof(cova::g_err), "%s", msg);
    return code;
}

using cova::host::Bbox;
using cova::host::KalmanBoxTracker;
using cova::host::Sort;

struct cova_sorttracker {
    uint32_t maxage, minhits;
    float iou;
    Sort *sort;  // created by set_caps (sorttracker/imp.rs:214-236), like the element
    std::vector<Bbox> scratch;
};

static int emit(const std::vector<KalmanBoxTracker> &tracks, uint8_t *out, size_t cap, size_t *out_len, std::vector<Bbox> &flat) {
    flat.clear();
    for (const auto &t : tracks) flat.insert(flat.end(), t.history.begin(), t.history.end());
    size_t need = cova::host::boxes_wire_size(flat);
    if (out_len) *out_len = need;
    if (need > cap || !out) return fail(COVA_E_TOOSMALL, "output buffer too small for the serialized tracks");
    cova::host::encode_boxes_into(flat, out);
    return COVA_OK;
}

extern "C" int cova_sorttracker_new(cova_sorttracker **out) {
    if (!out) return fail(COVA_E_INVAL, "null out");
    cova_sorttracker *s = new (std::nothrow) cova_sorttracker{30, 30, 0.1f, nullptr, {}};
    if (!s) return fail(COVA_E_NOMEM, "host allocation failed");
    *out = s;
    return COVA_OK;
}
extern "C" void cova_sorttracker_free(cova_sorttracker *s) {
    if (!s) return;
    delete s->sort;
    delete s;
}
extern "C" int cova_sorttracker_set_property(cova_sorttracker *s, const char *name, double value) {
    if (!s || !name) return fail(COVA_E_INVAL, "null argument");
    if (!strcmp(name, "iou-threshold")) {
        if (!(value >= 0.0 && value <= 1.0)) return fail(COVA_E_INVAL, "iou-threshold is a float in [0, 1]");
        s->iou = (float)value;
    } else if (!strcmp(name, "maxage")) {
        if (!(value >= 0.0 && value <= 4294967295.0)) return fail(COVA_E_INVAL, "maxage is a u32");
        s->maxage = (uint32_t)value;
    } else if (!strcmp(name, "minhits")) {
        if (!(value >= 0.0 && value <= 4294967295.0)) return fail(COVA_E_INVAL, "minhits is a u32");
        s->minhits = (uint32_t)value;
    } else {
        return fail(COVA_E_INVAL, "unknown property (iou-threshold, maxage, minhits)");
    }
    return COVA_OK;
}
extern "C" int cova_sorttracker_get_property(const cova_sorttracker *s, const char *name, double *value) {
    if (!s || !name || !value) return fail(COVA_E_INVAL, "null argument");
    if (!strcmp(name, "iou-threshold")) *value = s->iou;
    else if (!strcmp(name, "maxage")) *value = s->maxage;
    else if (!strcmp(name, "minhits")) *value = s->minhits;
    else return fail(COVA_E_INVAL, "unknown property (iou-threshold, maxage, minhits)");
    return COVA_OK;
}
extern "C" int cova_sorttracker_set_caps(cova_sorttracker *s, int32_t width, int32_t height) {
    if (!s) return fail(COVA_E_INVAL, "null handle");
    if (width < 0 || height < 0) return fail(COVA_E_INVAL, "caps width/height are in [0, i32::MAX]");
    delete s->sort;
    s->sort = new (std::nothrow) Sort(s->maxage, s->minhits, s->iou);
    return s->sort ? COVA_OK : fail(COVA_E_NOMEM, "host allocation failed");
}
extern "C" int cova_sorttracker_transform(cova_sorttracker *s, const uint8_t *boxes, size_t boxes_len, uint64_t pts_ns,
                                          uint8_t *out, size_t out_cap, size_t *out_len) {
    if (!s || !boxes) return fail(COVA_E_INVAL, "null argument");
    if (!s->sort) return fail(COVA_E_INVAL, "transform before set_caps");
    std::vector<Bbox> dets;
    if (!cova::host::decode_boxes(boxes, boxes_len, dets)) return fail(COVA_E_INVAL, "input is not bincode(Vec<Bbox>)");
    std::vector<KalmanBoxTracker> dead;
    if (!s->sort->update(std::move(dets), pts_ns, dead)) return fail(COVA_E_NUMERIC, "Kalman update: innovation covariance not positive definite");
    return emit(dead, out, out_cap, out_len, s->scratch);
}
extern "C" int cova_sorttracker_eos(cova_sorttracker *s, uint8_t *out, size_t out_cap, size_t *out_len) {
    if (!s) return fail(COVA_E_INVAL, "null handle");
    if (!s->sort) return fail(COVA_E_INVAL, "eos before set_caps");
    // the tracks leave the tracker only when the caller's buffer can take them
    std::vector<KalmanBoxTracker> keep = s->sort->trackers;
    std::vector<KalmanBoxTracker> fin = s->sort->finalize();
    int rc = emit(fin, out, out_cap, out_len, s->scratch);
    if (rc != COVA_OK) s->sort->trackers.swap(keep);
    return rc;
}
extern "C" int cova_sorttracker_n_tracks(const cova_sorttracker *s, uint32_t *n_total, uint32_t *n_active) {
    if (!s || !s->sort) return fail(COVA_E_INVAL, "no tracker state");
    uint32_t a = 0;
    for (const auto &t : s->sort->trackers) a += t.active;
    if (n_total) *n_total = (uint32_t)s->sort->trackers.size();
    if (n_active) *n_active = a;
    return COVA_OK;
}

// building blocks, exported so that the reference's own unit tests can be replayed through the ABI
extern "C" int cova_sort_linear_assignment(const float *cost, uint32_t n_trk, uint32_t n_det, int32_t *pairs, uint32_t *n_pairs) {
    if (!cost || !pairs || !n_pairs) return fail(COVA_E_INVAL, "null argument");
    std::vector<float> c(cost, cost + (size_t)n_trk * n_det);
    auto m = cova::host::linear_assignment(c, (int)n_trk, (int)n_det);
    for (size_t i = 0; i < m.size(); i++) pairs[2 * i] = m[i].first, pairs[2 * i + 1] = m[i].second;
    *n_pairs = (uint32_t)m.size();
    return COVA_OK;
}
extern "C" int cova_sort_iou_matrix(const float *preds, uint32_t n_preds, const float *dets, uint32_t n_dets, float *out) {
    if ((!preds && n_preds) || (!dets && n_dets) || !out) return fail(COVA_E_INVAL, "null argument");
    std::vector<Bbox> p, d;
    for (uint32_t i = 0; i < n_preds; i++) p.push_back(Bbox::make(preds[4 * i], preds[4 * i + 1], preds[4 * i + 2], preds[4 * i + 3]));
    for (uint32_t i = 0; i < n_dets; i++) d.push_back(Bbox::make(dets[4 * i], dets[4 * i + 1], dets[4 * i + 2], dets[4 * i + 3]));
    auto c = Sort::iou_cost(p, d);
    memcpy(out, c.data(), c.size() * sizeof(float));
    return COVA_OK;
}
extern "C" int cova_sort_match_dets(const float *preds, const uint8_t *active, uint32_t n_preds, const float *dets, uint32_t n_dets,
                                    float iou_threshold, int32_t *pairs, uint32_t *n_pairs) {
    if ((!preds && n_preds) || (!active && n_preds) || (!dets && n_dets) || !pairs || !n_pairs) return fail(COVA_E_INVAL, "null argument");
    std::vector<Bbox> p, d;
    std::vector<char> a(active, active + n_preds);
    for (uint32_t i = 0; i < n_preds; i++) p.push_back(Bbox::make(preds[4 * i], preds[4 * i + 1], preds[4 * i + 2], preds[4 * i + 3]));
    for (uint32_t i = 0; i < n_dets; i++) d.push_back(Bbox::make(dets[4 * i], dets[4 * i + 1], dets[4 * i + 2], dets[4 * i + 3]));
    auto m = Sort::match_dets(p, a, d, iou_threshold);
    for (size_t i = 0; i < m.size(); i++) pairs[2 * i] = m[i].first, pairs[2 * i + 1] = m[i].second;
    *n_pairs = (uint32_t)m.size();
    return COVA_OK;
}

// =================================================================================================
// cova element: frame selection (cova_select.hpp)
// =================================================================================================
using cova::host::CovaSelect;
using cova::host::Pushed;

struct cova_select {
    CovaSelect c;
    std::vector<Pushed> pending;
};

static int take_pushed(cova_select *s, cova_pushed_buffer *out, size_t cap, size_t *n) {
    if (n) *n = s->pending.size();
    if (s->pending.size() > cap || (!out && !s->pending.empty()))
        return fail(COVA_E_TOOSMALL, "pushed-buffer array too small; call cova_select_take_pushed with the reported count");
    for (size_t i = 0; i < s->pending.size(); i++) {
        out[i].id = s->pending[i].id, out[i].pts_ns = s->pending[i].pts;
        out[i].flags = s->pending[i].flags, out[i].list = s->pending[i].list;
    }
    s->pending.clear();
    return COVA_OK;
}

extern "C" int cova_select_new(cova_select **out) {
    if (!out) return fail(COVA_E_INVAL, "null out");
    cova_select *s = new (std::nothrow) cova_select();
    if (!s) return fail(COVA_E_NOMEM, "host allocation failed");
    *out = s;
    return COVA_OK;
}
extern "C" void cova_select_free(cova_select *s) { delete s; }
extern "C" int cova_select_set_property(cova_select *s, const char *name, double v) {
    if (!s || !name) return fail(COVA_E_INVAL, "null argument");
    const bool u32 = v >= 0.0 && v <= 4294967295.0;
    if (!strcmp(name, "sort-iou")) {
        if (!(v >= 0.0 && v <= 1.0)) return fail(COVA_E_INVAL, "sort-iou is a float in [0, 1]");
        s->c.sort_iou = (float)v;
    } else if (!strcmp(name, "sort-maxage") && u32) s->c.sort_maxage = (uint32_t)v;
    else if (!strcmp(name, "sort-minhits") && u32) s->c.sort_minhits = (uint32_t)v;
    else if (!strcmp(name, "port") && u32) s->c.port = (uint32_t)v;
    else if (!strcmp(name, "alpha") && u32) s->c.alpha = (uint32_t)v;
    else if (!strcmp(name, "beta") && u32) s->c.beta = (uint32_t)v;
    else if (!strcmp(name, "infer-i")) s->c.infer_i = v != 0.0;
    else if (!strcmp(name, "debug")) s->c.debug = v != 0.0;
    else return fail(COVA_E_INVAL, "unknown or read-only property, or value out of range");
    return COVA_OK;
}
extern "C" int cova_select_get_property(const cova_select *s, const char *name, double *v) {
    if (!s || !name || !v) return fail(COVA_E_INVAL, "null argument");
    if (!strcmp(name, "sort-iou")) *v = s->c.sort_iou;
    else if (!strcmp(name, "sort-maxage")) *v = s->c.sort_maxage;
    else if (!strcmp(name, "sort-minhits")) *v = s->c.sort_minhits;
    else if (!strcmp(name, "port")) *v = s->c.port;
    else if (!strcmp(name, "alpha")) *v = s->c.alpha;
    else if (!strcmp(name, "beta")) *v = s->c.beta;
    else if (!strcmp(name, "infer-i")) *v = s->c.infer_i;
    else if (!strcmp(name, "debug")) *v = s->c.debug;
    else if (!strcmp(name, "dropped")) *v = (double)s->c.dropped;
    else if (!strcmp(name, "decoded-dependency")) *v = (double)s->c.decoded_dependency;
    else if (!strcmp(name, "decoded-inference")) *v = (double)s->c.decoded_inference;
    else return fail(COVA_E_INVAL, "unknown property");
    return COVA_OK;
}
extern "C" int cova_select_sink_enc(cova_select *s, uint64_t buf_id, uint64_t pts_ns, uint32_t flags) {
    if (!s) return fail(COVA_E_INVAL, "null handle");
    if (!s->c.push_enc(buf_id, pts_ns, (flags & COVA_BUFFER_FLAG_DELTA_UNIT) != 0))
        return fail(COVA_E_INVAL, "delta unit before the first key frame (the reference unwraps an empty GoP list)");
    return COVA_OK;
}
extern "C" int cova_select_sink_mask(cova_select *s, const uint8_t *boxes, size_t boxes_len, uint64_t pts_ns,
                                     cova_pushed_buffer *out, size_t out_cap, size_t *n_out) {
    if (!s || !boxes) return fail(COVA_E_INVAL, "null argument");
    std::vector<Bbox> dets;
    if (!cova::host::decode_boxes(boxes, boxes_len, dets)) return fail(COVA_E_INVAL, "input is not bincode(Vec<Bbox>)");
    const int rc = s->c.push_boxes(std::move(dets), pts_ns, s->pending);
    if (rc == -1) return fail(COVA_E_NUMERIC, "Kalman update: innovation covariance not positive definite");
    if (rc == -2) return fail(COVA_E_STATE, "no frame could be selected for a dead track (assert!(track_inferenced > 0), cova/imp.rs:239)");
    return take_pushed(s, out, out_cap, n_out);
}
extern "C" int cova_select_eos(cova_select *s, int pad, cova_pushed_buffer *out, size_t out_cap, size_t *n_out) {
    if (!s || (pad != 0 && pad != 1)) return fail(COVA_E_INVAL, "pad is 0 (sink_enc) or 1 (sink_mask)");
    const bool drained = s->c.on_eos(pad, s->pending);
    const int rc = take_pushed(s, out, out_cap, n_out);
    if (rc) return rc;
    return drained ? COVA_OK : COVA_DROPPED;
}
extern "C" int cova_select_take_pushed(cova_select *s, cova_pushed_buffer *out, size_t out_cap, size_t *n_out) {
    if (!s) return fail(COVA_E_INVAL, "null handle");
    return take_pushed(s, out, out_cap, n_out);
}
extern "C" int cova_select_take_wire(cova_select *s, uint8_t *out, size_t out_cap, size_t *out_len) {
    if (!s) return fail(COVA_E_INVAL, "null handle");
    if (out_len) *out_len = s->c.wire.size();
    if (s->c.wire.size() > out_cap || (!out && !s->c.wire.empty())) return fail(COVA_E_TOOSMALL, "wire buffer too small");
    if (!s->c.wire.empty()) memcpy(out, s->c.wire.data(), s->c.wire.size());
    s->c.wire.clear();
    return COVA_OK;
}

// =================================================================================================
// demux + gopsplit (gop_demux.hpp)
// =================================================================================================
static int emit_samples(const std::vector<cova::host::Sample> &v, cova_sample *out, size_t cap, size_t *n) {
    if (n) *n = v.size();
    if (v.size() > cap || (!out && !v.empty())) return fail(COVA_E_TOOSMALL, "sample array too small");
    for (size_t i = 0; i < v.size(); i++) {
        out[i].offset = v[i].offset, out[i].size = v[i].size, out[i].flags = v[i].flags;
        out[i].dts = v[i].dts, out[i].pts = v[i].pts;
    }
    return COVA_OK;
}
extern "C" int cova_demux_mp4_samples(const uint8_t *data, size_t len, cova_sample *out, size_t out_cap, size_t *n_out,
                                      cova_mp4_info *info) {
    if (!data) return fail(COVA_E_INVAL, "null argument");
    std::vector<cova::host::Sample> v;
    cova::host::Mp4Info mi;
    int rc;
    try {   // nothing throws across the C ABI: the sample tables are sized from file contents
        rc = cova::host::mp4_video_samples(data, len, v, mi);
    } catch (const std::bad_alloc &) {
        return fail(COVA_E_NOMEM, "sample table too large");
    }
    if (rc == -1) return fail(COVA_E_INVAL, "malformed or truncated ISO media file (moov / stbl)");
    if (rc == -2) return fail(COVA_E_UNSUPPORTED, "no video track with an avc1 sample entry");
    if (info) info->timescale = mi.timescale, info->width = mi.width, info->height = mi.height, info->nal_length_size = mi.nal_length_size;
    return emit_samples(v, out, out_cap, n_out);
}
extern "C" int cova_demux_annexb_frames(const uint8_t *data, size_t len, cova_sample *out, size_t out_cap, size_t *n_out) {
    if (!data && len) return fail(COVA_E_INVAL, "null argument");
    std::vector<cova::host::Sample> v;
    try {
        cova::host::annexb_frames(data, len, v);
    } catch (const std::bad_alloc &) {
        return fail(COVA_E_NOMEM, "access-unit table too large");
    }
    return emit_samples(v, out, out_cap, n_out);
}
extern "C" int cova_gopsplit_ranges(const uint32_t *flags, size_t n_frames, uint32_t n_pads, uint64_t *first_frame, uint64_t *end_frame) {
    if ((!flags && n_frames) || !first_frame || !end_frame) return fail(COVA_E_INVAL, "null argument");
    if (!cova::host::gopsplit_ranges(flags, n_frames, n_pads, first_frame, end_frame)) return fail(COVA_E_INVAL, "there are no pads");
    return COVA_OK;
}

// =================================================================================================
// host packer for COVA_FLAG_INPUT_PACKED16 (frame_packer.hpp)
// =================================================================================================
struct cova_packer {
    cova::host::Packer pk;
    explicit cova_packer(unsigned n) : pk(n) {}
};
extern "C" int cova_packer_new(cova_packer **out, uint32_t n_threads) {
    if (!out) return fail(COVA_E_INVAL, "null out");
    *out = nullptr;
    try {
        *out = new cova_packer(n_threads);
    } catch (const std::exception &) {      // bad_alloc, or std::system_error when a thread cannot be started
        return fail(COVA_E_NOMEM, "could not start the packer's worker threads");
    }
    return COVA_OK;
}
extern "C" void cova_packer_free(cova_packer *pk) { delete pk; }
extern "C" int cova_packer_pack(cova_packer *pk, const uint8_t *quads, uint16_t *out, size_t n_mb) {
    if (!pk || (!quads && n_mb) || (!out && n_mb)) return fail(COVA_E_INVAL, "null argument");
    pk->pk.pack(quads, out, n_mb);
    return COVA_OK;
}
static_assert(COVA_SPARSE_MAX_FRAME_BYTES(3600) == cova::sparse::max_record_bytes(3600) &&
                  COVA_SPARSE_MAX_FRAME_BYTES(8160) == cova::sparse::max_record_bytes(8160) &&
                  COVA_SPARSE_MAX_FRAME_BYTES(129600) == cova::sparse::max_record_bytes(129600),
              "COVA_SPARSE_MAX_FRAME_BYTES and sparse_format.hpp disagree");
extern "C" int cova_packer_pack_sparse(cova_packer *pk, const uint8_t *quads, uint32_t n_frames, uint32_t w_mb, uint32_t h_mb,
                                       uint8_t *out, size_t out_cap, size_t *out_len) {
    if (!pk || !out_len || (!quads && n_frames)) return fail(COVA_E_INVAL, "null argument");
    if (!w_mb || !h_mb) return fail(COVA_E_INVAL, "empty macroblock grid");
    if ((uint64_t)w_mb * h_mb > UINT32_MAX / 2) return fail(COVA_E_INVAL, "macroblock grid too large");
    try {
        if (!pk->pk.pack_sparse(quads, n_frames, w_mb * h_mb, out, out_cap, out_len))
            return fail(COVA_E_TOOSMALL, "output buffer too small for the sparse batch; *out_len is the size it needs");
    } catch (const std::bad_alloc &) {
        return fail(COVA_E_NOMEM, "staging allocation failed");
    }
    return COVA_OK;
}
