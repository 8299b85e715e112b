/* cova_b200 - C ABI of the B200-native blob-detection path of CoVA.
 *
 * Everything a Rust (cgo / JNI / ctypes ...) host needs is plain pointers and sizes; no CUDA or
 * torch types appear in any signature.  A CUDA stream, where accepted, travels as void*.
 *
 * Conventions (SURVEY.md section 8b):
 *   return 0 (COVA_OK) on success, COVA_DROPPED (1) when an element produced no output for this
 *   input (GStreamer's BASE_TRANSFORM_FLOW_DROPPED), a negative COVA_E_* on error.  The library
 *   never aborts across the FFI boundary; cova_last_error() gives a thread-local detail string.
 *   Handles are single-caller (one streaming thread per element instance, as in the reference);
 *   different handles may be used concurrently from different threads.
 *
 * Each entry point cites the reference interface it replaces (paths relative to the reference tree).
 */
#ifndef COVA_B200_H
#define COVA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define COVA_OK 0
#define COVA_DROPPED 1
#define COVA_E_INVAL (-1)       /* bad argument */
#define COVA_E_CUDA (-2)        /* a CUDA call failed; see cova_last_error() */
#define COVA_E_NOMEM (-3)
#define COVA_E_TOOSMALL (-4)    /* output buffer too small; the required size is reported */
#define COVA_E_WEIGHTS (-5)     /* not a CVBN v1 weight container */
#define COVA_E_UNSUPPORTED (-6) /* e.g. timestep != 4 for BlobNet, grid too large for the CCL kernel (see COVA_FLAG_CCL_CLUSTER) */
#define COVA_E_NODEVICE (-7)    /* no CUDA device: there is no CPU fallback */
#define COVA_E_NUMERIC (-8)     /* host tracker: Kalman innovation covariance not positive definite */
#define COVA_E_STATE (-9)       /* host frame selection: a state the reference asserts can never happen */

const char *cova_version(void);
const char *cova_strerror(int code);
const char *cova_last_error(void);
int cova_device_count(int *n);
/* page-locked host memory: frame and box buffers in it let process_host overlap copies with kernels */
int cova_host_alloc(void **out, size_t bytes);
/* Multi-GPU, one process per GPU (the reference starts one pipeline process per `--cuda` device,
 * experiment/cova/launch.py:33-93):
 * restrict the calling thread to the CPUs local to `device` so that buffers it allocates afterwards are placed on the
 * GPU's NUMA node.  numa_node / n_cpus (optional) report what was found; no topology information = no change. */
int cova_bind_host_to_device(int device, int *numa_node, int *n_cpus);
void cova_host_free(void *ptr);

/* ------------------------------------------------------------------------------------------------
 * metapreprocess element   (cova-rs/gst-plugins/src/metapreprocess/imp.rs)
 *   properties timestep, gamma            imp.rs:57-133  (u32 >= 1, defaults 1)
 *   caps: I420 WxH -> RGBA (W/16) x (H/16*timestep), integer division   imp.rs:247-286
 *   transform(): sliding window, first timestep-1 buffers dropped, gamma sub-sampling  imp.rs:288-332
 * One handle == one element instance == one stream.  The window lives in device memory; the stacking
 * is done by the tensorise kernel (csrc/tensorise.cuh).
 * ------------------------------------------------------------------------------------------------ */
typedef struct cova_metapreprocess cova_metapreprocess;

int cova_metapreprocess_new(cova_metapreprocess **out, int device, uint32_t width_px, uint32_t height_px,
                            uint32_t timestep, uint32_t gamma);
void cova_metapreprocess_free(cova_metapreprocess *mp);
/* mutable like the GObject property (imp.rs:104-113) */
int cova_metapreprocess_set_gamma(cova_metapreprocess *mp, uint32_t gamma);
/* transform_caps(): output RGBA width/height and buffer size in bytes */
int cova_metapreprocess_out_caps(const cova_metapreprocess *mp, uint32_t *width, uint32_t *height, size_t *size);
/* transform(): reads the first size/timestep bytes of inbuf (host memory).  COVA_OK: outbuf holds the
 * stacked RGBA image (row block k = frame t-k).  COVA_DROPPED: nothing written. */
int cova_metapreprocess_transform(cova_metapreprocess *mp, const uint8_t *inbuf, size_t in_len, uint8_t *outbuf,
                                  size_t out_cap);

/* ------------------------------------------------------------------------------------------------
 * bboxcc element   (cova-rs/gst-plugins/src/bboxcc/imp.rs, process.rs)
 *   property cc-threshold u32, default 30, mutable while PLAYING      imp.rs:16,51-101
 *   transform_ip(): mask (height rows of len/height bytes, any non-zero byte = foreground)
 *     -> 8-connected components (cv::connectedComponentsWithStats order) -> keep pixel-area >= threshold
 *     -> bincode(Vec<Bbox>) replaces the buffer content                imp.rs:232-272, process.rs:5-49
 *   wire format: u64 LE count, then per box 5 x f32 LE (left, top, width, height, width*height) and
 *   four 0x00 Option tags = 24 bytes                                   cova-rs/bbox/src/bbox.rs:3-29,84-86
 * ------------------------------------------------------------------------------------------------ */
typedef struct cova_bboxcc cova_bboxcc;

int cova_bboxcc_new(cova_bboxcc **out, int device, uint32_t width, uint32_t height, uint32_t cc_threshold);
/* as cova_bboxcc_new (which is new2 with flags 0), with COVA_FLAG_CCL_CLUSTER / COVA_FLAG_CCL_BANDS(k) (see below);
 * any other bit is COVA_E_INVAL */
int cova_bboxcc_new2(cova_bboxcc **out, int device, uint32_t width, uint32_t height, uint32_t cc_threshold,
                     uint32_t flags);
void cova_bboxcc_free(cova_bboxcc *cc);
int cova_bboxcc_set_cc_threshold(cova_bboxcc *cc, uint32_t cc_threshold);
int cova_bboxcc_get_cc_threshold(const cova_bboxcc *cc, uint32_t *cc_threshold);
/* upper bound of the serialized size for this grid: 8 + 24*ceil(H/2)*ceil(W/2) */
size_t cova_bboxcc_max_out_size(const cova_bboxcc *cc);
/* COVA_E_TOOSMALL sets *out_len to the required size (the reference re-allocates, imp.rs:253-258) */
int cova_bboxcc_transform_ip(cova_bboxcc *cc, const uint8_t *mask, size_t mask_len, uint8_t *out, size_t out_cap,
                             size_t *out_len);
/* parity helper: what cv::connectedComponentsWithStats returns.  labels: i32[H*W]; stats: i32[n*5]
 * (left, top, width, height, area) with row 0 (background) zeroed; stats capacity must be
 * (ceil(H/2)*ceil(W/2)+1)*5 ints.  *n_labels counts the background. */
int cova_bboxcc_labels(cova_bboxcc *cc, const uint8_t *mask, size_t mask_len, int32_t *labels, int32_t *stats,
                       int32_t *n_labels);

/* ------------------------------------------------------------------------------------------------
 * Fused batch path: tensorise -> BlobNet -> threshold -> CCL on device, boxes only come back.
 * Replaces the chain metapreprocess -> nvvideoconvert -> nvstreammux -> nvinfer(TensorRT BlobNet)
 * -> nvstreamdemux -> maskcopy -> bboxcc (pipeline/cova/pipeline.py:101-250), for many chains at once.
 *
 * A batch is n_streams independent chains of frames_per_stream consecutive frames each, every chain
 * starting with an empty window exactly like a freshly started element (gopsplit hands every chain
 * whole GoPs, gst-plugins/gst-gopsplit/gstgopsplit.cpp:557-630); cova_pipeline_submit_host2 below continues
 * named streams across batches instead.  Windows are emitted in stream-major,
 * time-minor order; window w of a stream is the one whose newest frame is (timestep-1) + w*gamma.
 * ------------------------------------------------------------------------------------------------ */
typedef struct cova_pipeline cova_pipeline;

#define COVA_IMPL_TCGEN05 0u /* product path: tcgen05/TMEM implicit GEMM */
#define COVA_IMPL_SIMT 1u    /* validation kernels (CUDA cores, fp32 weights) used by the tests */
#define COVA_FLAG_KEEP_LOGITS 0x100u  /* also store fp32 logits (parity tests) */
#define COVA_FLAG_KEEP_STACKED 0x200u /* also materialise the stacked RGBA windows (parity tests) */
/* Frames arrive in the 2-byte packed format instead of the decoder's 4-byte quads: one little-endian u16 per macroblock,
 * bits 0-2 min(mb_weight, 6), bits 3-5 min(|mv_x|, 6), bits 6-8 min(|mv_y|, 6), the rest 0 (cova_packer_pack produces it).
 * Exact for BlobNet - its first operation is clip(x, 0, 6) (utils/model/preprocessing.py:5-8) and byte 3 never reaches it
 * (nvinfer drops the alpha channel, config/blobnet/amsterdam_b128.txt:7,9) - and half the host->device bytes of a path
 * whose end-to-end rate is bound by exactly those.  Every frames argument of such a pipeline is
 * [n_streams][frames][h_mb][w_mb] u16.  Not combinable with COVA_FLAG_KEEP_STACKED; w_mb must be even. */
#define COVA_FLAG_INPUT_PACKED16 0x400u
#define COVA_FLAG_CHUNKS(n) (((uint32_t)(n) & 0xffu) << 16) /* process a batch in n chunks of whole chains (0 = auto) */
/* Masks larger than one CTA's shared memory (8K video: 480x270 macroblocks = 32,400 2x2 blocks).  The CCL normally holds a
 * whole mask in one CTA's shared memory and such grids are refused with COVA_E_UNSUPPORTED at creation.  With this flag
 * (for cova_pipeline_new and cova_bboxcc_new2) a grid that fits one CTA still runs the single-CTA kernel; a larger one
 * runs a thread-block-cluster kernel: one cluster of k = 2..8 CTAs per mask, each CTA owning a band of ceil(nby/k) block
 * rows and reaching its peers through distributed shared memory (8K: k = 4).  Outputs are byte-identical to what the
 * single-CTA kernel would produce; under profiling the kernel is named "ccl_bbox_cluster".  Still COVA_E_UNSUPPORTED: a
 * grid that needs more than 8 bands (about 65,000 blocks), and a device on which no such cluster can be resident
 * (creation checks cudaOccupancyMaxActiveClusters).  Opt-in because the cluster kernel needs k CTAs of up to ~220 KB of
 * shared memory to be co-resident in one GPC, which the single-CTA kernel never does. */
#define COVA_FLAG_CCL_CLUSTER 0x800u
/* Forces the cluster kernel with bands of ceil(ceil(H/2) / k) block rows (k bands, fewer when the rows run out) on any
 * grid, so that tests and measurements can put seams into small masks.  COVA_E_INVAL, before any device call: without
 * COVA_FLAG_CCL_CLUSTER, k = 1 or k > 8, k > ceil(H/2), and any flag bit that no COVA_FLAG_* / COVA_IMPL_* defines. */
#define COVA_FLAG_CCL_BANDS(k) (((uint32_t)(k) & 0xfu) << 24)

int cova_pipeline_new(cova_pipeline **out, int device, uint32_t w_mb, uint32_t h_mb, uint32_t timestep,
                      uint32_t gamma, uint32_t max_streams, uint32_t max_frames_per_stream, const void *weights,
                      size_t weights_len, uint32_t cc_threshold, uint32_t flags);
void cova_pipeline_free(cova_pipeline *p);
int cova_pipeline_set_cc_threshold(cova_pipeline *p, uint32_t cc_threshold);
/* run all kernels on this stream (a cudaStream_t / CUstream as void*); NULL = the pipeline's own */
int cova_pipeline_set_stream(cova_pipeline *p, void *cuda_stream);
/* number of windows a batch of this shape produces */
int cova_pipeline_n_windows(const cova_pipeline *p, uint32_t n_streams, uint32_t frames_per_stream, uint32_t *n);

/* stage 0: put a batch of frames [n_streams][frames_per_stream][h_mb][w_mb][4] into the device frame pool.
 * is_device != 0: frames is a device pointer (device-to-device copy). Asynchronous on the stream.
 * The stage-wise calls (load_frames, load_masks, tensorise, blobnet, run_layer, ccl, run) share the pipeline's buffers
 * with submitted batches: while a submit waits for its collect they return COVA_E_INVAL before any device call. */
int cova_pipeline_load_frames(cova_pipeline *p, const uint8_t *frames, uint32_t n_streams,
                              uint32_t frames_per_stream, int is_device);
/* stages, each asynchronous on the stream, operating on the loaded batch */
int cova_pipeline_tensorise(cova_pipeline *p); /* frame pool -> BlobNet input layout (+ stacked RGBA if kept) */
int cova_pipeline_blobnet(cova_pipeline *p);   /* -> mask u8 {0,1} [n_windows][h_mb][w_mb] on device */
int cova_pipeline_ccl(cova_pipeline *p);       /* mask -> bincode blobs + offsets on device */
int cova_pipeline_run(cova_pipeline *p);       /* the three above */
int cova_pipeline_sync(cova_pipeline *p);
/* copy the boxes back: blob = concatenation of per-window bincode(Vec<Bbox>); window i occupies
 * [offsets[i], offsets[i] + lens[i]).  offsets/lens have n_windows entries.  Synchronises. */
int cova_pipeline_fetch_boxes(cova_pipeline *p, uint8_t *blob, size_t blob_cap, size_t *blob_len, uint64_t *offsets,
                              uint64_t *lens);
/* one call, host buffers in and out (the call a GStreamer element would make per batch) */
int cova_pipeline_process_host(cova_pipeline *p, const uint8_t *frames, uint32_t n_streams,
                               uint32_t frames_per_stream, uint8_t *blob, size_t blob_cap, size_t *blob_len,
                               uint64_t *offsets, uint64_t *lens, uint32_t *n_windows);

/* Asynchronous form of process_host for steady-state streaming: at most four batches in flight.  submit returns
 * once the copies and kernels are enqueued (frames must stay valid, ideally page-locked, until the matching
 * collect); collect blocks for the oldest batch and copies its boxes out.  submit(k+1) before collect(k) hides
 * the host<->device copies of one batch behind the kernels of the other; submit(k+3) before collect(k) keeps the
 * host->device copy engine busy back to back (the steady state is then bound by PCIe, not by a batch's latency). */
int cova_pipeline_submit_host(cova_pipeline *p, const uint8_t *frames, uint32_t n_streams, uint32_t frames_per_stream);
int cova_pipeline_collect_host(cova_pipeline *p, uint8_t *blob, size_t blob_cap, size_t *blob_len, uint64_t *offsets,
                               uint64_t *lens, uint32_t *n_windows);

/* Stream continuity (metapreprocess/imp.rs:38-42,302-330: State.prev_buffers and gamma_idx live for the whole stream; an
 * element instance never restarts its window between buffers).  submit_host / process_host treat every chain of every
 * batch as a freshly started element - right for GoP shards, each of which the reference also feeds to a fresh chain
 * (gstgopsplit.cpp:557-630), but a stream that is fed in SEVERAL batches would lose timestep-1 windows at every seam
 * and shift its gamma phase.  submit_host2 names the streams:
 *   stream_ids[n_streams]  ids in [0, max_streams), distinct within a batch; NULL = 0, 1, 2, ...
 *   pts[n_streams * frames_per_stream]  optional presentation time of every frame, echoed per window by collect_host2
 *   flags  COVA_SUBMIT_CONTINUE: chain s continues stream stream_ids[s]: the last timestep-1 frames of the stream (kept on
 *          the device) precede the new ones and the gamma phase carries on, so the batch yields exactly the windows the
 *          uncut stream would have produced for these frames (frames_per_stream windows per chain at gamma 1).
 *          Without the flag the named streams (re)start with an empty window.  Either way their state is recorded.
 *          COVA_SUBMIT_STAGGERED (only together with COVA_SUBMIT_CONTINUE): the streams of the batch need not be in
 *          lock-step.  Each chain continues its stream from that stream's own state - its own history
 *          h_s = min(seen_s, timestep-1) and its own gamma phase; a stream never seen (or reset) starts with an empty
 *          window - and yields exactly the windows its uncut stream would yield for these frames.  Chains may therefore
 *          yield different numbers of windows: map windows to streams with collect_host2's win_stream_ids.
 *          Any other flag bit, or STAGGERED without CONTINUE: COVA_E_INVAL before any device call.
 * Constraints: without COVA_SUBMIT_STAGGERED the streams of one CONTINUED batch must advance in lock-step (same history
 * length min(seen, timestep-1) and same gamma phase) - COVA_E_INVAL otherwise; pass COVA_SUBMIT_STAGGERED to lift this
 * rule.  frames_per_stream is the same for every stream of a call, and frames_per_stream + max_s h_s must fit
 * max_frames_per_stream.  Window order stays stream-major, time-minor.
 * collect_host2: as collect_host, plus per window the stream id and the PTS of its newest frame (the PTS the
 * reference's metapreprocess output buffer carries, BaseTransform default; cova/imp.rs:110-112 requires it).
 * Both arrays have n_windows entries; win_pts is only written when the submit passed pts. */
#define COVA_SUBMIT_CONTINUE 1u
#define COVA_SUBMIT_STAGGERED 2u
int cova_pipeline_submit_host2(cova_pipeline *p, const uint8_t *frames, uint32_t n_streams, uint32_t frames_per_stream,
                               const uint32_t *stream_ids, const uint64_t *pts, uint32_t flags);
int cova_pipeline_collect_host2(cova_pipeline *p, uint8_t *blob, size_t blob_cap, size_t *blob_len, uint64_t *offsets,
                                uint64_t *lens, uint32_t *n_windows, uint32_t *win_stream_ids, uint64_t *win_pts);
/* forget the state of the given streams (NULL = all): their next CONTINUED batch starts with an empty window */
int cova_pipeline_reset_streams(cova_pipeline *p, const uint32_t *stream_ids, uint32_t n);

/* Host-side packer for COVA_FLAG_INPUT_PACKED16: n_mb macroblock quads (the decoder's [mb_weight, |mv_x|, |mv_y|, stale]
 * bytes, h264_mb.c:822-855) -> n_mb u16.  A packer owns n_threads worker threads (0 = one per online CPU, at most 64);
 * pack() splits the range evenly over them and returns when all are done.  AVX2 when the CPU has it.  Host C++, no CUDA. */
typedef struct cova_packer cova_packer;
int cova_packer_new(cova_packer **out, uint32_t n_threads);
void cova_packer_free(cova_packer *pk);
int cova_packer_pack(cova_packer *pk, const uint8_t *quads, uint16_t *out, size_t n_mb);

/* Sparse input for COVA_FLAG_INPUT_PACKED16 pipelines: only the macroblocks that differ from a per-frame background cross
 * PCIe.  One frame = one record, 4-byte aligned, little-endian, n_mb = w_mb * h_mb macroblocks in raster order y*w_mb + x:
 *   bytes 0-3   u32 background: a packed16 value in bits 0-8, bits 9-31 zero
 *   bytes 4-7   u32 count: macroblocks whose value is not the background
 *   then        u32 bitmap[ceil(n_mb / 32)]: bit i % 32 of word i / 32 set = macroblock i differs; bits >= n_mb zero
 *   then        u16 values[count]: the packed16 values of the set macroblocks in raster order, zero-padded to 4 bytes
 * Record size = 8 + 4*ceil(n_mb/32) + 4*ceil(count/2).  A batch is the records of n_streams x frames_per_stream frames,
 * stream-major and time-minor like a dense frames argument, without gaps.  Any background is valid (a decoder can use its
 * skip value); the values follow the packed16 contract, which is documented and not checked. */
#define COVA_SPARSE_MAX_FRAME_BYTES(n_mb) \
    (8u + 4u * (((size_t)(n_mb) + 31u) / 32u) + 4u * (((size_t)(n_mb) + 1u) / 2u)) /* a record with count = n_mb */
/* Encodes n_frames frames of decoder quads [n_frames][h_mb][w_mb][4] into a sparse batch, reading every quad once, on the
 * packer's threads (contiguous ranges of frames per thread).  Canonical output: background = the frame's most frequent
 * packed16 value (ties: the smallest), zero padding.  *out_len = the batch size; COVA_E_TOOSMALL (nothing written) when it
 * exceeds out_cap.  It never exceeds n_frames * COVA_SPARSE_MAX_FRAME_BYTES(w_mb * h_mb). */
int cova_packer_pack_sparse(cova_packer *pk, const uint8_t *quads, uint32_t n_frames, uint32_t w_mb, uint32_t h_mb,
                            uint8_t *out, size_t out_cap, size_t *out_len);
/* As cova_pipeline_submit_host2 (stream ids, PTS echo, COVA_SUBMIT_CONTINUE / _STAGGERED, the same rules and errors;
 * collect with collect_host / collect_host2), with the frames as a sparse batch of data_len bytes.  Only on a
 * COVA_FLAG_INPUT_PACKED16 pipeline (COVA_E_INVAL otherwise).  Before any device call every record is checked - reserved
 * background bits, count == popcount(bitmap), no bit at or past n_mb, zero padding, and records ending exactly at
 * data_len - and a malformed batch is COVA_E_INVAL with nothing in flight.  data must stay valid until the collect. */
int cova_pipeline_submit_sparse(cova_pipeline *p, const uint8_t *data, size_t data_len, uint32_t n_streams,
                                uint32_t frames_per_stream, const uint32_t *stream_ids, const uint64_t *pts, uint32_t flags);

/* feed a mask batch straight to the CCL stage (u8 [n][h_mb][w_mb]; is_device as above) */
int cova_pipeline_load_masks(cova_pipeline *p, const uint8_t *masks, uint32_t n, int is_device);

/* parity / inspection (synchronise; host output buffers) */
int cova_pipeline_read_stacked(cova_pipeline *p, uint8_t *out, size_t cap);  /* [n_windows][T*h][w][4] */
int cova_pipeline_read_mask(cova_pipeline *p, uint8_t *out, size_t cap);     /* [n_windows][h][w] */
int cova_pipeline_read_logits(cova_pipeline *p, float *out, size_t cap_floats); /* [n_windows][h][w] */
/* activation `layer` (0 = BlobNet input, 1..4 = encoder outputs, 5..7 = decoder concat inputs dec1..dec3)
 * de-permuted to float [n_windows][C][T][H][W]; dims returned in shape[5] = {N, C, T, H, W} */
int cova_pipeline_read_activation(cova_pipeline *p, int layer, float *out, size_t cap_floats, uint32_t shape[5]);
/* run ONE BlobNet layer (0..3 = enc1..enc4, 4..6 = dec0..dec2, 7 = dec3 + head) with the chosen
 * implementation on whatever its input buffer currently holds - lets the tests compare the tcgen05
 * kernel of a layer against the validation kernel of the same layer on identical inputs */
int cova_pipeline_run_layer(cova_pipeline *p, int layer, uint32_t impl);
/* development switches.  Results become garbage with bit 0 (skip the MMAs) or bit 1 (skip the epilogue math); the others
 * select alternative, equally correct code paths for A/B measurements (tools/ab_step.py, tools/layer_timing.py):
 * bit 2 positions-as-M kernels for encoder blocks 2 and 4, bit 3 weights-stationary kernel for block 3, bit 5 plain
 * stream-ordered launches instead of programmatic dependent launch (this handle only), bit 6 whole-tile accumulators for
 * dec0 / dec1 */
int cova_pipeline_set_debug(cova_pipeline *p, int flags);

/* Diagnostics: the launch plan of each tcgen05 BlobNet layer, out[layer] for the layers of cova_pipeline_run_layer.  Each
 * layer picks its plan at run time from a list of candidate tile configurations, by what fits shared memory for the
 * grid WIDTH (the operand strips hold TPS tiles plus two rows of halo); height does not matter, the window count only
 * sets the number of tile groups and CTAs.  The widest grid every layer has a plan for at debug 0 is w_mb = 736
 * macroblocks (block 4 runs out first); cova_pipeline_new refuses a wider one with COVA_E_UNSUPPORTED before it touches
 * the device, and a debug route (cova_pipeline_set_debug bits 2 and 3) without a plan at the pipeline's width makes the
 * run calls return COVA_E_UNSUPPORTED before they launch any BlobNet layer. */
#define COVA_PLAN_ENC1 1 /* the fused block-1 kernel */
#define COVA_PLAN_POS 2  /* positions-as-M kernel (output positions in the MMA's M) */
#define COVA_PLAN_WS 3   /* weights-stationary kernel (blocks 2-4; weights in tensor memory) */
typedef struct cova_layer_plan {
    int32_t family;   /* COVA_PLAN_*; 0 = no plan / not launched yet */
    int32_t config;   /* index of the tile configuration in the layer's candidate list for that family */
    int32_t tps;      /* tiles per operand-ring stage */
    int32_t tile;     /* output positions per tile */
    int32_t n_stage;  /* operand-ring depth */
    int32_t n_groups; /* tile groups (block 1: frame steps of tile pairs) that pass through the ring */
    int32_t ctas;     /* CTAs launched */
} cova_layer_plan;
/* The plans the library would launch for a batch of `windows` windows (one chain of windows + timestep - 1 frames, gamma
 * 1) of a w_mb x h_mb grid, with debug bits `debug`, on a device of n_sms SMs.  Host arithmetic only: needs no device.
 * COVA_E_UNSUPPORTED, with the layer named in cova_last_error(), when some layer has no plan: out[] then holds the plans of
 * the layers before it and zeros from it on. */
int cova_blobnet_plan(uint32_t w_mb, uint32_t h_mb, uint32_t windows, int debug, int n_sms, cova_layer_plan out[8]);
/* the plan each layer used at its last tcgen05 launch on this handle (family 0 for a layer not launched yet) */
int cova_pipeline_last_plan(const cova_pipeline *p, cova_layer_plan out[8]);
/* kernels launched by this handle since creation */
int cova_pipeline_launch_count(const cova_pipeline *p, uint64_t *count);
/* per-kernel device time of the last cova_pipeline_run* with profiling enabled: names is a
 * ';'-separated list, ms has one entry per name.  enable != 0 records CUDA events around every kernel. */
int cova_pipeline_set_profiling(cova_pipeline *p, int enable);
int cova_pipeline_last_timings(cova_pipeline *p, char *names, size_t names_cap, float *ms, uint32_t *n);

/* ------------------------------------------------------------------------------------------------
 * sorttracker element   (cova-rs/gst-plugins/src/sorttracker/imp.rs; SURVEY.md section 8f row f2)
 * The step AFTER the GPU path: host C++ (no CUDA), consumes the per-frame bincode(Vec<Bbox>) blobs that
 * cova_pipeline_collect_host / cova_bboxcc_transform_ip produce and returns the histories of the tracks that
 * died on this frame.
 *   properties iou-threshold f32 [0,1] default 0.1, maxage u32 default 30, minhits u32 default 30, all
 *     mutable while PLAYING but read only when caps are set                      imp.rs:10-12,53-137,214-236
 *   set_caps(): (re)creates the Sort state                                       imp.rs:214-236
 *   transform(): Bbox::deserialize_vec -> Sort::update(boxes, pts ns) -> bincode of the dead tracks'
 *     histories, flattened in tracker order                                      imp.rs:238-266
 *   EOS: Sort::finalize() -> one extra buffer                                    imp.rs:268-287
 * Tracker semantics: cova-rs/sort/src/lib.rs:25-213, tracker/mod.rs:33-153, state.rs:10-27.
 * ------------------------------------------------------------------------------------------------ */
typedef struct cova_sorttracker cova_sorttracker;

int cova_sorttracker_new(cova_sorttracker **out);
void cova_sorttracker_free(cova_sorttracker *s);
/* GObject-style properties by name ("iou-threshold", "maxage", "minhits") */
int cova_sorttracker_set_property(cova_sorttracker *s, const char *name, double value);
int cova_sorttracker_get_property(const cova_sorttracker *s, const char *name, double *value);
int cova_sorttracker_set_caps(cova_sorttracker *s, int32_t width, int32_t height);
/* COVA_E_TOOSMALL reports the required size in *out_len; the tracker state has advanced regardless, so size
 * the buffer like the element does (transform_size: 2 MiB, imp.rs:322-332) */
int cova_sorttracker_transform(cova_sorttracker *s, const uint8_t *boxes, size_t boxes_len, uint64_t pts_ns,
                               uint8_t *out, size_t out_cap, size_t *out_len);
/* sink_event(EOS).  On COVA_E_TOOSMALL nothing is consumed and the call can be repeated. */
int cova_sorttracker_eos(cova_sorttracker *s, uint8_t *out, size_t out_cap, size_t *out_len);
int cova_sorttracker_n_tracks(const cova_sorttracker *s, uint32_t *n_total, uint32_t *n_active);

/* building blocks of Sort, exported so that the reference's unit tests (sort/src/lib.rs:230-408) can be replayed.
 * boxes are float[n][4] = (left, top, width, height); matrices are row-major [n_trk][n_det]; pairs is
 * int32[min(n_trk,n_det)][2] = (tracker, detection), sorted by tracker. */
int cova_sort_linear_assignment(const float *cost, uint32_t n_trk, uint32_t n_det, int32_t *pairs, uint32_t *n_pairs);
int cova_sort_iou_matrix(const float *preds, uint32_t n_preds, const float *dets, uint32_t n_dets, float *out);
int cova_sort_match_dets(const float *preds, const uint8_t *active, uint32_t n_preds, const float *dets, uint32_t n_dets,
                         float iou_threshold, int32_t *pairs, uint32_t *n_pairs);

/* ------------------------------------------------------------------------------------------------
 * cova element: frame selection   (cova-rs/gst-plugins/src/cova/imp.rs, cova/tracker.rs; SURVEY 8f row f3)
 * Two sink pads: sink_enc receives every ENCODED frame (kept per GoP), sink_mask the per-frame boxes of the
 * blob-detection path.  The element tracks the boxes (SORT) and pushes, per GoP, the list of encoded frames a
 * pixel decoder must still decode: the first frame at/after the start of every track that died unseen
 * (counted as decoded-inference), preceded by the frames it depends on (flag DROPPABLE, decoded-dependency);
 * everything else is dropped.  Host C++; buffers are referred to by a caller-chosen 64-bit id.
 *   properties: sort-iou f32 0.1, sort-maxage u32 30, sort-minhits u32 30, port u32 0, infer-i bool false,
 *     debug bool false, alpha u32 0, beta u32 0; read-only counters dropped, decoded-dependency,
 *     decoded-inference (u64)                                                          imp.rs:22-56, 536-790
 *   sink_enc chain: a buffer without DELTA_UNIT opens a GoP (its copy gets DISCONT)     imp.rs:292-331
 *   sink_mask chain: Tracker::update -> selection -> GoPs older than 250 frames pushed  imp.rs:90-289
 *   EOS on both pads: every GoP's list is pushed (even when empty), Tracker::flush      imp.rs:332-431
 *   port != 0: dead / final tracks go to the aggregator as length-delimited (u32 BE) bincode
 *     Frame{range_start, oldest, bboxes}; here the bytes are queued for cova_select_take_wire
 *                                                              cova/tracker.rs:43-125, bbox/src/lib.rs:7-22
 * ------------------------------------------------------------------------------------------------ */
typedef struct cova_select cova_select;

#define COVA_BUFFER_FLAG_DELTA_UNIT 1u /* gst::BufferFlags::DELTA_UNIT: not a key frame */
#define COVA_BUFFER_FLAG_DISCONT 2u    /* set on the first frame of every GoP (imp.rs:305-307) */
#define COVA_BUFFER_FLAG_DROPPABLE 4u  /* decode for reference only, no inference (imp.rs:186,211,221) */

typedef struct cova_pushed_buffer {
    uint64_t id;     /* the id given to cova_select_sink_enc; UINT64_MAX marks an EMPTY list pushed at EOS */
    uint64_t pts_ns;
    uint32_t flags;  /* COVA_BUFFER_FLAG_* */
    uint32_t list;   /* index of the gst::BufferList within this call (one list per GoP) */
} cova_pushed_buffer;

int cova_select_new(cova_select **out);
void cova_select_free(cova_select *s);
int cova_select_set_property(cova_select *s, const char *name, double value);
int cova_select_get_property(const cova_select *s, const char *name, double *value);
int cova_select_sink_enc(cova_select *s, uint64_t buf_id, uint64_t pts_ns, uint32_t flags);
/* On COVA_E_TOOSMALL the element state HAS advanced and *n_out is the number of entries waiting:
 * fetch them with cova_select_take_pushed. */
int cova_select_sink_mask(cova_select *s, const uint8_t *boxes, size_t boxes_len, uint64_t pts_ns,
                          cova_pushed_buffer *out, size_t out_cap, size_t *n_out);
/* pad: 0 = sink_enc, 1 = sink_mask.  COVA_DROPPED until both pads have seen EOS, COVA_OK when drained. */
int cova_select_eos(cova_select *s, int pad, cova_pushed_buffer *out, size_t out_cap, size_t *n_out);
int cova_select_take_pushed(cova_select *s, cova_pushed_buffer *out, size_t out_cap, size_t *n_out);
int cova_select_take_wire(cova_select *s, uint8_t *out, size_t out_cap, size_t *out_len);

/* ------------------------------------------------------------------------------------------------
 * demux + gopsplit   (gst-plugins/gst-gopsplit/gstgopsplit.cpp:500-729, pipeline/cova/pipeline.py:60-92;
 * SURVEY 8f row f4).  Host C++.  Finds the frames and key frames of a stream the way the front of the reference
 * pipeline (filesrc ! qtdemux ! h264parse) labels them, and cuts them into per-pad (= per-GPU) runs of whole GoPs
 * exactly as gopsplit assigns them: floor(G/P) GoPs per pad, the remainder to the last pad; with fewer GoPs than pads,
 * pad i gets GoP i.
 * ------------------------------------------------------------------------------------------------ */
typedef struct cova_sample {
    uint64_t offset; /* byte offset of the frame in the input */
    uint32_t size;
    uint32_t flags;  /* COVA_BUFFER_FLAG_DELTA_UNIT unless the frame is a key frame */
    uint64_t dts, pts; /* MP4: track timescale units; Annex B: frame index */
} cova_sample;
typedef struct cova_mp4_info {
    uint32_t timescale, width, height, nal_length_size;
} cova_mp4_info;

/* sample table of the first H.264 video track of an ISO media file (the whole file, or at least its moov box);
 * key frames = the stss sync samples, like qtdemux */
int cova_demux_mp4_samples(const uint8_t *data, size_t len, cova_sample *out, size_t out_cap, size_t *n_out,
                           cova_mp4_info *info);
/* access units of an Annex-B byte stream; key frames = units holding an IDR slice, like h264parse */
int cova_demux_annexb_frames(const uint8_t *data, size_t len, cova_sample *out, size_t out_cap, size_t *n_out);
/* flags[n_frames] as above -> [first_frame[p], end_frame[p]) for every pad p (empty range = 0, 0) */
int cova_gopsplit_ranges(const uint32_t *flags, size_t n_frames, uint32_t n_pads, uint64_t *first_frame, uint64_t *end_frame);

#ifdef __cplusplus
}
#endif
#endif /* COVA_B200_H */
