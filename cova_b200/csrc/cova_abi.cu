// C ABI of libcova_b200.so (see include/cova_b200.h).  One translation unit: kernels + host plumbing.
// There is NO CPU fallback anywhere in this file: without a CUDA device every constructor fails with
// COVA_E_NODEVICE.
#include <ctype.h>
#include <math.h>
#include <sched.h>

#include <algorithm>
#include <mutex>

// The fp32 CUDA-core validation kernels (COVA_IMPL_SIMT: layer-by-layer comparison partner of the tcgen05 kernels in the
// tests) are only compiled into libcova_b200_val.so (-DCOVA_VALIDATION); the shipped library holds the hot path alone.
#ifdef COVA_VALIDATION
#include "blobnet_simt.cuh"
#endif
#include "blobnet_tc.cuh"
#include "blobnet_enc.cuh"
#include "blobnet_enc1.cuh"
#include "ccl.cuh"
#include "common.cuh"
#include "sparse_expand.cuh"
#include "tensorise.cuh"
#include "weights_pack.cuh"

namespace cova {
thread_local char g_err[512] = "";

static int check_device(int device) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) return set_err(COVA_E_NODEVICE, "no CUDA device (%s); cova_b200 has no CPU fallback", cudaGetErrorString(e));
    if (device < 0 || device >= n) return set_err(COVA_E_INVAL, "device index out of range");
    COVA_CUDA(cudaSetDevice(device));
    return COVA_OK;
}

// newest-frame ring used by the metapreprocess element: slot of frame t-k = (head - k) mod T
__global__ void __launch_bounds__(256) stack_ring_kernel(const uint32_t *__restrict__ ring, uint32_t *__restrict__ out,
                                                         int words_per_frame, int T, int head) {
    const int total = words_per_frame * T;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        int k = i / words_per_frame, e = i - k * words_per_frame;
        int slot = (head - k + T) % T;
        out[i] = ring[(size_t)slot * words_per_frame + e];
    }
}
}  // namespace cova

using namespace cova;

// =================================================================================================
// misc
// =================================================================================================
extern "C" const char *cova_version(void) { return "cova_b200 0.1 (sm_100a)"; }
extern "C" const char *cova_last_error(void) { return g_err; }
extern "C" const char *cova_strerror(int code) {
    switch (code) {
        case COVA_OK: return "ok";
        case COVA_DROPPED: return "dropped (no output for this input)";
        case COVA_E_INVAL: return "invalid argument";
        case COVA_E_CUDA: return "CUDA error";
        case COVA_E_NOMEM: return "out of memory";
        case COVA_E_TOOSMALL: return "output buffer too small";
        case COVA_E_WEIGHTS: return "bad weight container";
        case COVA_E_UNSUPPORTED: return "unsupported configuration";
        case COVA_E_NODEVICE: return "no CUDA device (no CPU fallback)";
        case COVA_E_NUMERIC: return "numerical failure in the host tracker";
        case COVA_E_STATE: return "inconsistent frame-selection state";
        default: return "unknown error";
    }
}
extern "C" int cova_host_alloc(void **out, size_t bytes) {
    if (!out || !bytes) return set_err(COVA_E_INVAL, "null argument");
    *out = nullptr;
    cudaError_t e = cudaMallocHost(out, bytes);
    if (e != cudaSuccess) { cudaGetLastError(); return set_err(e == cudaErrorMemoryAllocation ? COVA_E_NOMEM : COVA_E_NODEVICE, "cudaMallocHost: %s", cudaGetErrorString(e)); }
    return COVA_OK;
}
extern "C" void cova_host_free(void *ptr) {
    if (ptr) cudaFreeHost(ptr);
}
// One process per GPU (DESIGN.md "Multi-GPU"): the frames of a rank travel host -> device at PCIe rate, so its pinned
// buffers must live on the NUMA node the GPU hangs off - with 8 ranks on a two-socket box the inter-socket link is
// otherwise shared by up to 4 x 55 GB/s of remote reads.  Restricting the calling thread to the GPU's local CPUs
// (sysfs local_cpulist) before it allocates makes first-touch placement do that without libnuma.
extern "C" int cova_bind_host_to_device(int device, int *numa_node, int *n_cpus) {
    if (numa_node) *numa_node = -1;
    if (n_cpus) *n_cpus = 0;
    char bus[32] = "";
    cudaError_t e = cudaDeviceGetPCIBusId(bus, (int)sizeof(bus), device);
    if (e != cudaSuccess) { cudaGetLastError(); return set_err(COVA_E_NODEVICE, "cudaDeviceGetPCIBusId: %s", cudaGetErrorString(e)); }
    for (char *c = bus; *c; c++) *c = (char)tolower(*c);
    const std::string base = std::string("/sys/bus/pci/devices/") + bus;
    if (FILE *f = fopen((base + "/numa_node").c_str(), "r")) {
        int node = -1;
        if (fscanf(f, "%d", &node) == 1 && numa_node) *numa_node = node;
        fclose(f);
    }
    FILE *f = fopen((base + "/local_cpulist").c_str(), "r");
    if (!f) return COVA_OK;                                   // no topology information: leave the affinity alone
    char list[4096] = "";
    const bool got = fgets(list, sizeof(list), f) != nullptr;
    fclose(f);
    if (!got) return COVA_OK;
    cpu_set_t set;
    CPU_ZERO(&set);
    int count = 0;
    for (char *tok = strtok(list, ",\n"); tok; tok = strtok(nullptr, ",\n")) {
        int a = 0, b = 0;
        const int k = sscanf(tok, "%d-%d", &a, &b);
        if (k < 1) continue;
        if (k == 1) b = a;
        for (int c = a; c <= b && c < CPU_SETSIZE; c++) { CPU_SET(c, &set); count++; }
    }
    if (!count) return COVA_OK;
    cpu_set_t cur;
    if (sched_getaffinity(0, sizeof(cur), &cur) == 0) {        // stay inside what the launcher (cgroup, taskset) allows
        cpu_set_t both;
        CPU_AND(&both, &set, &cur);
        if (CPU_COUNT(&both) == 0) return COVA_OK;
        set = both;
        count = CPU_COUNT(&both);
    }
    if (sched_setaffinity(0, sizeof(set), &set) != 0) return COVA_OK;
    if (n_cpus) *n_cpus = count;
    return COVA_OK;
}
extern "C" int cova_device_count(int *n) {
    if (!n) return set_err(COVA_E_INVAL, "null argument");
    int c = 0;
    if (cudaGetDeviceCount(&c) != cudaSuccess) { cudaGetLastError(); c = 0; }
    *n = c;
    return COVA_OK;
}

// =================================================================================================
// metapreprocess element
// =================================================================================================
struct cova_metapreprocess {
    int device;
    uint32_t w_mb, h_mb, timestep, gamma, gamma_idx, n_prev;
    int head;             // ring slot of the newest stored frame
    size_t S;             // size_per_buf (imp.rs:233)
    uint8_t *d_ring = nullptr, *d_out = nullptr;
    cudaStream_t stream = nullptr;
};

extern "C" int cova_metapreprocess_new(cova_metapreprocess **out, int device, uint32_t width_px, uint32_t height_px,
                                       uint32_t timestep, uint32_t gamma) {
    if (!out) return set_err(COVA_E_INVAL, "null out");
    *out = nullptr;
    if (timestep < 1 || gamma < 1) return set_err(COVA_E_INVAL, "timestep and gamma are u32 >= 1");
    if (width_px / 16 == 0 || height_px / 16 == 0) return set_err(COVA_E_INVAL, "frame smaller than one macroblock");
    int rc = check_device(device);
    if (rc) return rc;
    auto *mp = new (std::nothrow) cova_metapreprocess();
    if (!mp) return set_err(COVA_E_NOMEM, "host allocation failed");
    mp->device = device;
    mp->w_mb = width_px / 16;   // imp.rs:262-268: integer division
    mp->h_mb = height_px / 16;
    mp->timestep = timestep; mp->gamma = gamma; mp->gamma_idx = 0; mp->n_prev = 0; mp->head = -1;
    mp->S = (size_t)mp->w_mb * mp->h_mb * 4;
    cudaError_t e = cudaMalloc(&mp->d_ring, mp->S * timestep);
    if (e == cudaSuccess) e = cudaMalloc(&mp->d_out, mp->S * timestep);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&mp->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        cova_metapreprocess_free(mp);
        return set_err(COVA_E_CUDA, "metapreprocess allocation: %s", cudaGetErrorString(e));
    }
    *out = mp;
    return COVA_OK;
}
extern "C" void cova_metapreprocess_free(cova_metapreprocess *mp) {
    if (!mp) return;
    cudaSetDevice(mp->device);
    if (mp->d_ring) cudaFree(mp->d_ring);
    if (mp->d_out) cudaFree(mp->d_out);
    if (mp->stream) cudaStreamDestroy(mp->stream);
    delete mp;
}
extern "C" int cova_metapreprocess_set_gamma(cova_metapreprocess *mp, uint32_t gamma) {
    if (!mp || gamma < 1) return set_err(COVA_E_INVAL, "gamma is a u32 >= 1");
    mp->gamma = gamma;
    return COVA_OK;
}
extern "C" int cova_metapreprocess_out_caps(const cova_metapreprocess *mp, uint32_t *width, uint32_t *height, size_t *size) {
    if (!mp) return set_err(COVA_E_INVAL, "null handle");
    if (width) *width = mp->w_mb;
    if (height) *height = mp->h_mb * mp->timestep;
    if (size) *size = mp->S * mp->timestep;
    return COVA_OK;
}
extern "C" int cova_metapreprocess_transform(cova_metapreprocess *mp, const uint8_t *inbuf, size_t in_len, uint8_t *outbuf,
                                             size_t out_cap) {
    if (!mp || !inbuf) return set_err(COVA_E_INVAL, "null argument");
    if (in_len < mp->S) return set_err(COVA_E_INVAL, "input buffer shorter than size_per_buf");
    COVA_CUDA(cudaSetDevice(mp->device));
    const int T = (int)mp->timestep;
    // every branch of imp.rs:302-330 stores the incoming buffer as the newest one
    const int slot = (mp->head + 1) % T;
    COVA_CUDA(cudaMemcpyAsync(mp->d_ring + (size_t)slot * mp->S, inbuf, mp->S, cudaMemcpyHostToDevice, mp->stream));
    mp->head = slot;
    if (mp->n_prev < mp->timestep - 1) {          // imp.rs:302-305
        mp->n_prev++;
        COVA_CUDA(cudaStreamSynchronize(mp->stream));
        return COVA_DROPPED;
    }
    if (mp->gamma_idx != 0) {                      // imp.rs:325-330
        mp->gamma_idx--;
        COVA_CUDA(cudaStreamSynchronize(mp->stream));
        return COVA_DROPPED;
    }
    if (!outbuf || out_cap < mp->S * T) {
        // keep element state consistent with "this buffer was consumed", but tell the caller
        mp->gamma_idx = mp->gamma - 1;
        cudaStreamSynchronize(mp->stream);
        return set_err(COVA_E_TOOSMALL, "output buffer smaller than the RGBA stack");
    }
    const int words = (int)(mp->S / 4);
    int blocks = std::min(1024, (words * T + 255) / 256);
    stack_ring_kernel<<<blocks, 256, 0, mp->stream>>>(reinterpret_cast<const uint32_t *>(mp->d_ring),
                                                      reinterpret_cast<uint32_t *>(mp->d_out), words, T, mp->head);
    COVA_CUDA(cudaGetLastError());
    COVA_CUDA(cudaMemcpyAsync(outbuf, mp->d_out, mp->S * T, cudaMemcpyDeviceToHost, mp->stream));
    COVA_CUDA(cudaStreamSynchronize(mp->stream));
    mp->gamma_idx = mp->gamma - 1;                 // imp.rs:323
    return COVA_OK;
}

// =================================================================================================
// CCL launch shared by the bboxcc element and the pipeline
// =================================================================================================
struct CclBuffers {
    int H = 0, W = 0, nbx = 0, nby = 0, nb = 0, max_masks = 0;
    uint8_t *d_masks = nullptr, *d_blob = nullptr;
    size_t blob_cap = 0;
    unsigned long long *d_cursor = nullptr, *d_offsets = nullptr, *d_lens = nullptr;
    int32_t *d_labels = nullptr, *d_stats = nullptr, *d_nlabels = nullptr;
    size_t smem = 0;
    int threads = 0;
    bool compact = false;     // 13-byte-per-block shared-memory layout (ccl.cuh): two CTAs per SM at 4K
    int k = 1, rows = 0;      // k > 1: ccl_cluster_kernel, one cluster of k CTAs per mask, bands of `rows` block rows
};

constexpr int kCclSmemLimit = tc::kSmemLimit - 1024;   // dynamic part: the kernel also has a few bytes of static shared memory

// COVA_FLAG_CCL_CLUSTER / COVA_FLAG_CCL_BANDS: checked before any device call
static int ccl_check_flags(uint32_t flags) {
    const uint32_t bands = (flags >> 24) & 0xfu;
    if (bands && !(flags & COVA_FLAG_CCL_CLUSTER)) return set_err(COVA_E_INVAL, "COVA_FLAG_CCL_BANDS needs COVA_FLAG_CCL_CLUSTER");
    if (bands == 1 || bands > 8) return set_err(COVA_E_INVAL, "COVA_FLAG_CCL_BANDS(k) takes k = 2..8");
    return COVA_OK;
}
static int ccl_check_bands(uint32_t flags, uint32_t height) {
    if (((flags >> 24) & 0xfu) > (height + 1) / 2) return set_err(COVA_E_INVAL, "COVA_FLAG_CCL_BANDS(k) needs k <= ceil(height / 2) block rows");
    return COVA_OK;
}

// Can one cluster of b.k CTAs of b.smem bytes be resident at all?  (k CTAs of ~220 KB on SMs of one GPC, which the
// single-CTA kernel never needs.)
static int ccl_cluster_ok(const CclBuffers &b) {
    COVA_CUDA(cudaFuncSetAttribute(ccl_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kCclSmemLimit));
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3((unsigned)b.k); cfg.blockDim = dim3((unsigned)b.threads); cfg.dynamicSmemBytes = b.smem;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = (unsigned)b.k; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    int n = 0;
    COVA_CUDA(cudaOccupancyMaxActiveClusters(&n, ccl_cluster_kernel, &cfg));
    if (n < 1) {
        char msg[160];
        snprintf(msg, sizeof(msg), "no cluster of %d CTAs with %zu bytes of shared memory each fits this device", b.k, b.smem);
        return set_err(COVA_E_UNSUPPORTED, "%s", msg);
    }
    return COVA_OK;
}

static int ccl_alloc(CclBuffers &b, int H, int W, int max_masks, bool own_masks, uint32_t flags = 0) {
    b.H = H; b.W = W; b.nbx = (W + 1) / 2; b.nby = (H + 1) / 2; b.nb = b.nbx * b.nby; b.max_masks = max_masks;
    b.threads = ccl_threads_for(b.nb);
    // The compact layout would give 4K masks two CTAs per SM (204 KB -> 106 KB), but measured it does not pay: its
    // compare-and-swap statistics cost more than the second CTA brings (4K network masks 0.40 -> 0.44 ms per 1024, dense
    // 0.83 -> 0.86; only empty / all-ones masks gain).  It is used where the wide layout does not fit at all.
    b.compact = false;
    static const char *force = getenv("COVA_CCL_COMPACT");         // development knob: "0" / "1"
    if (force && (force[0] == '0' || force[0] == '1')) b.compact = force[0] == '1';
    b.smem = ccl_smem_bytes(b.nb, b.threads, b.compact);
    if (b.smem > (size_t)kCclSmemLimit && !b.compact) { b.compact = true; b.smem = ccl_smem_bytes(b.nb, b.threads, true); }
    const bool one_cta = b.smem <= (size_t)kCclSmemLimit && b.nb < 0x7FFF;   // block indices travel in 15 bits of the foreground lists
    const int forced = (int)((flags >> 24) & 0xfu);
    b.k = 1;
    if ((flags & COVA_FLAG_CCL_CLUSTER) && (forced || !one_cta)) {
        // bands in the wide layout: the fewest (2..8) that fit, or exactly the forced count of rows ceil(nby / k) - which
        // may leave fewer than k bands when the rows run out (nby = 5, k = 4: 2 + 2 + 1)
        for (int k = forced ? forced : 2; k <= (forced ? forced : 8) && b.k == 1; k++) {
            const int rows = (b.nby + k - 1) / k, band_nb = rows * b.nbx, threads = ccl_threads_for(band_nb);
            const size_t smem = ccl_smem_bytes(band_nb, threads, false);
            if (smem > (size_t)kCclSmemLimit || band_nb >= 0x7FFF) continue;
            b.k = (b.nby + rows - 1) / rows; b.rows = rows; b.threads = threads; b.smem = smem; b.compact = false;
        }
        if (b.k == 1) return set_err(COVA_E_UNSUPPORTED, "mask grid too large for the cluster CCL kernel (8 bands of the shared-memory layout)");
        int rc = ccl_cluster_ok(b);
        if (rc) return rc;
    } else if (!one_cta) {
        return set_err(COVA_E_UNSUPPORTED, "mask grid too large for the shared-memory CCL kernel");
    }
    b.blob_cap = (size_t)max_masks * (8 + 24 * (size_t)b.nb);
    if (own_masks) COVA_CUDA(cudaMalloc(&b.d_masks, (size_t)max_masks * H * W));
    COVA_CUDA(cudaMalloc(&b.d_blob, b.blob_cap));
    COVA_CUDA(cudaMalloc(&b.d_cursor, 2 * sizeof(unsigned long long)));
    COVA_CUDA(cudaMalloc(&b.d_offsets, (size_t)max_masks * sizeof(unsigned long long)));
    COVA_CUDA(cudaMalloc(&b.d_lens, (size_t)max_masks * sizeof(unsigned long long)));
    return COVA_OK;
}
static void ccl_free(CclBuffers &b, bool own_masks) {
    if (own_masks && b.d_masks) cudaFree(b.d_masks);
    if (b.d_blob) cudaFree(b.d_blob);
    if (b.d_cursor) cudaFree(b.d_cursor);
    if (b.d_offsets) cudaFree(b.d_offsets);
    if (b.d_lens) cudaFree(b.d_lens);
    if (b.d_labels) cudaFree(b.d_labels);
    if (b.d_stats) cudaFree(b.d_stats);
    if (b.d_nlabels) cudaFree(b.d_nlabels);
}
// merge-phase choice and tiling of a grid of a.nbx x nby blocks (the whole mask, or one band of it)
static void ccl_grid_args(CclArgs &a, int nby, int threads) {
    a.nby = nby;
    const int nb = a.nbx * nby;
    a.div_nbx = make_fastdiv((uint32_t)std::max(2, a.nbx));
    a.step_by = threads / a.nbx; a.step_bx = threads % a.nbx;
    // merge phase: tile scan (ccl.cuh, 2a/2b; about one tile of 32 columns per warp) for large grids, the concurrent
    // union-find over all foreground blocks for small ones.  Measured per 1024 4K masks (tools/ccl_timing.py): network masks
    // 0.35 -> 0.31 ms, dense network masks 0.86 -> 0.66, dense noise 0.88 -> 0.74 (all-ones 0.35 -> 0.55, empty 0.09 -> 0.11);
    // at 720p / 1080p the row-serial scan loses to the union-find (0.160 -> 0.189 / 0.156 -> 0.191 ms), so it is off there.
    // COVA_CCL_SCAN=0/1 forces either (development knob; both pass the golden and stress suites).
    static const char *scan_env = getenv("COVA_CCL_SCAN");
    a.scan = nb >= 4096;
    if (scan_env && (scan_env[0] == '0' || scan_env[0] == '1')) a.scan = scan_env[0] == '1';
    a.tiles_x = (a.nbx + 31) / 32;
    a.tiles_y = std::max(1, std::min(nby, (threads / 32) / a.tiles_x));
    a.tile_rows = (nby + a.tiles_y - 1) / a.tiles_y;
    a.tiles_y = (nby + a.tile_rows - 1) / a.tile_rows;
    a.div_tile_rows = make_fastdiv((uint32_t)std::max(2, a.tile_rows));
}

static int ccl_launch(CclBuffers &b, const uint8_t *d_masks, int n, uint32_t cc_threshold, bool want_labels, cudaStream_t st,
                      size_t first = 0, bool reset_cursor = true, bool pdl = true) {
    if (n <= 0) return COVA_OK;
    CclArgs a;
    a.masks = d_masks + first * (size_t)b.H * b.W; a.H = b.H; a.W = b.W; a.nbx = b.nbx;
    a.area_thresh = (int)cc_threshold;   // `settings.cc_threshold as i32` (imp.rs:248)
    a.blob = b.d_blob; a.blob_cap = b.blob_cap; a.cursor = b.d_cursor; a.offsets = b.d_offsets + first; a.lens = b.d_lens + first;
    a.labels = want_labels ? b.d_labels : nullptr;
    a.stats = want_labels ? b.d_stats : nullptr;
    a.n_labels = want_labels ? b.d_nlabels : nullptr;
    if (reset_cursor) COVA_CUDA(cudaMemsetAsync(b.d_cursor, 0, 2 * sizeof(unsigned long long), st));
    if (b.k > 1) {
        CclClusterArgs c;
        c.H = b.H; c.nb = b.nb; c.rows = b.rows; c.band_nb = b.rows * b.nbx;
        c.div_band = make_fastdiv((uint32_t)std::max(2, c.band_nb));
        c.band[0] = a; c.band[0].H = 2 * b.rows;
        ccl_grid_args(c.band[0], b.rows, b.threads);
        const int last_rows = b.nby - (b.k - 1) * b.rows;
        c.band[1] = a; c.band[1].H = b.H - 2 * (b.k - 1) * b.rows;
        ccl_grid_args(c.band[1], last_rows, b.threads);
        // same attribute policy as below: always the architectural maximum
        COVA_CUDA(cudaFuncSetAttribute(ccl_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kCclSmemLimit));
        cudaLaunchConfig_t cfg;
        memset(&cfg, 0, sizeof(cfg));
        cfg.gridDim = dim3((unsigned)(n * b.k)); cfg.blockDim = dim3((unsigned)b.threads); cfg.dynamicSmemBytes = b.smem; cfg.stream = st;
        cudaLaunchAttribute at[2];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = (unsigned)b.k; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[1].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = at; cfg.numAttrs = pdl ? 2 : 1;
        COVA_CUDA(cudaLaunchKernelEx(&cfg, ccl_cluster_kernel, c));
        return COVA_OK;
    }
    ccl_grid_args(a, b.nby, b.threads);
    // the attribute is per function AND per device, last write wins: handles of different grids (or on different devices,
    // or on different threads) share ccl_bbox_kernel, so it is set for every launch and always to the same value, the
    // architectural maximum (see tc::try_launch)
    auto kernel = b.compact ? ccl_bbox_kernel<true> : ccl_bbox_kernel<false>;
    COVA_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kCclSmemLimit));
    COVA_CUDA(launch_pdl(kernel, dim3((unsigned)n), dim3((unsigned)b.threads), b.smem, st, pdl, a));
    return COVA_OK;
}

// =================================================================================================
// bboxcc element
// =================================================================================================
struct cova_bboxcc {
    int device;
    uint32_t width, height, cc_threshold, flags;
    CclBuffers b;
    cudaStream_t stream = nullptr;
};

extern "C" int cova_bboxcc_new2(cova_bboxcc **out, int device, uint32_t width, uint32_t height, uint32_t cc_threshold,
                                uint32_t flags) {
    if (!out) return set_err(COVA_E_INVAL, "null out");
    *out = nullptr;
    if (!width || !height) return set_err(COVA_E_INVAL, "empty mask");
    if (flags & ~(COVA_FLAG_CCL_CLUSTER | COVA_FLAG_CCL_BANDS(0xf))) return set_err(COVA_E_INVAL, "unknown bboxcc flag");
    int rc = ccl_check_flags(flags);
    if (!rc) rc = ccl_check_bands(flags, height);
    if (rc) return rc;
    rc = check_device(device);
    if (rc) return rc;
    auto *cc = new (std::nothrow) cova_bboxcc();
    if (!cc) return set_err(COVA_E_NOMEM, "host allocation failed");
    cc->device = device; cc->width = width; cc->height = height; cc->cc_threshold = cc_threshold; cc->flags = flags;
    rc = ccl_alloc(cc->b, (int)height, (int)width, 1, true, flags);
    if (rc == COVA_OK && cudaStreamCreateWithFlags(&cc->stream, cudaStreamNonBlocking) != cudaSuccess)
        rc = set_err(COVA_E_CUDA, "stream creation failed");
    if (rc) { cova_bboxcc_free(cc); return rc; }
    *out = cc;
    return COVA_OK;
}
extern "C" int cova_bboxcc_new(cova_bboxcc **out, int device, uint32_t width, uint32_t height, uint32_t cc_threshold) {
    return cova_bboxcc_new2(out, device, width, height, cc_threshold, 0);
}
extern "C" void cova_bboxcc_free(cova_bboxcc *cc) {
    if (!cc) return;
    cudaSetDevice(cc->device);
    ccl_free(cc->b, true);
    if (cc->stream) cudaStreamDestroy(cc->stream);
    delete cc;
}
extern "C" int cova_bboxcc_set_cc_threshold(cova_bboxcc *cc, uint32_t t) {
    if (!cc) return set_err(COVA_E_INVAL, "null handle");
    cc->cc_threshold = t;
    return COVA_OK;
}
extern "C" int cova_bboxcc_get_cc_threshold(const cova_bboxcc *cc, uint32_t *t) {
    if (!cc || !t) return set_err(COVA_E_INVAL, "null argument");
    *t = cc->cc_threshold;
    return COVA_OK;
}
extern "C" size_t cova_bboxcc_max_out_size(const cova_bboxcc *cc) { return cc ? 8 + 24 * (size_t)cc->b.nb : 0; }

extern "C" int cova_bboxcc_transform_ip(cova_bboxcc *cc, const uint8_t *mask, size_t mask_len, uint8_t *out, size_t out_cap,
                                        size_t *out_len) {
    if (!cc || !mask || !out_len) return set_err(COVA_E_INVAL, "null argument");
    // process.rs:14-15: reshape(1, height) -> rows of len/height bytes; the element is configured per caps
    if (mask_len != (size_t)cc->width * cc->height) return set_err(COVA_E_INVAL, "mask length != width*height of the caps");
    COVA_CUDA(cudaSetDevice(cc->device));
    COVA_CUDA(cudaMemcpyAsync(cc->b.d_masks, mask, mask_len, cudaMemcpyHostToDevice, cc->stream));
    int rc = ccl_launch(cc->b, cc->b.d_masks, 1, cc->cc_threshold, false, cc->stream);
    if (rc) return rc;
    // One synchronisation per buffer: the length and as much of the blob as the caller's buffer (or the worst case of this
    // grid) can hold travel back together; the single mask's blob starts at offset 0 of the arena.
    unsigned long long len = 0;
    const size_t spec = out ? std::min(out_cap, cc->b.blob_cap) : 0;
    COVA_CUDA(cudaMemcpyAsync(&len, cc->b.d_lens, sizeof(len), cudaMemcpyDeviceToHost, cc->stream));
    if (spec) COVA_CUDA(cudaMemcpyAsync(out, cc->b.d_blob, spec, cudaMemcpyDeviceToHost, cc->stream));
    COVA_CUDA(cudaStreamSynchronize(cc->stream));
    *out_len = (size_t)len;
    if (!out || out_cap < len) return set_err(COVA_E_TOOSMALL, "serialized boxes need a larger buffer");
    return COVA_OK;
}

extern "C" int cova_bboxcc_labels(cova_bboxcc *cc, const uint8_t *mask, size_t mask_len, int32_t *labels, int32_t *stats,
                                  int32_t *n_labels) {
    if (!cc || !mask || !labels || !stats || !n_labels) return set_err(COVA_E_INVAL, "null argument");
    if (mask_len != (size_t)cc->width * cc->height) return set_err(COVA_E_INVAL, "mask length != width*height");
    COVA_CUDA(cudaSetDevice(cc->device));
    CclBuffers &b = cc->b;
    if (!b.d_labels) {
        COVA_CUDA(cudaMalloc(&b.d_labels, mask_len * sizeof(int32_t)));
        COVA_CUDA(cudaMalloc(&b.d_stats, (size_t)(b.nb + 1) * 5 * sizeof(int32_t)));
        COVA_CUDA(cudaMalloc(&b.d_nlabels, sizeof(int32_t)));
    }
    COVA_CUDA(cudaMemcpyAsync(b.d_masks, mask, mask_len, cudaMemcpyHostToDevice, cc->stream));
    int rc = ccl_launch(b, b.d_masks, 1, cc->cc_threshold, true, cc->stream);
    if (rc) return rc;
    COVA_CUDA(cudaMemcpyAsync(n_labels, b.d_nlabels, sizeof(int32_t), cudaMemcpyDeviceToHost, cc->stream));
    COVA_CUDA(cudaMemcpyAsync(labels, b.d_labels, mask_len * sizeof(int32_t), cudaMemcpyDeviceToHost, cc->stream));
    COVA_CUDA(cudaStreamSynchronize(cc->stream));
    COVA_CUDA(cudaMemcpyAsync(stats, b.d_stats, (size_t)(*n_labels) * 5 * sizeof(int32_t), cudaMemcpyDeviceToHost, cc->stream));
    COVA_CUDA(cudaStreamSynchronize(cc->stream));
    return COVA_OK;
}

// =================================================================================================
// fused batch pipeline
// =================================================================================================
struct DevLayer {
    uint4 *wpack = nullptr;
    float *epi = nullptr;
    int n_cols = 0;
};

constexpr int kSlots = 4;

// chains [stream0, stream0 + n_streams) of a batch, which yield its windows [window0, window0 + windows)
struct Chunk { uint32_t stream0, n_streams, window0, windows; };

struct cova_pipeline {
    int device = 0, n_sms = 0;
    uint32_t W = 0, H = 0, T = 0, gamma = 1, max_streams = 0, max_fps = 0, max_windows = 0, flags = 0, impl = 0;
    uint32_t cc_threshold = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    size_t frame_bytes = 0;              // bytes of one frame in the pool: 4 per macroblock, or 2 with COVA_FLAG_INPUT_PACKED16
    bool packed = false;
    // per-stream state for CONTINUED batches (metapreprocess/imp.rs:38-42: prev_buffers and gamma_idx live as long as the
    // stream): the last T - 1 frames of every stream id on the device, frames seen so far on the host
    uint8_t *d_carry = nullptr;
    std::vector<uint64_t> n_seen, id_mark;
    uint64_t id_epoch = 0;
    std::vector<uint32_t> first_scratch, hist_scratch;   // per chain of the batch being submitted
    std::vector<uint64_t> off_scratch;                   // record offsets of the sparse batch being submitted
    // A batch is processed in chunks of whole chains: the activation buffers are sized for ONE chunk, and
    // process_host() overlaps the H2D copy of chunk c+1, the kernels of chunk c and the D2H of chunk c-1.
    uint32_t chunk_streams = 0;          // chains per chunk (capacity)
    Chunk last_chunk = {};               // the chunk whose activations the buffers hold (cova_pipeline_read_activation)
    cudaStream_t s_in = nullptr, s_out = nullptr;
    // Four batch slots (frame pool + box arena + events): submit_host(k+3) can be queued before collect_host(k).  A
    // batch's host-visible latency is H2D + kernels + D2H of the boxes (whose size the host must first learn): measured
    // 2.25 + 2.05 + 0.65 ms for 8192 windows of 720p.  With k batches ahead the loop sustains one batch per
    // max(H2D, kernels, latency / k): two ahead = 2.47 ms (measured 2.46), three ahead = the PCIe time, 2.25 ms.
    // The synchronous entry points use slot 0.
    struct Slot {
        uint8_t *d_frames = nullptr;
        CclBuffers ccl;
        std::vector<cudaEvent_t> ev_in, ev_done;
        unsigned long long *h_cursor = nullptr;      // pinned: per-chunk cursor snapshots (2 words each)
        uint32_t n_streams = 0, fps = 0, n_windows = 0;  // n_streams = 0, n_windows = n: masks loaded directly, no chains
        bool busy = false, failed = false;
        uint32_t *h_ids = nullptr, *d_ids = nullptr;   // stream ids of a submit_host2 batch (pinned staging + device copy)
        std::vector<uint64_t> win_pts;                 // per window: PTS of its newest frame / stream id (submit_host2)
        std::vector<uint32_t> win_ids;
        // Window shape of the slot's batch (set_batch_shape).  Chain s yields windows [win0[s], win0[s+1]) of the batch; its
        // first one has its newest frame at device index first_s, the next ones follow every gamma frames.
        //   tab[s]     = (first_s, win0[s] - win0[first chain of s's chunk])      read by enc1_fused_kernel
        //   newest[w]  = index of window w's newest frame among its chunk's frames  read by the gather kernels
        // Each slot owns pinned staging and a device copy, uploaded on the compute stream in order with the batch's
        // kernels: batches of different shapes can be in flight together without draining the pipeline.
        std::vector<uint32_t> win0;
        int2 *h_tab = nullptr, *d_tab = nullptr;
        int *h_newest = nullptr, *d_newest = nullptr;
        cudaEvent_t ev_tab = nullptr;                  // recorded after the upload: the staging may be rewritten after it
        std::vector<uint32_t> tab_first;               // what the tables hold: per-chain first, frames per chain, stream
        uint32_t tab_fps = 0;
        cudaStream_t tab_stream = nullptr;
        // sparse input (cova_pipeline_submit_sparse), allocated on the slot's first sparse submit: the batch's records at
        // their host byte offsets, and the record offsets (pinned staging + device copy, uploaded on the compute stream)
        uint8_t *d_sparse = nullptr;
        unsigned long long *h_off = nullptr, *d_off = nullptr;
        cudaEvent_t ev_off = nullptr;                  // recorded after the offsets upload: the staging may be rewritten after it
    } slot[kSlots];
    int next_submit = 0, next_collect = 0, last_slot = 0;   // last_slot: given the last batch, read by stage-wise and read_*
    int sizes_h[5], sizes_w[5];          // extents: [0] input, [1..4] encoder outputs
    Geom gx[4];                          // X0..X3 (Tn = 4): inputs of enc1..enc4
    Geom gd[4];                          // D0in..D3in (Tn = 1): inputs of dec0..dec3
    Geom gx0f;                           // per-FRAME first-conv input (x-pair packed, Tn = 1, N = frames)
    uint4 *x0f = nullptr;
    uint4 *x[4] = {nullptr, nullptr, nullptr, nullptr};
    uint4 *d[4] = {nullptr, nullptr, nullptr, nullptr};
    uint8_t *d_mask = nullptr, *d_stacked = nullptr;
    float *d_logits = nullptr;
    HostWeights hw;
    float *d_wraw = nullptr;
    DevLayer enc[4], dec[4];
    DevLayer encs[4];                    // blocks 2..4, weights-stationary kernel (blobnet_enc.cuh)
    unsigned int *d_watchdog = nullptr;
    bool profiling = false;
    std::vector<cudaEvent_t> events;
    std::vector<std::string> names, last_names;
    std::vector<float> last_ms;
    size_t ev_used = 0;
    uint64_t launches = 0;
    int dbg = 0;
    cova_layer_plan last_plan[8] = {};   // per layer: the plan of its last tcgen05 launch (cova_pipeline_last_plan)
};
using Slot = cova_pipeline::Slot;

// windows of a device chain of `fps` frames whose first window has its newest frame at index `first`
static uint32_t windows_from(uint32_t fps, uint32_t first, uint32_t gamma) { return fps > first ? (fps - 1 - first) / gamma + 1 : 0; }

static void prof_mark(cova_pipeline *p, const char *name) {
    if (!p->profiling) return;
    if (p->ev_used >= p->events.size()) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        p->events.push_back(e);
    }
    cudaEventRecord(p->events[p->ev_used++], p->stream);
    p->names.push_back(name);
}

template <typename T>
static int dev_upload(T **dst, const void *src, size_t bytes) {
    COVA_CUDA(cudaMalloc(dst, bytes));
    COVA_CUDA(cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice));
    return COVA_OK;
}

static int upload_layer(DevLayer &dl, const PackedLayer *halves, int n_halves) {
    size_t hb = halves[0].b.size() * sizeof(__half);
    COVA_CUDA(cudaMalloc(&dl.wpack, hb * n_halves));
    for (int h = 0; h < n_halves; h++)
        COVA_CUDA(cudaMemcpy(reinterpret_cast<char *>(dl.wpack) + hb * h, halves[h].b.data(), hb, cudaMemcpyHostToDevice));
    int rc = dev_upload(&dl.epi, halves[0].epi.data(), halves[0].epi.size() * sizeof(float));
    dl.n_cols = halves[0].n_cols;
    return rc;
}

// chains per chunk: ~1024 windows per chunk, at most 16 chunks; tiny pipelines stay single-chunk
static uint32_t chunk_streams_for(uint32_t max_streams, uint32_t max_windows, uint32_t flags) {
    uint32_t chunks = std::min<uint32_t>(16, std::max<uint32_t>(1, max_windows / 1024));
    const uint32_t hint = (flags >> 16) & 0xffu;
    if (hint) chunks = hint;
    chunks = std::min(chunks, max_streams);
    return (max_streams + chunks - 1) / chunks;
}
static int ensure_slot(cova_pipeline *p, int k) {
    auto &sl = p->slot[k];
    if (!sl.d_frames) COVA_CUDA(cudaMalloc(&sl.d_frames, p->frame_bytes * p->max_streams * p->max_fps));
    if (!sl.ccl.d_blob) {
        sl.ccl.d_masks = p->d_mask;
        int rc = ccl_alloc(sl.ccl, (int)p->H, (int)p->W, std::max<int>(1, (int)p->max_windows), false, p->flags);
        if (rc) { ccl_free(sl.ccl, false); sl.ccl = CclBuffers(); return rc; }    // a later submit retries from scratch
    }
    return COVA_OK;
}
static void blobnet_geoms(int h_mb, int w_mb, int N, int F, int sizes_h[5], int sizes_w[5], Geom gx[4], Geom gd[4], Geom &gx0f);
static int plan_blobnet(int h_mb, int w_mb, int N, int n_chains, int fps, int gamma, int dbg, int n_sms, cova_layer_plan out[8]);

extern "C" int cova_pipeline_new(cova_pipeline **out, int device, uint32_t w_mb, uint32_t h_mb, uint32_t timestep,
                                 uint32_t gamma, uint32_t max_streams, uint32_t max_fps, const void *weights,
                                 size_t weights_len, uint32_t cc_threshold, uint32_t flags) {
    if (!out) return set_err(COVA_E_INVAL, "null out");
    *out = nullptr;
    if (timestep != (uint32_t)kT) return set_err(COVA_E_UNSUPPORTED, "BlobNet is built for timestep = 4 (utils/train-blobnet.py:58)");
    if (gamma < 1 || !max_streams || max_fps < timestep) return set_err(COVA_E_INVAL, "need gamma >= 1, max_streams >= 1, max_frames_per_stream >= timestep");
    if (w_mb < 16 || h_mb < 16) return set_err(COVA_E_UNSUPPORTED, "macroblock grid must be at least 16x16 for four 2x poolings");
    if ((flags & 0xffu) > COVA_IMPL_SIMT) return set_err(COVA_E_INVAL, "unknown implementation selector");
    if (flags & ~(0xffu | COVA_FLAG_KEEP_LOGITS | COVA_FLAG_KEEP_STACKED | COVA_FLAG_INPUT_PACKED16 | COVA_FLAG_CCL_CLUSTER |
                  COVA_FLAG_CHUNKS(0xff) | COVA_FLAG_CCL_BANDS(0xf)))
        return set_err(COVA_E_INVAL, "unknown pipeline flag");
    int rc = ccl_check_flags(flags);
    if (!rc) rc = ccl_check_bands(flags, h_mb);
    if (rc) return rc;
    const uint32_t chain_windows = windows_from(max_fps, timestep - 1, gamma);   // of a chain of max_fps frames
    const uint32_t max_windows = max_streams * chain_windows;
    const uint32_t chunk_streams = chunk_streams_for(max_streams, max_windows, flags);
    {   // every layer must have a tile plan for a chunk of this grid (the widest grids run out of shared memory for the
        // strips of block 4 first).  Whether a plan fits does not depend on the SM count.
        cova_layer_plan plans[8];
        rc = plan_blobnet((int)h_mb, (int)w_mb, (int)(chunk_streams * chain_windows), (int)chunk_streams,
                          (int)max_fps, (int)gamma, 0, 1, plans);
        if (rc) return rc;
    }
    if (flags & COVA_FLAG_INPUT_PACKED16) {
        if (flags & COVA_FLAG_KEEP_STACKED) return set_err(COVA_E_INVAL, "the stacked RGBA windows cannot be rebuilt from packed input (byte 3 and values above 6 are gone)");
        if ((flags & 0xffu) == COVA_IMPL_SIMT) return set_err(COVA_E_UNSUPPORTED, "the validation kernels read the 4-byte input format");
        if (w_mb & 1) return set_err(COVA_E_UNSUPPORTED, "packed input needs an even macroblock-grid width");
    }
#ifndef COVA_VALIDATION
    if ((flags & 0xffu) == COVA_IMPL_SIMT)
        return set_err(COVA_E_UNSUPPORTED, "the validation kernels (COVA_IMPL_SIMT) are not part of this build; use libcova_b200_val.so");
#endif
    rc = check_device(device);
    if (rc) return rc;
    auto *p = new (std::nothrow) cova_pipeline();
    if (!p) return set_err(COVA_E_NOMEM, "host allocation failed");
    p->device = device; p->W = w_mb; p->H = h_mb; p->T = timestep; p->gamma = gamma;
    p->max_streams = max_streams; p->max_fps = max_fps; p->flags = flags; p->impl = flags & 0xffu;
    p->cc_threshold = cc_threshold;
    p->max_windows = max_windows;
    auto fail = [&](int code) { cova_pipeline_free(p); return code; };
    if ((rc = parse_weights(weights, weights_len, p->hw))) return fail(rc);
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return fail(set_err(COVA_E_CUDA, "cudaGetDeviceProperties failed"));
    p->n_sms = prop.multiProcessorCount;
    if (p->impl == COVA_IMPL_TCGEN05 && prop.major != 10)
        return fail(set_err(COVA_E_UNSUPPORTED, "the tcgen05 path needs an sm_100 device"));
    if (cudaStreamCreateWithFlags(&p->own_stream, cudaStreamNonBlocking) != cudaSuccess) return fail(set_err(COVA_E_CUDA, "stream creation failed"));
    p->stream = p->own_stream;

    {
        p->chunk_streams = chunk_streams;
        const uint32_t chunks = (max_streams + p->chunk_streams - 1) / p->chunk_streams;
        if (cudaStreamCreateWithFlags(&p->s_in, cudaStreamNonBlocking) != cudaSuccess ||
            cudaStreamCreateWithFlags(&p->s_out, cudaStreamNonBlocking) != cudaSuccess)
            return fail(set_err(COVA_E_CUDA, "stream creation failed"));
        for (auto &sl : p->slot) {
            if (cudaEventCreateWithFlags(&sl.ev_tab, cudaEventDisableTiming) != cudaSuccess)
                return fail(set_err(COVA_E_CUDA, "event creation failed"));
            sl.ev_in.resize(chunks); sl.ev_done.resize(chunks);
            for (uint32_t c = 0; c < chunks; c++)
                if (cudaEventCreateWithFlags(&sl.ev_in[c], cudaEventDisableTiming) != cudaSuccess ||
                    cudaEventCreateWithFlags(&sl.ev_done[c], cudaEventDisableTiming) != cudaSuccess)
                    return fail(set_err(COVA_E_CUDA, "event creation failed"));
        }
    }
    const int N = (int)(p->chunk_streams * chain_windows);                                  // windows per chunk
    const int NB = (int)p->max_windows;                                                       // windows per batch
    const int F = (int)(p->chunk_streams * max_fps);
    blobnet_geoms((int)h_mb, (int)w_mb, N, F, p->sizes_h, p->sizes_w, p->gx, p->gd, p->gx0f);
    auto alloc_zero = [&](uint4 **ptr, const Geom &g) -> int {
        size_t bytes = (size_t)geom_rows(g) * 16;
        COVA_CUDA(cudaMalloc(ptr, bytes));
        COVA_CUDA(cudaMemset(*ptr, 0, bytes));
        return COVA_OK;
    };
    for (int i = 0; i < 4; i++) {
        // X0 in window layout is only consumed by the validation kernels; the tcgen05 path works per frame
        if (i > 0 || p->impl == COVA_IMPL_SIMT)
            if ((rc = alloc_zero(&p->x[i], p->gx[i]))) return fail(rc);
        if ((rc = alloc_zero(&p->d[i], p->gd[i]))) return fail(rc);
    }
    if ((rc = alloc_zero(&p->x0f, p->gx0f))) return fail(rc);
    p->packed = (flags & COVA_FLAG_INPUT_PACKED16) != 0;
    p->frame_bytes = (size_t)w_mb * h_mb * (p->packed ? 2 : 4);
    cudaError_t e = cudaMalloc(&p->d_mask, (size_t)std::max(1, NB) * w_mb * h_mb);
    for (auto &sl : p->slot) {
        if (e == cudaSuccess) e = cudaMallocHost(&sl.h_tab, sizeof(int2) * max_streams);
        if (e == cudaSuccess) e = cudaMalloc(&sl.d_tab, sizeof(int2) * max_streams);
        if (e == cudaSuccess) e = cudaMallocHost(&sl.h_newest, sizeof(int) * std::max(1, NB));
        if (e == cudaSuccess) e = cudaMalloc(&sl.d_newest, sizeof(int) * std::max(1, NB));
        if (e == cudaSuccess) e = cudaMallocHost(&sl.h_cursor, sizeof(unsigned long long) * 2 * 256);
    }
    if (e == cudaSuccess) e = cudaMemset(p->d_mask, 0, (size_t)std::max(1, NB) * w_mb * h_mb);
    if (e == cudaSuccess && (flags & COVA_FLAG_KEEP_LOGITS)) e = cudaMalloc(&p->d_logits, sizeof(float) * (size_t)NB * w_mb * h_mb);
    if (e == cudaSuccess && (flags & COVA_FLAG_KEEP_STACKED)) e = cudaMalloc(&p->d_stacked, p->frame_bytes * timestep * (size_t)NB);
    if (e == cudaSuccess) e = cudaMalloc(&p->d_watchdog, sizeof(unsigned int));
    if (e == cudaSuccess) e = cudaMemset(p->d_watchdog, 0, sizeof(unsigned int));
    if (e != cudaSuccess) return fail(set_err(COVA_E_CUDA, "pipeline allocation: %s", cudaGetErrorString(e)));
    // slot 0 now, the others on their first submit; a CCL grid that does not fit is refused here
    if ((rc = ensure_slot(p, 0))) return fail(rc);

    // weights: raw fp32 for the validation kernels, packed fp16 operand blocks for the tcgen05 path
    if ((rc = dev_upload(&p->d_wraw, p->hw.storage.data(), p->hw.storage.size() * sizeof(float)))) return fail(rc);
    for (int i = 0; i < 4; i++) {
        PackedLayer pl;
        pack_encoder(p->hw, i, pl);
        if ((rc = upload_layer(p->enc[i], &pl, 1))) return fail(rc);
        if (i >= 1) {
            PackedLayer ws;
            pack_encoder_ws(p->hw, i, i == 1 ? 2 : 1, i <= 2 ? 2 : 1, ws);
            if ((rc = upload_layer(p->encs[i], &ws, 1))) return fail(rc);
        }
    }
    for (int i = 0; i < 4; i++) {
        const int nsplit = i == 0 ? 2 : 1;
        PackedLayer pl[2];
        for (int h = 0; h < nsplit; h++) pack_decoder(p->hw, i, nsplit, h, pl[h]);
        if ((rc = upload_layer(p->dec[i], pl, nsplit))) return fail(rc);
    }
    *out = p;
    return COVA_OK;
}

extern "C" void cova_pipeline_free(cova_pipeline *p) {
    if (!p) return;
    cudaSetDevice(p->device);
    cudaDeviceSynchronize();
    for (int i = 0; i < 4; i++) {
        if (p->x[i]) cudaFree(p->x[i]);
        if (i == 0 && p->x0f) cudaFree(p->x0f);
        if (p->d[i]) cudaFree(p->d[i]);
        if (p->enc[i].wpack) cudaFree(p->enc[i].wpack);
        if (p->enc[i].epi) cudaFree(p->enc[i].epi);
        if (p->encs[i].wpack) cudaFree(p->encs[i].wpack);
        if (p->encs[i].epi) cudaFree(p->encs[i].epi);
        if (p->dec[i].wpack) cudaFree(p->dec[i].wpack);
        if (p->dec[i].epi) cudaFree(p->dec[i].epi);
    }
    for (auto &sl : p->slot) {
        if (sl.d_frames) cudaFree(sl.d_frames);
        ccl_free(sl.ccl, false);
        if (sl.h_cursor) cudaFreeHost(sl.h_cursor);
        if (sl.h_ids) cudaFreeHost(sl.h_ids);
        if (sl.d_ids) cudaFree(sl.d_ids);
        if (sl.h_tab) cudaFreeHost(sl.h_tab);
        if (sl.d_tab) cudaFree(sl.d_tab);
        if (sl.h_newest) cudaFreeHost(sl.h_newest);
        if (sl.d_newest) cudaFree(sl.d_newest);
        if (sl.ev_tab) cudaEventDestroy(sl.ev_tab);
        if (sl.d_sparse) cudaFree(sl.d_sparse);
        if (sl.h_off) cudaFreeHost(sl.h_off);
        if (sl.d_off) cudaFree(sl.d_off);
        if (sl.ev_off) cudaEventDestroy(sl.ev_off);
        for (auto e : sl.ev_in) cudaEventDestroy(e);
        for (auto e : sl.ev_done) cudaEventDestroy(e);
    }
    if (p->d_carry) cudaFree(p->d_carry);
    if (p->d_mask) cudaFree(p->d_mask);
    if (p->d_logits) cudaFree(p->d_logits);
    if (p->d_stacked) cudaFree(p->d_stacked);
    if (p->d_wraw) cudaFree(p->d_wraw);
    if (p->d_watchdog) cudaFree(p->d_watchdog);
    for (auto e : p->events) cudaEventDestroy(e);
    if (p->s_in) cudaStreamDestroy(p->s_in);
    if (p->s_out) cudaStreamDestroy(p->s_out);
    if (p->own_stream) cudaStreamDestroy(p->own_stream);
    cudaGetLastError();
    delete p;
}

extern "C" int cova_pipeline_set_cc_threshold(cova_pipeline *p, uint32_t t) {
    if (!p) return set_err(COVA_E_INVAL, "null handle");
    p->cc_threshold = t;
    return COVA_OK;
}
extern "C" int cova_pipeline_set_stream(cova_pipeline *p, void *s) {
    if (!p) return set_err(COVA_E_INVAL, "null handle");
    p->stream = s ? reinterpret_cast<cudaStream_t>(s) : p->own_stream;
    return COVA_OK;
}
extern "C" int cova_pipeline_n_windows(const cova_pipeline *p, uint32_t n_streams, uint32_t fps, uint32_t *n) {
    if (!p || !n) return set_err(COVA_E_INVAL, "null argument");
    *n = n_streams * windows_from(fps, p->T - 1, p->gamma);
    return COVA_OK;
}

// checked before the first device call of a submit or load_frames
static int check_batch_bounds(const cova_pipeline *p, uint32_t n_streams, uint32_t fps) {
    if (!n_streams || n_streams > p->max_streams || fps > p->max_fps)
        return set_err(COVA_E_INVAL, "batch exceeds max_streams / max_frames_per_stream of the pipeline");
    return COVA_OK;
}

// Window shape of a batch of n_streams device chains of fps frames each, into slot k.  first[s] is the index
// (inside device chain s) of the newest frame of the chain's first window; nullptr = T - 1 for every chain, i.e. chains
// that start with an empty window.  CONTINUED chains (submit_host2) start later, where their carried history and gamma
// phase put them.  Lock-step and staggered batches go through the same tables and kernels.
static int set_batch_shape(cova_pipeline *p, int k, uint32_t n_streams, uint32_t fps, const uint32_t *first = nullptr) {
    auto &sl = p->slot[k];
    const uint32_t t1 = p->T - 1, cs = p->chunk_streams;
    uint64_t total = 0;
    for (uint32_t s = 0; s < n_streams; s++) total += windows_from(fps, first ? first[s] : t1, p->gamma);
    if (total > p->max_windows) return set_err(COVA_E_INVAL, "batch produces more windows than the pipeline was sized for");
    sl.win0.resize(n_streams + 1);
    sl.win0[0] = 0;
    for (uint32_t s = 0; s < n_streams; s++) sl.win0[s + 1] = sl.win0[s] + windows_from(fps, first ? first[s] : t1, p->gamma);
    sl.n_streams = n_streams; sl.fps = fps; sl.n_windows = (uint32_t)total;
    bool same = sl.tab_fps == fps && sl.tab_stream == p->stream && sl.tab_first.size() == n_streams;
    for (uint32_t s = 0; same && s < n_streams; s++) same = sl.tab_first[s] == (first ? first[s] : t1);
    if (same) return COVA_OK;                                      // the slot's device tables already hold this shape
    // The staging may still be read by this slot's previous upload when synchronous entry points reuse slot 0 back to back.
    // On the submit path that upload has completed: the slot's previous batch was collected.
    COVA_CUDA(cudaEventSynchronize(sl.ev_tab));
    sl.tab_first.clear();                                          // invalid until the upload below is enqueued
    for (uint32_t s = 0; s < n_streams; s++) {
        const uint32_t f = first ? first[s] : t1, c0 = s / cs * cs;
        sl.h_tab[s] = make_int2((int)f, (int)(sl.win0[s] - sl.win0[c0]));
        for (uint32_t w = sl.win0[s]; w < sl.win0[s + 1]; w++)
            sl.h_newest[w] = (int)((s - c0) * fps + f + (w - sl.win0[s]) * p->gamma);
    }
    COVA_CUDA(cudaMemcpyAsync(sl.d_tab, sl.h_tab, sizeof(int2) * n_streams, cudaMemcpyHostToDevice, p->stream));
    if (total) COVA_CUDA(cudaMemcpyAsync(sl.d_newest, sl.h_newest, sizeof(int) * total, cudaMemcpyHostToDevice, p->stream));
    COVA_CUDA(cudaEventRecord(sl.ev_tab, p->stream));
    if (first) sl.tab_first.assign(first, first + n_streams);
    else sl.tab_first.assign(n_streams, t1);
    sl.tab_fps = fps; sl.tab_stream = p->stream;
    return COVA_OK;
}

static Chunk chunk_of(const Slot &sl, uint32_t c, uint32_t chunk_streams) {
    const uint32_t s0 = c * chunk_streams, ns = std::min(chunk_streams, sl.n_streams - s0);
    if (!ns) return Chunk{s0, 0, 0, 0};                            // masks loaded directly: no chains
    return Chunk{s0, ns, sl.win0[s0], sl.win0[s0 + ns] - sl.win0[s0]};
}
// The stage-wise calls share the device buffers and slot 0 with the submitted batches: refused while one is in flight.
static int require_idle(const cova_pipeline *p) {
    for (auto &sl : p->slot)
        if (sl.busy) return set_err(COVA_E_INVAL, "batches submitted asynchronously are still in flight");
    return COVA_OK;
}
// What tensorise / blobnet / run_layer work on: the one chunk of the last batch, or ck.windows = 0 if it has no windows.
static int stage_chunk(cova_pipeline *p, Chunk &ck) {
    if (!p) return set_err(COVA_E_INVAL, "null handle");
    if (int rc = require_idle(p)) return rc;
    const Slot &sl = p->slot[p->last_slot];
    ck = Chunk{};
    if (!sl.n_windows) return COVA_OK;
    COVA_CUDA(cudaSetDevice(p->device));
    if (sl.n_streams > p->chunk_streams)
        return set_err(COVA_E_UNSUPPORTED, "stage-wise calls need a batch that fits one chunk; use cova_pipeline_run / process_host");
    ck = p->last_chunk = chunk_of(sl, 0, p->chunk_streams);
    return COVA_OK;
}

extern "C" int cova_pipeline_load_frames(cova_pipeline *p, const uint8_t *frames, uint32_t n_streams, uint32_t fps, int is_device) {
    if (!p || !frames) return set_err(COVA_E_INVAL, "null argument");
    int rc = require_idle(p);
    if (!rc) rc = check_batch_bounds(p, n_streams, fps);
    if (rc) return rc;
    COVA_CUDA(cudaSetDevice(p->device));
    if ((rc = set_batch_shape(p, 0, n_streams, fps))) return rc;
    p->last_slot = 0;
    COVA_CUDA(cudaMemcpyAsync(p->slot[0].d_frames, frames, p->frame_bytes * n_streams * fps,
                              is_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, p->stream));
    return COVA_OK;
}

extern "C" int cova_pipeline_load_masks(cova_pipeline *p, const uint8_t *masks, uint32_t n, int is_device) {
    if (!p || !masks) return set_err(COVA_E_INVAL, "null argument");
    if (!n || n > p->max_windows) return set_err(COVA_E_INVAL, "mask batch exceeds the pipeline's window capacity");
    if (int rc = require_idle(p)) return rc;
    COVA_CUDA(cudaSetDevice(p->device));
    p->slot[0].n_streams = 0; p->slot[0].n_windows = n;
    p->last_slot = 0;
    COVA_CUDA(cudaMemcpyAsync(p->d_mask, masks, (size_t)n * p->W * p->H, is_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, p->stream));
    return COVA_OK;
}

static int tensorise_chunk(cova_pipeline *p, const Slot &sl, const Chunk &ck) {
    const int N = (int)ck.windows;
    if (!N) return COVA_OK;
    const uint8_t *frames = sl.d_frames + (size_t)ck.stream0 * sl.fps * p->frame_bytes;
    const int *newest = sl.d_newest + ck.window0;                   // chunk-relative, like the frames
    if (p->d_stacked) {
        const size_t S = p->frame_bytes;
        uint8_t *dst = p->d_stacked + (size_t)ck.window0 * p->T * S;
        if (S % 16 == 0) {
            long long total = (long long)N * p->T * (S / 16);
            int blocks = (int)std::min<long long>((total + 255) / 256, (long long)p->n_sms * 16);
            stack_rgba_kernel<uint4><<<blocks, 256, 0, p->stream>>>(reinterpret_cast<const uint4 *>(frames), newest,
                                                                   reinterpret_cast<uint4 *>(dst), (int)(S / 16), (int)p->T, total);
        } else {
            long long total = (long long)N * p->T * (S / 4);
            int blocks = (int)std::min<long long>((total + 255) / 256, (long long)p->n_sms * 16);
            stack_rgba_kernel<uint32_t><<<blocks, 256, 0, p->stream>>>(reinterpret_cast<const uint32_t *>(frames), newest,
                                                                      reinterpret_cast<uint32_t *>(dst), (int)(S / 4), (int)p->T, total);
        }
        COVA_CUDA(cudaGetLastError());
        p->launches++;
        prof_mark(p, "stack_rgba");
    }
    {   // per-frame first-conv input (tcgen05 path)
        const int F = (int)(ck.n_streams * sl.fps);
        long long total = (long long)F * p->H * p->gx0f.Wh;
        int blocks = (int)std::min<long long>((total + 255) / 256, (long long)p->n_sms * 32);
        if (total >= (1ll << 32)) return set_err(COVA_E_UNSUPPORTED, "chunk too large for the frame tensorisation kernel (32-bit index)");
        COVA_CUDA(launch_pdl(p->packed ? tensorise_frames_kernel<true> : tensorise_frames_kernel<false>, dim3((unsigned)blocks), dim3(256), 0,
                             p->stream, !(p->dbg & kDbgNoPdl), reinterpret_cast<const uint32_t *>(frames), p->x0f, p->gx0f, F,
                             make_fastdiv((uint32_t)std::max(2, p->gx0f.Wh)), make_fastdiv((uint32_t)std::max<uint32_t>(2u, p->H))));
        p->launches++;
        prof_mark(p, "tensorise_frames");
    }
#ifdef COVA_VALIDATION
    if (p->x[0]) {   // window-layout input of the validation kernels
        long long total = (long long)N * p->H * p->gx[0].Wh * kT;
        int blocks = (int)std::min<long long>((total + 255) / 256, (long long)p->n_sms * 32);
        tensorise_x0_kernel<<<blocks, 256, 0, p->stream>>>(reinterpret_cast<const uint32_t *>(frames), newest, p->x[0], p->gx[0], N);
        COVA_CUDA(cudaGetLastError());
        p->launches++;
        prof_mark(p, "tensorise_x0");
    }
#endif
    return COVA_OK;
}

extern "C" int cova_pipeline_tensorise(cova_pipeline *p) {
    Chunk ck;
    int rc = stage_chunk(p, ck);
    return rc ? rc : tensorise_chunk(p, p->slot[p->last_slot], ck);
}

// ---- layer launchers -------------------------------------------------------------------------------
static void crop_for(int in_extent, int target, int &crop_lo) {
    int pad = (2 * in_extent + 2) - target;     // decoder.py:42-59: (pad//2 + pad%2, pad//2)
    crop_lo = pad / 2 + pad % 2;
}

#ifndef COVA_VALIDATION
static int simt_layer(cova_pipeline *, const Chunk &, int) {
    return set_err(COVA_E_UNSUPPORTED, "the validation kernels (COVA_IMPL_SIMT) are not part of this build; use libcova_b200_val.so");
}
#else
static int simt_layer(cova_pipeline *p, const Chunk &ck, int layer) {
    const int N = (int)ck.windows;
    const float *w = p->d_wraw;
    if (layer == 0 && !p->x[0]) return set_err(COVA_E_UNSUPPORTED, "validation kernel of layer 0 needs a pipeline created with COVA_IMPL_SIMT");
    if (layer < 4) {
        const int i = layer;
        SimtEncArgs a;
        a.in = reinterpret_cast<const Row8 *>(p->x[i]); a.gin = p->gx[i];
        a.out = i < 3 ? reinterpret_cast<Row8 *>(p->x[i + 1]) : nullptr;
        a.gout = i < 3 ? p->gx[i + 1] : p->gx[3];
        // skip of enc(i+1) feeds dec(3-i): enc1 -> D3in, enc2 -> D2in, enc3 -> D1in, enc4 -> D0in (whole input)
        a.out2 = reinterpret_cast<Row8 *>(p->d[3 - i]); a.gout2 = p->gd[3 - i];
        a.out2_cb = i < 3 ? kDecCout[2 - i] / 8 : 0;
        a.w = w + p->hw.off_enc[i][0]; a.b = w + p->hw.off_enc[i][1]; a.gamma = w + p->hw.off_enc[i][2];
        a.beta = w + p->hw.off_enc[i][3]; a.mean = w + p->hw.off_enc[i][4]; a.var = w + p->hw.off_enc[i][5];
        a.w1 = w + p->hw.off_enc[i][6]; a.w2 = w + p->hw.off_enc[i][7];
        a.Cin = kEncCin[i]; a.Cout = kEncCout[i]; a.N = N;
        a.in_scale = i == 0 ? 1.0f / 6.0f : 1.0f;
        long long total = (long long)N * (a.gin.H / 2) * (a.gin.W / 2) * (a.Cout / 8);
        simt_encoder_kernel<<<(unsigned)((total + 127) / 128), 128, 0, p->stream>>>(a);
        COVA_CUDA(cudaGetLastError());
        p->launches++;
        prof_mark(p, i == 0 ? "simt_enc1" : i == 1 ? "simt_enc2" : i == 2 ? "simt_enc3" : "simt_enc4");
        return COVA_OK;
    }
    const int i = layer - 4;
    SimtDecArgs a;
    a.in = reinterpret_cast<const Row8 *>(p->d[i]); a.gin = p->gd[i];
    a.out = i < 3 ? reinterpret_cast<Row8 *>(p->d[i + 1]) : nullptr;
    a.gout = i < 3 ? p->gd[i + 1] : p->gd[3];
    a.w = w + p->hw.off_dec[i][0]; a.b = w + p->hw.off_dec[i][1];
    a.gamma = w + p->hw.off_dec[i][2]; a.beta = w + p->hw.off_dec[i][3]; a.mean = w + p->hw.off_dec[i][4]; a.var = w + p->hw.off_dec[i][5];
    a.head_w = w + p->hw.off_head[0]; a.head_b = w + p->hw.off_head[1];
    a.mask = p->d_mask + (size_t)ck.window0 * p->W * p->H;
    a.logits = p->d_logits ? p->d_logits + (size_t)ck.window0 * p->W * p->H : nullptr;
    a.Cin = kDecCin[i]; a.Cout = kDecCout[i]; a.N = N;
    a.Ht = p->sizes_h[3 - i]; a.Wt = p->sizes_w[3 - i];
    crop_for(a.gin.H, a.Ht, a.crop_t);
    crop_for(a.gin.W, a.Wt, a.crop_l);
    if (i < 3) {
        long long total = (long long)N * a.Ht * a.Wt * (a.Cout / 8);
        simt_decoder_kernel<<<(unsigned)((total + 127) / 128), 128, 0, p->stream>>>(a);
    } else {
        long long total = (long long)N * a.Ht * a.Wt;
        simt_head_kernel<<<(unsigned)((total + 127) / 128), 128, 0, p->stream>>>(a);
    }
    COVA_CUDA(cudaGetLastError());
    p->launches++;
    prof_mark(p, i == 0 ? "simt_dec0" : i == 1 ? "simt_dec1" : i == 2 ? "simt_dec2" : "simt_dec3_head");
    return COVA_OK;
}
#endif

// ---- launch plans ------------------------------------------------------------------------------------
// The candidate tile configurations of every tcgen05 layer, in order of preference.  Each list is written once:
// plan_layer() picks an entry and launch_layer() launches that entry of the same list.
template <class... Cs>
struct Cands {};
using tc::Cfg;
using tc::MODE_DEC;
using tc::MODE_ENC;
using tc::MODE_HEAD;
using tcs::ECfg;
//                       CIN_CB COUT LA LB NP TPS
using Enc2Ws = Cands<ECfg<2, 32, 2, 2, 192, 3>, ECfg<2, 32, 2, 2, 192, 2>, ECfg<2, 32, 2, 2, 192, 1>>;
using Enc3Ws = Cands<ECfg<4, 64, 1, 2, 128, 2>, ECfg<4, 64, 1, 2, 128, 1>>;
using Enc4Ws = Cands<ECfg<8, 128, 1, 1, 64, 2>, ECfg<8, 128, 1, 1, 64, 1>>;
//                    MODE   CIN_CB NCOLS TPS KCH COUT
using Enc2Pos = Cands<Cfg<MODE_ENC, 2, 32, 4, 2, 32>, Cfg<MODE_ENC, 2, 32, 2, 2, 32>, Cfg<MODE_ENC, 2, 32, 1, 2, 32>>;
using Enc3Pos = Cands<Cfg<MODE_ENC, 4, 64, 1, 4, 64>, Cfg<MODE_ENC, 4, 64, 1, 2, 64>>;
using Enc4Pos = Cands<Cfg<MODE_ENC, 8, 128, 1, 2, 128>>;
using Dec0Pos = Cands<Cfg<MODE_DEC, 16, 128, 1, 2, 64>>;
using Dec1Pos = Cands<Cfg<MODE_DEC, 16, 128, 1, 2, 32>>;
using Dec2Pos = Cands<Cfg<MODE_DEC, 8, 64, 1, 4, 16>, Cfg<MODE_DEC, 8, 64, 1, 2, 16>>;
using Dec3Pos = Cands<Cfg<MODE_HEAD, 4, 16, 2, 4, 16>, Cfg<MODE_HEAD, 4, 16, 1, 4, 16>, Cfg<MODE_HEAD, 4, 16, 1, 2, 16>>;

static const char *const kLayerName[8] = {"enc1", "enc2", "enc3", "enc4", "dec0", "dec1", "dec2", "dec3+head"};

// One layer's plan: the public record, the layer parameters with their tiling fields filled, and the grid.
struct LayerPlan {
    cova_layer_plan info;
    tc::LayerParams lp;
    tc1::Enc1Extra ex;        // block 1 only
    tc::Grid grid;
};

template <bool WS, class C0, class... Cs>
static bool fit(LayerPlan &pl, int n_sms, int min_stage, int idx = 0) {
    tc::LayerParams q = pl.lp;
    bool ok;
    if constexpr (WS) ok = tcs::plan_e<C0>(q, n_sms, min_stage, pl.grid);
    else ok = tc::plan<C0>(q, n_sms, min_stage, pl.grid);
    if (ok) {
        pl.lp = q;
        pl.info.config = idx;
        pl.info.tps = C0::TPS;
        if constexpr (WS) pl.info.tile = C0::NP;
        else pl.info.tile = kTileM;
        return true;
    }
    if constexpr (sizeof...(Cs) > 0) return fit<WS, Cs...>(pl, n_sms, min_stage, idx + 1);
    else return false;
}
// first fit in list order, except that a configuration that can double-buffer its strips (ring depth >= 2) beats an
// earlier one that cannot
template <bool WS, class... Cs>
static bool first_fit(Cands<Cs...>, LayerPlan &pl, int n_sms) {
    pl.info.family = WS ? COVA_PLAN_WS : COVA_PLAN_POS;
    return fit<WS, Cs...>(pl, n_sms, 2) || fit<WS, Cs...>(pl, n_sms, 1);
}
template <bool WS, class C0, class... Cs>
static cudaError_t launch_nth(const LayerPlan &pl, int idx, cudaStream_t st) {
    if (idx == 0) {
        if constexpr (WS) return tcs::launch_e<C0>(pl.lp, pl.grid, st);
        else return tc::launch<C0>(pl.lp, pl.grid, st);
    }
    if constexpr (sizeof...(Cs) > 0) return launch_nth<WS, Cs...>(pl, idx - 1, st);
    else return cudaErrorInvalidValue;
}
template <bool WS, class... Cs>
static cudaError_t launch_entry(Cands<Cs...>, const LayerPlan &pl, cudaStream_t st) {
    return launch_nth<WS, Cs...>(pl, pl.info.config, st);
}

// The geometry part of a layer's parameters, all a plan depends on: N windows (block 1: n_chains chains of fps frames).
static void plan_input(LayerPlan &pl, int layer, const Geom gx[4], const Geom gd[4], const Geom &gx0f, int N, int n_chains,
                       int fps, int gamma) {
    memset(&pl, 0, sizeof(pl));
    tc::LayerParams &lp = pl.lp;
    lp.N = N;
    lp.nsplit = 1;
    if (layer == 0) {
        lp.gin = gx0f; lp.gout = gx[1]; lp.gout2 = gd[3]; lp.N = n_chains * fps;
        pl.ex.n_chains = n_chains; pl.ex.fps = fps; pl.ex.gamma = gamma;
    } else if (layer < 4) {
        const int i = layer;
        lp.gin = gx[i]; lp.gout = i < 3 ? gx[i + 1] : gx[3]; lp.gout2 = gd[3 - i];
    } else {
        const int i = layer - 4;
        lp.gin = gd[i]; lp.gout = i < 3 ? gd[i + 1] : gd[3];
        lp.nsplit = i == 0 ? 2 : 1;
    }
}

// THE launch decision of a tcgen05 layer: kernel family and candidate for the geometry in pl (plan_input).  tc_layer launches
// what it returns, cova_blobnet_plan and cova_pipeline_new report or check it.  Depends on the grid width (the strip length
// grows with the row pitch), the debug bits 2 and 3, and the window count only through the SM count and 32-bit limits.
static int plan_layer(int layer, int dbg, int n_sms, LayerPlan &pl) {
    bool ok = false;
    if (layer == 0) {
        // first block: frame-level conv + PointWiseTN over a register ring of 4 frames, one kernel (blobnet_enc1.cuh)
        ok = tc1::plan_enc1(pl.lp, pl.ex, n_sms, pl.grid);
        pl.info.family = COVA_PLAN_ENC1; pl.info.tps = 2; pl.info.tile = kTileM;
    } else if (layer < 4) {
        const int i = layer;
        // block 3 (Cout = 64) stays on the positions-as-M kernel: measured 0.335 ms vs 0.376 ms per 8192 windows at 720p
        // (profiles/r1c_layer_timing.txt); dbg bit 3 forces the weights-stationary variant for experiments, dbg bit 2 the
        // positions-as-M kernel for blocks 2 and 4
        if (!(dbg & 4) && (i != 2 || (dbg & 8))) {
            // weights-stationary kernel first; the positions-as-M kernel below remains the fallback for grids
            // whose strips do not fit shared memory
            ok = i == 1 ? first_fit<true>(Enc2Ws{}, pl, n_sms) : i == 2 ? first_fit<true>(Enc3Ws{}, pl, n_sms) : first_fit<true>(Enc4Ws{}, pl, n_sms);
        }
        if (!ok) ok = i == 1 ? first_fit<false>(Enc2Pos{}, pl, n_sms) : i == 2 ? first_fit<false>(Enc3Pos{}, pl, n_sms) : first_fit<false>(Enc4Pos{}, pl, n_sms);
    } else {
        const int i = layer - 4;
        ok = i == 0 ? first_fit<false>(Dec0Pos{}, pl, n_sms) : i == 1 ? first_fit<false>(Dec1Pos{}, pl, n_sms)
           : i == 2 ? first_fit<false>(Dec2Pos{}, pl, n_sms) : first_fit<false>(Dec3Pos{}, pl, n_sms);
    }
    if (!ok) {
        pl.info = cova_layer_plan{};
        return set_err(COVA_E_UNSUPPORTED, "%s: no tcgen05 tile configuration fits shared memory for this macroblock grid", kLayerName[layer]);
    }
    pl.info.n_stage = pl.lp.n_stage;
    pl.info.n_groups = layer == 0 ? pl.ex.total : pl.lp.n_groups;
    pl.info.ctas = pl.grid.ctas;
    return COVA_OK;
}

static cudaError_t launch_layer(int layer, const LayerPlan &pl, cudaStream_t st) {
    const bool ws = pl.info.family == COVA_PLAN_WS;
    switch (layer) {
        case 0: return tc1::launch_enc1(pl.lp, pl.ex, pl.grid, st);
        case 1: return ws ? launch_entry<true>(Enc2Ws{}, pl, st) : launch_entry<false>(Enc2Pos{}, pl, st);
        case 2: return ws ? launch_entry<true>(Enc3Ws{}, pl, st) : launch_entry<false>(Enc3Pos{}, pl, st);
        case 3: return ws ? launch_entry<true>(Enc4Ws{}, pl, st) : launch_entry<false>(Enc4Pos{}, pl, st);
        case 4: return launch_entry<false>(Dec0Pos{}, pl, st);
        case 5: return launch_entry<false>(Dec1Pos{}, pl, st);
        case 6: return launch_entry<false>(Dec2Pos{}, pl, st);
        default: return launch_entry<false>(Dec3Pos{}, pl, st);
    }
}

// extents and activation geometries of a grid: N windows, F frames (block-1 input) per chunk
static void blobnet_geoms(int h_mb, int w_mb, int N, int F, int sizes_h[5], int sizes_w[5], Geom gx[4], Geom gd[4], Geom &gx0f) {
    sizes_h[0] = h_mb; sizes_w[0] = w_mb;
    for (int i = 1; i <= 4; i++) { sizes_h[i] = (sizes_h[i - 1] + 1) / 2; sizes_w[i] = (sizes_w[i - 1] + 1) / 2; }
    // encoder inputs (Tn = 4): X0 (8 ch incl. padding), X1 (16), X2 (32), X3 (64)
    const int xc[4] = {8, 16, 32, 64};
    for (int i = 0; i < 4; i++) gx[i] = make_geom(sizes_h[i], sizes_w[i], xc[i], kT, N);
    // decoder inputs (Tn = 1): D0in = enc4 t0 (128 @ s4), D1in (128 @ s3), D2in (64 @ s2), D3in (32 @ s1)
    for (int i = 0; i < 4; i++) gd[i] = make_geom(sizes_h[4 - i], sizes_w[4 - i], kDecCin[i], 1, N);
    // per-FRAME first-conv input (x-pair packed, Tn = 1, N = frames)
    gx0f = make_geom(sizes_h[0], sizes_w[0], 8, 1, F);
}

// plans of all eight layers for chunks of n_chains chains of fps frames that yield N windows
static int plan_blobnet(int h_mb, int w_mb, int N, int n_chains, int fps, int gamma, int dbg, int n_sms, cova_layer_plan out[8]) {
    int sh[5], sw[5];
    Geom gx[4], gd[4], gx0f;
    blobnet_geoms(h_mb, w_mb, N, n_chains * fps, sh, sw, gx, gd, gx0f);
    for (int layer = 0; layer < 8; layer++) {
        LayerPlan pl;
        plan_input(pl, layer, gx, gd, gx0f, N, n_chains, fps, gamma);
        int rc = plan_layer(layer, dbg, n_sms, pl);
        if (rc) return rc;
        out[layer] = pl.info;
    }
    return COVA_OK;
}

extern "C" int cova_blobnet_plan(uint32_t w_mb, uint32_t h_mb, uint32_t windows, int debug, int n_sms, cova_layer_plan out[8]) {
    if (!out) return set_err(COVA_E_INVAL, "null argument");
    memset(out, 0, 8 * sizeof(cova_layer_plan));
    if (!windows || windows > (1u << 24) || n_sms < 1) return set_err(COVA_E_INVAL, "need 1 <= windows <= 2^24 and n_sms >= 1");
    if (w_mb < 16 || h_mb < 16 || w_mb > (1u << 16) || h_mb > (1u << 16))
        return set_err(COVA_E_UNSUPPORTED, "macroblock grid must be at least 16x16 for four 2x poolings");
    // one chain of windows + timestep - 1 frames at gamma 1
    return plan_blobnet((int)h_mb, (int)w_mb, (int)windows, 1, (int)windows + kT - 1, 1, debug, n_sms, out);
}

static int tc_plan(cova_pipeline *p, const Slot &sl, const Chunk &ck, int layer, LayerPlan &pl) {
    plan_input(pl, layer, p->gx, p->gd, p->gx0f, (int)ck.windows, (int)ck.n_streams, (int)sl.fps, (int)p->gamma);
    return plan_layer(layer, p->dbg, p->n_sms, pl);
}

// launch a planned layer: everything but the plan's geometry and tiling fields is filled here
static int tc_launch(cova_pipeline *p, const Slot &sl, const Chunk &ck, int layer, LayerPlan &pl) {
    tc::LayerParams &lp = pl.lp;
    lp.watchdog = p->d_watchdog; lp.dbg = p->dbg;
    if (layer < 4) {
        const int i = layer;
        lp.in = p->x[i];
        lp.out = i < 3 ? p->x[i + 1] : nullptr;
        lp.out2 = p->d[3 - i];
        lp.out2_cb = i < 3 ? kDecCout[2 - i] / 8 : 0;
        const DevLayer &dl = pl.info.family == COVA_PLAN_WS ? p->encs[i] : p->enc[i];
        lp.wpack = dl.wpack; lp.epi = dl.epi;
        memcpy(lp.tn_w1, p->hw.enc[i].tn_w1, 64);
        memcpy(lp.tn_w2, p->hw.enc[i].tn_w2, 64);
        lp.bn_nonneg = 1;
        for (int c = 0; c < kEncCout[i]; c++)
            if (!(p->hw.enc[i].gamma[c] >= 0.f)) lp.bn_nonneg = 0;
        if (i == 0) {
            lp.in = p->x0f;
            pl.ex.tab = sl.d_tab + ck.stream0;
        }
    } else {
        const int i = layer - 4;
        lp.in = p->d[i];
        lp.out = i < 3 ? p->d[i + 1] : nullptr;
        lp.wpack = p->dec[i].wpack; lp.epi = p->dec[i].epi;
        lp.psplit = (p->dbg & 64) ? 0 : 1;     // dbg bit 6: whole-tile accumulators for dec0 / dec1 (experiments)
        lp.Ht = p->sizes_h[3 - i]; lp.Wt = p->sizes_w[3 - i];
        crop_for(lp.gin.H, lp.Ht, lp.crop_t);
        crop_for(lp.gin.W, lp.Wt, lp.crop_l);
        lp.mask = p->d_mask + (size_t)ck.window0 * p->W * p->H;
        lp.logits = p->d_logits ? p->d_logits + (size_t)ck.window0 * p->W * p->H : nullptr;
    }
    cudaError_t err = launch_layer(layer, pl, p->stream);
    if (err != cudaSuccess) return set_err(COVA_E_CUDA, "%s launch: %s", kLayerName[layer], cudaGetErrorString(err));
    p->last_plan[layer] = pl.info;
    p->launches++;
    static const char *const prof_name[8] = {"tc_enc1_fused", "tc_enc2", "tc_enc3", "tc_enc4", "tc_dec0", "tc_dec1", "tc_dec2", "tc_dec3_head"};
    prof_mark(p, prof_name[layer]);
    return COVA_OK;
}

extern "C" int cova_pipeline_run_layer(cova_pipeline *p, int layer, uint32_t impl) {
    if (!p) return set_err(COVA_E_INVAL, "null handle");
    if (layer < 0 || layer > 7 || impl > COVA_IMPL_SIMT) return set_err(COVA_E_INVAL, "layer must be 0..7, impl 0 or 1");
    Chunk ck;
    int rc = stage_chunk(p, ck);
    if (rc || !ck.windows) return rc;
    if (impl == COVA_IMPL_SIMT) return simt_layer(p, ck, layer);
    LayerPlan pl;
    if ((rc = tc_plan(p, p->slot[p->last_slot], ck, layer, pl))) return rc;
    return tc_launch(p, p->slot[p->last_slot], ck, layer, pl);
}

static int blobnet_chunk(cova_pipeline *p, const Slot &sl, const Chunk &ck) {
    if (!ck.windows) return COVA_OK;
    if (p->impl == COVA_IMPL_SIMT) {
        for (int layer = 0; layer < 8; layer++) {
            int rc = simt_layer(p, ck, layer);
            if (rc) return rc;
        }
        return COVA_OK;
    }
    // every layer is planned before the first one is launched: a grid (or debug route) that one of them cannot take is
    // refused on the host, with nothing of the chunk's network enqueued
    LayerPlan plans[8];
    for (int layer = 0; layer < 8; layer++) {
        int rc = tc_plan(p, sl, ck, layer, plans[layer]);
        if (rc) return rc;
    }
    for (int layer = 0; layer < 8; layer++) {
        int rc = tc_launch(p, sl, ck, layer, plans[layer]);
        if (rc) return rc;
    }
    return COVA_OK;
}

extern "C" int cova_pipeline_blobnet(cova_pipeline *p) {
    Chunk ck;
    int rc = stage_chunk(p, ck);
    return rc ? rc : blobnet_chunk(p, p->slot[p->last_slot], ck);
}

static int ccl_range(cova_pipeline *p, Slot &sl, size_t first, int n, bool reset_cursor) {
    int rc = ccl_launch(sl.ccl, p->d_mask, n, p->cc_threshold, false, p->stream, first, reset_cursor, !(p->dbg & kDbgNoPdl));
    if (rc) return rc;
    if (n > 0) {
        p->launches++;
        prof_mark(p, sl.ccl.k > 1 ? "ccl_bbox_cluster" : "ccl_bbox");
    }
    return COVA_OK;
}

extern "C" int cova_pipeline_ccl(cova_pipeline *p) {
    if (!p) return set_err(COVA_E_INVAL, "null handle");
    if (int rc = require_idle(p)) return rc;
    COVA_CUDA(cudaSetDevice(p->device));
    Slot &sl = p->slot[p->last_slot];
    // ccl_range resets the box arena's cursor only when it launches
    if (!sl.n_windows) COVA_CUDA(cudaMemsetAsync(sl.ccl.d_cursor, 0, 2 * sizeof(unsigned long long), p->stream));
    return ccl_range(p, sl, 0, (int)sl.n_windows, true);
}

static void prof_begin(cova_pipeline *p) {
    if (!p->profiling) return;
    p->ev_used = 0;
    p->names.clear();
    prof_mark(p, "start");
}

// all kernels of one chunk, on p->stream
static int run_chunk(cova_pipeline *p, Slot &sl, const Chunk &ck) {
    p->last_chunk = ck;
    // the box arena's cursor is reset ahead of the batch's first kernel, not between the last layer and the CCL
    // kernel: a memset node there would break the chain of programmatic dependent launches (common.cuh)
    if (ck.stream0 == 0) COVA_CUDA(cudaMemsetAsync(sl.ccl.d_cursor, 0, 2 * sizeof(unsigned long long), p->stream));
    int rc = tensorise_chunk(p, sl, ck);
    if (!rc) rc = blobnet_chunk(p, sl, ck);
    if (!rc) rc = ccl_range(p, sl, ck.window0, (int)ck.windows, false);
    return rc;
}

extern "C" int cova_pipeline_run(cova_pipeline *p) {
    if (!p) return set_err(COVA_E_INVAL, "null handle");
    if (int rc = require_idle(p)) return rc;
    COVA_CUDA(cudaSetDevice(p->device));
    prof_begin(p);
    Slot &sl = p->slot[p->last_slot];
    if (!sl.n_streams || !sl.n_windows) return cova_pipeline_ccl(p);   // masks loaded directly, or no window at all
    for (uint32_t c = 0; c * p->chunk_streams < sl.n_streams; c++)
        if (int rc = run_chunk(p, sl, chunk_of(sl, c, p->chunk_streams))) return rc;
    return COVA_OK;
}

static int sync_stream(cova_pipeline *p, cudaStream_t st) {
    cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) {
        unsigned int code = 0;
        cudaMemcpy(&code, p->d_watchdog, sizeof(code), cudaMemcpyDeviceToHost);
        char extra[64];
        snprintf(extra, sizeof(extra), " (barrier watchdog code %u)", code);
        return set_err(COVA_E_CUDA, "stream synchronize: %s%s", cudaGetErrorString(e), extra);
    }
    return COVA_OK;
}

extern "C" int cova_pipeline_sync(cova_pipeline *p) {
    if (!p) return set_err(COVA_E_INVAL, "null handle");
    COVA_CUDA(cudaSetDevice(p->device));
    int rc = sync_stream(p, p->stream);
    if (rc) return rc;
    if (p->profiling && p->ev_used > 1) {
        // per-kernel device time, summed over the chunks of the batch
        p->last_ms.clear();
        p->last_names.clear();
        for (size_t i = 1; i < p->ev_used; i++) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, p->events[i - 1], p->events[i]);
            size_t k = 0;
            for (; k < p->last_names.size(); k++)
                if (p->last_names[k] == p->names[i]) break;
            if (k == p->last_names.size()) { p->last_names.push_back(p->names[i]); p->last_ms.push_back(0.f); }
            p->last_ms[k] += ms;
        }
        p->ev_used = 0;
        p->names.clear();
    }
    return COVA_OK;
}

extern "C" int cova_pipeline_fetch_boxes(cova_pipeline *p, uint8_t *blob, size_t blob_cap, size_t *blob_len, uint64_t *offsets, uint64_t *lens) {
    if (!p || !blob_len) return set_err(COVA_E_INVAL, "null argument");
    COVA_CUDA(cudaSetDevice(p->device));
    Slot &sl = p->slot[p->last_slot];
    const size_t n = sl.n_windows;
    COVA_CUDA(cudaMemcpyAsync(sl.h_cursor, sl.ccl.d_cursor, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, p->stream));
    int rc = cova_pipeline_sync(p);
    if (rc) return rc;
    if (sl.h_cursor[1]) return set_err(COVA_E_CUDA, "device box arena overflow (internal sizing error)");
    const unsigned long long end = sl.h_cursor[0];
    *blob_len = (size_t)end;
    if (offsets && n) COVA_CUDA(cudaMemcpyAsync(offsets, sl.ccl.d_offsets, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, p->stream));
    if (lens && n) COVA_CUDA(cudaMemcpyAsync(lens, sl.ccl.d_lens, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, p->stream));
    const bool fits = blob && blob_cap >= end;
    if (fits && end) COVA_CUDA(cudaMemcpyAsync(blob, sl.ccl.d_blob, (size_t)end, cudaMemcpyDeviceToHost, p->stream));
    COVA_CUDA(cudaStreamSynchronize(p->stream));
    if (!fits) return set_err(COVA_E_TOOSMALL, "box blob needs a larger buffer");
    return COVA_OK;
}

// Per-stream carry-over for CONTINUED batches.  carry[id] holds the last T - 1 frames of stream `id`, newest last.
//   mode 0 (restore): device chain s gets the newest h carried frames of stream ids[s] in front of its new frames;
//   mode 1 (save):    the last min(fps_dev, T - 1) frames of device chain s become the carry of stream ids[s].
__global__ void __launch_bounds__(256) carry_kernel(uint32_t *__restrict__ pool, uint32_t *__restrict__ carry, const uint32_t *__restrict__ ids,
                                                    int n_streams, int words_per_frame, int fps_dev, int h, int t1, int mode) {
    const int k = mode ? min(fps_dev, t1) : h;                     // frames moved per stream
    const long long per_stream = (long long)k * words_per_frame, total = per_stream * n_streams;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int s = (int)(i / per_stream);
        const long long e = i - (long long)s * per_stream;
        uint32_t *c = carry + ((long long)ids[s] * t1 + (t1 - k)) * words_per_frame + e;
        uint32_t *f = pool + ((long long)s * fps_dev + (mode ? fps_dev - k : 0)) * words_per_frame + e;
        if (mode) *c = *f; else *f = *c;
    }
}

// Host frames in, boxes out, asynchronously.  Three streams: the H2D copy of chunk c+1, the kernels of chunk c and
// the D2H copy of earlier boxes overlap; with up to four batches in flight (submit k+3 before collect k) the copies
// of one batch hide behind the kernels of another and the H2D engine is never idle.  A chunk's boxes occupy one contiguous range of the slot's device
// arena (the cursor is only reset at the start of a batch), so each chunk needs exactly one blob copy of exactly
// the bytes it produced.
//
// submit_host2 adds the stream identity the reference's elements have implicitly (one element instance per stream,
// State.prev_buffers / gamma_idx alive for the whole stream, metapreprocess/imp.rs:38-42,302-330): with
// COVA_SUBMIT_CONTINUE the chains of this batch continue the streams `stream_ids` from where their previous batch left
// them - the carried T - 1 frames are put in front of the new ones on the device and the gamma phase continues, so a
// stream cut into batches yields exactly the windows of the uncut stream.
//
// COVA_SUBMIT_STAGGERED lets the continued streams of one batch differ in history h_s = min(seen_s, T - 1) and gamma phase.
// Every device chain then has fps + lead frames, lead = max_s h_s: the new frames start at index lead, the carried ones sit
// right-aligned in front of them at [lead - h_s, lead), and what lies before that is never read by an emitted window.  So
// the copies and the per-frame kernels see one uniform chain length, and only the window -> frame tables differ per chain.
//
// Sparse input (submit_sparse, sparse_len != nullptr: `frames` is a batch of *sparse_len bytes of records) differs only in
// the copy stage of a chunk: the host validates every record first and keeps their offsets; chunk c's records are one
// contiguous byte range, copied as such, and sparse_expand_kernel writes them into the frame pool where the dense copy
// would have put them.  Everything after that is shared.

// Argument checks and per-chain plan of a submit, before any device call: fills first_scratch, hist_scratch and
// off_scratch, and raises lead (0 on entry) to the longest carried history
static int plan_submit(cova_pipeline *p, const uint8_t *frames, uint32_t n_streams, uint32_t fps, const uint32_t *stream_ids,
                       uint32_t flags, bool stateful, const size_t *sparse_len, uint32_t &lead) {
    if (flags & ~(COVA_SUBMIT_CONTINUE | COVA_SUBMIT_STAGGERED)) return set_err(COVA_E_INVAL, "unknown submit flag");
    if ((flags & COVA_SUBMIT_STAGGERED) && !(flags & COVA_SUBMIT_CONTINUE))
        return set_err(COVA_E_INVAL, "COVA_SUBMIT_STAGGERED needs COVA_SUBMIT_CONTINUE");
    if (sparse_len && !p->packed) return set_err(COVA_E_INVAL, "sparse input needs a COVA_FLAG_INPUT_PACKED16 pipeline");
    int rc = check_batch_bounds(p, n_streams, fps);
    if (rc) return rc;
    if (sparse_len) {
        const uint64_t n_frames = (uint64_t)n_streams * fps;
        p->off_scratch.resize(n_frames + 1);
        uint64_t bad = 0;
        if (const char *why = sparse::validate_batch(frames, *sparse_len, n_frames, p->W * p->H, p->off_scratch.data(), &bad)) {
            char frame[32];
            snprintf(frame, sizeof(frame), "%llu", (unsigned long long)bad);
            return set_err(COVA_E_INVAL, "malformed sparse batch at frame %s: %s", frame, why);
        }
    }
    const uint32_t t1 = p->T - 1;
    std::vector<uint32_t> &first = p->first_scratch, &hist = p->hist_scratch;
    first.assign(n_streams, t1);
    hist.assign(n_streams, 0);
    if (stateful) {
        if (!fps) return set_err(COVA_E_INVAL, "a stream batch needs at least one frame per stream");
        if (p->n_seen.empty()) { p->n_seen.assign(p->max_streams, 0); p->id_mark.assign(p->max_streams, 0); }
        p->id_epoch++;                                              // "seen in this batch" marks without clearing the array
        for (uint32_t s = 0; s < n_streams; s++) {
            const uint32_t id = stream_ids ? stream_ids[s] : s;
            if (id >= p->max_streams) return set_err(COVA_E_INVAL, "stream id out of range (ids are 0 .. max_streams-1)");
            if (p->id_mark[id] == p->id_epoch) return set_err(COVA_E_INVAL, "a stream id appears twice in one batch");
            p->id_mark[id] = p->id_epoch;
            if (!(flags & COVA_SUBMIT_CONTINUE)) continue;
            const uint64_t seen = p->n_seen[id];
            const uint32_t hs = (uint32_t)std::min<uint64_t>(seen, t1);
            const uint64_t base = seen - hs;                        // frames of the stream in front of its carried ones
            // smallest index i' >= T-1 of the unpadded chain with (base + i' - (T-1)) % gamma == 0 (imp.rs:321-330)
            hist[s] = hs;
            first[s] = t1 + (uint32_t)((p->gamma - base % p->gamma) % p->gamma);
            lead = std::max(lead, hs);
            // without COVA_SUBMIT_STAGGERED the streams of a batch advance in lock-step: same history, same gamma phase
            if (!(flags & COVA_SUBMIT_STAGGERED) && s && (hs != hist[0] || first[s] != first[0]))
                return set_err(COVA_E_INVAL, "streams of one CONTINUED batch must have the same history length and gamma phase "
                                             "(or pass COVA_SUBMIT_STAGGERED)");
        }
        for (uint32_t s = 0; s < n_streams; s++) first[s] += lead - hist[s];   // chain s is padded by lead - h_s frames
    }
    if (fps + lead > p->max_fps)
        return set_err(COVA_E_INVAL, "carried frames + new frames exceed max_frames_per_stream of the pipeline");
    return COVA_OK;
}

// slot k takes the planned batch: buffers on first use, window shape, per-window stream ids and PTS, frames seen per stream
static int setup_slot(cova_pipeline *p, int k, uint32_t n_streams, uint32_t fps, uint32_t lead, const uint32_t *stream_ids,
                      const uint64_t *pts, uint32_t flags, bool stateful, bool sparse) {
    int rc = ensure_slot(p, k);
    if (rc) return rc;
    auto &sl = p->slot[k];
    const uint32_t t1 = p->T - 1;
    if (stateful) {
        if (!p->d_carry && t1) {
            COVA_CUDA(cudaMalloc(&p->d_carry, (size_t)p->max_streams * t1 * p->frame_bytes));
            COVA_CUDA(cudaMemsetAsync(p->d_carry, 0, (size_t)p->max_streams * t1 * p->frame_bytes, p->stream));
        }
        if (!sl.h_ids) {
            COVA_CUDA(cudaMallocHost(&sl.h_ids, sizeof(uint32_t) * p->max_streams));
            COVA_CUDA(cudaMalloc(&sl.d_ids, sizeof(uint32_t) * p->max_streams));
        }
    }
    if (sparse && !sl.ev_off) {        // dense users never pay for these
        const size_t max_frames = (size_t)p->max_streams * p->max_fps;
        if (!sl.d_sparse) COVA_CUDA(cudaMalloc(&sl.d_sparse, max_frames * COVA_SPARSE_MAX_FRAME_BYTES(p->W * p->H)));
        if (!sl.h_off) COVA_CUDA(cudaMallocHost(&sl.h_off, sizeof(unsigned long long) * (max_frames + 1)));
        if (!sl.d_off) COVA_CUDA(cudaMalloc(&sl.d_off, sizeof(unsigned long long) * (max_frames + 1)));
        COVA_CUDA(cudaEventCreateWithFlags(&sl.ev_off, cudaEventDisableTiming));
    }
    const std::vector<uint32_t> &first = p->first_scratch;
    if ((rc = set_batch_shape(p, k, n_streams, fps + lead, first.data()))) return rc;
    p->last_slot = k;
    sl.win_pts.clear(); sl.win_ids.clear();
    if (stateful) {
        // window w of chain s has its newest frame at device index first_s + w*gamma = new-frame index first_s + w*gamma - lead
        sl.win_ids.resize(sl.n_windows);
        if (pts) sl.win_pts.resize(sl.n_windows);
        for (uint32_t s = 0; s < n_streams; s++) {
            const uint32_t id = stream_ids ? stream_ids[s] : s;
            sl.h_ids[s] = id;
            for (uint32_t w = sl.win0[s]; w < sl.win0[s + 1]; w++) {
                sl.win_ids[w] = id;
                if (pts) sl.win_pts[w] = pts[(size_t)s * fps + (first[s] + (w - sl.win0[s]) * p->gamma - lead)];
            }
            p->n_seen[id] = ((flags & COVA_SUBMIT_CONTINUE) ? p->n_seen[id] : 0) + fps;
        }
    }
    return COVA_OK;
}

// copy stage, on s_in: per chunk the new frames (dense, padded behind lead carried frames, or sparse records), then ev_in[c]
static int copy_chunks(cova_pipeline *p, Slot &sl, const uint8_t *frames, uint32_t fps, uint32_t lead, bool sparse) {
    if (sparse) {
        // the slot's previous offsets upload has completed (its batch was collected); the event makes that explicit
        const size_t n_offs = (size_t)sl.n_streams * fps + 1;
        COVA_CUDA(cudaEventSynchronize(sl.ev_off));
        memcpy(sl.h_off, p->off_scratch.data(), sizeof(unsigned long long) * n_offs);
        COVA_CUDA(cudaMemcpyAsync(sl.d_off, sl.h_off, sizeof(unsigned long long) * n_offs, cudaMemcpyHostToDevice, p->stream));
        COVA_CUDA(cudaEventRecord(sl.ev_off, p->stream));
    }
    const size_t src_chain = p->frame_bytes * fps, dst_chain = p->frame_bytes * sl.fps, lead_bytes = p->frame_bytes * lead;
    for (uint32_t c = 0; c * p->chunk_streams < sl.n_streams; c++) {
        const Chunk ck = chunk_of(sl, c, p->chunk_streams);
        const size_t s0 = ck.stream0, ns = ck.n_streams;
        if (sparse) {      // chunk c's records: one contiguous byte range, to the same offset of the staging
            const uint64_t b0 = p->off_scratch[s0 * fps], b1 = p->off_scratch[(s0 + ns) * fps];
            COVA_CUDA(cudaMemcpyAsync(sl.d_sparse + b0, frames + b0, b1 - b0, cudaMemcpyHostToDevice, p->s_in));
        } else if (!lead) COVA_CUDA(cudaMemcpyAsync(sl.d_frames + s0 * dst_chain, frames + s0 * src_chain, ns * src_chain, cudaMemcpyHostToDevice, p->s_in));
        else COVA_CUDA(cudaMemcpy2DAsync(sl.d_frames + s0 * dst_chain + lead_bytes, dst_chain, frames + s0 * src_chain, src_chain, src_chain, ns,
                                         cudaMemcpyHostToDevice, p->s_in));
        COVA_CUDA(cudaEventRecord(sl.ev_in[c], p->s_in));
    }
    return COVA_OK;
}

// compute stage, on p->stream: per chunk after ev_in[c] sparse expansion, carry restore / save, kernels, cursor snapshot
static int compute_chunks(cova_pipeline *p, Slot &sl, uint32_t fps, uint32_t lead, bool stateful, bool sparse) {
    const uint32_t t1 = p->T - 1, fps_dev = sl.fps;
    const size_t dst_chain = p->frame_bytes * fps_dev;
    const int wpf = (int)(p->frame_bytes / 4);
    if (stateful) COVA_CUDA(cudaMemcpyAsync(sl.d_ids, sl.h_ids, sizeof(uint32_t) * sl.n_streams, cudaMemcpyHostToDevice, p->stream));
    for (uint32_t c = 0; c * p->chunk_streams < sl.n_streams; c++) {
        const Chunk ck = chunk_of(sl, c, p->chunk_streams);
        COVA_CUDA(cudaStreamWaitEvent(p->stream, sl.ev_in[c], 0));
        if (sparse) {      // a plain launch: tensorise_frames_kernel waits for it (pdl_wait) before reading the pool
            SparseExpandArgs ea{sl.d_sparse, sl.d_off, sl.d_frames, ck.stream0 * fps, fps, fps_dev, lead, p->W * p->H};
            sparse_expand_kernel<<<ck.n_streams * fps, kExpandThreads, 0, p->stream>>>(ea);
            p->launches++;
            COVA_CUDA(cudaGetLastError());
        }
        if (stateful && t1) {
            const int ns = (int)ck.n_streams;
            uint32_t *pool = reinterpret_cast<uint32_t *>(sl.d_frames + ck.stream0 * dst_chain);
            const int blocks = std::min(p->n_sms * 8, std::max(1, (int)(((long long)ns * t1 * wpf + 255) / 256)));
            if (lead) {     // lead frames for every chain: a chain with less history gets older carry bytes no window reads
                carry_kernel<<<blocks, 256, 0, p->stream>>>(pool, reinterpret_cast<uint32_t *>(p->d_carry), sl.d_ids + ck.stream0, ns, wpf, (int)fps_dev, (int)lead, (int)t1, 0);
                p->launches++;
            }
            carry_kernel<<<blocks, 256, 0, p->stream>>>(pool, reinterpret_cast<uint32_t *>(p->d_carry), sl.d_ids + ck.stream0, ns, wpf, (int)fps_dev, (int)lead, (int)t1, 1);
            p->launches++;
            COVA_CUDA(cudaGetLastError());
        }
        if (sl.n_windows) {
            int rc = run_chunk(p, sl, ck);
            if (rc) return rc;
            COVA_CUDA(cudaMemcpyAsync(sl.h_cursor + 2 * c, sl.ccl.d_cursor, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, p->stream));
        }
        COVA_CUDA(cudaEventRecord(sl.ev_done[c], p->stream));
    }
    return COVA_OK;
}

static int submit_impl(cova_pipeline *p, const uint8_t *frames, uint32_t n_streams, uint32_t fps, const uint32_t *stream_ids,
                       const uint64_t *pts, uint32_t flags, bool stateful, const size_t *sparse_len = nullptr) {
    if (!p || !frames) return set_err(COVA_E_INVAL, "null argument");
    const bool sparse = sparse_len != nullptr;
    uint32_t lead = 0;                                              // carried frames in front of every device chain
    int rc = plan_submit(p, frames, n_streams, fps, stream_ids, flags, stateful, sparse_len, lead);
    if (rc) return rc;
    COVA_CUDA(cudaSetDevice(p->device));
    const int k = p->next_submit;
    if (p->slot[k].busy) return set_err(COVA_E_INVAL, "four batches are already in flight: collect one first");
    if ((rc = setup_slot(p, k, n_streams, fps, lead, stream_ids, pts, flags, stateful, sparse))) return rc;
    auto &sl = p->slot[k];
    sl.busy = true; sl.failed = false;
    p->next_submit = (k + 1) % kSlots;
    if (!stateful && !sl.n_windows) return COVA_OK;                // chains shorter than a window: nothing to compute
    // from here on a failure leaves the slot marked failed: the matching collect reports it instead of reading events that
    // were never recorded
    if ((rc = copy_chunks(p, sl, frames, fps, lead, sparse)) || (rc = compute_chunks(p, sl, fps, lead, stateful, sparse)))
        sl.failed = true;
    return rc;
}

extern "C" int cova_pipeline_submit_host(cova_pipeline *p, const uint8_t *frames, uint32_t n_streams, uint32_t fps) {
    return submit_impl(p, frames, n_streams, fps, nullptr, nullptr, 0, false);
}
extern "C" int cova_pipeline_submit_host2(cova_pipeline *p, const uint8_t *frames, uint32_t n_streams, uint32_t fps,
                                          const uint32_t *stream_ids, const uint64_t *pts, uint32_t flags) {
    return submit_impl(p, frames, n_streams, fps, stream_ids, pts, flags, true);
}
extern "C" int cova_pipeline_submit_sparse(cova_pipeline *p, const uint8_t *data, size_t data_len, uint32_t n_streams,
                                           uint32_t fps, const uint32_t *stream_ids, const uint64_t *pts, uint32_t flags) {
    return submit_impl(p, data, n_streams, fps, stream_ids, pts, flags, true, &data_len);
}
extern "C" int cova_pipeline_reset_streams(cova_pipeline *p, const uint32_t *stream_ids, uint32_t n) {
    if (!p) return set_err(COVA_E_INVAL, "null handle");
    if (p->n_seen.empty()) return COVA_OK;
    if (!stream_ids) { std::fill(p->n_seen.begin(), p->n_seen.end(), 0); return COVA_OK; }
    for (uint32_t i = 0; i < n; i++) {
        if (stream_ids[i] >= p->max_streams) return set_err(COVA_E_INVAL, "stream id out of range");
        p->n_seen[stream_ids[i]] = 0;
    }
    return COVA_OK;
}

static int collect_impl(cova_pipeline *p, uint8_t *blob, size_t blob_cap, size_t *blob_len, uint64_t *offsets, uint64_t *lens,
                        uint32_t *n_windows, uint32_t *win_stream_ids, uint64_t *win_pts) {
    if (!p || !blob_len) return set_err(COVA_E_INVAL, "null argument");
    COVA_CUDA(cudaSetDevice(p->device));
    const int k = p->next_collect;
    auto &sl = p->slot[k];
    if (!sl.busy) return set_err(COVA_E_INVAL, "no batch in flight");
    sl.busy = false;
    p->next_collect = (k + 1) % kSlots;
    if (n_windows) *n_windows = sl.n_windows;
    *blob_len = 0;
    if (sl.failed) {
        sl.failed = false;
        cudaStreamSynchronize(p->stream);
        cudaGetLastError();
        return set_err(COVA_E_CUDA, "the submit of this batch failed part-way; its results are void");
    }
    if (win_stream_ids && !sl.win_ids.empty()) memcpy(win_stream_ids, sl.win_ids.data(), sl.win_ids.size() * sizeof(uint32_t));
    if (win_pts && !sl.win_pts.empty()) memcpy(win_pts, sl.win_pts.data(), sl.win_pts.size() * sizeof(uint64_t));
    const uint32_t nc = (sl.n_streams + p->chunk_streams - 1) / p->chunk_streams;
    if (!sl.n_windows) {
        // nothing to copy, but the batch's device work (carry-over of a short CONTINUED batch) must have completed before
        // the caller may reuse its frame buffer
        if (nc && cudaEventSynchronize(sl.ev_done[nc - 1]) != cudaSuccess) return sync_stream(p, p->stream);
        return COVA_OK;
    }
    unsigned long long prev = 0;
    bool too_small = false;
    for (uint32_t c = 0; c < nc; c++) {
        if (cudaEventSynchronize(sl.ev_done[c]) != cudaSuccess) return sync_stream(p, p->stream);
        if (sl.h_cursor[2 * c + 1]) return set_err(COVA_E_CUDA, "device box arena overflow (internal sizing error)");
        const unsigned long long end = sl.h_cursor[2 * c];
        const Chunk ck = chunk_of(sl, c, p->chunk_streams);
        const size_t w0 = ck.window0, nw = ck.windows;
        if (offsets) COVA_CUDA(cudaMemcpyAsync(offsets + w0, sl.ccl.d_offsets + w0, nw * sizeof(uint64_t), cudaMemcpyDeviceToHost, p->s_out));
        if (lens) COVA_CUDA(cudaMemcpyAsync(lens + w0, sl.ccl.d_lens + w0, nw * sizeof(uint64_t), cudaMemcpyDeviceToHost, p->s_out));
        if (blob && end <= blob_cap) {
            if (end > prev) COVA_CUDA(cudaMemcpyAsync(blob + prev, sl.ccl.d_blob + prev, (size_t)(end - prev), cudaMemcpyDeviceToHost, p->s_out));
        } else {
            too_small = true;
        }
        prev = end;
    }
    COVA_CUDA(cudaStreamSynchronize(p->s_out));
    *blob_len = (size_t)prev;
    if (too_small) return set_err(COVA_E_TOOSMALL, "box blob needs a larger buffer");
    return COVA_OK;
}

extern "C" int cova_pipeline_collect_host(cova_pipeline *p, uint8_t *blob, size_t blob_cap, size_t *blob_len, uint64_t *offsets,
                                          uint64_t *lens, uint32_t *n_windows) {
    return collect_impl(p, blob, blob_cap, blob_len, offsets, lens, n_windows, nullptr, nullptr);
}
extern "C" int cova_pipeline_collect_host2(cova_pipeline *p, uint8_t *blob, size_t blob_cap, size_t *blob_len, uint64_t *offsets,
                                           uint64_t *lens, uint32_t *n_windows, uint32_t *win_stream_ids, uint64_t *win_pts) {
    return collect_impl(p, blob, blob_cap, blob_len, offsets, lens, n_windows, win_stream_ids, win_pts);
}

extern "C" int cova_pipeline_process_host(cova_pipeline *p, const uint8_t *frames, uint32_t n_streams, uint32_t fps, uint8_t *blob,
                                          size_t blob_cap, size_t *blob_len, uint64_t *offsets, uint64_t *lens, uint32_t *n_windows) {
    if (!p || !frames || !blob_len) return set_err(COVA_E_INVAL, "null argument");
    int rc = require_idle(p);
    if (rc) return rc;
    p->next_submit = p->next_collect = 0;
    prof_begin(p);
    rc = cova_pipeline_submit_host(p, frames, n_streams, fps);
    if (!rc) rc = cova_pipeline_collect_host(p, blob, blob_cap, blob_len, offsets, lens, n_windows);
    else if (p->slot[0].busy) { p->slot[0].busy = false; p->slot[0].failed = false; p->next_submit = p->next_collect = 0; }
    if (!rc) rc = cova_pipeline_sync(p);
    return rc;
}

// ---- inspection ------------------------------------------------------------------------------------
// the last batch's [n_windows][per_window] array of elem_bytes elements on the device -> out (cap elements)
static int read_windows(cova_pipeline *p, const void *src, size_t per_window, size_t elem_bytes, void *out, size_t cap) {
    const size_t n = per_window * p->slot[p->last_slot].n_windows;
    if (cap < n) return set_err(COVA_E_TOOSMALL, "buffer too small");
    int rc = cova_pipeline_sync(p);
    if (rc) return rc;
    COVA_CUDA(cudaMemcpy(out, src, n * elem_bytes, cudaMemcpyDeviceToHost));
    return COVA_OK;
}
extern "C" int cova_pipeline_read_stacked(cova_pipeline *p, uint8_t *out, size_t cap) {
    if (!p || !out) return set_err(COVA_E_INVAL, "null argument");
    if (!p->d_stacked) return set_err(COVA_E_INVAL, "pipeline was created without COVA_FLAG_KEEP_STACKED");
    return read_windows(p, p->d_stacked, p->frame_bytes * p->T, 1, out, cap);
}
extern "C" int cova_pipeline_read_mask(cova_pipeline *p, uint8_t *out, size_t cap) {
    if (!p || !out) return set_err(COVA_E_INVAL, "null argument");
    return read_windows(p, p->d_mask, (size_t)p->W * p->H, 1, out, cap);
}
extern "C" int cova_pipeline_read_logits(cova_pipeline *p, float *out, size_t cap_floats) {
    if (!p || !out) return set_err(COVA_E_INVAL, "null argument");
    if (!p->d_logits) return set_err(COVA_E_INVAL, "pipeline was created without COVA_FLAG_KEEP_LOGITS");
    return read_windows(p, p->d_logits, (size_t)p->W * p->H, sizeof(float), out, cap_floats);
}

extern "C" int cova_pipeline_read_activation(cova_pipeline *p, int layer, float *out, size_t cap_floats, uint32_t shape[5]) {
    if (!p || !out || !shape) return set_err(COVA_E_INVAL, "null argument");
    if (layer < 0 || layer > 7) return set_err(COVA_E_INVAL, "layer must be 0..7");
    const bool enc_side = layer <= 3;
    const Geom &g = enc_side ? p->gx[layer] : p->gd[layer - 4];
    const uint4 *src = enc_side ? p->x[layer] : p->d[layer - 4];
    const int C = layer == 0 ? 3 : (enc_side ? kEncCout[layer - 1] : kDecCin[layer - 4]);
    const int N = (int)p->last_chunk.windows, Tn = g.Tn;
    shape[0] = N; shape[1] = C; shape[2] = Tn; shape[3] = g.H; shape[4] = g.W;
    size_t n = (size_t)N * C * Tn * g.H * g.W;
    if (cap_floats < n) return set_err(COVA_E_TOOSMALL, "buffer too small");
    int rc = cova_pipeline_sync(p);
    if (rc) return rc;
    if (layer == 0 && !p->x[0]) {
        // BlobNet input as the tcgen05 path sees it: per-frame x-pair-packed rows + the window table
        const Geom &gf = p->gx0f;
        std::vector<Row8> host((size_t)geom_rows(gf));
        COVA_CUDA(cudaMemcpy(host.data(), p->x0f, host.size() * sizeof(Row8), cudaMemcpyDeviceToHost));
        for (int nn = 0; nn < N; nn++)
            for (int c = 0; c < 3; c++)
                for (int t = 0; t < kT; t++)
                    for (int y = 0; y < gf.H; y++)
                        for (int x = 0; x < gf.W; x++) {
                            const int f = p->slot[p->last_slot].h_newest[p->last_chunk.window0 + nn] - t;
                            const Row8 &r = host[(size_t)geom_row(gf, 0, (y & 1) << 1, geom_pos(gf, f, y >> 1, x >> 1, 0))];
                            out[((((size_t)nn * 3 + c) * kT + t) * gf.H + y) * gf.W + x] = __half2float(r.v[(x & 1) * 4 + c]);
                        }
        shape[2] = kT;
        return COVA_OK;
    }
    std::vector<Row8> host((size_t)geom_rows(g));
    COVA_CUDA(cudaMemcpy(host.data(), src, host.size() * sizeof(Row8), cudaMemcpyDeviceToHost));
    for (int nn = 0; nn < N; nn++)
        for (int c = 0; c < C; c++)
            for (int t = 0; t < Tn; t++)
                for (int y = 0; y < g.H; y++)
                    for (int x = 0; x < g.W; x++) {
                        const Row8 &r = host[(size_t)geom_row_of(g, nn, t, c >> 3, y, x)];
                        out[((((size_t)nn * C + c) * Tn + t) * g.H + y) * g.W + x] = __half2float(r.v[c & 7]);
                    }
    return COVA_OK;
}

extern "C" int cova_pipeline_set_debug(cova_pipeline *p, int flags) {
    if (!p) return set_err(COVA_E_INVAL, "null handle");
    p->dbg = flags;
    // bit 5 (kDbgNoPdl): plain stream-ordered launches instead of programmatic dependent launch, for THIS handle only
    return COVA_OK;
}
extern "C" int cova_pipeline_last_plan(const cova_pipeline *p, cova_layer_plan out[8]) {
    if (!p || !out) return set_err(COVA_E_INVAL, "null argument");
    memcpy(out, p->last_plan, sizeof(p->last_plan));
    return COVA_OK;
}
extern "C" int cova_pipeline_launch_count(const cova_pipeline *p, uint64_t *count) {
    if (!p || !count) return set_err(COVA_E_INVAL, "null argument");
    *count = p->launches;
    return COVA_OK;
}
extern "C" int cova_pipeline_set_profiling(cova_pipeline *p, int enable) {
    if (!p) return set_err(COVA_E_INVAL, "null handle");
    p->profiling = enable != 0;
    p->ev_used = 0;
    p->names.clear();
    return COVA_OK;
}
extern "C" int cova_pipeline_last_timings(cova_pipeline *p, char *names, size_t names_cap, float *ms, uint32_t *n) {
    if (!p || !n) return set_err(COVA_E_INVAL, "null argument");
    uint32_t cap = *n;
    *n = (uint32_t)p->last_ms.size();
    std::string joined;
    for (size_t i = 0; i < p->last_names.size(); i++) { if (i) joined += ";"; joined += p->last_names[i]; }
    if (names && names_cap) { strncpy(names, joined.c_str(), names_cap - 1); names[names_cap - 1] = 0; }
    if (ms) for (uint32_t i = 0; i < std::min<uint32_t>(cap, *n); i++) ms[i] = p->last_ms[i];
    return COVA_OK;
}
