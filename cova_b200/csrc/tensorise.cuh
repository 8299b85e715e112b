// Tensorisation kernels: decoder metadata quads -> (a) the stacked RGBA window image the reference's
// metapreprocess element emits, (b) the BlobNet input in the phase-plane fp16 layout of common.cuh.
//
// Reference: cova-rs/gst-plugins/src/metapreprocess/imp.rs:307-320 (out[0:S] = current frame,
// out[kS:(k+1)S] = frame t-k) and the nvinfer pre-process + Reshape that follow it
// (config/blobnet/*.txt:7,9 - RGBA -> planar RGB, scale 1, byte 3 dropped;
//  utils/train-blobnet.py:113-116 - (3, T*H, W) -> (3, T, H, W)); utils/model/preprocessing.py:5-8
// (clip(x, 0, 6); the 1/6 is folded into the first convolution's weights).
#pragma once
#include "common.cuh"

namespace cova {

// (a) stacked RGBA: pure gather/copy, HBM bound.  One element = one 32-bit macroblock quad, or one
// 128-bit vector of four quads when the frame size allows it.
template <typename V>
__global__ void __launch_bounds__(256) stack_rgba_kernel(const V *__restrict__ frames, const int *__restrict__ newest,
                                                         V *__restrict__ out, int vec_per_frame, int T,
                                                         long long total) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < total; i += stride) {
        int e = (int)(i % vec_per_frame);
        long long r = i / vec_per_frame;
        int k = (int)(r % T);
        int n = (int)(r / T);
        long long src = (long long)(newest[n] - k) * vec_per_frame + e;
        out[i] = __ldg(frames + src);
    }
}

#ifdef COVA_VALIDATION
// (b) BlobNet input layout (validation build only).  Thread <-> (window n, row y, column pair x2, time t); the four t of one
// (y, x2) are adjacent lanes so that the 16-byte rows they write are contiguous (64 B), and a warp
// reads 8 consecutive 8-byte pixel pairs from each of the 4 frames.
__global__ void __launch_bounds__(256) tensorise_x0_kernel(const uint32_t *__restrict__ frames,
                                                           const int *__restrict__ newest, uint4 *__restrict__ x0,
                                                           Geom g, int n_windows) {
    const int Wh = g.Wh;
    const long long total = (long long)n_windows * g.H * Wh * kT;
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const int px_per_frame = g.H * g.W;
    for (; i < total; i += stride) {
        int t = (int)(i & 3);
        long long r = i >> 2;
        int x2 = (int)(r % Wh);
        r /= Wh;
        int y = (int)(r % g.H);
        int n = (int)(r / g.H);
        const uint32_t *f = frames + (long long)(newest[n] - t) * px_per_frame + (long long)y * g.W;
        int x = 2 * x2;
        uint32_t q0 = __ldg(f + x);
        uint32_t q1 = (x + 1 < g.W) ? __ldg(f + x + 1) : 0u;
        long long pos = geom_pos(g, n, y >> 1, x2, t);
        int ph = (y & 1) << 1;
#pragma unroll
        for (int b = 0; b < 2; b++) {
            if (b == 1 && x + 1 >= g.W) break;
            uint32_t q = b ? q1 : q0;
            // bytes: 0 mb_weight, 1 |mv_x|, 2 |mv_y|, 3 stale (dropped).  clip(., 0, 6) of a u8 = min(., 6)
            __half2 c01 = __floats2half2_rn((float)min(q & 0xffu, 6u), (float)min((q >> 8) & 0xffu, 6u));
            __half2 c2z = __floats2half2_rn((float)min((q >> 16) & 0xffu, 6u), 0.f);
            uint4 row;
            row.x = *reinterpret_cast<uint32_t *>(&c01);
            row.y = *reinterpret_cast<uint32_t *>(&c2z);
            row.z = 0u;
            row.w = 0u;
            x0[geom_row(g, 0, ph | b, pos)] = row;
        }
    }
}

#endif  // COVA_VALIDATION

// (c) per-FRAME BlobNet input for the tcgen05 path: one 16-byte row per horizontal pixel pair,
//     [c0 c1 c2 0 | c0' c1' c2' 0] (fp16, clipped to 6), in the two row-parity planes (ph = 0 and 2) of a
//     Tn = 1 phase-plane geometry whose "windows" are the frames of the pool.  The first convolution runs once
//     per frame on this; the window structure (newest-first stacking of `timestep` frames) is applied afterwards
//     by enc1_fused_kernel as it walks each chain through time (blobnet_enc1.cuh).
// fp16 of the clipped bytes without integer->float conversions: 0x6400 | n is the half 1024 + n for n < 1024, and
// subtracting 1024 in half arithmetic is exact.  q = [mb_weight, |mv_x|, |mv_y|, stale]; returns (c0 c1 | c2 0) as two half2.
__device__ __forceinline__ uint2 quad_to_half4(uint32_t q) {
    // clip(., 0, 6) of a u8 = min(., 6), all four bytes at once.  __vminu4 is emulated on sm_100 (a dozen instructions);
    // SWAR: bit 7 of byte i of `ge` is set iff byte i >= 7 (low 7 bits + 121 carry into bit 7, or bit 7 already set)
    const uint32_t ge = (((q & 0x7f7f7f7fu) + 0x79797979u) | q) & 0x80808080u;
    const uint32_t sel = (ge >> 7) * 0xffu;                            // 0xff in every byte that is >= 7
    const uint32_t m = (q & ~sel) | (0x06060606u & sel);
    const uint32_t lo = __byte_perm(m, 0u, 0x4140) | 0x64006400u;      // bytes 0, 1 into the low byte of each half
    const uint32_t hi = __byte_perm(m, 0u, 0x4442) | 0x64006400u;      // byte 2; the fourth channel stays 0 (byte 3 is dropped)
    const __half2 k = __half2half2(__ushort_as_half((unsigned short)0x6400));
    const __half2 a = __hsub2(*reinterpret_cast<const __half2 *>(&lo), k), b = __hsub2(*reinterpret_cast<const __half2 *>(&hi), k);
    return make_uint2(*reinterpret_cast<const uint32_t *>(&a), *reinterpret_cast<const uint32_t *>(&b));
}

// PACKED: the frames are in the 2-byte packed input format (include/cova_b200.h, COVA_FLAG_INPUT_PACKED16): one u16 per
// macroblock, bits 0-2 mb_weight, 3-5 |mv_x|, 6-8 |mv_y|, each already clipped to 6 by the host packer - exact for BlobNet,
// whose first operation is clip(., 0, 6) (utils/model/preprocessing.py:5-8), and half the host->device bytes.  W is even.
__device__ __forceinline__ uint32_t unpack16(uint32_t p) { return (p & 7u) | ((p & 0x38u) << 5) | ((p & 0x1c0u) << 10); }

// fmap (chunks of a ragged batch, cova_pipeline_submit_ragged): frame f of the n_frames that exist is frame fmap[f] of the
// pool, whose chains have one stride but end at different frames; nullptr = every frame of the pool exists (fmap[f] = f).
// The thread count scales with the frames that exist: a chain's dead tail is neither read nor written.
template <bool PACKED>
__global__ void __launch_bounds__(256) tensorise_frames_kernel(const uint32_t *__restrict__ frames, uint4 *__restrict__ x0f,
                                                               Geom g, int n_frames, FastDiv div_wh, FastDiv div_h,
                                                               const int *__restrict__ fmap) {
    pdl_launch_dependents();
    pdl_wait();              // x0f is still being read by the previous batch's first block until that batch has completed
    const uint32_t Wh = (uint32_t)g.Wh, H = (uint32_t)g.H, W = (uint32_t)g.W;
    const uint32_t total = (uint32_t)n_frames * H * Wh;                 // host guarantees < 2^32
    const uint32_t stride = gridDim.x * blockDim.x;
    const bool pair_aligned = (W & 1u) == 0u;                          // then an x pair is one aligned 8-byte load
    // four x pairs per thread and iteration, loads first: a thread keeps 4 x 8 bytes in flight (with one load per
    // iteration a full SM has 16 KB outstanding, half of what the HBM latency-bandwidth product asks for)
    constexpr int U = 4;
    for (uint32_t i0 = blockIdx.x * blockDim.x + threadIdx.x; i0 < total; i0 += U * stride) {
        uint32_t q0[U], q1[U], rr[U], xx[U];
#pragma unroll
        for (int k = 0; k < U; k++) {
            const uint32_t i = i0 + (uint32_t)k * stride;
            q0[k] = q1[k] = 0u; rr[k] = xx[k] = 0u;
            if (i < total) {
                uint32_t r = Wh > 1 ? fast_div(i, div_wh) : i;                           // r = f * H + y
                const uint32_t x2 = i - r * Wh;
                if (fmap) {                                                                  // -> row of the pool
                    const uint32_t f = H > 1 ? fast_div(r, div_h) : r;
                    r += ((uint32_t)__ldg(fmap + f) - f) * H;
                }
                const uint32_t *src = frames + ((size_t)r * W + 2 * x2);
                rr[k] = r; xx[k] = x2;
                if constexpr (PACKED) {
                    const uint32_t pp = __ldg(frames + ((size_t)r * (W >> 1) + x2));     // one x pair = two u16
                    q0[k] = unpack16(pp & 0xffffu); q1[k] = unpack16(pp >> 16);
                } else if (pair_aligned) {
                    const uint2 q = __ldg(reinterpret_cast<const uint2 *>(src));
                    q0[k] = q.x; q1[k] = q.y;
                } else {
                    q0[k] = __ldg(src);
                    q1[k] = (2 * x2 + 1 < W) ? __ldg(src + 1) : 0u;
                }
            }
        }
#pragma unroll
        for (int k = 0; k < U; k++) {
            if (i0 + (uint32_t)k * stride >= total) break;
            const uint32_t f = H > 1 ? fast_div(rr[k], div_h) : rr[k], y = rr[k] - f * H;
            const uint2 a = quad_to_half4(q0[k]), b = quad_to_half4(q1[k]);
            x0f[geom_row(g, 0, (int)((y & 1u) << 1), geom_pos(g, (int)f, (int)(y >> 1), (int)xx[k], 0))] = make_uint4(a.x, a.y, b.x, b.y);
        }
    }
}

}  // namespace cova
