// Sparse input (sparse_format.hpp, cova_pipeline_submit_sparse) -> the slot's packed16 frame pool.
//
// One CTA per frame.  The bitmap is taken in tiles of kExpandTileWords words (one tile up to 4K, 4 tiles at 8K): the
// popcounts of a tile's words get an exclusive block scan, which with the count of the tiles before gives every word the
// rank of its first set bit among the record's values.  Then each thread writes macroblock pairs - one u32 of the pool,
// consecutive threads consecutive words - as `bit ? values[rank] : background`.  w_mb is even, so a frame is a whole
// number of u32 (not necessarily of 16 bytes).
//
// Frame i = (s, f) of the batch lands at chain-relative index lead + f of device chain s, exactly where the dense H2D copy
// puts packed16 frames: carry-over, staggering and every later kernel see the same pool.  The record offsets come from
// the host's validation walk; the kernel reads nothing outside [off[i], off[i+1]) even if the caller's buffer changed
// after it was validated (a value rank past the record's end yields the background instead).
#pragma once
#include "common.cuh"
#include "sparse_format.hpp"

namespace cova {

constexpr int kExpandThreads = 256;
constexpr int kExpandTileWords = 4 * kExpandThreads;   // 32,768 macroblocks per tile

struct SparseExpandArgs {
    const uint8_t *data;                 // device copy of the batch, records at their host byte offsets
    const unsigned long long *off;       // n_frames + 1 record offsets of the batch
    uint8_t *pool;                       // the slot's frame pool: chains of fps_dev frames of 2 * n_mb bytes
    uint32_t frame0;                     // first batch frame of this launch (the chunk's first)
    uint32_t fps, fps_dev, lead, n_mb;
};

__global__ void __launch_bounds__(kExpandThreads) sparse_expand_kernel(SparseExpandArgs a) {
    __shared__ uint32_t s_words[kExpandTileWords];
    __shared__ uint32_t s_rank[kExpandTileWords];      // values before word j's first bit
    __shared__ uint32_t s_warp[kExpandThreads / 32];
    __shared__ uint32_t s_tile_total;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const uint32_t i = a.frame0 + blockIdx.x;
    const uint32_t s = i / a.fps, f = i - s * a.fps;
    const unsigned long long lo = a.off[i], rec_len = a.off[i + 1] - lo;
    const uint8_t *rec = a.data + lo;
    const uint32_t nw = sparse::bitmap_words(a.n_mb), vo = sparse::values_offset(a.n_mb);
    const uint32_t bg = *reinterpret_cast<const uint32_t *>(rec) & 0xffffu;
    const uint32_t *bits = reinterpret_cast<const uint32_t *>(rec + sparse::kHeaderBytes);
    const uint16_t *vals = reinterpret_cast<const uint16_t *>(rec + vo);
    const uint32_t n_vals = (uint32_t)((rec_len - vo) / 2);            // values the record holds (validated: rec_len >= vo)
    uint32_t *dst = reinterpret_cast<uint32_t *>(a.pool + ((size_t)s * a.fps_dev + a.lead + f) * (size_t)a.n_mb * 2);
    const uint32_t n_pairs = a.n_mb / 2;
    uint32_t carry = 0;                                                 // set bits in the tiles before
    for (uint32_t w0 = 0; w0 < nw; w0 += kExpandTileWords) {
        const uint32_t nt = min((uint32_t)kExpandTileWords, nw - w0);
        uint32_t c[4], sum = 0;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const uint32_t j = 4 * t + k;
            const uint32_t x = j < nt ? __ldg(bits + w0 + j) : 0u;
            s_words[j] = x;
            c[k] = sum;
            sum += __popc(x);
        }
        uint32_t incl = sum;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += y;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            const uint32_t v = lane < kExpandThreads / 32 ? s_warp[lane] : 0u;
            uint32_t x = v;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t y = __shfl_up_sync(0xffffffffu, x, d);
                if (lane >= d) x += y;
            }
            if (lane < kExpandThreads / 32) s_warp[lane] = x - v;
            if (lane == 31) s_tile_total = x;
        }
        __syncthreads();
        const uint32_t base = carry + s_warp[warp] + incl - sum;
#pragma unroll
        for (int k = 0; k < 4; k++) s_rank[4 * t + k] = base + c[k];
        __syncthreads();
        const uint32_t p0 = w0 * 16, p1 = min(n_pairs, (w0 + nt) * 16);
        for (uint32_t p = p0 + t; p < p1; p += kExpandThreads) {
            const uint32_t j = p - p0, word = j >> 4, sh = (j & 15) * 2;
            const uint32_t x = s_words[word];
            uint32_t r = s_rank[word] + __popc(x & ((1u << sh) - 1u));
            const uint32_t b = x >> sh;
            uint32_t v0 = bg, v1 = bg;
            if (b & 1u) { if (r < n_vals) v0 = __ldg(vals + r); r++; }
            if ((b & 2u) && r < n_vals) v1 = __ldg(vals + r);
            dst[p] = v0 | (v1 << 16);
        }
        carry += s_tile_total;
        __syncthreads();                                                // the next tile rewrites the shared arrays
    }
}

}  // namespace cova
