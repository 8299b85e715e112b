// The sparse input format (include/cova_b200.h, cova_pipeline_submit_sparse): the one place that knows its layout.
// The host encoder (frame_packer.hpp), the submit path's validation walk (cova_abi.cu) and the expansion kernel
// (sparse_expand.cuh) all take the constants and the record arithmetic from here.
//
// One frame = one record, 4-byte aligned, little-endian, n_mb = w_mb * h_mb macroblocks in raster order:
//   u32 background      bits 0-8 a packed16 value, bits 9-31 zero
//   u32 count           macroblocks whose value is not the background
//   u32 bitmap[ceil(n_mb / 32)]   bit i % 32 of word i / 32 set = macroblock i differs; bits at or past n_mb are zero
//   u16 values[count]   the differing macroblocks' packed16 values in raster order, zero-padded to a multiple of 4 bytes
// A batch is the records of n_streams x frames_per_stream frames, stream-major and time-minor, without gaps.
#pragma once
#include <stddef.h>
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define COVA_SPARSE_HD __host__ __device__ __forceinline__ constexpr
#else
#define COVA_SPARSE_HD inline constexpr
#endif

namespace cova {
namespace sparse {

constexpr uint32_t kHeaderBytes = 8;         // background + count
constexpr uint32_t kValueBits = 9;           // a packed16 value: three 3-bit fields
constexpr uint32_t kValueBins = 1u << kValueBits;

COVA_SPARSE_HD uint32_t bitmap_words(uint32_t n_mb) { return (n_mb + 31) / 32; }
// byte offset of the values inside a record
COVA_SPARSE_HD uint32_t values_offset(uint32_t n_mb) { return kHeaderBytes + 4 * bitmap_words(n_mb); }
COVA_SPARSE_HD uint64_t record_bytes(uint32_t n_mb, uint32_t count) {
    return (uint64_t)values_offset(n_mb) + 4 * (((uint64_t)count + 1) / 2);
}
COVA_SPARSE_HD uint64_t max_record_bytes(uint32_t n_mb) { return record_bytes(n_mb, n_mb); }

inline uint32_t load_u32(const uint8_t *p) {
    uint32_t v;
    memcpy(&v, p, 4);       // the caller's buffer need not be 4-byte aligned
    return v;
}

// Walks a batch of n_frames records of n_mb macroblocks and checks every rule of the format: reserved background bits,
// count == popcount(bitmap), no bit at or past n_mb, zero padding, and records that end exactly at len.  On success
// off[0 .. n_frames] holds the byte offset of every record plus the total (off[n_frames] == len) and the function
// returns nullptr; otherwise it returns what is wrong, and *bad_frame (if given) is the frame.
inline const char *validate_batch(const uint8_t *data, size_t len, uint64_t n_frames, uint32_t n_mb, uint64_t *off,
                                  uint64_t *bad_frame = nullptr) {
    const uint32_t nw = bitmap_words(n_mb), tail = n_mb % 32;
    const uint32_t tail_mask = tail ? ~((1u << tail) - 1) : 0u;       // bits past n_mb in the last word
    uint64_t pos = 0;
    for (uint64_t f = 0; f < n_frames; f++) {
        if (bad_frame) *bad_frame = f;
        off[f] = pos;
        if (len - pos < values_offset(n_mb)) return "batch ends inside a record's header or bitmap";
        const uint8_t *r = data + pos;
        const uint32_t bg = load_u32(r), count = load_u32(r + 4);
        if (bg >> kValueBits) return "background has bits set above bit 8";
        if (count > n_mb) return "count exceeds the number of macroblocks";
        uint32_t pop = 0;
        for (uint32_t w = 0; w < nw; w++) pop += (uint32_t)__builtin_popcount(load_u32(r + kHeaderBytes + 4 * w));
        if (tail && (load_u32(r + kHeaderBytes + 4 * (nw - 1)) & tail_mask)) return "bitmap has a bit at or past n_mb";
        if (pop != count) return "count differs from the number of bits set in the bitmap";
        const uint64_t size = record_bytes(n_mb, count);
        if (len - pos < size) return "batch ends inside a record's values";
        if (count & 1) {
            uint16_t pad;
            memcpy(&pad, r + size - 2, 2);
            if (pad) return "record padding is not zero";
        }
        pos += size;
    }
    off[n_frames] = pos;
    if (bad_frame) *bad_frame = n_frames;
    if (pos != len) return "data_len is not the sum of the record sizes";
    return nullptr;
}

}  // namespace sparse
}  // namespace cova
