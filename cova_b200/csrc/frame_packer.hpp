// Host-side packer for the 2-byte input format (include/cova_b200.h, COVA_FLAG_INPUT_PACKED16).  Plain C++17, no CUDA.
//
// The decoder writes 4 bytes per macroblock - mb_weight, |mv_x|, |mv_y| and one stale byte
// (third_parties/FFmpeg/libavcodec/h264_mb.c:822-855) - and BlobNet's first operation is clip(x, 0, 6)
// (utils/model/preprocessing.py:5-8), so 9 bits per macroblock carry everything the network can see.  Packing on the
// host halves the bytes that cross PCIe, which is what bounds the end-to-end rate of the path (DESIGN.md, "Measurement").
//     u16 = min(b0, 6) | min(b1, 6) << 3 | min(b2, 6) << 6
// A packer owns its worker threads for its lifetime (a thread start per batch would cost as much as the packing).
// It also encodes the sparse format (sparse_format.hpp) straight from the quads: pack_sparse().
#pragma once
#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <new>
#include <thread>
#include <vector>

#if defined(__x86_64__)
#include <immintrin.h>
#endif

#include "sparse_format.hpp"

namespace cova {
namespace host {

inline void pack_scalar(const uint8_t *q, uint16_t *out, size_t n) {
    for (size_t i = 0; i < n; i++) {
        const uint32_t a = q[4 * i], b = q[4 * i + 1], c = q[4 * i + 2];
        out[i] = (uint16_t)((a < 6 ? a : 6) | ((b < 6 ? b : 6) << 3) | ((c < 6 ? c : 6) << 6));
    }
}

#if defined(__x86_64__)
// 16 macroblocks per iteration: byte-wise min with 6, then (b0 + 8*b1) and (64*b2 + 0*b3) by one multiply-add of adjacent
// bytes, their sum by one multiply-add of adjacent words, and a saturating pack 32 -> 16 bits.
__attribute__((target("avx2"))) inline void pack_avx2(const uint8_t *q, uint16_t *out, size_t n) {
    const __m256i six = _mm256_set1_epi8(6);
    const __m256i coef = _mm256_set1_epi32(0x00400801);       // bytes 1, 8, 64, 0
    const __m256i ones = _mm256_set1_epi16(1);
    size_t i = 0;
    for (; i + 16 <= n; i += 16) {
        __m256i a = _mm256_loadu_si256(reinterpret_cast<const __m256i *>(q + 4 * i));
        __m256i b = _mm256_loadu_si256(reinterpret_cast<const __m256i *>(q + 4 * i + 32));
        a = _mm256_madd_epi16(_mm256_maddubs_epi16(_mm256_min_epu8(a, six), coef), ones);
        b = _mm256_madd_epi16(_mm256_maddubs_epi16(_mm256_min_epu8(b, six), coef), ones);
        __m256i p = _mm256_permute4x64_epi64(_mm256_packus_epi32(a, b), 0xD8);   // packus interleaves the 128-bit lanes
        _mm256_storeu_si256(reinterpret_cast<__m256i *>(out + i), p);
    }
    pack_scalar(q + 4 * i, out + i, n - i);
}
inline bool have_avx2() { return __builtin_cpu_supports("avx2"); }
#else
inline bool have_avx2() { return false; }
#endif

inline void pack_range(const uint8_t *q, uint16_t *out, size_t n) {
#if defined(__x86_64__)
    if (have_avx2()) { pack_avx2(q, out, n); return; }
#endif
    pack_scalar(q, out, n);
}

#if defined(__x86_64__)
// The first n_groups whole groups of 16 macroblocks of a sparse record: one compare and movemask per group gives the
// group's 16 bitmap bits (two mask bits per u16 lane, gathered by pext); the differing values are appended lane by lane.
__attribute__((target("avx2,bmi2"))) inline uint32_t sparse_groups_avx2(const uint16_t *v, uint32_t n_groups, uint16_t bg,
                                                                       uint16_t *bits, uint16_t *vals) {
    const __m256i b = _mm256_set1_epi16((short)bg);
    uint32_t n = 0;
    for (uint32_t g = 0; g < n_groups; g++) {
        const __m256i x = _mm256_loadu_si256(reinterpret_cast<const __m256i *>(v + 16 * g));
        uint32_t m = ~(uint32_t)_mm256_movemask_epi8(_mm256_cmpeq_epi16(x, b));
        bits[g] = (uint16_t)_pext_u32(m, 0x55555555u);
        while (m) {
            const uint32_t j = (uint32_t)__builtin_ctz(m) >> 1;
            vals[n++] = v[16 * g + j];
            m &= ~(3u << (2 * j));
        }
    }
    return n;
}
inline bool have_avx2_bmi2() { return __builtin_cpu_supports("avx2") && __builtin_cpu_supports("bmi2"); }
#endif

// Sparse records (sparse_format.hpp) of one frame from its quads, read once: pack into `v` (n_mb u16), count the values
// (four interleaved histograms, so that runs of one value do not serialise on one counter), take the most frequent value
// (ties: the smallest) as the background, then write the bitmap and the differing values.  Returns the record size.
// `hist` holds 4 * kValueBins zeroed counters and is left zeroed.
inline size_t encode_sparse_frame(const uint8_t *q, uint32_t n_mb, uint16_t *v, uint32_t *hist, uint8_t *rec) {
    pack_range(q, v, n_mb);
    uint32_t i = 0;
    for (; i + 4 <= n_mb; i += 4) {
        hist[v[i]]++; hist[sparse::kValueBins + v[i + 1]]++;
        hist[2 * sparse::kValueBins + v[i + 2]]++; hist[3 * sparse::kValueBins + v[i + 3]]++;
    }
    for (; i < n_mb; i++) hist[v[i]]++;
    uint32_t bg = 0, best = 0;
    for (uint32_t b = 0; b < sparse::kValueBins; b++) {
        const uint32_t c = hist[b] + hist[sparse::kValueBins + b] + hist[2 * sparse::kValueBins + b] + hist[3 * sparse::kValueBins + b];
        hist[b] = hist[sparse::kValueBins + b] = hist[2 * sparse::kValueBins + b] = hist[3 * sparse::kValueBins + b] = 0;
        if (c > best) best = c, bg = b;
    }
    // bitmap as u16 halves: bit i % 16 of half i / 16 is bit i % 32 of word i / 32 (little-endian)
    const uint32_t nw = sparse::bitmap_words(n_mb);
    uint16_t *bits = reinterpret_cast<uint16_t *>(rec + sparse::kHeaderBytes);
    uint16_t *vals = reinterpret_cast<uint16_t *>(rec + sparse::values_offset(n_mb));
    uint32_t n = 0, g = 0;
#if defined(__x86_64__)
    if (have_avx2_bmi2()) { n = sparse_groups_avx2(v, n_mb / 16, (uint16_t)bg, bits, vals); g = n_mb / 16; }
#endif
    for (; g < 2 * nw; g++) {
        const uint32_t lo = 16 * g, hi = std::min(n_mb, lo + 16);
        uint32_t m = 0;
        for (uint32_t j = lo; j < hi; j++) {
            const uint32_t d = v[j] != bg;
            m |= d << (j - lo);
            vals[n] = v[j];
            n += d;
        }
        bits[g] = (uint16_t)m;
    }
    if (n & 1) vals[n] = 0;
    const uint32_t hdr[2] = {bg, n};
    memcpy(rec, hdr, sizeof(hdr));
    return (size_t)sparse::record_bytes(n_mb, n);
}

class Packer {
   public:
    explicit Packer(unsigned n_threads) {
        if (!n_threads) n_threads = std::thread::hardware_concurrency();
        if (!n_threads) n_threads = 1;
        if (n_threads > 64) n_threads = 64;
        n_ = n_threads;
        for (unsigned t = 1; t < n_; t++) workers_.emplace_back([this, t] { loop(t); });   // the caller is worker 0
    }
    ~Packer() {
        {
            std::lock_guard<std::mutex> lk(m_);
            stop_ = true;
            gen_++;
        }
        cv_.notify_all();
        for (auto &w : workers_) w.join();
    }
    unsigned threads() const { return n_; }
    void pack(const uint8_t *q, uint16_t *out, size_t n) {
        if (n_ == 1 || n < 65536) { pack_range(q, out, n); return; }
        // contiguous shares in multiples of 64 macroblocks (whole cache lines of output)
        const size_t per = ((n + n_ - 1) / n_ + 63) / 64 * 64;
        run(n_, [&](unsigned t) {
            const size_t lo = std::min(n, per * t), hi = std::min(n, lo + per);
            if (hi > lo) pack_range(q + 4 * lo, out + lo, hi - lo);
        });
    }
    // Sparse batch of n_frames frames of n_mb quads.  Every thread encodes a contiguous range of frames into its own
    // staging area; the threads' totals then give each range its place and the threads copy their records there.  So the
    // quads are read once, whatever the record sizes turn out to be.  Returns false (nothing written) when the batch
    // needs more than cap bytes; *len is the batch size either way.
    bool pack_sparse(const uint8_t *q, uint64_t n_frames, uint32_t n_mb, uint8_t *out, size_t cap, size_t *len) {
        const unsigned nt = (unsigned)std::min<uint64_t>(n_, std::max<uint64_t>(1, n_frames));
        const uint64_t per = (n_frames + nt - 1) / nt;
        const size_t max_rec = (size_t)sparse::max_record_bytes(n_mb);
        if (sp_.size() < nt) sp_.resize(nt);
        run(nt, [&](unsigned t) {
            SparseScratch &s = sp_[t];
            const uint64_t lo = std::min(n_frames, per * t), hi = std::min(n_frames, lo + per);
            s.used = 0;
            s.oom = false;
            try {           // an exception must not leave a worker thread
                if (s.v.size() < n_mb) s.v.resize(n_mb);
                if (s.hist.empty()) s.hist.assign(4 * sparse::kValueBins, 0);
                for (uint64_t f = lo; f < hi; f++) {
                    if (s.stage.size() < s.used + max_rec) s.stage.resize(std::max(s.used + max_rec, 2 * s.stage.size()));
                    s.used += encode_sparse_frame(q + 4 * (size_t)n_mb * f, n_mb, s.v.data(), s.hist.data(), s.stage.data() + s.used);
                }
            } catch (const std::bad_alloc &) {
                s.oom = true;
            }
        });
        for (unsigned t = 0; t < nt; t++)
            if (sp_[t].oom) throw std::bad_alloc();
        size_t total = 0;
        for (unsigned t = 0; t < nt; t++) sp_[t].at = total, total += sp_[t].used;
        *len = total;
        if (total > cap || (!out && total)) return false;
        run(nt, [&](unsigned t) {
            if (sp_[t].used) memcpy(out + sp_[t].at, sp_[t].stage.data(), sp_[t].used);
        });
        return true;
    }

   private:
    struct SparseScratch {
        std::vector<uint16_t> v;           // one frame, packed
        std::vector<uint32_t> hist;        // 4 x kValueBins counters, zero between frames
        std::vector<uint8_t> stage;        // this thread's records
        size_t used = 0, at = 0;           // bytes staged, their place in the batch
        bool oom = false;
    };
    // job(t) on threads 0 .. nt-1 (0 = the caller); returns when all are done
    void run(unsigned nt, const std::function<void(unsigned)> &job) {
        if (nt <= 1) { job(0); return; }
        {
            std::lock_guard<std::mutex> lk(m_);
            job_ = &job; active_ = nt; pending_ = n_ - 1;
            gen_++;
        }
        cv_.notify_all();
        job(0);
        std::unique_lock<std::mutex> lk(m_);
        done_.wait(lk, [this] { return pending_ == 0; });
    }
    void loop(unsigned t) {
        uint64_t seen = 0;
        for (;;) {
            const std::function<void(unsigned)> *job;
            bool mine;
            {
                std::unique_lock<std::mutex> lk(m_);
                cv_.wait(lk, [&] { return gen_ != seen; });
                seen = gen_;
                if (stop_) return;
                job = job_;
                mine = t < active_;
            }
            if (mine) (*job)(t);
            {
                std::lock_guard<std::mutex> lk(m_);
                if (--pending_ == 0) done_.notify_one();
            }
        }
    }
    unsigned n_ = 1;
    std::vector<std::thread> workers_;
    std::mutex m_;
    std::condition_variable cv_, done_;
    const std::function<void(unsigned)> *job_ = nullptr;
    unsigned active_ = 0, pending_ = 0;
    uint64_t gen_ = 0;
    bool stop_ = false;
    std::vector<SparseScratch> sp_;
};

}  // namespace host
}  // namespace cova
