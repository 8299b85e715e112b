// BlobNet encoder block 1, fused: first conv (+ bias, ReLU, BatchNorm, 2x2 max-pool) once per FRAME and
// PointWiseTN once per WINDOW in ONE tcgen05 kernel, sm_100a.
//
// The first convolution has kernel depth 1 (reference utils/model/encoder.py:33-44), so the pooled activation of
// a frame is shared by the four windows the frame appears in; PointWiseTN (utils/model/pointwise.py:10-26) then
// mixes the four frames of a window per (pixel, channel).  A CTA therefore walks ONE chain through time for a
// fixed pair of 128-position tiles: every step brings in the two input strips of the next frame (cp.async.bulk),
// runs the 12 MMAs of the frame-level conv (same operand layout as tc::issue_tile<ENCF>), and the epilogue thread
// that owns (position, channel block) keeps the pooled fp16 activations of the three previous frames in REGISTERS -
// so the window's PointWiseTN input never touches shared memory or HBM.  Per step the kernel writes the window's
// four time planes of X1 (next encoder input) and the t = 0 skip row of the decoder concat buffer; no per-frame pooled
// tensor goes through HBM (it would be 0.3 GB written + 0.3 GB read per 8192 windows at 720p).
//
// Work item = (chain, tile pair, segment of frames); a segment after the first re-computes 3 warm-up frames.
// Warp roles as in blobnet_tc.cuh: warp 0 producer, warp 1 TMEM owner + MMA issuer, 16 epilogue warps
// (TMEM lane quarter x channel block x tile of the pair).
#pragma once
#include <type_traits>

#include "blobnet_tc.cuh"

namespace cova {
namespace tc1 {

using tc::LayerParams;
using C1 = tc::Cfg<tc::MODE_ENCF, 1, 16, 2, 1, 16>;   // two 128-position tiles per strip, N = 4 phases x 16 channels

constexpr int kMaxStage1 = 8;
constexpr int kSlots1 = 4;                 // frame-steps of accumulators in TMEM: 2 tiles x 64 columns each
constexpr int kEpiWarps1 = 16;
constexpr int kThreads1 = 64 + 32 * kEpiWarps1;
constexpr int kPairRows = 2 * kTileM;

struct Enc1Extra {
    int n_chains, fps, gamma;               // chains of this chunk, frame stride of a chain in the pool, sub-sampling
    // per chain of the chunk: (x = index of the newest frame of its first window, y = index of that window in the chunk,
    // z = end: the chain's frames are [0, end), w = frames of the chunk's chains before it, sum of their ends).  Chains of a
    // staggered batch differ in x and y, chains of a ragged batch in z (cova_abi.cu, set_batch_shape); a chain's window
    // n + k has its newest frame at x + k * gamma, with the chain's own gamma when `gam` is given
    const int4 *tab;
    const int *gam;                         // per chain of the chunk: its gamma (nullptr: every chain has `gamma`)
    int ntp;                                // tile pairs per frame
    int n_items;                            // (chain, tile pair) items = n_chains * ntp, item (c, j) is end_c frame steps long
    int full_items;                         // items handed out whole, round-robin: a multiple of the grid size
    int total, span;                        // frame steps in all items / consecutive steps of the REMAINING items per CTA
    int g0;                                 // frame steps of the whole items: where the remaining items' steps begin
};

struct SmemPlan1 {
    uint32_t w_off, stage_off, stage_bytes, epi_off, bar_off, total;
};
__host__ __device__ inline SmemPlan1 plan_smem1(int Ls, int n_stage, int w_bytes) {
    SmemPlan1 s;
    s.w_off = 0;
    s.stage_off = (uint32_t)((w_bytes + 127) / 128 * 128);
    s.stage_bytes = (uint32_t)(2 * Ls * 16);
    s.epi_off = s.stage_off + (uint32_t)n_stage * s.stage_bytes;
    s.bar_off = s.epi_off + 3 * 16 * 4;
    s.total = s.bar_off + 8 * (2 * kMaxStage1 + 2 * kSlots1 + 1) + 16;
    return s;
}

struct Item {
    int chain, jp, i0, i1, start;
};
// Work partition.  An item = one (chain, tile pair) walked through the chain's end_c frames; consecutive items are the
// tile pairs of one chain, and handing them out round-robin keeps the CTAs that run concurrently on the same few chains (the
// four tile pairs of a frame read and write neighbouring DRAM pages - a flat split of the whole step sequence into 148
// spans balanced better and ran 12 % slower).  Only the items left over after the last whole round (items mod grid size)
// are cut: their steps form one sequence that is split evenly, and a CTA whose piece starts inside an item re-computes the
// kT - 1 warm-up frames the register ring needs.  At the benchmark size: 3 whole items + a 31-step piece = 235 steps per
// CTA for 232 of work (whole items only: 268; two fixed segments per item: 259).  Item (c, j) starts at step
// ntp * tab[c].w + j * tab[c].z of the sequence, so a piece finds its item by a binary search over the chunk's chains;
// with equal ends this is exactly the division by the chain length it replaces.
struct WorkIter {
    int item, g, g1;
};
__device__ __forceinline__ WorkIter work_begin(const Enc1Extra &ex, int cta) {
    WorkIter wi;
    wi.item = cta;
    wi.g = ex.g0 + cta * ex.span;
    wi.g1 = min(ex.total, wi.g + ex.span);
    return wi;
}
__device__ __forceinline__ bool work_next(const Enc1Extra &ex, int n_cta, WorkIter &wi, Item &it) {
    if (wi.item < ex.full_items) {                                   // a whole item
        it.jp = wi.item % ex.ntp; it.chain = wi.item / ex.ntp; it.i0 = 0; it.i1 = __ldg(&ex.tab[it.chain].z); it.start = 0;
        wi.item += n_cta;
        return true;
    }
    if (wi.g >= wi.g1) return false;
    int lo = 0, hi = ex.n_chains - 1;                                 // the last chain that starts at or before step g
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (ex.ntp * __ldg(&ex.tab[mid].w) <= wi.g) lo = mid; else hi = mid - 1;
    }
    const int end = __ldg(&ex.tab[lo].z), r = wi.g - ex.ntp * __ldg(&ex.tab[lo].w);
    const int jp = r / end, i = r - jp * end;                         // a piece of a left-over item
    const int len = min(end - i, wi.g1 - wi.g);
    it.jp = jp; it.chain = lo; it.i0 = i; it.i1 = i + len; it.start = max(0, i - (kT - 1));
    wi.g += len;
    return true;
}

__device__ __forceinline__ void stg256(uint4 *dst, const uint4 &a, const uint4 &b) {
    asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                 ::"l"(dst), "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w), "r"(b.x), "r"(b.y), "r"(b.z), "r"(b.w) : "memory");
}

__global__ void __launch_bounds__(kThreads1, 1) enc1_fused_kernel(const __grid_constant__ LayerParams p, const __grid_constant__ Enc1Extra ex) {
    extern __shared__ __align__(1024) unsigned char smem[];
    const SmemPlan1 sp = plan_smem1(p.Ls, p.n_stage, p.w_bytes);
    const uint32_t smem_base = tc::smem_u32(smem);
    float *epi = reinterpret_cast<float *>(smem + sp.epi_off);
    const uint32_t bar0 = smem_base + sp.bar_off;
    const uint32_t full0 = bar0, empty0 = bar0 + 8u * kMaxStage1, tfull0 = bar0 + 8u * 2 * kMaxStage1,
                   tempty0 = tfull0 + 8u * kSlots1, w_bar = tempty0 + 8u * kSlots1;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + sp.bar_off + 8 * (2 * kMaxStage1 + 2 * kSlots1 + 1));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int cta = (int)blockIdx.x, n_cta = (int)gridDim.x;
    pdl_launch_dependents();

    for (int i = threadIdx.x; i < 3 * 16; i += kThreads1) epi[i] = p.epi[i];     // bias | scale | shift
    if (threadIdx.x == 0) {
        for (int s = 0; s < kMaxStage1; s++) { tc::mbar_init(full0 + 8u * s, 1); tc::mbar_init(empty0 + 8u * s, 1); }
        for (int s = 0; s < kSlots1; s++) { tc::mbar_init(tfull0 + 8u * s, 1); tc::mbar_init(tempty0 + 8u * s, kEpiWarps1); }
        tc::mbar_init(w_bar, 1);
        tc::fence_barrier_init();
    }
    if (warp == 1) {
        tc::tmem_alloc(tc::smem_u32(tmem_slot), 512);
        tc::tmem_relinquish();
    }
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (warp == 0 && tc::elect_one()) {          // weights do not depend on the preceding kernel: fetch them before the wait
        tc::mbar_expect_tx(w_bar, (uint32_t)p.w_bytes);
        tc::bulk_g2s(smem_base + sp.w_off, p.wpack, (uint32_t)p.w_bytes, w_bar);
    }
    __syncwarp();
    pdl_wait();

    if (warp == 0) {
        // ===== producer: the two row-parity strips of one frame per step =====
        if (tc::elect_one()) {
            uint32_t it = 0;
            Item w;
            for (WorkIter wi = work_begin(ex, cta); work_next(ex, n_cta, wi, w);) {
                for (int i = w.start; i < w.i1; i++, it++) {
                    const int s = (int)(it % (uint32_t)p.n_stage);
                    tc::mbar_wait(empty0 + 8u * s, ((it / (uint32_t)p.n_stage) & 1u) ^ 1u, p.watchdog, 1u);
                    tc::mbar_expect_tx(full0 + 8u * s, sp.stage_bytes);
                    const uint32_t dst0 = smem_base + sp.stage_off + (uint32_t)s * sp.stage_bytes;
                    const long long pos0 = p.gin.guard + ((long long)w.chain * ex.fps + i) * p.gin.S + w.jp * kPairRows - p.gin.halo;
#pragma unroll
                    for (int pl = 0; pl < 2; pl++)
                        tc::bulk_g2s(dst0 + (uint32_t)(pl * p.Ls) * 16u, p.in + geom_row(p.gin, 0, pl * 2, pos0), (uint32_t)p.Ls * 16u,
                                     full0 + 8u * s);
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer (one elected thread) =====
        if (tc::elect_one()) {
            constexpr uint32_t idesc = tc::make_idesc(C1::BLOCK_N);
            tc::mbar_wait(w_bar, 0u, p.watchdog, 2u);
            uint32_t it = 0;
            Item w;
            for (WorkIter wi = work_begin(ex, cta); work_next(ex, n_cta, wi, w);) {
                for (int i = w.start; i < w.i1; i++, it++) {
                    const int s = (int)(it % (uint32_t)p.n_stage);
                    tc::mbar_wait(full0 + 8u * s, (it / (uint32_t)p.n_stage) & 1u, p.watchdog, 3u);
                    const int slot = (int)(it % (uint32_t)kSlots1);
                    tc::mbar_wait(tempty0 + 8u * slot, ((it / (uint32_t)kSlots1) & 1u) ^ 1u, p.watchdog, 4u);
                    tc::tc_fence_after();
                    const uint32_t stage_addr = smem_base + sp.stage_off + (uint32_t)s * sp.stage_bytes;
                    if (!(p.dbg & 1)) {
#pragma unroll
                        for (int j = 0; j < 2; j++)
                            tc::issue_tile<C1>(p, stage_addr, smem_base + sp.w_off, tmem_base + (uint32_t)(slot * 128 + j * 64), j, 0, idesc);
                    }
                    tc::umma_commit(tfull0 + 8u * slot);
                    tc::umma_commit(empty0 + 8u * s);
                }
            }
        }
    } else {
        // ===== epilogue: TMEM -> pool/ReLU/BN -> register ring of 4 frames -> PointWiseTN -> X1 + skip =====
        const int q = warp & 3, gidx = (warp - 2) >> 2;
        const int cg = gidx & 1, tg = gidx >> 1;              // channel block, tile of the pair
        const Geom &gi = p.gin;
        const float4 *c4 = reinterpret_cast<const float4 *>(epi);
        uint32_t it = 0;
        Item w;
        for (WorkIter wi = work_begin(ex, cta); work_next(ex, n_cta, wi, w);) {
            const int r = w.jp * kPairRows + tg * kTileM + q * 32 + lane;
            const int y2 = r / gi.P, x2 = r - y2 * gi.P;
            const bool valid = r < gi.S && y2 < (gi.H >> 1) && x2 < (gi.W >> 1);
            const bool warp_live = __any_sync(0xffffffffu, valid);       // warps that only cover padding rows skip the arithmetic
            // (first, window 0) of the chain: one load per item; window 0 goes into the base addresses, only first stays live
            const int2 cw = *reinterpret_cast<const int2 *>(&ex.tab[w.chain]);
            const int Y = y2 + (gi.H & 1), X = x2 + (gi.W & 1);          // zero-pad top / left when odd (encoder.py:68-76)
            const int pho = ((Y & 1) << 1) | (X & 1);
            const long long base_o = (long long)(cg * 4 + pho) * p.gout.Lp + p.gout.guard + ((long long)(Y >> 1) * p.gout.P + (X >> 1)) * kT +
                                   (long long)cw.y * p.gout.S * kT;
            const long long base_s = (long long)((p.out2_cb + cg) * 4 + pho) * p.gout2.Lp + p.gout2.guard + (long long)(Y >> 1) * p.gout2.P + (X >> 1) +
                                   (long long)cw.y * p.gout2.S;
            const int first = cw.x;
            const int gam = ex.gam ? __ldg(&ex.gam[w.chain]) : ex.gamma;
            // Ring of the last four pooled frames: ring[s][k] = channel pair (2k, 2k+1) of the frame whose index is s mod 4,
            // as fp32 values already rounded to fp16 (the pooled activation is an fp16 tensor).  The frame loop is
            // unrolled four times over the ring phase R, so "frame i - t" is the compile-time slot (R - t) & 3: no
            // rotation moves, and one fp16 round trip per frame instead of one conversion per frame and window.
            float2 ring[4][4];
#pragma unroll
            for (int sl = 0; sl < 4; sl++)
#pragma unroll
                for (int k = 0; k < 4; k++) ring[sl][k] = make_float2(0.f, 0.f);
            auto step = [&](auto R_, int i) {
                constexpr int R = decltype(R_)::value;
                const int slot = (int)(it % (uint32_t)kSlots1);
                tc::mbar_wait(tfull0 + 8u * slot, (it / (uint32_t)kSlots1) & 1u, p.watchdog, 5u);
                tc::tc_fence_after();
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(slot * 128 + tg * 64 + cg * 8);
                uint32_t v[4][8];
#pragma unroll
                for (int ph = 0; ph < 4; ph++) tc::tmem_ld8(taddr + (uint32_t)(ph * 16), v[ph]);
                tc::tmem_wait_ld();
                tc::tc_fence_before();
                __syncwarp();
                if (lane == 0) tc::mbar_arrive(tempty0 + 8u * slot);       // accumulators are in registers: release the slot early
                it++;
                if ((p.dbg & 2) || !warp_live) return;
                {
                    float bs[8], sc[8], sh[8], ext[8];
                    *reinterpret_cast<float4 *>(bs) = c4[cg * 2]; *reinterpret_cast<float4 *>(bs + 4) = c4[cg * 2 + 1];
                    *reinterpret_cast<float4 *>(sc) = c4[4 + cg * 2]; *reinterpret_cast<float4 *>(sc + 4) = c4[4 + cg * 2 + 1];
                    *reinterpret_cast<float4 *>(sh) = c4[8 + cg * 2]; *reinterpret_cast<float4 *>(sh + 4) = c4[8 + cg * 2 + 1];
#pragma unroll
                    for (int j = 0; j < 8; j++) {
                        // MaxPool(BN(ReLU(x + b))) = BN(ReLU(max x + b)) for a non-negative BN scale, of min x otherwise
                        // (see tc::epilogue_enc_pool): one activation per channel instead of four
                        const float a0 = __uint_as_float(v[0][j]), a1 = __uint_as_float(v[1][j]);
                        const float a2 = __uint_as_float(v[2][j]), a3 = __uint_as_float(v[3][j]);
                        ext[j] = fmaxf(fmax3(a0, a1, a2), a3);
                        if (!p.bn_nonneg) {
                            const float lo = fminf(fminf(a0, a1), fminf(a2, a3));
                            ext[j] = sc[j] >= 0.f ? ext[j] : lo;
                        }
                    }
#pragma unroll
                    for (int k = 0; k < 4; k++) {                        // bias -> ReLU -> BatchNorm on channel pairs (packed fp32)
                        const float2 o = ffma2(relu2(fadd2(make_float2(ext[2 * k], ext[2 * k + 1]), make_float2(bs[2 * k], bs[2 * k + 1]))),
                                               make_float2(sc[2 * k], sc[2 * k + 1]), make_float2(sh[2 * k], sh[2 * k + 1]));
                        ring[R][k] = __half22float2(__floats2half2_rn(o.x, o.y));   // the pooled activation is an fp16 tensor
                    }
                }
                const int rel = i - first;
                const bool emit = i >= w.i0 && rel >= 0 && (gam == 1 || rel % gam == 0);   // warp-uniform
                if (emit && valid) {
                    const long long n = gam == 1 ? rel : rel / gam;                     // window of the chain
                    uint32_t o32[4][4];
#pragma unroll
                    for (int k = 0; k < 4; k++) {                        // channel pair (2k, 2k+1) in the two packed fp32 lanes
                        const float2 x[4] = {ring[R][k], ring[(R + 3) & 3][k], ring[(R + 2) & 3][k], ring[(R + 1) & 3][k]};   // frames i, i-1, i-2, i-3
                        float2 h1[4];
#pragma unroll
                        for (int m = 0; m < 4; m++) {                    // h1[m] = relu(sum_t x[t] W1[t][m])  (pointwise.py:18-21)
                            float2 h = fmul2(x[0], bc2(p.tn_w1[m]));
#pragma unroll
                            for (int t = 1; t < 4; t++) h = ffma2(x[t], bc2(p.tn_w1[t * 4 + m]), h);
                            h1[m] = relu2(h);
                        }
#pragma unroll
                        for (int to = 0; to < 4; to++) {                 // relu(x + relu(h2)) = max(x + h2, x, 0)  (pointwise.py:22-26)
                            float2 h = x[to];
#pragma unroll
                            for (int m = 0; m < 4; m++) h = ffma2(h1[m], bc2(p.tn_w2[m * 4 + to]), h);
                            o32[to][k] = tc::pack_half2(fmax3(h.x, x[to].x, 0.f), fmax3(h.y, x[to].y, 0.f));
                        }
                    }
                    uint4 *dst = p.out + (base_o + n * (long long)p.gout.S * kT);   // rows t = 0..3 are consecutive: 64 bytes
                    const uint4 t0 = make_uint4(o32[0][0], o32[0][1], o32[0][2], o32[0][3]);
                    stg256(dst, t0, make_uint4(o32[1][0], o32[1][1], o32[1][2], o32[1][3]));
                    stg256(dst + 2, make_uint4(o32[2][0], o32[2][1], o32[2][2], o32[2][3]), make_uint4(o32[3][0], o32[3][1], o32[3][2], o32[3][3]));
                    p.out2[base_s + n * (long long)p.gout2.S] = t0;
                }
            };
            for (int i = w.start; i < w.i1;) {
                step(std::integral_constant<int, 0>{}, i); if (++i >= w.i1) break;
                step(std::integral_constant<int, 1>{}, i); if (++i >= w.i1) break;
                step(std::integral_constant<int, 2>{}, i); if (++i >= w.i1) break;
                step(std::integral_constant<int, 3>{}, i); ++i;
            }
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 1) tc::tmem_dealloc(tmem_base, 512);
}

// as tc::plan / tc::launch: the ring depth is the only choice (as deep as fits, at least 2).  htab: the host copy of the
// chunk's chain table (ends and their prefix sums); nullptr = every chain ends at ex.fps.
inline bool plan_enc1(LayerParams &p, Enc1Extra &ex, const int4 *htab, int n_sms, tc::Grid &g) {
    p.Ls = kPairRows + 2 * p.gin.halo;
    if (p.gin.P >= 16384) return false;                                            // LBO field: 14 bits of 16-byte units
    ex.ntp = (p.gin.S + kPairRows - 1) / kPairRows;
    const long long F = (long long)ex.n_chains * ex.fps;
    if (F < 1 || F * p.gin.S >= (1ll << 31)) return false;
    if (p.gin.guard + (F - 1) * p.gin.S + (long long)ex.ntp * kPairRows + p.gin.halo > p.gin.Lp) return false;   // strip over-read stays inside the plane
    if ((p.gout.Lp & 1) || (p.gout.guard & 1)) return false;                       // 256-bit stores need 32-byte aligned rows
    p.w_bytes = C1::BLOCKS * C1::BLOCK_N * 32;
    if (F * ex.ntp >= (1ll << 31)) return false;
    // frames that exist: the chains' ends (every end is at most the stride, so the bounds above hold)
    const long long frames = htab ? (long long)htab[ex.n_chains - 1].w + htab[ex.n_chains - 1].z : F;
    ex.total = (int)(frames * ex.ntp);
    ex.n_items = ex.n_chains * ex.ntp;
    const int ctas = std::max(1, std::min(n_sms, ex.total));
    ex.full_items = (ex.n_items / ctas) * ctas;
    const int c = ex.full_items / ex.ntp, j = ex.full_items - c * ex.ntp;           // the first left-over item
    ex.g0 = htab ? (c < ex.n_chains ? ex.ntp * htab[c].w + j * htab[c].z : ex.total) : ex.full_items * ex.fps;
    ex.span = (ex.total - ex.g0 + ctas - 1) / ctas;
    for (p.n_stage = kMaxStage1; p.n_stage >= 2; p.n_stage--)
        if (plan_smem1(p.Ls, p.n_stage, p.w_bytes).total <= (uint32_t)tc::kSmemLimit) break;
    if (p.n_stage < 2) return false;
    // more than half of the SM's shared memory: one CTA per SM (the CTA allocates all 512 TMEM columns)
    g.smem = std::max<uint32_t>(plan_smem1(p.Ls, p.n_stage, p.w_bytes).total, 120u * 1024u);
    g.ctas = ctas;
    return true;
}

inline cudaError_t launch_enc1(const LayerParams &p, const Enc1Extra &ex, const tc::Grid &g, cudaStream_t st) {
    cudaError_t err = cudaFuncSetAttribute(enc1_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::kSmemLimit);   // see tc::launch
    if (err != cudaSuccess) return err;
    return launch_pdl(enc1_fused_kernel, dim3((unsigned)g.ctas), dim3(kThreads1), g.smem, st, !(p.dbg & kDbgNoPdl), p, ex);
}

}  // namespace tc1
}  // namespace cova
