// BlobNet layers as tcgen05 / TMEM implicit GEMMs ("shift-GEMM"), sm_100a.
//
// Every layer is   D[pos, n] = sum_{tap} sum_{c} A[pos + shift(tap), c] * W[tap][c][n]
// over 128-position tiles of the phase-plane layout (common.cuh): because a spatial shift is a
// constant row offset there, the A operand of every tap is just a different START ADDRESS into one
// shared-memory strip that a bulk-async copy (cp.async.bulk, SASS UBLKCP) brought in once - no im2col,
// no re-load per tap.  Operands use the canonical K-major no-swizzle core-matrix layout
// (8 rows x 16 bytes; SBO = 128 B between 8-row groups, LBO = distance between the two 8-channel
// halves of a K=16 step).  Four accumulators per tile live in TMEM, one per output phase:
//   encoder: the four conv outputs a 2x2 max-pool window needs -> bias+ReLU+BN+max are done in
//            registers straight out of TMEM, then PointWiseTN across the 4 frames of a window, which
//            sit in 4 adjacent TMEM lanes (quad shuffles);
//   decoder: the four input phases of a stride-2 transposed conv; N = 4 output parities x Cout.
// Warp roles: warp 0 = bulk-copy producer, warp 1 = TMEM owner + single-thread MMA issuer,
// warps 2..5 = epilogue (TMEM lane quarter = warp_id % 4).  Persistent CTAs, one per SM.
//
// Reference for the math: utils/model/encoder.py:33-76, pointwise.py:10-26, decoder.py:5-64,106-134.
#pragma once
#include "common.cuh"
#include "weights_pack.cuh"

namespace cova {
namespace tc {

constexpr int MODE_ENC = 0, MODE_DEC = 1, MODE_HEAD = 2, MODE_ENCF = 3;   // ENCF: first conv, per FRAME (MMAs of blobnet_enc1.cuh)
constexpr int kMaxStage = 4;
constexpr int kEpiWarps = 16;                 // 4 groups of 4 warps (one per TMEM lane quarter)
constexpr int kThreads = 64 + 32 * kEpiWarps;
constexpr int kDecScratchRows = 68;            // decoder epilogue: 16-byte rows of transposition scratch per epilogue warp (epilogue_dec)
constexpr int kPairPitch = 72;                 // floats per channel-PAIR row of the quad-exchange scratch: 32 lanes x 2 channels + 8
constexpr int kScratchPitch = kPairPitch / 2;  // per channel: the scratch of a warp is 8 channels x kScratchPitch floats

struct LayerParams {
    const uint4 *in; Geom gin;
    uint4 *out; Geom gout;             // ENC: Tn=4 output (may be null); DEC: next concat buffer
    uint4 *out2; Geom gout2;           // ENC: Tn=1 copy of t=0 (skip / dec0 input)
    int out2_cb;                       // ENC: channel-block offset of the skip inside the concat buffer
    const uint4 *wpack;                // B blocks (fp16), per N-half contiguous
    const float *epi;                  // epilogue constants
    float tn_w1[16], tn_w2[16];        // ENC: PointWiseTN matrices [T_in][T_out]
    int N;                             // windows in this batch
    int n_tiles, n_groups;             // 128-position tiles / groups of TPS tiles
    int Ls;                            // strip rows per (cb, phase) in one stage = TPS*128 + 2*halo
    int n_stage;                       // ring depth actually used (<= kMaxStage)
    int w_bytes;                       // bytes of B blocks per N-half
    int nsplit;                        // DEC: N split over CTAs (dec0: 2)
    int Ht, Wt, crop_t, crop_l;        // DEC/HEAD: target extent and crop
    uint8_t *mask; float *logits;      // HEAD
    const float *seg; float seg_tau;   // HEAD: pixel is foreground when logit > (seg ? seg[n] : seg_tau), n = window of the chunk
    unsigned int *watchdog;            // set to a non-zero code if a barrier wait times out
    int bn_nonneg;                     // ENC: every BatchNorm scale of the layer is >= 0 (skips the min-pool path)
    int dbg;                           // experiments only: bit0 = skip the MMAs, bit1 = skip the epilogue math (results are garbage)
    FastDiv divS, divP;                // exact division by gin.S and gin.P (epilogue position decode)
    int psplit;                        // DEC with 512 accumulator columns per tile: two half-tiles of two input phases each (see Cfg::CAN_SPLIT)
};

// ------------------------------------------------------------------------------------------------ PTX
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
// Bounded wait: a descriptor / protocol bug must fail the launch, never hang the GPU box.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, unsigned int *watchdog, unsigned int code) {
    for (uint32_t spin = 0; !mbar_try(bar, parity); ++spin) {
        if (spin > (1u << 22)) {
            if (watchdog) atomicExch(watchdog, code);
            __trap();
        }
    }
}
// One elected lane of a fully converged warp.  Unlike `lane == 0`, elect.sync tells ptxas that exactly one
// thread runs the guarded code, so descriptors can go to uniform registers without a waterfall loop.
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred P1;\n\t"
        "elect.sync _|P1, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, P1;\n\t}"
        : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() { asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, uint32_t (&r)[4]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(taddr));
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// The same wait, carrying a data dependence on the registers an EARLIER tcgen05.ld filled: in a double-buffered epilogue
// the consumer of r[] is separated from its load by another load, and nothing else would keep the compiler from
// scheduling the arithmetic on r[] above the wait.
__device__ __forceinline__ void tmem_wait_ld_dep(uint32_t (&r)[8]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7])::"memory");
}

// shared-memory matrix descriptor, K-major, no swizzle, sm_100 version bit (cute SmemDescriptor)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}
// instruction descriptor: fp16 x fp16 -> fp32, A and B K-major, M = 128
__host__ __device__ constexpr uint32_t make_idesc(int n) { return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((128u >> 4) << 24); }

__host__ __device__ constexpr int fdiv2(int v) { return v >= 0 ? v / 2 : -((1 - v) / 2); }
__host__ __device__ constexpr int pow2_cols(int c) { return c <= 32 ? 32 : c <= 64 ? 64 : c <= 128 ? 128 : c <= 256 ? 256 : 512; }

template <int MODE_, int CIN_CB_, int NCOLS_, int TPS_, int KCH_, int COUT_>
struct Cfg {
    static constexpr int MODE = MODE_, CIN_CB = CIN_CB_, NCOLS = NCOLS_, TPS = TPS_, KCH = KCH_, COUT = COUT_;
    static constexpr bool ENCF = MODE == MODE_ENCF;
    static constexpr int NKC = CIN_CB / KCH;
    static constexpr int NPLANE = ENCF ? 2 : 4;                          // phase planes staged per channel block
    static constexpr int COLS_TILE = 4 * NCOLS;
    static constexpr int NSLOT = (512 / COLS_TILE) < 8 ? (512 / COLS_TILE) : 8;
    // the 4 epilogue warp groups split a tile by channel group (CG) and, when a tile has fewer than 4
    // channel blocks, also take alternate tiles (TG); decoder / head groups take one input phase each
    static constexpr int CG = (MODE_ == MODE_ENC || ENCF) ? ((COUT_ / 8) < 4 ? (COUT_ / 8) : 4) : 4;
    static constexpr int TG = 4 / CG;
    static constexpr int TMEM_COLS = pow2_cols(NSLOT * COLS_TILE);
    static constexpr int NTAP = MODE == MODE_ENC ? 9 : 4;
    static constexpr int KP = ENCF ? 1 : KCH / 2;                        // K=16 steps per tap inside a stage
    // Encoder blocks with Cout <= 64: the two column phases of a pooling window that read the same input column are
    // fed by ONE MMA of N = 2*Cout (weights_pack.cuh, pack_encoder): per row phase 3 x {N, 2N, 2N, N} MMAs per K step
    // instead of 18 of N.  An MMA with the A operand in shared memory costs ~43 + N/2 cycles (section 3.1 of DESIGN.md),
    // so halving the count of the N = 64 MMAs of block 3 saves a fifth of its tensor time.
    static constexpr bool PAIR = MODE == MODE_ENC && NCOLS <= 64;
    // Transposed convs whose doubled weights still fit shared memory (dec2, head) pair their column phases the same way:
    // 3 MMAs {2N, N, N} per (row phase, row tap, K step) instead of 4 of N (weights_pack.cuh, pack_decoder).
    static constexpr bool PAIRD = (MODE == MODE_DEC || MODE == MODE_HEAD) && NCOLS * CIN_CB <= 512;
    static constexpr int BLOCKS = ENCF ? 6 : (PAIR ? 18 * (CIN_CB / 2) : (PAIRD ? 2 : 1) * NTAP * (CIN_CB / 2));   // B blocks (of BLOCK_N rows) per N-half
    static constexpr int BLOCK_N = ENCF ? 4 * NCOLS : NCOLS;             // rows of one B block (= N of one MMA)
    // A decoder tile whose four phase accumulators fill all 512 TMEM columns (dec0, dec1) cannot be double-buffered as a
    // whole: its MMAs and its epilogue would alternate.  Such a tile is processed as two half-tiles (input phases 0,1 and
    // 2,3; 256 columns each, own full/empty barriers): the strips pass through the stage ring once per half, and the
    // epilogue of one half runs under the MMAs of the other.  Accumulation order per phase is unchanged (bit-identical).
    static constexpr bool CAN_SPLIT = MODE == MODE_DEC && COLS_TILE == 512 && TPS == 1;
    static_assert(NKC == 1 || TPS == 1, "accumulating over k-chunks needs one tile per stage");
    static_assert(ENCF || (KCH % 2 == 0), "a K=16 step spans two channel blocks");
    static_assert(COLS_TILE <= 512, "accumulators exceed TMEM");
    static_assert(NSLOT >= TG, "tile-parallel epilogue groups need their own accumulator slots");
};

struct SmemPlan {
    uint32_t w_off, stage_off, stage_bytes, epi_off, bar_off, total;
};
template <class C>
__host__ __device__ inline SmemPlan plan_smem(int Ls, int n_stage, int w_bytes, int epi_floats) {
    SmemPlan s;
    s.w_off = 0;
    s.stage_off = (uint32_t)((w_bytes + 127) / 128 * 128);
    s.stage_bytes = (uint32_t)(C::KCH * C::NPLANE * Ls * 16);
    s.epi_off = s.stage_off + (uint32_t)n_stage * s.stage_bytes;
    s.bar_off = s.epi_off + (uint32_t)((epi_floats * 4 + 15) / 16 * 16);
    s.total = s.bar_off + 8 * (2 * kMaxStage + 2 * 8 + 1) + 16;
    return s;
}
template <class C>
__host__ __device__ constexpr int epi_floats() {
    // encoder: bias|scale|shift, two 4x4 TN matrices, then 256 floats of exchange scratch per epilogue warp
    return C::MODE == MODE_ENC ? 3 * C::COUT + 32 + kEpiWarps * 8 * kScratchPitch
                               : (C::MODE == MODE_DEC ? 2 * C::COUT + kEpiWarps * kDecScratchRows * 4 : 4);
}

// ------------------------------------------------------------------------------------------------ MMA issue
// All MMAs of one tile for one stage (k-chunk kc).  Fully unrolled: plane/shift of every tap are
// compile-time, only P, Tn, Ls are runtime.
template <class C, int PH0 = 0, int NPH = 4>
__device__ __forceinline__ void issue_tile(const LayerParams &p, uint32_t stage_addr, uint32_t w_addr, uint32_t d_tmem,
                                           int tile_in_stage, int kc, uint32_t idesc) {
    const int Ls = p.Ls, P = p.gin.P, Tn = p.gin.Tn;
    const int row0 = p.gin.halo + tile_in_stage * kTileM;
    if constexpr (C::ENCF) {
        // First conv on x-pair-packed rows ([c0 c1 c2 0 | c0' c1' c2' 0] = pixels (y, 2*x2), (y, 2*x2+1)), two row-parity
        // planes.  An operand tile is (u = a+dy in -1..2, sx in -1..1); every MMA pairs two tiles through LBO (K = 16)
        // and feeds all four phase accumulators at once (N = 64; unused (phase, tile) pairs have zero weights):
        //   steps 0..3: (u, sx=-1) | (u, sx=0)  -> second K half is the next row, LBO = 16 B
        //   steps 4..5: (u_lo, sx=+1) | (u_lo+2, sx=+1), same plane, one image row apart, LBO = P rows
        const uint64_t bdesc0 = make_desc(w_addr, (uint32_t)C::BLOCK_N * 16u, 128u);
#pragma unroll
        for (int st = 0; st < 6; st++) {
            const int u = st < 4 ? st - 1 : (st == 4 ? 0 : -1);
            const int slot = u & 1;                                     // staged plane: row parity a'
            const int r0 = slot * Ls + row0 + fdiv2(u) * P + (st < 4 ? -1 : 1);
            const uint64_t adesc = make_desc(stage_addr + (uint32_t)r0 * 16u, st < 4 ? 16u : (uint32_t)P * 16u, 128u);
            umma_f16(d_tmem, adesc, bdesc0 + (uint64_t)(st * C::BLOCK_N * 2), idesc, st > 0 ? 1u : 0u);
        }
    } else if constexpr (C::PAIR) {
        const uint32_t a_lbo = (uint32_t)(4 * Ls * 16);
        constexpr uint32_t idesc2 = make_idesc(2 * C::NCOLS);
        constexpr int voff[4] = {0, 1, 3, 5};
#pragma unroll
        for (int pa = 0; pa < 2; pa++) {
#pragma unroll
            for (int dy = -1; dy <= 1; dy++) {
                const int u = pa + dy;
#pragma unroll
                for (int ivi = 0; ivi < 4; ivi++) {
                    const int iv = (ivi + 1) & 3, v = iv - 1;              // order v = 0, 1, 2, -1: the first MMA of a row phase covers both accumulators
                    const bool two = iv == 1 || iv == 2;
                    const int plane = ((u & 1) << 1) | (v & 1);
                    const int r0 = plane * Ls + row0 + (fdiv2(u) * P + fdiv2(v)) * Tn;
                    const uint32_t d = d_tmem + (uint32_t)((pa * 2 + (iv == 3 ? 1 : 0)) * C::NCOLS);
#pragma unroll
                    for (int kpl = 0; kpl < C::KP; kpl++) {
                        const uint64_t adesc = make_desc(stage_addr + (uint32_t)((2 * kpl * 4) * Ls + r0) * 16u, a_lbo, 128u);
                        const int kp = kc * C::KP + kpl;
                        const uint32_t boff = (uint32_t)((((dy + 1) * (C::CIN_CB / 2) + kp) * 6 + voff[iv]) * C::NCOLS * 32);
                        const uint64_t bdesc = make_desc(w_addr + boff, (uint32_t)(two ? 2 * C::NCOLS : C::NCOLS) * 16u, 128u);
                        umma_f16(d, adesc, bdesc, two ? idesc2 : idesc, (kc > 0 || dy > -1 || ivi > 0 || kpl > 0) ? 1u : 0u);
                    }
                }
            }
        }
    } else if constexpr (C::PAIRD) {
        // transposed conv, column phases paired (weights_pack.cuh, pack_decoder): per row phase pa and row tap a, the input
        // column offsets w = 0 (both column phases, N = 2*NCOLS), w = -1 (pb = 0) and w = +1 (pb = 1)
        static_assert(PH0 % 2 == 0 && NPH % 2 == 0, "half-tiles are row phases");
        const uint32_t a_lbo = (uint32_t)(4 * Ls * 16);
        constexpr uint32_t idesc2 = make_idesc(2 * C::NCOLS);
#pragma unroll
        for (int pa = PH0 / 2; pa < (PH0 + NPH) / 2; pa++) {
#pragma unroll
            for (int a = 0; a < 2; a++) {
#pragma unroll
                for (int wi = 0; wi < 3; wi++) {
                    const int w = wi == 0 ? 0 : (wi == 1 ? -1 : 1);        // paired block first: it initialises both accumulators
                    const int plane = (((pa - a) & 1) << 1) | (w & 1);
                    const int r0 = plane * Ls + row0 + (fdiv2(pa - a) * P + fdiv2(w)) * Tn;
                    const uint32_t d = d_tmem + (uint32_t)((pa * 2 + (wi == 2 ? 1 : 0)) * C::NCOLS);
#pragma unroll
                    for (int kpl = 0; kpl < C::KP; kpl++) {
                        const uint64_t adesc = make_desc(stage_addr + (uint32_t)((2 * kpl * 4) * Ls + r0) * 16u, a_lbo, 128u);
                        const int kp = kc * C::KP + kpl;
                        const uint32_t boff = (uint32_t)(((a * (C::CIN_CB / 2) + kp) * 4 + (wi == 0 ? 0 : wi + 1)) * C::NCOLS * 32);
                        const uint64_t bdesc = make_desc(w_addr + boff, (uint32_t)(wi == 0 ? 2 * C::NCOLS : C::NCOLS) * 16u, 128u);
                        umma_f16(d, adesc, bdesc, wi == 0 ? idesc2 : idesc, (kc > 0 || a > 0 || wi > 0 || kpl > 0) ? 1u : 0u);
                    }
                }
            }
        }
    } else {
        const uint32_t a_lbo = (uint32_t)(4 * Ls * 16);
        const uint64_t bdesc0 = make_desc(w_addr, (uint32_t)C::NCOLS * 16u, 128u);
#pragma unroll
        for (int ph = PH0; ph < PH0 + NPH; ph++) {
            const int pa = ph >> 1, pb = ph & 1;
            const uint32_t d = d_tmem + (uint32_t)(ph * C::NCOLS);
#pragma unroll
            for (int tp = 0; tp < C::NTAP; tp++) {
                int plane, sy, sx;
                if constexpr (C::MODE == MODE_ENC) {
                    const int dy = tp / 3 - 1, dx = tp % 3 - 1;
                    plane = (((pa + dy) & 1) << 1) | ((pb + dx) & 1);
                    sy = fdiv2(pa + dy); sx = fdiv2(pb + dx);
                } else {
                    const int a = tp >> 1, b = tp & 1;
                    plane = (((pa - a) & 1) << 1) | ((pb - b) & 1);
                    sy = fdiv2(pa - a); sx = fdiv2(pb - b);
                }
                const int r0 = plane * Ls + row0 + (sy * P + sx) * Tn;
#pragma unroll
                for (int kpl = 0; kpl < C::KP; kpl++) {
                    const uint64_t adesc = make_desc(stage_addr + (uint32_t)((2 * kpl * 4) * Ls + r0) * 16u, a_lbo, 128u);
                    const int block = tp * (C::CIN_CB / 2) + kc * C::KP + kpl;
                    const uint64_t bdesc = bdesc0 + (uint64_t)(block * C::NCOLS * 2);
                    umma_f16(d, adesc, bdesc, idesc, (kc > 0 || tp > 0 || kpl > 0) ? 1u : 0u);
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------ epilogues
__device__ __forceinline__ uint32_t pack_half2(float a, float b) {
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t *>(&h);
}

// Encoder tail for one 128-position tile and one group of channel blocks.  Lane = (position, t): the four
// frames of a window position are the four lanes of a quad.
//   1. bias -> ReLU -> BatchNorm -> 2x2 max-pool over the four phase accumulators, per lane, in registers;
//   2. PointWiseTN needs all four t of a (position, channel): the quad exchanges its 8 channels x 4 t through a
//      1.1 KB per-warp shared-memory scratch ([channel][lane] floats, padded rows: conflict-free stores, one 128-bit load per
//      channel) and each lane then computes TWO channels for ALL four output frames - no redundant 4x4
//      products and no shuffles;
//   3. each lane stores its 2-channel slice (4 bytes) of the four 16-byte output rows of the quad.
// Part 1 (epilogue_enc_pool): drain this warp's accumulators, keeping only the pooled extremum per channel in registers -
// the caller then hands the TMEM slot back to the MMA warp BEFORE part 2 (epilogue_enc) does the arithmetic and the stores,
// so the MMAs of the tile after next never wait for a finalisation.
template <class C>
__device__ __forceinline__ void epilogue_enc_pool(const LayerParams &p, const float *epi, uint32_t taddr, int cg,
                                                  float (&ext)[(C::COUT / 8) / C::CG][8]) {
    constexpr int CB_PER = (C::COUT / 8) / C::CG;
    const float *scale = epi + C::COUT;
#pragma unroll
    for (int i = 0; i < CB_PER; i++) {
        const int cb = cg * CB_PER + i;
        uint32_t v[4][8];
#pragma unroll
        for (int ph = 0; ph < 4; ph++) tmem_ld8(taddr + (uint32_t)(ph * C::NCOLS + cb * 8), v[ph]);
        tmem_wait_ld();
#pragma unroll
        for (int j = 0; j < 8; j++) {
            // MaxPool(BN(ReLU(x + b))): x -> fma(max(x + b, 0), s, sh) is monotone (non-decreasing for s >= 0,
            // non-increasing for s < 0), so the pool maximum is attained at max(x) resp. min(x): bit-identical
            // to pooling the four activated values, with a quarter of the arithmetic.
            const float a0 = __uint_as_float(v[0][j]), a1 = __uint_as_float(v[1][j]);
            const float a2 = __uint_as_float(v[2][j]), a3 = __uint_as_float(v[3][j]);
            ext[i][j] = fmaxf(fmax3(a0, a1, a2), a3);
            if (!p.bn_nonneg) {
                const float lo = fminf(fminf(a0, a1), fminf(a2, a3));
                ext[i][j] = scale[cb * 8 + j] >= 0.f ? ext[i][j] : lo;
            }
        }
    }
}

template <class C>
__device__ __forceinline__ void epilogue_enc(const LayerParams &p, const float *epi, float *scratch, const float (&ext)[(C::COUT / 8) / C::CG][8],
                                             int pp, int lane, int cg) {
    const Geom &gi = p.gin;
    const int t = pp & 3;
    const int qq = pp >> 2;
    const int n = (int)fast_div((uint32_t)qq, p.divS);
    const int r = qq - n * gi.S;
    const int y2 = (int)fast_div((uint32_t)r, p.divP), x2 = r - y2 * gi.P;
    const bool valid = n < p.N && y2 < (gi.H >> 1) && x2 < (gi.W >> 1);   // same for the 4 lanes of a quad
    const int Y = y2 + (gi.H & 1), X = x2 + (gi.W & 1);          // zero-pad top / left when odd (encoder.py:68-76)
    const int pho = ((Y & 1) << 1) | (X & 1);
    uint32_t *dst1 = nullptr, *dst2 = nullptr;                   // this lane's 4-byte slice of row (quad, t' = 0)
    if (valid) {
        if (p.out) dst1 = reinterpret_cast<uint32_t *>(p.out + geom_row(p.gout, 0, pho, geom_pos(p.gout, n, Y >> 1, X >> 1, 0))) + t;
        if (p.out2) dst2 = reinterpret_cast<uint32_t *>(p.out2 + geom_row(p.gout2, p.out2_cb, pho, geom_pos(p.gout2, n, Y >> 1, X >> 1, 0))) + t;
    }
    const float4 *bias4 = reinterpret_cast<const float4 *>(epi), *scale4 = reinterpret_cast<const float4 *>(epi + C::COUT),
                 *shift4 = reinterpret_cast<const float4 *>(epi + 2 * C::COUT);
    const int qbase = lane & ~3;
    constexpr int CB_PER = (C::COUT / 8) / C::CG;                 // channel blocks of this warp group
    // PointWiseTN matrices as packed broadcast pairs are taken straight from the kernel parameters (uniform registers)
#pragma unroll
    for (int i = 0; i < CB_PER; i++) {
        const int cb = cg * CB_PER + i;
        float bs[8], sc[8], sh[8];
        *reinterpret_cast<float4 *>(bs) = bias4[cb * 2]; *reinterpret_cast<float4 *>(bs + 4) = bias4[cb * 2 + 1];
        *reinterpret_cast<float4 *>(sc) = scale4[cb * 2]; *reinterpret_cast<float4 *>(sc + 4) = scale4[cb * 2 + 1];
        *reinterpret_cast<float4 *>(sh) = shift4[cb * 2]; *reinterpret_cast<float4 *>(sh + 4) = shift4[cb * 2 + 1];
#pragma unroll
        for (int jp = 0; jp < 4; jp++) {
            // bias -> ReLU -> BatchNorm on the pooled extremum, channel pairs in packed fp32 lanes
            const float2 act = relu2(fadd2(make_float2(ext[i][2 * jp], ext[i][2 * jp + 1]), make_float2(bs[2 * jp], bs[2 * jp + 1])));
            *reinterpret_cast<float2 *>(scratch + jp * kPairPitch + 2 * lane) =
                ffma2(act, make_float2(sc[2 * jp], sc[2 * jp + 1]), make_float2(sh[2 * jp], sh[2 * jp + 1]));
        }
        __syncwarp();
        // PointWiseTN (pointwise.py:18-26) for the channel pair t of this quad's position, all four output frames:
        // x[ti] = (channel 2t, channel 2t+1) of frame ti
        const float4 xa = *reinterpret_cast<const float4 *>(scratch + t * kPairPitch + 2 * qbase);
        const float4 xb = *reinterpret_cast<const float4 *>(scratch + t * kPairPitch + 2 * qbase + 4);
        const float2 x[4] = {make_float2(xa.x, xa.y), make_float2(xa.z, xa.w), make_float2(xb.x, xb.y), make_float2(xb.z, xb.w)};
        float2 h1[4];
#pragma unroll
        for (int m = 0; m < 4; m++) {
            float2 h = fmul2(x[0], bc2(p.tn_w1[m]));
#pragma unroll
            for (int ti = 1; ti < 4; ti++) h = ffma2(x[ti], bc2(p.tn_w1[ti * 4 + m]), h);
            h1[m] = relu2(h);
        }
        uint32_t packed[4];
#pragma unroll
        for (int to = 0; to < 4; to++) {                              // relu(x + relu(h2)) = max(x + h2, x, 0)
            float2 h = x[to];
#pragma unroll
            for (int m = 0; m < 4; m++) h = ffma2(h1[m], bc2(p.tn_w2[m * 4 + to]), h);
            packed[to] = pack_half2(fmax3(h.x, x[to].x, 0.f), fmax3(h.y, x[to].y, 0.f));
        }
        if (valid) {
            if (p.out) {
                uint32_t *d = dst1 + (long long)cb * 4 * p.gout.Lp * 4;   // rows are 4 x u32
#pragma unroll
                for (int to = 0; to < 4; to++) d[to * 4] = packed[to];    // rows t' = 0..3 are consecutive
            }
            if (p.out2) dst2[(long long)cb * 4 * p.gout2.Lp * 4] = packed[0];
        }
        __syncwarp();
    }
}

// Decoder tail.  Warp group g takes the input-row phase pa = g >> 1, BOTH column phases pb, and every second output parity
// of the CTA (pl = g & 1, g & 1 + 2, ...).  Why both pb: output column X = 4*x2 + 2*pb + px - crop_l, so within one output
// phase plane the rows of consecutive input positions x2 alternate between pb = 0 and pb = 1.  A warp that stores one pb
// writes 16 bytes of every other 32-byte sector (measured: dec2 0.149 ms with that pattern, 0.100 ms with the same
// stores coalesced); a warp that holds both writes whole sectors.  The rows go through a per-warp shared-memory scratch
// (pb = 0 rows at [lane], pb = 1 rows at [36 + lane]: conflict-free both ways) so that lane L stores row L of a 32-row
// run (positions 0..15 of the warp, then 16..31): each store instruction covers 512 contiguous bytes wherever the
// positions of the warp are contiguous in the output plane.
template <class C>
__device__ __forceinline__ void epilogue_dec(const LayerParams &p, const float *epi, uint4 *scratch, uint32_t taddr, int pp, int half,
                                             int g, int lane) {
    const Geom &gi = p.gin;
    const int n = (int)fast_div((uint32_t)pp, p.divS);
    const int r = pp - n * gi.S;
    const int y2 = (int)fast_div((uint32_t)r, p.divP), x2 = r - y2 * gi.P;
    constexpr int PARN = C::NCOLS / C::COUT;   // output parities handled by this CTA
    constexpr int CBN = C::COUT / 8;
    static_assert(PARN % 2 == 0, "the two warp groups of a row phase split the parities");
    const float4 *scale4 = reinterpret_cast<const float4 *>(epi), *offs4 = reinterpret_cast<const float4 *>(epi + C::COUT);
    const int pa = g >> 1;
    const int oy = 2 * y2 + pa, ox0 = 4 * x2;                      // sub-pixel grid position for pb = 0 is (oy, 2*x2); pb = 1 one to the right
    const bool vrow = n < p.N && oy <= gi.H;
    const int src_a = lane >> 1, src_b = 16 + (lane >> 1), my_pb = lane & 1;
    const uint32_t acc0 = taddr + (uint32_t)((pa * 2) * C::NCOLS), acc1 = acc0 + (uint32_t)C::NCOLS;
#pragma unroll 1
    for (int pl = g & 1; pl < PARN; pl += 2) {
        const int par = half * PARN + pl, py = par >> 1, px = par & 1;
        const int Y = 2 * oy + py - p.crop_t, X0 = ox0 + px - p.crop_l;             // pb = 1: X0 + 2, i.e. the next row of the same plane
        const bool vy = vrow && Y >= 0 && Y < p.Ht;
        const bool v0 = vy && X0 >= 0 && X0 < p.Wt && 2 * x2 <= gi.W;
        const bool v1 = vy && X0 + 2 >= 0 && X0 + 2 < p.Wt && 2 * x2 + 1 <= gi.W;
        const int plane = (((py - p.crop_t) & 1) << 1) | ((px - p.crop_l) & 1);     // warp-uniform
        const int pos0 = (int)p.gout.guard + (n * p.gout.S + (Y >> 1) * p.gout.P + (X0 >> 1));   // arithmetic shifts: X0 may be -1
        const unsigned m0 = __ballot_sync(0xffffffffu, v0), m1 = __ballot_sync(0xffffffffu, v1);
        const unsigned mine = my_pb ? m1 : m0;
        const bool va = (mine >> src_a) & 1u, vb = (mine >> src_b) & 1u;
        const long long plane_row = (long long)plane * p.gout.Lp;
        uint4 *dst_a = p.out + (plane_row + (__shfl_sync(0xffffffffu, pos0, src_a) + my_pb));
        uint4 *dst_b = p.out + (plane_row + (__shfl_sync(0xffffffffu, pos0, src_b) + my_pb));
        if (!(m0 | m1)) continue;                                                   // warp-uniform: nothing of this warp survives the crop
#pragma unroll
        for (int cb = 0; cb < CBN; cb++) {
            uint32_t a0[8], a1[8];
            tmem_ld8(acc0 + (uint32_t)(pl * C::COUT + cb * 8), a0);
            tmem_ld8(acc1 + (uint32_t)(pl * C::COUT + cb * 8), a1);
            const float4 s0 = scale4[cb * 2], s1 = scale4[cb * 2 + 1], f0 = offs4[cb * 2], f1 = offs4[cb * 2 + 1];
            tmem_wait_ld();
            uint4 rw[2];
#pragma unroll
            for (int b = 0; b < 2; b++) {
                const uint32_t(&a)[8] = b ? a1 : a0;
                // bias+BN folded into (scale, offs), then the consumer's ReLU
                const float2 o01 = relu2(ffma2(make_float2(__uint_as_float(a[0]), __uint_as_float(a[1])), make_float2(s0.x, s0.y), make_float2(f0.x, f0.y)));
                const float2 o23 = relu2(ffma2(make_float2(__uint_as_float(a[2]), __uint_as_float(a[3])), make_float2(s0.z, s0.w), make_float2(f0.z, f0.w)));
                const float2 o45 = relu2(ffma2(make_float2(__uint_as_float(a[4]), __uint_as_float(a[5])), make_float2(s1.x, s1.y), make_float2(f1.x, f1.y)));
                const float2 o67 = relu2(ffma2(make_float2(__uint_as_float(a[6]), __uint_as_float(a[7])), make_float2(s1.z, s1.w), make_float2(f1.z, f1.w)));
                rw[b].x = pack_half2(o01.x, o01.y); rw[b].y = pack_half2(o23.x, o23.y);
                rw[b].z = pack_half2(o45.x, o45.y); rw[b].w = pack_half2(o67.x, o67.y);
            }
            scratch[lane] = rw[0];
            scratch[36 + lane] = rw[1];
            __syncwarp();
            const uint4 ra = scratch[my_pb * 36 + src_a], rb = scratch[my_pb * 36 + src_b];
            __syncwarp();
            const long long cb_row = (long long)cb * 4 * p.gout.Lp;
            if (va) dst_a[cb_row] = ra;
            if (vb) dst_b[cb_row] = rb;
        }
    }
}

template <class C>
__device__ __forceinline__ void epilogue_head(const LayerParams &p, const float *epi, uint32_t taddr, int pp, int ph) {
    const Geom &gi = p.gin;
    const int n = (int)fast_div((uint32_t)pp, p.divS);
    const int r = pp - n * gi.S;
    const int y2 = (int)fast_div((uint32_t)r, p.divP), x2 = r - y2 * gi.P;
    const float c0 = epi[0];
    uint32_t v[4];
    tmem_ld4(taddr + (uint32_t)(ph * C::NCOLS), v);
    tmem_wait_ld();
    const int oy = 2 * y2 + (ph >> 1), ox = 2 * x2 + (ph & 1);
    const bool vpos = n < p.N && oy <= gi.H && ox <= gi.W;
    // tau = logit(segmentation-threshold), 0 at the default 0.5; per window only for a batch whose streams set their own
    const float tau = vpos && p.seg ? __ldg(p.seg + n) : p.seg_tau;
#pragma unroll
    for (int par = 0; par < 4; par++) {
        const int Y = 2 * oy + (par >> 1) - p.crop_t, X = 2 * ox + (par & 1) - p.crop_l;
        if (vpos && Y >= 0 && Y < p.Ht && X >= 0 && X < p.Wt) {
            const float z = __uint_as_float(v[par]) + c0;
            const size_t o = ((size_t)n * p.Ht + Y) * p.Wt + X;
            p.mask[o] = z > tau ? 1 : 0;      // sigmoid(z) > segmentation-threshold (nvinfer), +1 of maskcopy folded
            if (p.logits) p.logits[o] = z;
        }
    }
}

// ------------------------------------------------------------------------------------------------ kernel
template <class C>
__global__ void __launch_bounds__(kThreads, 1) shiftgemm_kernel(const __grid_constant__ LayerParams p) {
    static_assert(!C::ENCF, "the first block runs tc1::enc1_fused_kernel");
    extern __shared__ __align__(1024) unsigned char smem[];
    const SmemPlan sp = plan_smem<C>(p.Ls, p.n_stage, p.w_bytes, epi_floats<C>());
    const uint32_t smem_base = smem_u32(smem);
    float *epi = reinterpret_cast<float *>(smem + sp.epi_off);
    const uint32_t bar0 = smem_base + sp.bar_off;
    auto full_bar = [&](int s) { return bar0 + 8u * (uint32_t)s; };
    auto empty_bar = [&](int s) { return bar0 + 8u * (uint32_t)(kMaxStage + s); };
    auto tfull_bar = [&](int s) { return bar0 + 8u * (uint32_t)(2 * kMaxStage + s); };
    auto tempty_bar = [&](int s) { return bar0 + 8u * (uint32_t)(2 * kMaxStage + 8 + s); };
    const uint32_t w_bar = bar0 + 8u * (uint32_t)(2 * kMaxStage + 16);
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + sp.bar_off + 8 * (2 * kMaxStage + 17));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nsplit = C::MODE == MODE_DEC ? p.nsplit : 1;
    const int half = (int)blockIdx.x % nsplit;
    const int cta = (int)blockIdx.x / nsplit, n_cta = (int)gridDim.x / nsplit;
    int nh = 1;                                   // half-tiles per tile
    if constexpr (C::CAN_SPLIT) nh = p.psplit ? 2 : 1;
    pdl_launch_dependents();

    // epilogue constants -> smem (generic proxy)
    constexpr int kEpiConst = C::MODE == MODE_ENC ? 3 * C::COUT + 32 : (C::MODE == MODE_DEC ? 2 * C::COUT : epi_floats<C>());
    for (int i = threadIdx.x; i < kEpiConst; i += kThreads) {
        float v;
        if (C::MODE == MODE_ENC && i >= 3 * C::COUT) v = (i - 3 * C::COUT < 16) ? p.tn_w1[i - 3 * C::COUT] : p.tn_w2[i - 3 * C::COUT - 16];
        else v = p.epi[i];
        epi[i] = v;
    }
    if (threadIdx.x == 0) {
        for (int s = 0; s < kMaxStage; s++) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
        for (int s = 0; s < 8; s++) { mbar_init(tfull_bar(s), 1); mbar_init(tempty_bar(s), 4 * C::CG / nh); }
        mbar_init(w_bar, 1);
        fence_barrier_init();
    }
    if (warp == 1) {
        tmem_alloc(smem_u32(tmem_slot), C::TMEM_COLS);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (warp == 0 && elect_one()) {              // weights do not depend on the preceding kernel: fetch them before the wait
        mbar_expect_tx(w_bar, (uint32_t)p.w_bytes);
        bulk_g2s(smem_base + sp.w_off, reinterpret_cast<const unsigned char *>(p.wpack) + (size_t)half * p.w_bytes,
                 (uint32_t)p.w_bytes, w_bar);
    }
    __syncwarp();
    pdl_wait();

    if (warp == 0) {
        // ===== producer: one strip per (group, k-chunk) =====
        if (elect_one()) {
            uint32_t it = 0;
            for (int g = cta; g < p.n_groups; g += n_cta) {
                const long long pos0 = p.gin.guard + (long long)g * C::TPS * kTileM - p.gin.halo;
                for (int kc = 0; kc < C::NKC * nh; kc++, it++) {     // half-tiles: the k-chunks pass through the ring once per half
                    const int s = (int)(it % (uint32_t)p.n_stage);
                    mbar_wait(empty_bar(s), ((it / (uint32_t)p.n_stage) & 1u) ^ 1u, p.watchdog, 1u);
                    mbar_expect_tx(full_bar(s), sp.stage_bytes);
                    const uint32_t dst0 = smem_base + sp.stage_off + (uint32_t)s * sp.stage_bytes;
#pragma unroll 1
                    for (int cbi = 0; cbi < C::KCH; cbi++)
#pragma unroll
                        for (int pl = 0; pl < C::NPLANE; pl++)
                            bulk_g2s(dst0 + (uint32_t)((cbi * C::NPLANE + pl) * p.Ls) * 16u,
                                     p.in + geom_row(p.gin, (kc % C::NKC) * C::KCH + cbi, pl * (4 / C::NPLANE), pos0), (uint32_t)p.Ls * 16u, full_bar(s));
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer (one elected thread) =====
        if (elect_one()) {
            constexpr uint32_t idesc = make_idesc(C::BLOCK_N);
            mbar_wait(w_bar, 0u, p.watchdog, 2u);
            uint32_t it = 0, tile_it = 0;
            for (int g = cta; g < p.n_groups; g += n_cta) {
                const uint32_t tile_it0 = tile_it;
                if constexpr (C::CAN_SPLIT) {
                    if (nh == 2) {
                        // two half-tiles (input phases 0,1 | 2,3), each with its own accumulator barriers
                        for (int hh = 0; hh < 2; hh++) {
                            for (int kc = 0; kc < C::NKC; kc++, it++) {
                                const int s = (int)(it % (uint32_t)p.n_stage);
                                mbar_wait(full_bar(s), (it / (uint32_t)p.n_stage) & 1u, p.watchdog, 3u);
                                if (kc == 0) mbar_wait(tempty_bar(hh), (tile_it & 1u) ^ 1u, p.watchdog, 4u);
                                tc_fence_after();
                                const uint32_t stage_addr = smem_base + sp.stage_off + (uint32_t)s * sp.stage_bytes;
                                if (!(p.dbg & 1)) {
                                    if (hh == 0) issue_tile<C, 0, 2>(p, stage_addr, smem_base + sp.w_off, tmem_base, 0, kc, idesc);
                                    else issue_tile<C, 2, 2>(p, stage_addr, smem_base + sp.w_off, tmem_base, 0, kc, idesc);
                                }
                                if (kc == C::NKC - 1) umma_commit(tfull_bar(hh));
                                umma_commit(empty_bar(s));
                            }
                        }
                        tile_it++;
                        continue;
                    }
                }
                for (int kc = 0; kc < C::NKC; kc++, it++) {
                    const int s = (int)(it % (uint32_t)p.n_stage);
                    mbar_wait(full_bar(s), (it / (uint32_t)p.n_stage) & 1u, p.watchdog, 3u);
                    tc_fence_after();
                    const uint32_t stage_addr = smem_base + sp.stage_off + (uint32_t)s * sp.stage_bytes;
                    tile_it = tile_it0;
#pragma unroll 1
                    for (int j = 0; j < C::TPS; j++) {
                        if ((g * C::TPS + j) >= p.n_tiles) break;
                        const int slot = (int)(tile_it % (uint32_t)C::NSLOT);
                        if (kc == 0) {
                            mbar_wait(tempty_bar(slot), ((tile_it / (uint32_t)C::NSLOT) & 1u) ^ 1u, p.watchdog, 4u);
                            tc_fence_after();
                        }
                        if (!(p.dbg & 1)) issue_tile<C>(p, stage_addr, smem_base + sp.w_off, tmem_base + (uint32_t)(slot * C::COLS_TILE), j, kc, idesc);
                        if (kc == C::NKC - 1) umma_commit(tfull_bar(slot));
                        tile_it++;
                    }
                    umma_commit(empty_bar(s));   // strip may be overwritten once these MMAs have read it
                }
            }
        }
    } else {
        // ===== epilogue warps: TMEM -> registers -> fused layer tail -> HBM =====
        const int q = warp & 3;                       // TMEM lane quarter this warp may read
        const int gidx = (warp - 2) >> 2;             // warp group 0..3
        const int cg = gidx % C::CG, tg = gidx / C::CG;
        float *scratch = epi + 3 * C::COUT + 32 + (warp - 2) * 8 * kScratchPitch;   // encoder only
        uint32_t tile_it = 0;
        for (int g = cta; g < p.n_groups; g += n_cta) {
#pragma unroll 1
            for (int j = 0; j < C::TPS; j++) {
                const int tile = g * C::TPS + j;
                if (tile >= p.n_tiles) break;
                if ((int)(tile_it % (uint32_t)C::TG) == tg) {
                    int slot = (int)(tile_it % (uint32_t)C::NSLOT);
                    uint32_t acc_col = (uint32_t)(slot * C::COLS_TILE);
                    if (nh == 2) { slot = cg >> 1; acc_col = 0u; }                 // half-tile of this group's input phase
                    mbar_wait(tfull_bar(slot), (nh == 2 ? tile_it : tile_it / (uint32_t)C::NSLOT) & 1u, p.watchdog, 5u);
                    tc_fence_after();
                    const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc_col;
                    const int pp = tile * kTileM + q * 32 + lane;
                    if constexpr (C::MODE == MODE_ENC) {
                        float ext[(C::COUT / 8) / C::CG][8];
                        if (!(p.dbg & 2)) epilogue_enc_pool<C>(p, epi, taddr, cg, ext);
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(tempty_bar(slot));          // accumulators are in registers: release the slot early
                        if (!(p.dbg & 2)) epilogue_enc<C>(p, epi, scratch, ext, pp, lane, cg);
                        tile_it++;
                        continue;
                    }
                    if (p.dbg & 2) {
                    }
                    else if constexpr (C::MODE == MODE_DEC)
                        epilogue_dec<C>(p, epi, reinterpret_cast<uint4 *>(epi + 2 * C::COUT) + (warp - 2) * kDecScratchRows, taddr, pp, half, cg, lane);
                    else epilogue_head<C>(p, epi, taddr, pp, cg);
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(tempty_bar(slot));
                }
                tile_it++;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, C::TMEM_COLS);
}

// ------------------------------------------------------------------------------------------------ launch
constexpr int kSmemLimit = 227 * 1024;

// Host-side part of a launch, split in two so that the choice can be queried without a device (cova_blobnet_plan).
// plan: fills the tiling fields of p (n_tiles, n_groups, Ls, n_stage, w_bytes, divS, divP) and the grid; false when C
// does not fit this geometry with at least min_stage strips in its ring.  launch: the attribute call and the launch.
struct Grid {
    int ctas;          // CTAs launched (all N-halves)
    uint32_t smem;     // dynamic shared memory per CTA
};

template <class C>
inline bool plan(LayerParams &p, int n_sms, int min_stage, Grid &g) {
    const long long mtot = (long long)p.N * p.gin.S * p.gin.Tn;
    p.n_tiles = (int)((mtot + kTileM - 1) / kTileM);
    p.n_groups = (p.n_tiles + C::TPS - 1) / C::TPS;
    p.Ls = C::TPS * kTileM + 2 * p.gin.halo;
    p.divS = make_fastdiv((uint32_t)p.gin.S);
    p.divP = make_fastdiv((uint32_t)p.gin.P);
    if (4 * p.Ls >= 16384 || p.gin.P >= 16384) return false;                       // LBO field: 14 bits of 16-byte units
    if (p.gin.guard + (long long)p.n_groups * C::TPS * kTileM + p.gin.halo > p.gin.Lp) return false;
    const int nsplit = C::MODE == MODE_DEC ? p.nsplit : 1;
    p.w_bytes = C::BLOCKS * C::BLOCK_N * 32;
    // ring depth: as deep as fits, up to 2 strips (whole-K stages) or 4 (k-chunked stages)
    const int target = C::NKC > 1 ? kMaxStage : 2;
    for (p.n_stage = target; p.n_stage >= 1; p.n_stage--)
        if (plan_smem<C>(p.Ls, p.n_stage, p.w_bytes, epi_floats<C>()).total <= (uint32_t)kSmemLimit) break;
    if (p.n_stage < min_stage) return false;
    g.smem = plan_smem<C>(p.Ls, p.n_stage, p.w_bytes, epi_floats<C>()).total;
    int ctas = n_sms / nsplit;
    if (ctas > p.n_groups) ctas = p.n_groups;
    if (ctas < 1) ctas = 1;
    g.ctas = ctas * nsplit;
    return true;
}

template <class C>
inline cudaError_t launch(const LayerParams &p, const Grid &g, cudaStream_t st) {
    // The attribute belongs to the FUNCTION (per device), not to a launch, and the last write wins: two handles with
    // different grids on two threads would otherwise lower it under each other's feet between "set" and "launch"
    // (seen as cudaErrorInvalidValue by tests/test_gpu_parity.py::test_two_threads_two_handles...).  Always the same value,
    // the architectural maximum, makes the call idempotent; occupancy follows the size actually requested at launch.
    cudaError_t err = cudaFuncSetAttribute(shiftgemm_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit);
    if (err != cudaSuccess) return err;
    return launch_pdl(shiftgemm_kernel<C>, dim3((unsigned)g.ctas), dim3(kThreads), g.smem, st, !(p.dbg & kDbgNoPdl), p);
}

}  // namespace tc
}  // namespace cova
