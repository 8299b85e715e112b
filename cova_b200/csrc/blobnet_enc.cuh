// BlobNet encoder blocks 2..4 as "weights-stationary" tcgen05 GEMMs, sm_100a.
//
// Measured on B200 (profiles/r1b_mma_bench.txt): one tcgen05.mma (M = 128, K = 16, fp16) costs
//   43 + N/2 cycles with the A operand in shared memory, 10 + N/2 cycles with A in TMEM.
// With positions as M and Cout = 32..128 as N (csrc/blobnet_tc.cuh) the fixed part dominates.  Here the
// roles are swapped:
//   D[m, n] = sum_k A[m, k] * B[n, k]        A = WEIGHTS, resident in TMEM for the CTA's lifetime
//                                             B = NP (112..192) consecutive positions of a phase-plane strip
// so the fixed cost is 10 cycles and is amortised over up to 192 positions.  M = 128 rows are filled with
// (pooling phase, output channel): the four conv outputs a 2x2 max-pool window needs read the input at 16
// distinct offsets (u, v) in [-1, 2]^2, and row (phase, cout) of the A block of offset (u, v) holds
// W[cout][.][u - a][v - b] (zero when that is not a tap of the phase) - "union of taps".
//   block 2: Cout = 32, 4 phases in M, 16 offsets, 1 pass per tile
//   block 3: Cout = 64, the 2 column phases in M, 12 offsets, 2 passes (row phase a = 0, 1)
//   block 4: Cout = 128, 9 taps, 4 passes
// Accumulators: D[lane = (cb_local, phase, channel), column = position].  The epilogue reads them with
// tcgen05.ld.16x256b, whose fragment layout hands thread i rows i/4 and i/4 + 8 of a 16-lane half: with the
// pooling phases placed 8 lanes apart, all phases of a channel land in ONE thread (max-pool = 3 FMNMX, no
// shuffles), and a thread owns two adjacent columns = two of the four frames of a window pixel; PointWiseTN is
// completed with one partner exchange (lane ^ 1).  Across passes pooling is a running maximum in registers.
// Negative BatchNorm scales (max-pool of a decreasing function = function of the minimum) are handled by
// negating the channel's weights on the host and using sgn = -1 in relu(sgn*x + b).
//
// Reference for the math: utils/model/encoder.py:33-76, utils/model/pointwise.py:10-26.
#pragma once
#include "blobnet_tc.cuh"

namespace cova {
namespace tcs {

using tc::LayerParams;

constexpr int kMaxStage = 4;
constexpr int kMaxSlot = 4;

__device__ __forceinline__ void umma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint4 &a, const uint4 &b) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                 ::"r"(taddr), "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w), "r"(b.x), "r"(b.y), "r"(b.z), "r"(b.w) : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

template <int CIN_CB_, int COUT_, int LA_, int LB_, int NP_, int TPS_, int EW_ = 16>
struct ECfg {
    static constexpr int EW = EW_, CS = EW_ / 4;           // epilogue warps: CS per TMEM lane quarter, each owning a column range of a tile
    static constexpr int THREADS = 64 + 32 * EW_;
    static constexpr int CIN_CB = CIN_CB_, COUT = COUT_, LA = LA_, LB = LB_, NP = NP_, TPS = TPS_;
    static constexpr int PL = LA * LB;                     // pooling phases that live in M (lanes)
    static constexpr int PA = 2 / LA, PB = 2 / LB, PASSES = PA * PB;
    static constexpr int NU = LA == 2 ? 4 : 3, NV = LB == 2 ? 4 : 3;
    static constexpr int KP = CIN_CB / 2;                  // K = 16 steps per offset
    static constexpr int NBLK = NU * NV * KP;              // A blocks (128 rows x 16 K) resident in TMEM
    static constexpr int A_COLS = NBLK * 8;
    static constexpr int NSLOT = ((512 - A_COLS) / NP) < kMaxSlot ? ((512 - A_COLS) / NP) : kMaxSlot;
    static constexpr int NUN = NP / 16;                    // 16-column units (4 pixels x 4 frames) per tile
    static constexpr int UB = NUN / CS, UR = NUN % CS;     // units per epilogue warp: UB (+1 for the first UR column ranges)
    static constexpr int MAXU = UB + (UR ? 1 : 0);
    static constexpr int NIT = 4 / PL;                     // (channel block) items per thread and group
    static constexpr int CBQ = COUT / 32;                  // output channel blocks per TMEM lane quarter (= NIT)
    // Block 4 (Cout = 128) is the last encoder block: it has no next-encoder output, only the t = 0 skip row of the
    // decoder input; blocks 2 and 3 always write both.  Compile-time, so the finalisation carries no pointer tests.
    static constexpr bool HAS_OUT = COUT < 128;
    static_assert(COUT * PL == 128, "M = 128 rows = lane phases x output channels");
    static_assert(CIN_CB % 2 == 0, "a K = 16 step spans two channel blocks");
    static_assert(NP % 16 == 0 && NP >= 16 && NP <= 256, "N of one MMA");
    static_assert(NSLOT >= 2, "accumulators must be double-buffered");
    static_assert(PASSES == 1 || NSLOT >= 2, "");
};

struct ELayerExtra {
    FastDiv divS, divP;
};

struct SmemPlanE {
    uint32_t stage_off, stage_bytes, epi_off, bar_off, total;
};
template <class C>
__host__ __device__ inline SmemPlanE plan_smem_e(int Ls, int n_stage) {
    SmemPlanE s;
    s.stage_off = 0;
    s.stage_bytes = (uint32_t)(C::CIN_CB * 4 * Ls * 16);
    s.epi_off = s.stage_off + (uint32_t)n_stage * s.stage_bytes;
    s.bar_off = s.epi_off + (uint32_t)((4 * C::COUT + 32) * 4);
    s.total = s.bar_off + 8 * (2 * kMaxStage + 2 * kMaxSlot) + 16;
    return s;
}

// all MMAs of one pass (pa, pb) of one tile
template <class C, int PASS>
__device__ __forceinline__ void issue_pass(const LayerParams &p, uint32_t stage_addr, uint32_t a_tmem, uint32_t d_tmem,
                                           int tile_in_stage, uint32_t idesc) {
    constexpr int pa = C::PA == 2 ? PASS / C::PB : 0, pb = C::PB == 2 ? PASS % C::PB : 0;
    const int Ls = p.Ls, P = p.gin.P;
    const int row0 = p.gin.halo + tile_in_stage * C::NP;
    const uint32_t lbo = (uint32_t)(4 * Ls * 16);
#pragma unroll
    for (int iu = 0; iu < C::NU; iu++) {
#pragma unroll
        for (int iv = 0; iv < C::NV; iv++) {
            const int u = C::LA == 2 ? iu - 1 : pa + iu - 1;
            const int v = C::LB == 2 ? iv - 1 : pb + iv - 1;
            const int plane = ((u & 1) << 1) | (v & 1);
            const int r0 = plane * Ls + row0 + (tc::fdiv2(u) * P + tc::fdiv2(v)) * kT;
#pragma unroll
            for (int kpl = 0; kpl < C::KP; kpl++) {
                const uint64_t bdesc = tc::make_desc(stage_addr + (uint32_t)((2 * kpl * 4) * Ls + r0) * 16u, lbo, 128u);
                umma_f16_ts(d_tmem, a_tmem + (uint32_t)(((iu * C::NV + iv) * C::KP + kpl) * 8), bdesc, idesc,
                            (iu > 0 || iv > 0 || kpl > 0) ? 1u : 0u);
            }
        }
    }
}

template <class C, int PASS>
__device__ __forceinline__ void issue_all_passes(const LayerParams &p, uint32_t stage_addr, uint32_t tmem_base, int tile_in_stage,
                                                 uint32_t idesc, uint32_t &slot_it, uint32_t tfull0, uint32_t tempty0) {
    if constexpr (PASS < C::PASSES) {
        const int slot = (int)(slot_it % (uint32_t)C::NSLOT);
        tc::mbar_wait(tempty0 + 8u * (uint32_t)slot, ((slot_it / (uint32_t)C::NSLOT) & 1u) ^ 1u, p.watchdog, 4u);
        tc::tc_fence_after();
        if (!(p.dbg & 1))
            issue_pass<C, PASS>(p, stage_addr, tmem_base, tmem_base + (uint32_t)(C::A_COLS + slot * C::NP), tile_in_stage, idesc);
        tc::umma_commit(tfull0 + 8u * (uint32_t)slot);
        slot_it++;
        issue_all_passes<C, PASS + 1>(p, stage_addr, tmem_base, tile_in_stage, idesc, slot_it, tfull0, tempty0);
    }
}

// ---- epilogue pieces ---------------------------------------------------------------------------------
// tcgen05.ld.16x256b.x2: of the 16-lane x 16-column block at taddr, thread i receives, for column block k = 0, 1
// (8 columns each): row (i/4), columns 8k + 2*(i%4) + {0,1} in r[4k + 0..1] and row (i/4 + 8), same columns, in
// r[4k + 2..3]  (layout verified by tools/tmem_layout_test.cu)
__device__ __forceinline__ void tmem_ld_16x256b_x2(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.16x256b.x2.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]) : "r"(taddr));
}
// One 16-column unit (4 pixels x 4 frames) of one accumulator slot: both 16-lane halves of this warp's TMEM lane
// quarter -> max over the pooling phases that live in lanes, folded into the running maximum over passes.
//   v[item][2k + c]: column block k (pixels 2k, 2k+1), this thread's column pair c = frames 2*(lane&1) + c of
//   pixel 2k + ((lane >> 1) & 1); item = channel block (NIT = 4/PL of them; channel = lane/4 of each block)
template <class C, bool FIRST>
__device__ __forceinline__ void pool_unit(const uint32_t (&a0)[8], const uint32_t (&a1)[8], float (&v)[C::NIT][4]) {
#pragma unroll
    for (int k = 0; k < 2; k++)
#pragma unroll
        for (int c = 0; c < 2; c++) {
            const float r00 = __uint_as_float(a0[4 * k + c]), r01 = __uint_as_float(a0[4 * k + 2 + c]);
            const float r10 = __uint_as_float(a1[4 * k + c]), r11 = __uint_as_float(a1[4 * k + 2 + c]);
            const int o = 2 * k + c;
            if constexpr (C::PL == 4) {
                v[0][o] = FIRST ? fmaxf(fmax3(r00, r01, r10), r11) : fmax3(fmax3(r00, r01, r10), r11, v[0][o]);
            } else if constexpr (C::PL == 2) {
                v[0][o] = FIRST ? fmaxf(r00, r01) : fmax3(r00, r01, v[0][o]);
                v[1][o] = FIRST ? fmaxf(r10, r11) : fmax3(r10, r11, v[1][o]);
            } else {
                v[0][o] = FIRST ? r00 : fmaxf(r00, v[0][o]); v[1][o] = FIRST ? r01 : fmaxf(r01, v[1][o]);
                v[2][o] = FIRST ? r10 : fmaxf(r10, v[2][o]); v[3][o] = FIRST ? r11 : fmaxf(r11, v[3][o]);
            }
        }
}

// 2-byte store to a global address held as an opaque 64-bit value (see the asm barrier on outb / out2b in the kernel)
template <int OFF>
__device__ __forceinline__ void stg_h(const unsigned char *addr, float v) {
    asm volatile("st.global.b16 [%0 + %2], %1;" ::"l"(addr), "h"(__half_as_ushort(__float2half_rn(v))), "n"(OFF) : "memory");
}

struct EpiItem {
    float sgn, bias, scale, shift;
};

// One unit, all items of this thread.  The lane pair (lane ^ 1) first swaps column pairs so that each thread owns
// all four frames of ONE pixel (th = 0: pixel of block 0, th = 1: pixel of block 1); then bias -> ReLU -> BatchNorm,
// PointWiseTN over the 4 frames entirely in registers (packed fp32 pairs, TN weights straight from the kernel
// parameters), fp16, store.  All lanes must call (shuffles); stores are predicated.
// orow / srow: 16-byte row index of (channel block 0, this thread's pixel, t = 0) in out / out2;
// outb / out2b: byte address of this thread's channel inside row 0 of out / out2.
template <class C>
__device__ __forceinline__ void finalize_unit(const LayerParams &p, const float (&v)[C::NIT][4], const EpiItem (&ecr)[C::NIT],
                                              const float4 *ecs, bool th, bool valid, unsigned char *outb, unsigned char *out2b,
                                              uint32_t orow, uint32_t srow, uint32_t step_o, uint32_t step_s) {
#pragma unroll
    for (int it = 0; it < C::NIT; it++) {
        // th = 0 keeps block 0 (frames 0,1 of its pixel) and receives frames 2,3 of it from the partner's block 0;
        // th = 1 keeps block 1 (frames 2,3) and receives frames 0,1 of that pixel from the partner's block 1
        const float g0 = th ? v[it][0] : v[it][2], g1 = th ? v[it][1] : v[it][3];
        const float k0 = th ? v[it][2] : v[it][0], k1 = th ? v[it][3] : v[it][1];
        const float r0 = __shfl_xor_sync(0xffffffffu, g0, 1), r1 = __shfl_xor_sync(0xffffffffu, g1, 1);
        const float2 in01 = make_float2(th ? r0 : k0, th ? r1 : k1), in23 = make_float2(th ? k0 : r0, th ? k1 : r1);
        EpiItem ec[1];
        if constexpr (C::NIT >= 4) {
            const float4 e = ecs[it * 8];
            ec[0].sgn = e.x; ec[0].bias = e.y; ec[0].scale = e.z; ec[0].shift = e.w;
        } else {
            ec[0] = ecr[it];
        }
        const float2 x01 = ffma2(relu2(ffma2(in01, bc2(ec[0].sgn), bc2(ec[0].bias))), bc2(ec[0].scale), bc2(ec[0].shift));
        const float2 x23 = ffma2(relu2(ffma2(in23, bc2(ec[0].sgn), bc2(ec[0].bias))), bc2(ec[0].scale), bc2(ec[0].shift));
        // h1[m] = relu(sum_t x[t] * W1[t][m])      (pointwise.py:18-21)
        float2 h01 = fmul2(bc2(x01.x), make_float2(p.tn_w1[0], p.tn_w1[1])), h23 = fmul2(bc2(x01.x), make_float2(p.tn_w1[2], p.tn_w1[3]));
        h01 = ffma2(bc2(x01.y), make_float2(p.tn_w1[4], p.tn_w1[5]), h01);   h23 = ffma2(bc2(x01.y), make_float2(p.tn_w1[6], p.tn_w1[7]), h23);
        h01 = ffma2(bc2(x23.x), make_float2(p.tn_w1[8], p.tn_w1[9]), h01);   h23 = ffma2(bc2(x23.x), make_float2(p.tn_w1[10], p.tn_w1[11]), h23);
        h01 = ffma2(bc2(x23.y), make_float2(p.tn_w1[12], p.tn_w1[13]), h01); h23 = ffma2(bc2(x23.y), make_float2(p.tn_w1[14], p.tn_w1[15]), h23);
        h01 = relu2(h01); h23 = relu2(h23);
        // y[to] = relu(x[to] + relu(sum_m h1[m] * W2[m][to]))      (pointwise.py:22-26); relu(x + relu(h)) = max(x + h, x, 0)
        float2 y01 = ffma2(bc2(h01.x), make_float2(p.tn_w2[0], p.tn_w2[1]), x01);
        y01 = ffma2(bc2(h01.y), make_float2(p.tn_w2[4], p.tn_w2[5]), y01);
        y01 = ffma2(bc2(h23.x), make_float2(p.tn_w2[8], p.tn_w2[9]), y01);
        y01 = ffma2(bc2(h23.y), make_float2(p.tn_w2[12], p.tn_w2[13]), y01);
        const float o0 = fmax3(y01.x, x01.x, 0.f), o1 = fmax3(y01.y, x01.y, 0.f);
        if constexpr (C::HAS_OUT) {
            float2 y23 = ffma2(bc2(h01.x), make_float2(p.tn_w2[2], p.tn_w2[3]), x23);
            y23 = ffma2(bc2(h01.y), make_float2(p.tn_w2[6], p.tn_w2[7]), y23);
            y23 = ffma2(bc2(h23.x), make_float2(p.tn_w2[10], p.tn_w2[11]), y23);
            y23 = ffma2(bc2(h23.y), make_float2(p.tn_w2[14], p.tn_w2[15]), y23);
            const float o2 = fmax3(y23.x, x23.x, 0.f), o3 = fmax3(y23.y, x23.y, 0.f);
            if (valid) {
                const unsigned char *dst = outb + (size_t)(orow + (uint32_t)it * step_o) * 16;     // rows t = 0..3 are consecutive
                stg_h<0>(dst, o0); stg_h<16>(dst, o1); stg_h<32>(dst, o2); stg_h<48>(dst, o3);
            }
        }
        if (valid) stg_h<0>(out2b + (size_t)(srow + (uint32_t)it * step_s) * 16, o0);
    }
}

// ------------------------------------------------------------------------------------------------ kernel
template <class C>
__global__ void __launch_bounds__(C::THREADS, 1) enc_ws_kernel(const __grid_constant__ LayerParams p, const __grid_constant__ ELayerExtra ex) {
    extern __shared__ __align__(1024) unsigned char smem[];
    const SmemPlanE sp = plan_smem_e<C>(p.Ls, p.n_stage);
    const uint32_t smem_base = tc::smem_u32(smem);
    float *epi = reinterpret_cast<float *>(smem + sp.epi_off);
    const uint32_t bar0 = smem_base + sp.bar_off;
    const uint32_t full0 = bar0, empty0 = bar0 + 8u * kMaxStage, tfull0 = bar0 + 8u * 2 * kMaxStage,
                   tempty0 = bar0 + 8u * (2 * kMaxStage + kMaxSlot);
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + sp.bar_off + 8 * (2 * kMaxStage + 2 * kMaxSlot));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int cta = (int)blockIdx.x, n_cta = (int)gridDim.x;
    pdl_launch_dependents();

    for (int i = threadIdx.x; i < 4 * C::COUT + 32; i += C::THREADS) {
        float v;
        if (i >= 4 * C::COUT) v = (i - 4 * C::COUT < 16) ? p.tn_w1[i - 4 * C::COUT] : p.tn_w2[i - 4 * C::COUT - 16];
        else v = p.epi[i];
        epi[i < 4 * C::COUT ? (i % C::COUT) * 4 + i / C::COUT : i] = v;      // per channel: {sgn, bias, scale, shift}
    }
    if (threadIdx.x == 0) {
        for (int s = 0; s < kMaxStage; s++) { tc::mbar_init(full0 + 8u * s, 1); tc::mbar_init(empty0 + 8u * s, 1); }
        for (int s = 0; s < kMaxSlot; s++) { tc::mbar_init(tfull0 + 8u * s, 1); tc::mbar_init(tempty0 + 8u * s, C::EW); }
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

    // weights -> TMEM (A operand): row m = 32*q + lane, 8 columns (16 fp16) per block
    if (warp >= 2) {
        const int q = warp & 3, cq = (warp - 2) >> 2;
        const uint4 *src = p.wpack + (size_t)(q * 32 + lane) * 2;
        for (int blk = cq; blk < C::NBLK; blk += C::CS) {
            const uint4 a = __ldg(src + (size_t)blk * 256), b = __ldg(src + (size_t)blk * 256 + 1);
            tmem_st8(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(blk * 8), a, b);
        }
        tmem_wait_st();
    }
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    pdl_wait();              // prologue done (weights in TMEM); activations of the preceding layer from here on

    if (warp == 0) {
        // ===== producer: one strip set per group of TPS tiles =====
        if (tc::elect_one()) {
            uint32_t it = 0;
            for (int g = cta; g < p.n_groups; g += n_cta, it++) {
                const long long pos0 = p.gin.guard + (long long)g * C::TPS * C::NP - p.gin.halo;
                const int s = (int)(it % (uint32_t)p.n_stage);
                tc::mbar_wait(empty0 + 8u * s, ((it / (uint32_t)p.n_stage) & 1u) ^ 1u, p.watchdog, 1u);
                tc::mbar_expect_tx(full0 + 8u * s, sp.stage_bytes);
                const uint32_t dst0 = smem_base + sp.stage_off + (uint32_t)s * sp.stage_bytes;
#pragma unroll 1
                for (int cbi = 0; cbi < C::CIN_CB; cbi++)
#pragma unroll
                    for (int pl = 0; pl < 4; pl++)
                        tc::bulk_g2s(dst0 + (uint32_t)((cbi * 4 + pl) * p.Ls) * 16u, p.in + geom_row(p.gin, cbi, pl, pos0),
                                     (uint32_t)p.Ls * 16u, full0 + 8u * s);
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        if (tc::elect_one()) {
            constexpr uint32_t idesc = tc::make_idesc(C::NP);
            uint32_t it = 0, slot_it = 0;
            for (int g = cta; g < p.n_groups; g += n_cta, it++) {
                const int s = (int)(it % (uint32_t)p.n_stage);
                tc::mbar_wait(full0 + 8u * s, (it / (uint32_t)p.n_stage) & 1u, p.watchdog, 3u);
                tc::tc_fence_after();
                const uint32_t stage_addr = smem_base + sp.stage_off + (uint32_t)s * sp.stage_bytes;
#pragma unroll 1
                for (int j = 0; j < C::TPS; j++) {
                    if ((g * C::TPS + j) >= p.n_tiles) break;
                    issue_all_passes<C, 0>(p, stage_addr, tmem_base, j, idesc, slot_it, tfull0, tempty0);
                }
                tc::umma_commit(empty0 + 8u * s);
            }
        }
    } else {
        // ===== epilogue warps =====
        const int q = warp & 3, cq = (warp - 2) >> 2;
        const uint32_t jch = (uint32_t)(lane >> 2);
        const bool th = lane & 1;
        const int pix_in_unit = 2 * (lane & 1) + ((lane >> 1) & 1);        // the pixel this thread finalises
        const int n_my = C::UB + (cq < C::UR ? 1 : 0);
        const int u_begin = cq * C::UB + (cq < C::UR ? cq : C::UR);
        // per-channel epilogue constants: in registers for one or two items, re-read from shared memory for four
        const float4 *ecs = reinterpret_cast<const float4 *>(epi) + (q * C::NIT * 8 + (int)jch);
        EpiItem ec[C::NIT];
#pragma unroll
        for (int it = 0; it < C::NIT; it++) {
            const float4 e = ecs[it * 8];
            ec[it].sgn = e.x; ec[it].bias = e.y; ec[it].scale = e.z; ec[it].shift = e.w;
        }
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(C::A_COLS + u_begin * 16);
        const uint32_t step_o = 4u * (uint32_t)p.gout.Lp, step_s = 4u * (uint32_t)p.gout2.Lp;
        const uint32_t base_o = (uint32_t)(q * C::NIT) * step_o + (uint32_t)p.gout.guard;
        const uint32_t base_s = (uint32_t)(p.out2_cb + q * C::NIT) * step_s + (uint32_t)p.gout2.guard;
        unsigned char *outb = reinterpret_cast<unsigned char *>(p.out) + jch * 2u;
        unsigned char *out2b = reinterpret_cast<unsigned char *>(p.out2) + jch * 2u;
        asm volatile("" : "+l"(outb), "+l"(out2b));          // keep both in registers: ptxas otherwise re-derives them per unit
        // Software pipeline over this CTA's tiles: the accumulators of tile i+1 are read (and the slot released) pass by
        // pass as they complete, interleaved with the finalisation of tile i out of registers - so the MMA warp never
        // waits for a finalisation and the epilogue never waits for a pass it could have had earlier.
        uint32_t slot_it = 0;
        // this CTA's tiles in order: groups cta, cta + n_cta, ... of TPS consecutive tiles; only the last group of the launch
        // can be partial, so the first tile index beyond n_tiles ends the sequence (the producer and the MMA warp walk the
        // same sequence).  Kept to a handful of instructions: the first version of this iterator was 11 % of the kernel's
        // warp instructions (profiles/r2v_enc2_lines.txt).
        int g_next = cta, jt_next = 0, t_next = cta * C::TPS;
        auto next_tile = [&]() -> int {
            if (g_next >= p.n_groups || t_next >= p.n_tiles) { g_next = p.n_groups; return -1; }
            const int t = t_next;
            if (++jt_next == C::TPS) { jt_next = 0; g_next += n_cta; t_next = g_next * C::TPS; } else { t_next++; }
            return t;
        };
        float run_cur[C::MAXU][C::NIT][4];
        uint32_t cur_o = 0, cur_s = 0, cur_vmask = 0, cur_vmine = 0;   // cur_vmine: validity bits of this thread's pixel of every unit
        bool have_cur = false;
        int tile = next_tile();
        while (tile >= 0 || have_cur) {
            float run_nxt[C::MAXU][C::NIT][4];
            uint32_t nxt_o = 0, nxt_s = 0, nxt_vmask = 0;
            if (tile >= 0) {
                // output rows of this warp's 4*n_my pixels: lane L computes pixel L once per tile, the units fetch theirs
                // with shuffles (every pixel is shared by 8 lanes x 4 lane quarters)
                bool tab_valid = false;
                if (lane < 4 * n_my) {
                    const Geom &gi = p.gin;
                    const uint32_t qq = (uint32_t)tile * (C::NP / 4) + (uint32_t)(u_begin * 4 + lane);
                    const uint32_t n = fast_div(qq, ex.divS);
                    const uint32_t r = qq - n * (uint32_t)gi.S;
                    const uint32_t y2 = fast_div(r, ex.divP), x2 = r - y2 * (uint32_t)gi.P;
                    tab_valid = (int)n < p.N && (int)y2 < (gi.H >> 1) && (int)x2 < (gi.W >> 1);
                    const uint32_t Y = y2 + (uint32_t)(gi.H & 1), X = x2 + (uint32_t)(gi.W & 1);   // zero-pad top / left when odd (encoder.py:68-76)
                    const uint32_t pho = ((Y & 1) << 1) | (X & 1);
                    nxt_o = base_o + pho * (uint32_t)p.gout.Lp + ((n * (uint32_t)p.gout.S + (Y >> 1) * (uint32_t)p.gout.P + (X >> 1)) << 2);
                    nxt_s = base_s + pho * (uint32_t)p.gout2.Lp + n * (uint32_t)p.gout2.S + (Y >> 1) * (uint32_t)p.gout2.P + (X >> 1);
                }
                nxt_vmask = __ballot_sync(0xffffffffu, tab_valid);
            }
#pragma unroll
            for (int ps = 0; ps < C::PASSES; ps++) {
                if (tile >= 0) {
                    const int slot = (int)(slot_it % (uint32_t)C::NSLOT);
                    tc::mbar_wait(tfull0 + 8u * slot, (slot_it / (uint32_t)C::NSLOT) & 1u, p.watchdog, 5u);
                    tc::tc_fence_after();
                    if (!(p.dbg & 2)) {
                        if constexpr (C::PASSES == 1) {
                            uint32_t a[C::MAXU][2][8];                        // all loads in flight, one wait
#pragma unroll
                            for (int u = 0; u < C::MAXU; u++)
                                if (u < n_my) {
                                    tmem_ld_16x256b_x2(lane_addr + (uint32_t)(slot * C::NP + u * 16), a[u][0]);
                                    tmem_ld_16x256b_x2(lane_addr + (16u << 16) + (uint32_t)(slot * C::NP + u * 16), a[u][1]);
                                }
                            tc::tmem_wait_ld();
#pragma unroll
                            for (int u = 0; u < C::MAXU; u++)
                                if (u < n_my) pool_unit<C, true>(a[u][0], a[u][1], run_nxt[u]);
                        } else {
#pragma unroll
                            for (int u = 0; u < C::MAXU; u++)
                                if (u < n_my) {
                                    uint32_t a[2][8];
                                    tmem_ld_16x256b_x2(lane_addr + (uint32_t)(slot * C::NP + u * 16), a[0]);
                                    tmem_ld_16x256b_x2(lane_addr + (16u << 16) + (uint32_t)(slot * C::NP + u * 16), a[1]);
                                    tc::tmem_wait_ld();
                                    if (ps == 0) pool_unit<C, true>(a[0], a[1], run_nxt[u]);
                                    else pool_unit<C, false>(a[0], a[1], run_nxt[u]);
                                }
                        }
                    }
                    tc::tc_fence_before();
                    __syncwarp();
                    if (lane == 0) tc::mbar_arrive(tempty0 + 8u * slot);
                    slot_it++;
                }
                if (have_cur && !(p.dbg & 2)) {
                    // finalise this pass's share of the previous tile's units
                    const int u_lo = ps * C::MAXU / C::PASSES, u_hi = (ps + 1) * C::MAXU / C::PASSES;
#pragma unroll
                    for (int u = 0; u < C::MAXU; u++)
                        if (u >= u_lo && u < u_hi && u < n_my && ((cur_vmask >> (4 * u)) & 15u)) {   // warp-uniform: skip padding units
                            const uint32_t orow = __shfl_sync(0xffffffffu, cur_o, 4 * u + pix_in_unit);
                            const uint32_t srow = __shfl_sync(0xffffffffu, cur_s, 4 * u + pix_in_unit);
                            finalize_unit<C>(p, run_cur[u], ec, ecs, th, (cur_vmine & (1u << (4 * u))) != 0u, outb, out2b, orow, srow, step_o, step_s);
                        }
                }
            }
            have_cur = tile >= 0;
            if (have_cur) {
#pragma unroll
                for (int u = 0; u < C::MAXU; u++)
#pragma unroll
                    for (int it = 0; it < C::NIT; it++)
#pragma unroll
                        for (int c = 0; c < 4; c++) run_cur[u][it][c] = run_nxt[u][it][c];
                cur_o = nxt_o; cur_s = nxt_s; cur_vmask = nxt_vmask; cur_vmine = nxt_vmask >> pix_in_unit;
                tile = next_tile();
            }
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 1) tc::tmem_dealloc(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------------ launch
// as tc::plan / tc::launch
template <class C>
inline bool plan_e(LayerParams &p, int n_sms, int min_stage, tc::Grid &g) {
    const long long mtot = (long long)p.N * p.gin.S * p.gin.Tn;
    if (mtot >= (1ll << 31)) return false;
    p.n_tiles = (int)((mtot + C::NP - 1) / C::NP);
    p.n_groups = (p.n_tiles + C::TPS - 1) / C::TPS;
    p.Ls = C::TPS * C::NP + 2 * p.gin.halo;
    if (4 * p.Ls >= 16384 || p.gin.P >= 16384) return false;
    if (p.gin.guard + (long long)p.n_groups * C::TPS * C::NP + p.gin.halo > p.gin.Lp) return false;
    for (p.n_stage = kMaxStage; p.n_stage >= 1; p.n_stage--)
        if (plan_smem_e<C>(p.Ls, p.n_stage).total <= (uint32_t)tc::kSmemLimit) break;
    if (p.n_stage < min_stage) return false;
    g.smem = plan_smem_e<C>(p.Ls, p.n_stage).total;
    g.ctas = std::max(1, std::min(n_sms, p.n_groups));
    return true;
}

template <class C>
inline cudaError_t launch_e(const LayerParams &p, const tc::Grid &g, cudaStream_t st) {
    if ((p.out != nullptr) != C::HAS_OUT || !p.out2) return cudaErrorInvalidValue;   // output set is part of the configuration (ECfg::HAS_OUT)
    cudaError_t err = cudaFuncSetAttribute(enc_ws_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::kSmemLimit);   // see tc::launch
    if (err != cudaSuccess) return err;
    ELayerExtra ex;
    ex.divS = make_fastdiv((uint32_t)p.gin.S);
    ex.divP = make_fastdiv((uint32_t)p.gin.P);
    return launch_pdl(enc_ws_kernel<C>, dim3((unsigned)g.ctas), dim3(C::THREADS), g.smem, st, !(p.dbg & kDbgNoPdl), p, ex);
}

}  // namespace tcs
}  // namespace cova
