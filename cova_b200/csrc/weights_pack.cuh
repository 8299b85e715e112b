// Host-side parsing of the CVBN v1 weight container and packing into the operand layouts the
// kernels consume.  Container layout: see cova_b200/weights.py (torch tensor layouts, fp32).
//
// What is folded here, in fp32, before the one rounding to fp16:
//   * preprocessing 1/6 (reference utils/model/preprocessing.py:5-8) into the first conv's weights
//     (the kernel feeds the clipped integers 0..6, which are exact in fp16);
//   * BatchNorm (eps 1e-3) into a per-channel scale/shift applied in the epilogues (it sits AFTER the
//     ReLU and BEFORE the max-pool in the encoder - reference encoder.py:63-66 - so it cannot be folded
//     into the conv weights there; in the decoder it directly follows the bias and is folded);
//   * the 1x1 head conv (reference decoder.py:118,131) into the last transposed conv: no
//     non-linearity sits between them, so dec3 + head is a transposed conv with ONE output channel.
#pragma once
#include "common.cuh"

namespace cova {

struct HostWeights {
    struct Enc { const float *conv_w, *conv_b, *gamma, *beta, *mean, *var, *tn_w1, *tn_w2; } enc[4];
    struct Dec { const float *convt_w, *convt_b, *gamma, *beta, *mean, *var; } dec[4];
    const float *head_w, *head_b;
    std::vector<float> storage;
    size_t off_enc[4][8], off_dec[4][6], off_head[2];   // float offsets into storage (mirrored on device)
};

// Finite values the kernels still cannot represent, refused instead of turning into NaN / Inf outputs: a negative
// variance (NaN BatchNorm scale), a BatchNorm scale, shift or offset that overflows fp32, and a weight whose fp16 image
// overflows (|v| >= 65520 rounds to Inf): W / 6 in block 1, W in the other layers, the head folded into dec3.  Each
// value is computed by the expression the packing (below) uses.  Keras never leaves a negative moving variance.
inline int check_weights(const HostWeights &hw) {
    char name[32];
    auto bad = [&](const char *what) { return set_err(COVA_E_WEIGHTS, "CVBN %s: %s", name, what); };
    auto fp16_ok = [](float v) { return fabsf(v) < 65520.f; };
    auto scale_ok = [&](const float *gamma, const float *var, int c, float &s) {
        s = gamma[c] / sqrtf(var[c] + kBnEps);
        return std::isfinite(s);
    };
    for (int i = 0; i < 4; i++) {
        const auto &e = hw.enc[i];
        const size_t co_n = kEncCout[i], n_w = co_n * kEncCin[i] * 9;
        snprintf(name, sizeof(name), "enc%d.conv_w", i);
        for (size_t k = 0; k < n_w; k++)
            if (!fp16_ok(i == 0 ? e.conv_w[k] / 6.0f : e.conv_w[k]))
                return bad(i == 0 ? "a weight / 6 overflows fp16" : "a weight overflows fp16");
        for (size_t c = 0; c < co_n; c++) {
            float s;
            snprintf(name, sizeof(name), "enc%d.bn_var", i);
            if (e.var[c] < 0.f) return bad("negative variance");
            snprintf(name, sizeof(name), "enc%d.bn_gamma", i);
            if (!scale_ok(e.gamma, e.var, (int)c, s)) return bad("the BatchNorm scale overflows fp32");
            snprintf(name, sizeof(name), "enc%d.bn_mean", i);
            if (!std::isfinite(e.beta[c] - e.mean[c] * s)) return bad("the BatchNorm shift overflows fp32");
        }
    }
    for (int i = 0; i < 4; i++) {
        const auto &d = hw.dec[i];
        const size_t co_n = kDecCout[i], n_w = co_n * kDecCin[i] * 16;
        snprintf(name, sizeof(name), "dec%d.convt_w", i);
        if (i < 3)
            for (size_t k = 0; k < n_w; k++)
                if (!fp16_ok(d.convt_w[k])) return bad("a weight overflows fp16");
        for (size_t c = 0; i < 3 && c < co_n; c++) {
            float s;
            snprintf(name, sizeof(name), "dec%d.bn_var", i);
            if (d.var[c] < 0.f) return bad("negative variance");
            snprintf(name, sizeof(name), "dec%d.bn_gamma", i);
            if (!scale_ok(d.gamma, d.var, (int)c, s)) return bad("the BatchNorm scale overflows fp32");
            snprintf(name, sizeof(name), "dec%d.bn_mean", i);
            if (!std::isfinite((d.convt_b[c] - d.mean[c]) * s + d.beta[c])) return bad("the BatchNorm offset overflows fp32");
        }
    }
    // dec3 + head: fold[ci][ky][kx] = sum_co W[ci][co][ky][kx] * head_w[co] in double, rounded to fp32 then fp16
    const int ci_n = kDecCin[3], co_n = kDecCout[3];
    snprintf(name, sizeof(name), "head_w");
    for (int ci = 0; ci < ci_n; ci++)
        for (int k = 0; k < 16; k++) {
            double acc = 0;
            for (int co = 0; co < co_n; co++) acc += (double)hw.dec[3].convt_w[((size_t)ci * co_n + co) * 16 + k] * hw.head_w[co];
            if (!fp16_ok((float)acc)) return bad("dec3.convt_w folded with the head overflows fp16");
        }
    double c0 = hw.head_b[0];
    for (int co = 0; co < co_n; co++) c0 += (double)hw.head_w[co] * hw.dec[3].convt_b[co];
    snprintf(name, sizeof(name), "head_b");
    if (!std::isfinite((float)c0)) return bad("head_b + head_w . dec3.convt_b overflows fp32");
    return COVA_OK;
}

inline int parse_weights(const void *blob, size_t len, HostWeights &hw) {
    if (!blob || len < 16) return set_err(COVA_E_WEIGHTS, "weight blob too short");
    const uint32_t *h = static_cast<const uint32_t *>(blob);
    if (h[0] != 0x4E425643u || h[1] != 1u || h[2] != (uint32_t)kT)
        return set_err(COVA_E_WEIGHTS, "not a CVBN v1 container (magic/version/timestep)");
    size_t need = 0;
    for (int i = 0; i < 4; i++) need += (size_t)kEncCout[i] * kEncCin[i] * 9 + 5 * (size_t)kEncCout[i] + 32;
    for (int i = 0; i < 4; i++) need += (size_t)kDecCin[i] * kDecCout[i] * 16 + (size_t)kDecCout[i] * (i < 3 ? 5 : 1);
    need += kDecCout[3] + 1;
    if (len != 16 + need * 4) return set_err(COVA_E_WEIGHTS, "CVBN container has the wrong length");
    hw.storage.resize(need);
    memset(hw.off_enc, 0, sizeof(hw.off_enc)); memset(hw.off_dec, 0, sizeof(hw.off_dec));
    memcpy(hw.storage.data(), static_cast<const char *>(blob) + 16, need * 4);
    size_t o = 0;
    auto take = [&](size_t n, size_t &slot) { slot = o; o += n; return hw.storage.data() + slot; };
    for (int i = 0; i < 4; i++) {
        size_t co = kEncCout[i], ci = kEncCin[i];
        hw.enc[i].conv_w = take(co * ci * 9, hw.off_enc[i][0]);
        hw.enc[i].conv_b = take(co, hw.off_enc[i][1]);
        hw.enc[i].gamma = take(co, hw.off_enc[i][2]);
        hw.enc[i].beta = take(co, hw.off_enc[i][3]);
        hw.enc[i].mean = take(co, hw.off_enc[i][4]);
        hw.enc[i].var = take(co, hw.off_enc[i][5]);
        hw.enc[i].tn_w1 = take(16, hw.off_enc[i][6]);
        hw.enc[i].tn_w2 = take(16, hw.off_enc[i][7]);
    }
    for (int i = 0; i < 4; i++) {
        size_t co = kDecCout[i], ci = kDecCin[i];
        hw.dec[i].convt_w = take(ci * co * 16, hw.off_dec[i][0]);
        hw.dec[i].convt_b = take(co, hw.off_dec[i][1]);
        if (i < 3) {
            hw.dec[i].gamma = take(co, hw.off_dec[i][2]);
            hw.dec[i].beta = take(co, hw.off_dec[i][3]);
            hw.dec[i].mean = take(co, hw.off_dec[i][4]);
            hw.dec[i].var = take(co, hw.off_dec[i][5]);
        } else {
            hw.dec[i].gamma = hw.dec[i].beta = hw.dec[i].mean = hw.dec[i].var = nullptr;
        }
    }
    hw.head_w = take(kDecCout[3], hw.off_head[0]);
    hw.head_b = take(1, hw.off_head[1]);
    for (float v : hw.storage)
        if (!(v == v) || v > 3e38f || v < -3e38f) return set_err(COVA_E_WEIGHTS, "CVBN container holds NaN/Inf");
    return check_weights(hw);
}

inline int floor_div2(int v) { return v >= 0 ? v / 2 : -((-v + 1) / 2); }

// ---- B-operand blocks: one block = N rows x 16 K, canonical K-major no-swizzle core matrices:
//      half index of (n, k) inside a block = ((k >> 3) * N + n) * 8 + (k & 7)
inline void put_b(std::vector<__half> &dst, size_t block, int N, int n, int k, float v) {
    dst[block * (size_t)N * 16 + ((size_t)(k >> 3) * N + n) * 8 + (k & 7)] = __float2half_rn(v);
}

struct PackedLayer {
    std::vector<__half> b;     // B blocks
    std::vector<float> epi;    // epilogue constants
    int n_cols = 0;            // N of one MMA
    int blocks = 0;
};

// Encoder layer i: blocks indexed [tap][kpair] (i >= 1) or [phase][step] (i == 0); epi = bias|scale|shift
inline void pack_encoder(const HostWeights &hw, int i, PackedLayer &pl) {
    const int ci_n = kEncCin[i], co_n = kEncCout[i];
    const auto &e = hw.enc[i];
    auto W = [&](int co, int ci, int dy, int dx) { return e.conv_w[((size_t)(co * ci_n + ci) * 3 + (dy + 1)) * 3 + (dx + 1)]; };
    pl.n_cols = co_n;
    if (i == 0) {
        // frame-level first conv on x-pair-packed rows (blobnet_tc.cuh, issue_tile<ENCF>): 6 blocks of N = 64
        // rows (4 phases x 16 channels) x K = 16 (two operand tiles of 8: [c0 c1 c2 0 | c0' c1' c2' 0]).
        pl.blocks = 6;
        pl.n_cols = 4 * co_n;
        pl.b.assign((size_t)pl.blocks * pl.n_cols * 16, __float2half_rn(0.f));
        for (int st = 0; st < 6; st++)
            for (int half = 0; half < 2; half++) {
                int u, sx;
                if (st < 4) { u = st - 1; sx = half - 1; }
                else { u = (st == 4 ? 0 : -1) + 2 * half; sx = 1; }
                for (int ph = 0; ph < 4; ph++) {
                    const int a = ph >> 1, b = ph & 1, dy = u - a;
                    if (dy < -1 || dy > 1) continue;
                    for (int bp = 0; bp < 2; bp++) {                 // b' = pixel of the pair
                        const int dx = 2 * sx + bp - b;
                        if (dx < -1 || dx > 1) continue;
                        for (int co = 0; co < co_n; co++)
                            for (int ci = 0; ci < ci_n; ci++)
                                put_b(pl.b, st, pl.n_cols, ph * co_n + co, half * 8 + bp * 4 + ci, W(co, ci, dy, dx) / 6.0f);
                    }
                }
            }
    } else if (co_n <= 64) {
        // "paired column phases" (blobnet_tc.cuh, Cfg::PAIR): per (dy, kpair) four operand blocks, one per input column
        // offset v = -1..2 relative to the pooled pixel: v = -1 feeds only column phase b = 0 (tap dx = -1), v = 2 only
        // b = 1 (dx = +1): N = Cout; v = 0 and v = 1 feed both phases with taps dx = v (b = 0) and dx = v - 1 (b = 1):
        // N = 2*Cout, rows [phase 0 | phase 1] - one MMA instead of two.  Rows of a (dy, kpair) group: Cout * {1, 2, 2, 1}.
        const int kp_n = ci_n / 16;
        pl.blocks = 3 * kp_n * 6;                                  // in units of Cout rows
        pl.b.assign((size_t)pl.blocks * co_n * 16, __float2half_rn(0.f));
        const int voff[4] = {0, 1, 3, 5};                          // start of block v + 1 inside its group, in units of Cout rows
        for (int dy = -1; dy <= 1; dy++)
            for (int kp = 0; kp < kp_n; kp++)
                for (int iv = 0; iv < 4; iv++) {
                    const int v = iv - 1, N = (iv == 1 || iv == 2) ? 2 * co_n : co_n;
                    __half *blk = pl.b.data() + ((size_t)((dy + 1) * kp_n + kp) * 6 + voff[iv]) * co_n * 16;
                    for (int n = 0; n < N; n++) {
                        const int b = iv == 3 ? 1 : n / co_n, co = n % co_n, dx = v - b;   // single-phase blocks: b = 0 (v = -1) or 1 (v = 2)
                        for (int k = 0; k < 16; k++)
                            blk[((size_t)(k >> 3) * N + n) * 8 + (k & 7)] = __float2half_rn(W(co, kp * 16 + k, dy, dx));
                    }
                }
    } else {
        const int kp_n = ci_n / 16;
        pl.blocks = 9 * kp_n;
        pl.b.assign((size_t)pl.blocks * co_n * 16, __float2half_rn(0.f));
        for (int tp = 0; tp < 9; tp++)
            for (int kp = 0; kp < kp_n; kp++)
                for (int co = 0; co < co_n; co++)
                    for (int k = 0; k < 16; k++)
                        put_b(pl.b, tp * kp_n + kp, co_n, co, k, W(co, kp * 16 + k, tp / 3 - 1, tp % 3 - 1));
    }
    pl.epi.resize(3 * co_n);
    for (int co = 0; co < co_n; co++) {
        float s = e.gamma[co] / sqrtf(e.var[co] + kBnEps);
        pl.epi[co] = e.conv_b[co];
        pl.epi[co_n + co] = s;
        pl.epi[2 * co_n + co] = e.beta[co] - e.mean[co] * s;
    }
}


// Encoder layer i (>= 1) for the weights-stationary kernel (blobnet_enc.cuh): A blocks [iu][iv][kpair], each
// 128 rows x 16 K (fp16, 32 bytes per row); row m = 32*q + cbl*(8*PL) + lph*8 + j holds output channel
// (q*CBQ + cbl)*8 + j of lane phase lph = (la, lb).  LA / LB = 2 puts the row / column pooling phase into M
// ("union of taps": offset u = iu - 1 in [-1, 2] serves tap dy = u - la when that is in [-1, 1]); otherwise the
// phase is a separate pass and iu indexes the tap directly.  Channels with a negative BatchNorm scale are
// negated (sgn = -1): max-pooling -conv yields -min(conv), which is what MaxPool(BN(ReLU(.))) needs there.
// epi = sgn | bias | scale | shift.
inline void pack_encoder_ws(const HostWeights &hw, int i, int LA, int LB, PackedLayer &pl) {
    const int ci_n = kEncCin[i], co_n = kEncCout[i], kp_n = ci_n / 16;
    const auto &e = hw.enc[i];
    auto W = [&](int co, int ci, int dy, int dx) { return e.conv_w[((size_t)(co * ci_n + ci) * 3 + (dy + 1)) * 3 + (dx + 1)]; };
    const int PL = LA * LB, NU = LA == 2 ? 4 : 3, NV = LB == 2 ? 4 : 3, CBQ = co_n / 32;
    pl.blocks = NU * NV * kp_n;
    pl.n_cols = 128;
    pl.b.assign((size_t)pl.blocks * 128 * 16, __float2half_rn(0.f));
    pl.epi.resize(4 * co_n);
    for (int co = 0; co < co_n; co++) {
        float s = e.gamma[co] / sqrtf(e.var[co] + kBnEps);
        pl.epi[co] = s >= 0.f ? 1.f : -1.f;
        pl.epi[co_n + co] = e.conv_b[co];
        pl.epi[2 * co_n + co] = s;
        pl.epi[3 * co_n + co] = e.beta[co] - e.mean[co] * s;
    }
    for (int iu = 0; iu < NU; iu++)
        for (int iv = 0; iv < NV; iv++)
            for (int kp = 0; kp < kp_n; kp++) {
                const size_t blk = (size_t)(iu * NV + iv) * kp_n + kp;
                for (int m = 0; m < 128; m++) {
                    const int q = m >> 5, l = m & 31, j = l & 7, lph = (l >> 3) & (PL - 1), cbl = l / (8 * PL);
                    const int co = (q * CBQ + cbl) * 8 + j;
                    const int lb = LB == 2 ? (lph & 1) : 0, la = LA == 2 ? (LB == 2 ? lph >> 1 : lph & 1) : 0;
                    const int dy = LA == 2 ? (iu - 1) - la : iu - 1, dx = LB == 2 ? (iv - 1) - lb : iv - 1;
                    if (dy < -1 || dy > 1 || dx < -1 || dx > 1) continue;
                    for (int k = 0; k < 16; k++)
                        pl.b[(blk * 128 + m) * 16 + k] = __float2half_rn(pl.epi[co] * W(co, kp * 16 + k, dy, dx));
                }
            }
}

// Decoder layer i (< 3), N-half `half` of `nsplit`: N = (4/nsplit) parities x Cout; epi = scale|offset (per Cout).
// Layer 3 (+ head): N = 16 (4 parities used); epi[0] = constant term.
// Blocks are grouped per (row tap a, kpair) by the input COLUMN offset w = pb - b they read (pb = column phase of the
// sub-pixel position, b = column tap), "paired column phases" as in pack_encoder: [w = 0: 2N rows = tap (a,0) for pb = 0 |
// tap (a,1) for pb = 1] [w = -1: N rows, tap (a,1), pb = 0] [w = +1: N rows, tap (a,0), pb = 1] - the same 4N rows as four
// separate taps TWICE (every tap serves both column phases), but three MMAs instead of four per (row phase, a, K step).
// Used where the doubled weights still fit shared memory: dec2 and the head (blobnet_tc.cuh, Cfg::PAIRD); dec0 / dec1
// keep one block per tap, [tap][kpair].
inline size_t dec_block_half(int N, int a, int kp_n, int kp, int unit) { return ((size_t)(a * kp_n + kp) * 4 + unit) * N * 16; }
inline void pack_decoder(const HostWeights &hw, int i, int nsplit, int half, PackedLayer &pl) {
    const int ci_n = kDecCin[i], co_n = kDecCout[i], kp_n = ci_n / 16;
    const auto &d = hw.dec[i];
    auto W = [&](int ci, int co, int ky, int kx) { return d.convt_w[((size_t)(ci * co_n + co) * 4 + ky) * 4 + kx]; };
    const bool paired = i >= 2;
    pl.blocks = (paired ? 8 : 4) * kp_n;
    if (i < 2) {
        const int par_n = 4 / nsplit;
        pl.n_cols = par_n * co_n;
        pl.b.assign((size_t)pl.blocks * pl.n_cols * 16, __float2half_rn(0.f));
        for (int tp = 0; tp < 4; tp++)
            for (int kp = 0; kp < kp_n; kp++)
                for (int pl_i = 0; pl_i < par_n; pl_i++) {
                    int par = half * par_n + pl_i, py = par >> 1, px = par & 1, a = tp >> 1, b = tp & 1;
                    for (int co = 0; co < co_n; co++)
                        for (int k = 0; k < 16; k++)
                            put_b(pl.b, tp * kp_n + kp, pl.n_cols, pl_i * co_n + co, k, W(kp * 16 + k, co, py + 2 * a, px + 2 * b));
                }
    } else if (i < 3) {
        const int par_n = 4 / nsplit;
        pl.n_cols = par_n * co_n;
        pl.b.assign((size_t)pl.blocks * pl.n_cols * 16, __float2half_rn(0.f));
        const int N = pl.n_cols;
        for (int a = 0; a < 2; a++)
            for (int kp = 0; kp < kp_n; kp++)
                for (int blk = 0; blk < 3; blk++) {                 // 0: w = 0 (paired, 2N rows), 1: w = -1, 2: w = +1
                    const int NB = blk == 0 ? 2 * N : N;
                    __half *dst = pl.b.data() + dec_block_half(N, a, kp_n, kp, blk == 0 ? 0 : blk + 1);
                    for (int n = 0; n < NB; n++) {
                        const int b = blk == 0 ? n / N : (blk == 1 ? 1 : 0), nn = n % N;
                        const int pl_i = nn / co_n, co = nn % co_n, par = half * par_n + pl_i, py = par >> 1, px = par & 1;
                        for (int k = 0; k < 16; k++)
                            dst[((size_t)(k >> 3) * NB + n) * 8 + (k & 7)] = __float2half_rn(W(kp * 16 + k, co, py + 2 * a, px + 2 * b));
                    }
                }
    } else {
        pl.n_cols = 16;
        pl.b.assign((size_t)pl.blocks * 16 * 16, __float2half_rn(0.f));
        for (int a = 0; a < 2; a++)
            for (int kp = 0; kp < kp_n; kp++)
                for (int blk = 0; blk < 3; blk++) {
                    const int NB = blk == 0 ? 32 : 16;
                    __half *dst = pl.b.data() + dec_block_half(16, a, kp_n, kp, blk == 0 ? 0 : blk + 1);
                    for (int n = 0; n < NB; n++) {
                        const int b = blk == 0 ? n / 16 : (blk == 1 ? 1 : 0), par = n % 16;
                        if (par >= 4) continue;                      // N = 16 is the smallest MMA; 4 parities are used
                        const int py = par >> 1, px = par & 1;
                        for (int k = 0; k < 16; k++) {
                            double acc = 0;
                            for (int co = 0; co < co_n; co++) acc += (double)W(kp * 16 + k, co, py + 2 * a, px + 2 * b) * hw.head_w[co];
                            dst[((size_t)(k >> 3) * NB + n) * 8 + (k & 7)] = __float2half_rn((float)acc);
                        }
                    }
                }
        double c0 = hw.head_b[0];
        for (int co = 0; co < co_n; co++) c0 += (double)hw.head_w[co] * d.convt_b[co];
        pl.epi.assign(4, (float)c0);
    }
    if (i < 3) {
        pl.epi.resize(2 * co_n);
        for (int co = 0; co < co_n; co++) {
            float s = d.gamma[co] / sqrtf(d.var[co] + kBnEps);
            pl.epi[co] = s;
            pl.epi[co_n + co] = (d.convt_b[co] - d.mean[co]) * s + d.beta[co];
        }
    }
}

}  // namespace cova
