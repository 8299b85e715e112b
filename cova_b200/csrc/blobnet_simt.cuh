// BlobNet on CUDA cores, written straight from the layer definitions (fp32 weights, fp32 math, fp16
// activations in the shared phase-plane layout).  VALIDATION KERNELS: the tests run them next to the
// tcgen05 path to localise descriptor / packing bugs layer by layer; bench.py never selects them.
//
// Reference: utils/model/encoder.py:33-76, pointwise.py:10-26, decoder.py:5-64,106-134.
#pragma once
#include "common.cuh"

namespace cova {

struct SimtEncArgs {
    const Row8 *in; Geom gin;
    Row8 *out; Geom gout;          // Tn = 4 output for the next encoder layer (may be null)
    Row8 *out2; Geom gout2;        // Tn = 1 copy of t = 0 for the decoder (skip / dec0 input)
    int out2_cb;                   // channel-block offset inside the concat buffer
    const float *w, *b, *gamma, *beta, *mean, *var, *w1, *w2;
    int Cin, Cout, N;
    float in_scale;                // 1/6 for the first layer (Preprocessing), 1 otherwise
};

__global__ void __launch_bounds__(128) simt_encoder_kernel(SimtEncArgs A) {
    const int Ho = A.gin.Hh, Wo = A.gin.Wh;                 // output extent after pool (+ pad)
    const int Hp = A.gin.H / 2, Wp = A.gin.W / 2;           // pooled extent ("valid" pooling floors)
    const int padT = A.gin.H & 1, padL = A.gin.W & 1;       // encoder.py:68-76
    const int cbo_n = A.Cout / 8;
    long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)A.N * Hp * Wp * cbo_n;
    if (idx >= total) return;
    int xo = (int)(idx % Wp); idx /= Wp;
    int yo = (int)(idx % Hp); idx /= Hp;
    int n = (int)(idx % A.N);
    int cbo = (int)(idx / A.N);
    float pooled[kT][8];
    for (int t = 0; t < kT; t++) {
        for (int j = 0; j < 8; j++) pooled[t][j] = -3.0e38f;
        for (int ph = 0; ph < 4; ph++) {
            float acc[8];
            for (int j = 0; j < 8; j++) acc[j] = A.b[cbo * 8 + j];
            for (int dy = -1; dy <= 1; dy++)
                for (int dx = -1; dx <= 1; dx++) {
                    int y = 2 * yo + (ph >> 1) + dy, x = 2 * xo + (ph & 1) + dx;
                    if (y < 0 || y >= A.gin.H || x < 0 || x >= A.gin.W) continue;   // "same" zero padding
                    for (int cbi = 0; cbi < A.gin.CB; cbi++) {
                        Row8 r = A.in[geom_row_of(A.gin, n, t, cbi, y, x)];
                        for (int k = 0; k < 8; k++) {
                            int ci = cbi * 8 + k;
                            if (ci >= A.Cin) break;
                            float v = __half2float(r.v[k]) * A.in_scale;
                            const float *wp = A.w + ((size_t)(cbo * 8) * A.Cin + ci) * 9 + (dy + 1) * 3 + (dx + 1);
                            for (int j = 0; j < 8; j++) acc[j] = fmaf(v, wp[(size_t)j * A.Cin * 9], acc[j]);
                        }
                    }
                }
            for (int j = 0; j < 8; j++) {
                int co = cbo * 8 + j;
                float s = A.gamma[co] / sqrtf(A.var[co] + kBnEps);
                float v = fmaxf(acc[j], 0.f) * s + (A.beta[co] - A.mean[co] * s);   // ReLU -> BN
                pooled[t][j] = fmaxf(pooled[t][j], v);                               // -> MaxPool
            }
        }
    }
    // PointWiseTN over T (pointwise.py:18-26); w1/w2 are [T_in][T_out]
    const int Y = yo + padT, X = xo + padL;
    for (int to = 0; to < kT; to++) {
        Row8 o;
        for (int j = 0; j < 8; j++) {
            float h2 = 0.f;
            for (int m = 0; m < kT; m++) {
                float h1 = 0.f;
                for (int ti = 0; ti < kT; ti++) h1 = fmaf(pooled[ti][j], A.w1[ti * kT + m], h1);
                h2 = fmaf(fmaxf(h1, 0.f), A.w2[m * kT + to], h2);
            }
            o.v[j] = __float2half_rn(fmaxf(pooled[to][j] + fmaxf(h2, 0.f), 0.f));
        }
        if (A.out) A.out[geom_row_of(A.gout, n, to, cbo, Y, X)] = o;
        if (to == 0 && A.out2) A.out2[geom_row_of(A.gout2, n, 0, A.out2_cb + cbo, Y, X)] = o;
    }
    (void)Ho; (void)Wo;
}

struct SimtDecArgs {
    const Row8 *in; Geom gin;      // concat input, Tn = 1
    Row8 *out; Geom gout;          // next concat buffer (channel blocks [0, Cout/8))
    const float *w, *b, *gamma, *beta, *mean, *var;   // convt_w [Cin][Cout][4][4]
    const float *head_w, *head_b;  // last layer only
    uint8_t *mask; float *logits;  // last layer only: [N][Ht][Wt]
    const float *seg; float seg_tau;   // last layer only: foreground when logit > (seg ? seg[n] : seg_tau), as tc epilogue_head
    int Cin, Cout, N, Ht, Wt, crop_t, crop_l;
};

// out[oy][ox] = sum_{iy,ix,ky,kx : oy = 2*iy + ky} relu(in[iy][ix]) * W[ci][co][ky][kx]   (stride 2, valid)
__device__ __forceinline__ void simt_convt_point(const SimtDecArgs &A, int n, int Y, int X, int co0, int nco, float *acc) {
    const int oy = Y + A.crop_t, ox = X + A.crop_l;
    for (int ky = 0; ky < 4; ky++) {
        int ty = oy - ky;
        if (ty < 0 || (ty & 1)) continue;
        int iy = ty >> 1;
        if (iy >= A.gin.H) continue;
        for (int kx = 0; kx < 4; kx++) {
            int tx = ox - kx;
            if (tx < 0 || (tx & 1)) continue;
            int ix = tx >> 1;
            if (ix >= A.gin.W) continue;
            for (int cbi = 0; cbi < A.gin.CB; cbi++) {
                Row8 r = A.in[geom_row_of(A.gin, n, 0, cbi, iy, ix)];
                for (int k = 0; k < 8; k++) {
                    int ci = cbi * 8 + k;
                    float v = fmaxf(__half2float(r.v[k]), 0.f);   // ReLU in front of the ConvT (decoder.py:12-13)
                    const float *wp = A.w + (((size_t)ci * A.Cout + co0) * 4 + ky) * 4 + kx;
                    for (int j = 0; j < nco; j++) acc[j] = fmaf(v, wp[(size_t)j * 16], acc[j]);
                }
            }
        }
    }
}

__global__ void __launch_bounds__(128) simt_decoder_kernel(SimtDecArgs A) {
    const int cbo_n = A.Cout / 8;
    long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)A.N * A.Ht * A.Wt * cbo_n;
    if (idx >= total) return;
    int X = (int)(idx % A.Wt); idx /= A.Wt;
    int Y = (int)(idx % A.Ht); idx /= A.Ht;
    int n = (int)(idx % A.N);
    int cbo = (int)(idx / A.N);
    float acc[8];
    for (int j = 0; j < 8; j++) acc[j] = A.b[cbo * 8 + j];
    simt_convt_point(A, n, Y, X, cbo * 8, 8, acc);
    Row8 o;
    for (int j = 0; j < 8; j++) {
        int co = cbo * 8 + j;
        float s = A.gamma[co] / sqrtf(A.var[co] + kBnEps);
        float v = (acc[j] - A.mean[co]) * s + A.beta[co];       // BatchNorm
        o.v[j] = __float2half_rn(fmaxf(v, 0.f));                 // stored post-ReLU: its only consumer starts with ReLU
    }
    A.out[geom_row_of(A.gout, n, 0, cbo, Y, X)] = o;
}

__global__ void __launch_bounds__(128) simt_head_kernel(SimtDecArgs A) {
    long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)A.N * A.Ht * A.Wt;
    if (idx >= total) return;
    int X = (int)(idx % A.Wt); idx /= A.Wt;
    int Y = (int)(idx % A.Ht);
    int n = (int)(idx / A.Ht);
    float acc[16];
    for (int j = 0; j < 16; j++) acc[j] = A.b[j];
    simt_convt_point(A, n, Y, X, 0, 16, acc);
    float z = A.head_b[0];
    for (int j = 0; j < 16; j++) z = fmaf(acc[j], A.head_w[j], z);
    size_t o = ((size_t)n * A.Ht + Y) * A.Wt + X;
    A.mask[o] = z > (A.seg ? A.seg[n] : A.seg_tau) ? 1 : 0;   // sigmoid(z) > segmentation-threshold; maskcopy's class_map + 1
    if (A.logits) A.logits[o] = z;
}

}  // namespace cova
