// ccd_synth.cu -- float tail of the Cool-chic decoder on sm_100a: learned upsampling,
// synthesis, final resize, frame quantisation.
//
// Replaces (reference, fp32 PyTorch CPU):
//   core/upsampling.py:189-196   pre-concat conv, TRAIN-mode kron form (zero pad, + x)
//   core/upsampling.py:306-325   transposed conv, TRAIN-mode kron form (replicate pad 4, crop 11)
//   core/upsampling.py:463-500   Upsampling.forward cascade
//   core/synthesis.py:61-76      SynthesisConv2d.forward (replicate pad, conv+bias, +x, ReLU)
//   core/synthesis.py:272-294    Synthesis.forward (trunk + stabiliser, output_transform)
//   component/coolchic.py:187-192 final F.interpolate + crop
//   bitstream/decode.py:191-206  round / 420 average / clamp / round
//
// Canonical fp32 order (identical to oracle/ccoracle.c, so GPU == oracle bit for bit):
// every output is acc = init; for ci, for ky, for kx: acc = fmaf(w, x, acc).
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "ccd_detmath.h"
#include "ccd_internal.h"

namespace {

__device__ __forceinline__ int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

struct K1d {
    float w[16];
};

__global__ void k_ups_first(const int8_t *__restrict__ lat, size_t n, float *__restrict__ out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (float)lat[i];
}

// hi = conv2d(x, kron(w, w), zero padding k/2) + x      (x = int8 latent as float)
__global__ void k_ups_pre(const int8_t *__restrict__ lat, int h, int w, K1d kw, int k, float *__restrict__ out) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= w || y >= h) return;
    const int p = k / 2;
    float acc = 0.0f;
    for (int a = 0; a < k; a++) {
        const int yy = y + a - p;
        if (yy < 0 || yy >= h) continue;
        for (int b = 0; b < k; b++) {
            const int xx = x + b - p;
            if (xx < 0 || xx >= w) continue;
            const float kk = __fmul_rn(kw.w[a], kw.w[b]);
            acc = __fmaf_rn(kk, (float)lat[(size_t)yy * w + xx], acc);
        }
    }
    out[(size_t)y * w + x] = __fadd_rn(acc, (float)lat[(size_t)y * w + x]);
}

// transposed conv stride 2 on the replicate-padded input, cropped (see oracle convt_kron)
__global__ void k_ups_convt(const float *__restrict__ in, int h, int w, K1d kw, int k, float *__restrict__ out,
                            int ht, int wt) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    const int u = blockIdx.y * blockDim.y + threadIdx.y;
    const int c = blockIdx.z;
    if (v >= wt || u >= ht) return;
    const int P0 = k / 2, C = 2 * P0 - 1 + k / 2;
    const float *src = in + (size_t)c * h * w;
    const int o1 = u + C, o2 = v + C;
    const int i1_lo = (o1 - (k - 1) < 0) ? 0 : (o1 - (k - 1) + 1) / 2, i1_hi = o1 / 2;
    const int i2_lo = (o2 - (k - 1) < 0) ? 0 : (o2 - (k - 1) + 1) / 2, i2_hi = o2 / 2;
    float acc = 0.0f;
    for (int i1 = i1_lo; i1 <= i1_hi; i1++) {
        const int a = o1 - 2 * i1;
        const int r = clampi(i1 - P0, 0, h - 1);
        for (int i2 = i2_lo; i2 <= i2_hi; i2++) {
            const int b = o2 - 2 * i2;
            const int cc = clampi(i2 - P0, 0, w - 1);
            const float kk = __fmul_rn(kw.w[a], kw.w[b]);
            acc = __fmaf_rn(kk, src[(size_t)r * w + cc], acc);
        }
    }
    out[((size_t)c * ht + u) * wt + v] = acc;
}

// One level of the upsampling cascade (Upsampling.forward, upsampling.py:463-500) for the default kernel
// sizes (8-tap transposed conv, 7-tap pre-concatenation conv) in ONE launch: blockIdx.z == 0 filters the
// target grid's own latent (k_ups_pre), z >= 1 upsamples channel z - 1 of the coarser stack (k_ups_convt).
// The separable kernels' 2-D products w[a] * w[b] are formed once on the host (one fp32 multiply each, the
// same value the per-tap __fmul_rn gives); a thread of the transposed part produces a 2 x 2 output block from
// one 5 x 5 clamped input window (25 loads for 64 FMAs).  Accumulation order per output = k_ups_convt / k_ups_pre.
struct UpsLevelParams {
    const int8_t *lat;  // target grid [th][tw]
    const float *in;    // coarser stack [cc][ch][cw]
    float *out;         // [cc + 1][th][tw]
    int cc, ch, cw, th, tw;
    float kt[8][8];     // transposed-conv taps
    float kc[7][7];     // pre-concatenation taps
};
__global__ void __launch_bounds__(256) k_ups_level(UpsLevelParams P) {
    const int th = P.th, tw = P.tw;
    if (blockIdx.z == 0) {
        const int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y;
        if (x >= tw || y >= th) return;
        float acc = 0.0f;
#pragma unroll
        for (int a = 0; a < 7; a++) {
            const int yy = y + a - 3;
#pragma unroll
            for (int b = 0; b < 7; b++) {
                const int xx = x + b - 3;
                if (yy >= 0 && yy < th && xx >= 0 && xx < tw) acc = __fmaf_rn(P.kc[a][b], (float)P.lat[(size_t)yy * tw + xx], acc);
            }
        }
        P.out[(size_t)y * tw + x] = __fadd_rn(acc, (float)P.lat[(size_t)y * tw + x]);
        return;
    }
    // transposed part: output block (2q .. 2q+1, 2s .. 2s+1)
    const int s0 = blockIdx.x * 32 + threadIdx.x, q = blockIdx.y * 8 + threadIdx.y;
    if (2 * s0 >= tw || 2 * q >= th) return;
    const int c = blockIdx.z - 1, h = P.ch, w = P.cw;
    const float *src = P.in + (size_t)c * h * w;
    float win[5][5];
#pragma unroll
    for (int i = 0; i < 5; i++) {
        const float *row = src + (size_t)clampi(q - 2 + i, 0, h - 1) * w;
#pragma unroll
        for (int j = 0; j < 5; j++) win[i][j] = __ldg(row + clampi(s0 - 2 + j, 0, w - 1));
    }
    float *dst = P.out + (size_t)(c + 1) * th * tw;
#pragma unroll
    for (int du = 0; du < 2; du++) {
        const int u = 2 * q + du;
        if (u >= th) continue;
#pragma unroll
        for (int dv = 0; dv < 2; dv++) {
            const int v = 2 * s0 + dv;
            if (v >= tw) continue;
            // u = 2q: input rows q-2 .. q+1 with taps a = 7, 5, 3, 1;  u = 2q+1: rows q-1 .. q+2, a = 6, 4, 2, 0
            float acc = 0.0f;
#pragma unroll
            for (int t1 = 0; t1 < 4; t1++)
#pragma unroll
                for (int t2 = 0; t2 < 4; t2++)
                    acc = __fmaf_rn(P.kt[(1 - du) + 6 - 2 * t1][(1 - dv) + 6 - 2 * t2], win[t1 + du][t2 + dv], acc);
            dst[(size_t)u * tw + v] = acc;
        }
    }
}

// generic SynthesisConv2d: one thread = one pixel, loops over output channels
__global__ void k_syn_layer(const float *__restrict__ in, int h, int w, int cin, int cout, int k, int residual,
                            int relu, const float *__restrict__ wt, const float *__restrict__ bias,
                            float *__restrict__ out) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= w || y >= h) return;
    const int p = (k - 1) / 2;
    const size_t plane = (size_t)h * w;
    for (int co = 0; co < cout; co++) {
        float acc = __ldg(bias + co);
        for (int ci = 0; ci < cin; ci++) {
            for (int ky = 0; ky < k; ky++) {
                const int yy = clampi(y + ky - p, 0, h - 1);
                for (int kx = 0; kx < k; kx++) {
                    const int xx = clampi(x + kx - p, 0, w - 1);
                    acc = __fmaf_rn(__ldg(wt + (((size_t)co * cin + ci) * k + ky) * k + kx),
                                    in[ci * plane + (size_t)yy * w + xx], acc);
                }
            }
        }
        if (residual) acc = __fadd_rn(acc, in[co * plane + (size_t)y * w + x]);
        if (relu) acc = fmaxf(acc, 0.0f);
        out[co * plane + (size_t)y * w + x] = acc;
    }
}

// two fused 1x1 layers (cin -> chid -> cout), hidden activations stay in registers.
// Same summation order as two sequential generic layers.
template <int CIN_MAX, int COUT_MAX>
__global__ void k_syn_pw2(const float *__restrict__ in, size_t plane, int cin, int chid, int cout, int relu0,
                          int relu1, const float *__restrict__ w0, const float *__restrict__ b0,
                          const float *__restrict__ w1, const float *__restrict__ b1, float *__restrict__ out) {
    extern __shared__ float s_w[];
    float *sw0 = s_w;                   // [chid][cin]
    float *sb0 = sw0 + chid * cin;      // [chid]
    float *sw1 = sb0 + chid;            // [cout][chid]
    float *sb1 = sw1 + cout * chid;     // [cout]
    for (int i = threadIdx.x; i < chid * cin; i += blockDim.x) sw0[i] = w0[i];
    for (int i = threadIdx.x; i < chid; i += blockDim.x) sb0[i] = b0[i];
    for (int i = threadIdx.x; i < cout * chid; i += blockDim.x) sw1[i] = w1[i];
    for (int i = threadIdx.x; i < cout; i += blockDim.x) sb1[i] = b1[i];
    __syncthreads();
    const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= plane) return;
    float x[CIN_MAX], o[COUT_MAX];
#pragma unroll
    for (int i = 0; i < CIN_MAX; i++) x[i] = (i < cin) ? in[(size_t)i * plane + p] : 0.0f;
#pragma unroll
    for (int c = 0; c < COUT_MAX; c++) o[c] = (c < cout) ? sb1[c] : 0.0f;
    for (int hcn = 0; hcn < chid; hcn++) {
        float a = sb0[hcn];
#pragma unroll
        for (int i = 0; i < CIN_MAX; i++)
            if (i < cin) a = __fmaf_rn(sw0[hcn * cin + i], x[i], a);
        if (relu0) a = fmaxf(a, 0.0f);
#pragma unroll
        for (int c = 0; c < COUT_MAX; c++)
            if (c < cout) o[c] = __fmaf_rn(sw1[c * chid + hcn], a, o[c]);
    }
#pragma unroll
    for (int c = 0; c < COUT_MAX; c++)
        if (c < cout) out[(size_t)c * plane + p] = relu1 ? fmaxf(o[c], 0.0f) : o[c];
}

// ---------------------------------------------------------------------------------------------------
// Fused synthesis (core/synthesis.py:272-294) for the architecture family every Cool-chic preset uses:
//   [1x1 cin -> hid (relu?)] [1x1 hid -> C (relu?)] then 0, 1 or 2 3x3 layers C -> C (residual? relu?)
//   + linear stabiliser (1x1 on the dense input) + output transform (1x1 C -> C).
// One CTA = one 32 x 16 output tile.  Stage A evaluates the two 1x1 layers on the tile plus a halo of one
// pixel per 3x3 layer (three positions per thread share each weight fetch), the 3x3 layers go from shared
// memory to shared memory, the stabiliser / residual adds / output transform happen in registers, and only
// the final C planes are written: the dense latent is read once and nothing else touches HBM.
// Replicate padding = every stage evaluates out-of-frame positions at their clamped coordinates.
// Same fp32 operation order per output as the unfused kernels (and oracle/ccoracle.c::syn_conv), so the
// result is bit-identical.
struct SynFusedParams {
    const float *in;    // dense latent [cin][h][w]
    float *out;         // [C][h][w]
    int h, w, cin, hid, n3;            // n3: number of 3x3 layers (0..2)
    int relu0, relu1, res3[2], relu3[2];
    int stab_in;                       // 0: no stabiliser
    const float *w0, *b0, *w1, *b1;    // [hid][cin], [hid], [C][hid], [C]
    const float *w3[2], *b3[2];        // [C][C][3][3], [C]
    const float *ws, *bs, *wo, *bo;    // [C][stab_in], [C], [C][C], [C]
};
constexpr int SF_TW = 32, SF_TH = 16, SF_THREADS = 256;

template <int CINP, int C>
__global__ void __launch_bounds__(SF_THREADS) k_syn_fused(SynFusedParams P) {
    extern __shared__ __align__(16) float sf_smem[];
    const int n3 = P.n3, hid = P.hid, cin = P.cin;
    const int RW = SF_TW + 2 * n3, RH = SF_TH + 2 * n3;  // stage-A region
    // shared memory: weights, then region buffers
    float *sw0 = sf_smem;                    // [hid][CINP]
    float *sb0 = sw0 + hid * CINP;           // [hid]
    float *sw1 = sb0 + hid;                  // [hid][4*ceil(C/4)]  (transposed: one vector load per hidden unit)
    constexpr int CP = (C + 3) & ~3;
    float *sb1 = sw1 + hid * CP;             // [CP]
    float *sw3 = sb1 + CP;                   // [2][C][C][9]
    float *sb3 = sw3 + 2 * C * C * 9;        // [2][CP]
    float *sws = sb3 + 2 * CP;               // [C][CINP]
    float *sbs = sws + C * CINP;             // [CP]
    float *swo = sbs + CP;                   // [C][CP]
    float *sbo = swo + C * CP;               // [CP]
    float *bufA = sbo + CP;                  // [C][RH][RW]
    float *bufB = bufA + C * RH * RW;        // [C][RH-2][RW-2]   (n3 == 2)
    float *sstab = bufB + (n3 == 2 ? C * (RH - 2) * (RW - 2) : 0);  // [C][SF_TH][SF_TW]
    const int tid = threadIdx.x;
    for (int i = tid; i < hid * CINP; i += SF_THREADS) {
        const int hh = i / CINP, ci = i - hh * CINP;
        sw0[i] = ci < cin ? P.w0[hh * cin + ci] : 0.0f;
    }
    for (int i = tid; i < hid; i += SF_THREADS) sb0[i] = P.b0[i];
    for (int i = tid; i < hid * CP; i += SF_THREADS) {
        const int hh = i / CP, c = i - hh * CP;
        sw1[i] = c < C ? P.w1[c * hid + hh] : 0.0f;
    }
    for (int i = tid; i < CP; i += SF_THREADS) {
        sb1[i] = i < C ? P.b1[i] : 0.0f;
        sbs[i] = (i < C && P.stab_in) ? P.bs[i] : 0.0f;
        sbo[i] = i < C ? P.bo[i] : 0.0f;
        for (int l = 0; l < 2; l++) sb3[l * CP + i] = (i < C && l < n3) ? P.b3[l][i] : 0.0f;
    }
    for (int l = 0; l < n3; l++)
        for (int i = tid; i < C * C * 9; i += SF_THREADS) sw3[l * C * C * 9 + i] = P.w3[l][i];
    for (int i = tid; i < C * CINP; i += SF_THREADS) {
        const int c = i / CINP, ci = i - c * CINP;
        sws[i] = (ci < P.stab_in) ? P.ws[c * P.stab_in + ci] : 0.0f;
    }
    for (int i = tid; i < C * CP; i += SF_THREADS) {
        const int c = i / CP, k = i - c * CP;
        swo[i] = k < C ? P.wo[c * C + k] : 0.0f;
    }
    __syncthreads();

    const int x0 = blockIdx.x * SF_TW, y0 = blockIdx.y * SF_TH;
    const int H = P.h, W = P.w;
    const size_t plane = (size_t)H * W;
    // ---- stage A: two 1x1 layers (+ stabiliser on the tile itself) on RH x RW positions, 3 per thread
    const int nA = RH * RW;
    for (int base = 0; base < nA; base += 3 * SF_THREADS) {
        float x[3][CINP], o[3][C];
        int pos[3];
#pragma unroll
        for (int q = 0; q < 3; q++) {
            const int pp = base + q * SF_THREADS + tid;
            pos[q] = pp;
            const int py = pp / RW, px = pp - py * RW;
            const int gy = clampi(y0 - n3 + py, 0, H - 1), gx = clampi(x0 - n3 + px, 0, W - 1);
            const float *src = P.in + (size_t)gy * W + gx;
#pragma unroll
            for (int ci = 0; ci < CINP; ci++) x[q][ci] = (pp < nA && ci < cin) ? __ldg(src + (size_t)ci * plane) : 0.0f;
#pragma unroll
            for (int c = 0; c < C; c++) o[q][c] = sb1[c];
        }
        for (int hh = 0; hh < hid; hh++) {
            float wv[CINP];
#pragma unroll
            for (int v = 0; v < CINP / 4; v++) {
                const float4 t = *reinterpret_cast<const float4 *>(sw0 + hh * CINP + 4 * v);
                wv[4 * v] = t.x; wv[4 * v + 1] = t.y; wv[4 * v + 2] = t.z; wv[4 * v + 3] = t.w;
            }
            float w1v[CP];
#pragma unroll
            for (int v = 0; v < CP / 4; v++) {
                const float4 t = *reinterpret_cast<const float4 *>(sw1 + hh * CP + 4 * v);
                w1v[4 * v] = t.x; w1v[4 * v + 1] = t.y; w1v[4 * v + 2] = t.z; w1v[4 * v + 3] = t.w;
            }
            const float bb = sb0[hh];
#pragma unroll
            for (int q = 0; q < 3; q++) {
                float a = bb;
#pragma unroll
                for (int ci = 0; ci < CINP; ci++)
                    if (ci < cin) a = __fmaf_rn(wv[ci], x[q][ci], a);
                if (P.relu0) a = fmaxf(a, 0.0f);
#pragma unroll
                for (int c = 0; c < C; c++) o[q][c] = __fmaf_rn(w1v[c], a, o[q][c]);
            }
        }
#pragma unroll
        for (int q = 0; q < 3; q++) {
            if (pos[q] >= nA) continue;
            const int py = pos[q] / RW, px = pos[q] - py * RW;
#pragma unroll
            for (int c = 0; c < C; c++) bufA[(c * RH + py) * RW + px] = P.relu1 ? fmaxf(o[q][c], 0.0f) : o[q][c];
            // stabiliser (synthesis.py:286-289) for positions of the tile itself
            const int ty = py - n3, tx = px - n3;
            if (P.stab_in && ty >= 0 && ty < SF_TH && tx >= 0 && tx < SF_TW) {
#pragma unroll
                for (int c = 0; c < C; c++) {
                    float a = sbs[c];
#pragma unroll
                    for (int ci = 0; ci < CINP; ci++)
                        if (ci < P.stab_in) a = __fmaf_rn(sws[c * CINP + ci], x[q][ci], a);
                    sstab[(c * SF_TH + ty) * SF_TW + tx] = a;
                }
            }
        }
    }
    __syncthreads();
    // ---- 3x3 layers, shared memory -> shared memory (the last one -> registers -> output)
    const float *cur = bufA;
    int cw = RW, chh = RH, off = n3;  // current buffer geometry; off = its halo w.r.t. the tile
    for (int l = 0; l < n3 - 1; l++) {
        // intermediate 3x3 layer on the region shrunk by one pixel
        const int ow = cw - 2, oh = chh - 2;
        const float *wl = sw3 + l * C * C * 9;
        for (int pp = tid; pp < ow * oh; pp += SF_THREADS) {
            const int py = pp / ow, px = pp - py * ow;
            // this position in frame coordinates, clamped (replicate padding of the NEXT layer), then back
            // to buffer coordinates of `cur`
            const int gy = clampi(y0 - (off - 1) + py, 0, H - 1), gx = clampi(x0 - (off - 1) + px, 0, W - 1);
            const int by = gy - (y0 - off), bx = gx - (x0 - off);
            float acc[C];
#pragma unroll
            for (int co = 0; co < C; co++) acc[co] = sb3[l * CP + co];
#pragma unroll
            for (int ci = 0; ci < C; ci++)
#pragma unroll
                for (int ky = 0; ky < 3; ky++)
#pragma unroll
                    for (int kx = 0; kx < 3; kx++) {
                        const float v = cur[(ci * chh + by + ky - 1) * cw + bx + kx - 1];
#pragma unroll
                        for (int co = 0; co < C; co++) acc[co] = __fmaf_rn(wl[((co * C + ci) * 3 + ky) * 3 + kx], v, acc[co]);
                    }
#pragma unroll
            for (int co = 0; co < C; co++) {
                float a = acc[co];
                if (P.res3[l]) a = __fadd_rn(a, cur[(co * chh + by) * cw + bx]);
                if (P.relu3[l]) a = fmaxf(a, 0.0f);
                bufB[(co * oh + py) * ow + px] = a;
            }
        }
        __syncthreads();
        cur = bufB;
        cw = ow;
        chh = oh;
        off -= 1;
    }
    // ---- last stage on the tile: last 3x3 layer (if any), + stabiliser, output transform, store
    for (int pp = tid; pp < SF_TW * SF_TH; pp += SF_THREADS) {
        const int ty = pp / SF_TW, tx = pp - ty * SF_TW;
        const int gy = y0 + ty, gx = x0 + tx;
        if (gy >= H || gx >= W) continue;
        const int by = ty + off, bx = tx + off;
        float t[C];
        if (n3 > 0) {
            const int l = n3 - 1;
            const float *wl = sw3 + l * C * C * 9;
#pragma unroll
            for (int co = 0; co < C; co++) t[co] = sb3[l * CP + co];
#pragma unroll
            for (int ci = 0; ci < C; ci++)
#pragma unroll
                for (int ky = 0; ky < 3; ky++)
#pragma unroll
                    for (int kx = 0; kx < 3; kx++) {
                        const float v = cur[(ci * chh + by + ky - 1) * cw + bx + kx - 1];
#pragma unroll
                        for (int co = 0; co < C; co++) t[co] = __fmaf_rn(wl[((co * C + ci) * 3 + ky) * 3 + kx], v, t[co]);
                    }
#pragma unroll
            for (int co = 0; co < C; co++) {
                if (P.res3[l]) t[co] = __fadd_rn(t[co], cur[(co * chh + by) * cw + bx]);
                if (P.relu3[l]) t[co] = fmaxf(t[co], 0.0f);
            }
        } else {
#pragma unroll
            for (int co = 0; co < C; co++) t[co] = cur[(co * chh + by) * cw + bx];
        }
        if (P.stab_in) {
#pragma unroll
            for (int co = 0; co < C; co++) t[co] = __fadd_rn(t[co], sstab[(co * SF_TH + ty) * SF_TW + tx]);
        }
#pragma unroll
        for (int co = 0; co < C; co++) {
            float a = sbo[co];
#pragma unroll
            for (int ci = 0; ci < C; ci++) a = __fmaf_rn(swo[co * CP + ci], t[ci], a);
            P.out[(size_t)co * plane + (size_t)gy * W + gx] = a;
        }
    }
}

// ===================================================================================================
// Batched float tail (BASELINE configs[2] / [4]: many streams in one call).
//
//   k_ups_level_b : one level of the cascade for ALL streams of a group in one launch
//                   (blockIdx.z = stream * planes + plane)
//   k_tail_syn2   : the LAST cascade level + the whole synthesis + the frame tail in one kernel.  The dense
//                   latent at image resolution (7 fp32 planes, 28 B / pixel written and read back by the
//                   unfused path) is never materialised: a CTA stages the int8 tile of the finest grid
//                   (zero padding = TMA out-of-bounds fill) and the tile of the half-resolution stack in shared
//                   memory -- with TMA (cp.async.bulk.tensor + mbarrier) when the row pitches allow it -- and
//                   evaluates the 7x7 pre-concatenation conv and the 8x8 stride-2 transposed conv on the fly
//                   for every position of the synthesis region.  Epilogue: output transform, then optionally
//                   decode_frame's round / (4:2:0 average) / clamp / round (bitstream/decode.py:191-206).
// Every output keeps the canonical fp32 operation order of the unfused kernels (bit-identical, tested).
// ===================================================================================================
struct UpsLevelJob {
    const int8_t *lat;  // target grid [th][tw]
    const float *in;    // coarser stack [cc][ch][cw] (fp32) ...
    const int8_t *in8;  // ... or, for the first level, the coarsest latent grid itself (cc == 1)
    float *out;         // [cc + 1][th][tw]
    int cc, ch, cw, th, tw;
    float kt[8][8];     // transposed-conv taps
    float kc[7][7];     // pre-concatenation taps
};
__global__ void __launch_bounds__(256) k_ups_level_b(const UpsLevelJob *__restrict__ jobs, int planes) {
    const int job = blockIdx.z / planes, plane = blockIdx.z - job * planes;
    const UpsLevelJob &P = jobs[job];
    if (plane > P.cc) return;
    const int th = P.th, tw = P.tw;
    if (plane == 0) {
        const int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y;
        if (x >= tw || y >= th) return;
        float acc = 0.0f;
#pragma unroll
        for (int a = 0; a < 7; a++) {
            const int yy = y + a - 3;
#pragma unroll
            for (int b = 0; b < 7; b++) {
                const int xx = x + b - 3;
                if (yy >= 0 && yy < th && xx >= 0 && xx < tw) acc = __fmaf_rn(P.kc[a][b], (float)P.lat[(size_t)yy * tw + xx], acc);
            }
        }
        P.out[(size_t)y * tw + x] = __fadd_rn(acc, (float)P.lat[(size_t)y * tw + x]);
        return;
    }
    const int s0 = blockIdx.x * 32 + threadIdx.x, q = blockIdx.y * 8 + threadIdx.y;
    if (2 * s0 >= tw || 2 * q >= th) return;
    const int c = plane - 1, h = P.ch, w = P.cw;
    float win[5][5];
    if (P.in8) {
        const int8_t *src = P.in8 + (size_t)c * h * w;
#pragma unroll
        for (int i = 0; i < 5; i++) {
            const int8_t *row = src + (size_t)clampi(q - 2 + i, 0, h - 1) * w;
#pragma unroll
            for (int j = 0; j < 5; j++) win[i][j] = (float)row[clampi(s0 - 2 + j, 0, w - 1)];
        }
    } else {
        const float *src = P.in + (size_t)c * h * w;
#pragma unroll
        for (int i = 0; i < 5; i++) {
            const float *row = src + (size_t)clampi(q - 2 + i, 0, h - 1) * w;
#pragma unroll
            for (int j = 0; j < 5; j++) win[i][j] = __ldg(row + clampi(s0 - 2 + j, 0, w - 1));
        }
    }
    float *dst = P.out + (size_t)(c + 1) * th * tw;
#pragma unroll
    for (int du = 0; du < 2; du++) {
        const int u = 2 * q + du;
        if (u >= th) continue;
#pragma unroll
        for (int dv = 0; dv < 2; dv++) {
            const int v = 2 * s0 + dv;
            if (v >= tw) continue;
            float acc = 0.0f;
#pragma unroll
            for (int t1 = 0; t1 < 4; t1++)
#pragma unroll
                for (int t2 = 0; t2 < 4; t2++)
                    acc = __fmaf_rn(P.kt[(1 - du) + 6 - 2 * t1][(1 - dv) + 6 - 2 * t2], win[t1 + du][t2 + dv], acc);
            dst[(size_t)u * tw + v] = acc;
        }
    }
}

struct alignas(64) TailSynJob {
    unsigned char tmap_lat[128];  // CUtensorMap: finest latent grid, uint8 [h][w], box LW x LH
    unsigned char tmap_stk[128];  // CUtensorMap: coarser stack, fp32 [cc][ch][cw], box SW x SH x cc
    const int8_t *lat;            // finest grid [h][w]
    const float *stk;             // coarser stack [cc][ch][cw] (cc = cin - 1), already upsampled to (ch, cw)
    const int8_t *stk8;           // ... or the coarsest latent itself when only two grids exist (cc == 1)
    float *out[3 + 2];            // output planes (C <= 5)
    int h, w, ch, cw, cin, hid, n3;
    int relu0, relu1, res3[2], relu3[2];
    int stab_in;
    int use_tma;
    int finish;                   // 0: raw synthesis output; 1: frame tail, three full planes; 2: frame tail 4:2:0
    float M;                      // 2^bitdepth - 1
    const float *w0, *b0, *w1, *b1;
    const float *w3[2], *b3[2];
    const float *ws, *bs, *wo, *bo;
    float kt[8][8], kc[7][7];
};
// (TMA needs the box to start on a 16-byte boundary in the innermost dimension: the tile origins are rounded down
// to a multiple of 16 int8 / 4 fp32 columns and the boxes widened accordingly)
__host__ __device__ inline int ts_lw(int n3) { return (SF_TW + 2 * n3 + 6 + 15 + 15) & ~15; }
__host__ __device__ inline int ts_lh(int n3) { return SF_TH + 2 * n3 + 6; }
__host__ __device__ inline int ts_sw(int n3) { return ((SF_TW + 2 * n3) / 2 + 5 + 3 + 3) & ~3; }
__host__ __device__ inline int ts_sh(int n3) { return (SF_TH + 2 * n3) / 2 + 5; }

__device__ __forceinline__ float quant(float v, float M);
__device__ __forceinline__ float clamp01(float v);

// ---------------------------------------------------------------------------------------------------------------
// k_tail_syn2, blocked for instruction efficiency (the first version of this kernel issued ~3 650 instructions per
// pixel for 862 FMAs):
//   * the halo of the stage-A region is rounded up to an even number of pixels, so that the region starts on even
//     frame coordinates and stage A works on 2 x 2 QUADS with compile-time parities: the 8x8 stride-2 transposed
//     conv reads ONE 5 x 5 window per channel for its four outputs, its taps come as 16 vector loads (re-laid
//     [du][t1][dv][t2]); the 7x7 pre-concatenation conv slides over 8 rows of 8 values (converted to fp32 once per
//     tile); the two 1x1 layers share every weight fetch between the four positions;
//   * out-of-frame positions of the region (replicate padding of the 3x3 layers) are copies of the clamped
//     position's values (the 1x1 layers are pointwise), filled by a fix-up pass on border tiles only;
//   * the 3x3 layers evaluate two horizontally adjacent outputs per thread from one 3 x 4 window per channel, their
//     weights re-laid [ci][ky][kx][co] (one vector load per tap); stores are 64-bit.
// Every output keeps its canonical accumulation order: bit-identical to k_syn_fused and the oracle.
__host__ __device__ inline int ts2_n3e(int n3) { return (n3 + 1) & ~1; }
constexpr int TS2_THREADS = 192;  // 180 quads per 32 x 16 tile with a 2-pixel halo; three CTAs per SM

template <int CINP, int C>
__global__ void __launch_bounds__(TS2_THREADS, 3) k_tail_syn2(const TailSynJob *__restrict__ jobs) {
    extern __shared__ __align__(128) unsigned char ts_raw[];
    const TailSynJob &P = jobs[blockIdx.z];
    const int H = P.h, W = P.w;
    const int x0 = blockIdx.x * SF_TW, y0 = blockIdx.y * SF_TH;
    if (x0 >= W || y0 >= H) return;
    const int n3 = P.n3, n3e = ts2_n3e(n3), hid = P.hid, cin = P.cin, cc = cin - 1;
    const int RW = SF_TW + 2 * n3e, RH = SF_TH + 2 * n3e;
    const int LW = ts_lw(n3e), LH = ts_lh(n3e), SW = ts_sw(n3e), SH = ts_sh(n3e);
    constexpr int CP = (C + 3) & ~3;  // output channels padded to a multiple of 4 (vector loads of weights)
    uint64_t *bar = reinterpret_cast<uint64_t *>(ts_raw);
    int8_t *Lt = reinterpret_cast<int8_t *>(ts_raw + 128);                          // [LH][LW] int8 (TMA destination)
    float *St = reinterpret_cast<float *>(ts_raw + 128 + ((LW * LH + 127) & ~127)); // [cc][SH][SW]
    float *Lf = St + ((cc * SH * SW + 31) & ~31);  // [LH][LW] the latent tile as fp32
    float *sw0 = Lf + LW * LH;               // [hid][CINP]
    float *sb0 = sw0 + hid * CINP;
    float *sw1 = sb0 + ((hid + 3) & ~3);     // [hid][CP]
    float *sb1 = sw1 + hid * CP;
    float *sw3 = sb1 + CP;                   // [2][C][3][3][CP]
    float *sb3 = sw3 + 2 * C * 9 * CP;
    float *sws = sb3 + 2 * CP;               // [C][CINP]
    float *sbs = sws + C * CINP;
    float *swo = sbs + CP;                   // [C][CP]
    float *sbo = swo + C * CP;
    float *skt = sbo + CP;                   // [2 du][4 t1][2 dv][4 t2]
    float *skc = skt + 64;                   // [7][8] (rows padded)
    float *bufA = skc + 56;                  // [C][RH][RW]
    float *bufB = bufA + C * RH * RW;        // [C][RH-2][RW-2]   (n3 == 2)
    float *sstab = bufB + (n3 == 2 ? C * (RH - 2) * (RW - 2) : 0);  // [C][SF_TH][SF_TW]
    const int tid = threadIdx.x;
    const int Y0 = y0 - n3e, X0 = x0 - n3e;                 // stage-A region origin (even frame coordinates)
    const int ly0 = Y0 - 3, lx0 = (X0 - 3) & ~15;           // latent tile (16-byte aligned start)
    const int sy0 = ((Y0 < 0 ? 0 : Y0) >> 1) - 2, sx0 = (((X0 < 0 ? 0 : X0) >> 1) - 2) & ~3;  // stack tile
    const int ch = P.ch, cw = P.cw;
    // ---- stage 0: tiles -> shared memory
    if (P.use_tma) {
        const uint32_t bar_a = (uint32_t)__cvta_generic_to_shared(bar);
        if (tid == 0) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_a));
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncthreads();
        if (tid == 0) {
            const uint32_t bytes = (uint32_t)(LW * LH + cc * SH * SW * 4);
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_a), "r"(bytes) : "memory");
            const uint64_t tm0 = reinterpret_cast<uint64_t>(P.tmap_lat), tm1 = reinterpret_cast<uint64_t>(P.tmap_stk);
            if (P.use_tma & 2) {
                asm volatile("fence.proxy.tensormap::generic.acquire.gpu [%0], 128;" ::"l"(tm0) : "memory");
                asm volatile("fence.proxy.tensormap::generic.acquire.gpu [%0], 128;" ::"l"(tm1) : "memory");
            }
            asm volatile(
                "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                ::"r"((uint32_t)__cvta_generic_to_shared(Lt)), "l"(tm0), "r"(lx0), "r"(ly0), "r"(bar_a)
                : "memory");
            asm volatile(
                "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                ::"r"((uint32_t)__cvta_generic_to_shared(St)), "l"(tm1), "r"(sx0), "r"(sy0), "r"(0), "r"(bar_a)
                : "memory");
        }
    } else {
        for (int i = tid; i < LW * LH; i += TS2_THREADS) {
            const int r = i / LW, c = i - r * LW;
            const int gy = ly0 + r, gx = lx0 + c;
            Lf[i] = (gy >= 0 && gy < H && gx >= 0 && gx < W) ? (float)P.lat[(size_t)gy * W + gx] : 0.0f;
        }
        for (int i = tid; i < cc * SH * SW; i += TS2_THREADS) {
            const int c = i / (SH * SW), rem = i - c * SH * SW, r = rem / SW, col = rem - r * SW;
            const int gy = sy0 + r, gx = sx0 + col;
            float v = 0.0f;
            if (gy >= 0 && gy < ch && gx >= 0 && gx < cw)
                v = P.stk8 ? (float)P.stk8[((size_t)c * ch + gy) * cw + gx] : __ldg(P.stk + ((size_t)c * ch + gy) * cw + gx);
            St[i] = v;
        }
    }
    // ---- weights (overlaps the bulk copies)
    for (int i = tid; i < hid * CINP; i += TS2_THREADS) {
        const int hh = i / CINP, ci = i - hh * CINP;
        sw0[i] = ci < cin ? P.w0[hh * cin + ci] : 0.0f;
    }
    for (int i = tid; i < hid; i += TS2_THREADS) sb0[i] = P.b0[i];
    for (int i = tid; i < hid * CP; i += TS2_THREADS) {
        const int hh = i / CP, c = i - hh * CP;
        sw1[i] = c < C ? P.w1[c * hid + hh] : 0.0f;
    }
    for (int i = tid; i < CP; i += TS2_THREADS) {
        sb1[i] = i < C ? P.b1[i] : 0.0f;
        sbs[i] = (i < C && P.stab_in) ? P.bs[i] : 0.0f;
        sbo[i] = i < C ? P.bo[i] : 0.0f;
        for (int l = 0; l < 2; l++) sb3[l * CP + i] = (i < C && l < n3) ? P.b3[l][i] : 0.0f;
    }
    for (int l = 0; l < n3; l++)
        for (int i = tid; i < C * 9 * CP; i += TS2_THREADS) {
            const int co = i % CP, t = i / CP;  // t = ci * 9 + ky * 3 + kx
            sw3[l * C * 9 * CP + i] = co < C ? P.w3[l][(co * C + t / 9) * 9 + t % 9] : 0.0f;
        }
    for (int i = tid; i < C * CINP; i += TS2_THREADS) {
        const int c = i / CINP, ci = i - c * CINP;
        sws[i] = (ci < P.stab_in) ? P.ws[c * P.stab_in + ci] : 0.0f;
    }
    for (int i = tid; i < C * CP; i += TS2_THREADS) {
        const int c = i / CP, k = i - c * CP;
        swo[i] = k < C ? P.wo[c * C + k] : 0.0f;
    }
    for (int i = tid; i < 64; i += TS2_THREADS) {
        const int t2 = i & 3, dv = (i >> 2) & 1, t1 = (i >> 3) & 3, du = i >> 5;
        skt[i] = P.kt[(1 - du) + 6 - 2 * t1][(1 - dv) + 6 - 2 * t2];
    }
    for (int i = tid; i < 56; i += TS2_THREADS) skc[i] = (i & 7) < 7 ? P.kc[i >> 3][i & 7] : 0.0f;
    if (P.use_tma) {
        const uint32_t bar_a = (uint32_t)__cvta_generic_to_shared(bar);
        uint32_t done = 0;
        while (!done) {
            asm volatile(
                "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n selp.u32 %0, 1, 0, p;\n}\n"
                : "=r"(done)
                : "r"(bar_a)
                : "memory");
        }
        for (int i = tid; i < LW * LH; i += TS2_THREADS) Lf[i] = (float)Lt[i];
    }
    __syncthreads();

    // ---- stage A on 2 x 2 quads of the region
    const int QW = RW / 2, nQ = (RH / 2) * QW;
    for (int q = tid; q < nQ; q += TS2_THREADS) {
        const int qy = q / QW, qx = q - qy * QW;
        const int u0 = Y0 + 2 * qy, v0 = X0 + 2 * qx;  // even
        bool in[4];
        bool any_in = false;
#pragma unroll
        for (int p = 0; p < 4; p++) {
            const int u = u0 + (p >> 1), v = v0 + (p & 1);
            in[p] = u >= 0 && u < H && v >= 0 && v < W;
            any_in |= in[p];
        }
        if (!any_in) continue;  // (filled by the fix-up pass)
        float x[4][CINP];
#pragma unroll
        for (int p = 0; p < 4; p++)
#pragma unroll
            for (int ci = 0; ci < CINP; ci++) x[p][ci] = 0.0f;
        {
            // channel 0: conv2d(latent, kron 7x7, zero padding) + latent (upsampling.py:189-196), sliding over the 8 rows
            // of the quad's 8 x 8 window; every output accumulates in (ka, kb) raster order
            const float *lp = Lf + (u0 - 3 - ly0) * LW + (v0 - 3 - lx0);
            float acc[4] = {0.0f, 0.0f, 0.0f, 0.0f}, centre[4] = {0.0f, 0.0f, 0.0f, 0.0f};
            float wprev[7];
#pragma unroll
            for (int a = 0; a < 8; a++) {
                float r[8];
#pragma unroll
                for (int b = 0; b < 8; b++) r[b] = lp[a * LW + b];
                float wcur[7];
                if (a < 7) {
#pragma unroll
                    for (int b = 0; b < 7; b++) wcur[b] = skc[a * 8 + b];
                }
#pragma unroll
                for (int b = 0; b < 7; b++) {
                    if (a < 7) {  // row a is tap row ka = a of the outputs with dy = 0
                        acc[0] = __fmaf_rn(wcur[b], r[b], acc[0]);
                        acc[1] = __fmaf_rn(wcur[b], r[b + 1], acc[1]);
                    }
                    if (a >= 1) {  // and tap row ka = a - 1 of the outputs with dy = 1
                        acc[2] = __fmaf_rn(wprev[b], r[b], acc[2]);
                        acc[3] = __fmaf_rn(wprev[b], r[b + 1], acc[3]);
                    }
                }
                if (a == 3) { centre[0] = r[3]; centre[1] = r[4]; }
                if (a == 4) { centre[2] = r[3]; centre[3] = r[4]; }
                if (a < 7) {
#pragma unroll
                    for (int b = 0; b < 7; b++) wprev[b] = wcur[b];
                }
            }
#pragma unroll
            for (int p = 0; p < 4; p++) x[p][0] = __fadd_rn(acc[p], centre[p]);
        }
        {
            // channels 1 .. cc: transposed conv (8x8 kron, stride 2, replicate-padded input, crop 11; upsampling.py:312-325)
            const int qy0 = u0 >> 1, qx0 = v0 >> 1;  // (arithmetic shifts: u0, v0 may be negative on border tiles)
            int ro[5], co[5];
#pragma unroll
            for (int t = 0; t < 5; t++) {
                ro[t] = (clampi(qy0 - 2 + t, 0, ch - 1) - sy0) * SW;
                co[t] = clampi(qx0 - 2 + t, 0, cw - 1) - sx0;
            }
#pragma unroll
            for (int c = 0; c < CINP - 1; c++) {
                if (c < cc) {
                    const float *sp = St + c * SH * SW;
                    float win[5][5];
#pragma unroll
                    for (int i = 0; i < 5; i++)
#pragma unroll
                        for (int j = 0; j < 5; j++) win[i][j] = sp[ro[i] + co[j]];
#pragma unroll
                    for (int du = 0; du < 2; du++)
#pragma unroll
                        for (int dv = 0; dv < 2; dv++) {
                            float acc = 0.0f;
#pragma unroll
                            for (int t1 = 0; t1 < 4; t1++) {
                                const float4 w4 = *reinterpret_cast<const float4 *>(skt + ((du * 4 + t1) * 2 + dv) * 4);
                                acc = __fmaf_rn(w4.x, win[t1 + du][0 + dv], acc);
                                acc = __fmaf_rn(w4.y, win[t1 + du][1 + dv], acc);
                                acc = __fmaf_rn(w4.z, win[t1 + du][2 + dv], acc);
                                acc = __fmaf_rn(w4.w, win[t1 + du][3 + dv], acc);
                            }
                            x[du * 2 + dv][c + 1] = acc;
                        }
                }
            }
        }
        float o[4][C];
#pragma unroll
        for (int p = 0; p < 4; p++)
#pragma unroll
            for (int c = 0; c < C; c++) o[p][c] = sb1[c];
        for (int hh = 0; hh < hid; hh++) {
            float wv[CINP];
#pragma unroll
            for (int v = 0; v < CINP / 4; v++) {
                const float4 t = *reinterpret_cast<const float4 *>(sw0 + hh * CINP + 4 * v);
                wv[4 * v] = t.x; wv[4 * v + 1] = t.y; wv[4 * v + 2] = t.z; wv[4 * v + 3] = t.w;
            }
            float w1v[CP];
#pragma unroll
            for (int v = 0; v < CP / 4; v++) {
                const float4 t = *reinterpret_cast<const float4 *>(sw1 + hh * CP + 4 * v);
                w1v[4 * v] = t.x; w1v[4 * v + 1] = t.y; w1v[4 * v + 2] = t.z; w1v[4 * v + 3] = t.w;
            }
            const float bb = sb0[hh];
#pragma unroll
            for (int p = 0; p < 4; p++) {
                float a = bb;
#pragma unroll
                // (inputs and weights beyond cin are +0: fma(0, 0, a) == a bit for bit -- a starts from a bias that is never
                // -0 and a sum is -0 only if both terms are --, so no per-term test: a predicate copy per FMA was a third
                // of this loop's instructions)
                for (int ci = 0; ci < CINP; ci++) a = __fmaf_rn(wv[ci], x[p][ci], a);
                if (P.relu0) a = fmaxf(a, 0.0f);
#pragma unroll
                for (int c = 0; c < C; c++) o[p][c] = __fmaf_rn(w1v[c], a, o[p][c]);
            }
        }
#pragma unroll
        for (int p = 0; p < 4; p++) {
            if (!in[p]) continue;
            const int py = 2 * qy + (p >> 1), px = 2 * qx + (p & 1);
#pragma unroll
            for (int c = 0; c < C; c++) bufA[(c * RH + py) * RW + px] = P.relu1 ? fmaxf(o[p][c], 0.0f) : o[p][c];
            const int ty = py - n3e, tx = px - n3e;
            if (P.stab_in && ty >= 0 && ty < SF_TH && tx >= 0 && tx < SF_TW) {
#pragma unroll
                for (int c = 0; c < C; c++) {
                    float a = sbs[c];
#pragma unroll
                    for (int ci = 0; ci < CINP; ci++) a = __fmaf_rn(sws[c * CINP + ci], x[p][ci], a);  // (zero-padded: as above)
                    sstab[(c * SF_TH + ty) * SF_TW + tx] = a;
                }
            }
        }
    }
    __syncthreads();
    // ---- replicate padding on border tiles: out-of-frame positions of the region copy the clamped position
    if (Y0 < 0 || X0 < 0 || Y0 + RH > H || X0 + RW > W) {
        for (int pp = tid; pp < RH * RW; pp += TS2_THREADS) {
            const int py = pp / RW, px = pp - py * RW;
            const int u = Y0 + py, v = X0 + px;
            if (u >= 0 && u < H && v >= 0 && v < W) continue;
            const int sy = clampi(u, 0, H - 1) - Y0, sx = clampi(v, 0, W - 1) - X0;
#pragma unroll
            for (int c = 0; c < C; c++) bufA[(c * RH + py) * RW + px] = bufA[(c * RH + sy) * RW + sx];
        }
        __syncthreads();
    }
    // ---- 3x3 layers: two horizontally adjacent outputs per thread
    const float *cur = bufA;
    int cwid = RW, chh = RH, off = n3e;
    for (int l = 0; l < n3 - 1; l++) {
        const int ow = cwid - 2, oh = chh - 2;
        const float *wl = sw3 + l * C * 9 * CP;
        for (int pp = tid; pp < (ow / 2) * oh; pp += TS2_THREADS) {
            const int py = pp / (ow / 2), px = 2 * (pp - py * (ow / 2));
            const int gy = clampi(y0 - (off - 1) + py, 0, H - 1);
            const int by = gy - (y0 - off);
            const int bx0 = clampi(x0 - (off - 1) + px, 0, W - 1) - (x0 - off);
            const int bx1 = clampi(x0 - (off - 1) + px + 1, 0, W - 1) - (x0 - off);
            float acc0[C], acc1[C];
#pragma unroll
            for (int co = 0; co < C; co++) acc0[co] = acc1[co] = sb3[l * CP + co];
#pragma unroll
            for (int ci = 0; ci < C; ci++)
#pragma unroll
                for (int ky = 0; ky < 3; ky++) {
                    const float *row = cur + (ci * chh + by + ky - 1) * cwid;
                    float v0[3], v1[3];
                    if (bx1 == bx0 + 1) {
                        v0[0] = row[bx0 - 1]; v0[1] = row[bx0]; v0[2] = row[bx0 + 1];
                        v1[0] = v0[1]; v1[1] = v0[2]; v1[2] = row[bx0 + 2];
                    } else {
                        v0[0] = row[bx0 - 1]; v0[1] = row[bx0]; v0[2] = row[bx0 + 1];
                        v1[0] = row[bx1 - 1]; v1[1] = row[bx1]; v1[2] = row[bx1 + 1];
                    }
#pragma unroll
                    for (int kx = 0; kx < 3; kx++) {
                        float w[CP];
#pragma unroll
                        for (int v = 0; v < CP / 4; v++) {
                            const float4 t = *reinterpret_cast<const float4 *>(wl + ((ci * 3 + ky) * 3 + kx) * CP + 4 * v);
                            w[4 * v] = t.x; w[4 * v + 1] = t.y; w[4 * v + 2] = t.z; w[4 * v + 3] = t.w;
                        }
#pragma unroll
                        for (int co = 0; co < C; co++) {
                            acc0[co] = __fmaf_rn(w[co], v0[kx], acc0[co]);
                            acc1[co] = __fmaf_rn(w[co], v1[kx], acc1[co]);
                        }
                    }
                }
#pragma unroll
            for (int co = 0; co < C; co++) {
                float a0 = acc0[co], a1 = acc1[co];
                if (P.res3[l]) {
                    a0 = __fadd_rn(a0, cur[(co * chh + by) * cwid + bx0]);
                    a1 = __fadd_rn(a1, cur[(co * chh + by) * cwid + bx1]);
                }
                if (P.relu3[l]) { a0 = fmaxf(a0, 0.0f); a1 = fmaxf(a1, 0.0f); }
                bufB[(co * oh + py) * ow + px] = a0;
                bufB[(co * oh + py) * ow + px + 1] = a1;
            }
        }
        __syncthreads();
        cur = bufB;
        cwid = ow;
        chh = oh;
        off -= 1;
    }
    // ---- last stage on the tile (one pair of pixels per thread): last 3x3 layer (if any), + stabiliser, output
    // transform, frame tail, 64-bit stores
    const float M = P.M;
    float *uvq = sstab;  // 4:2:0 tail: rounded U, V of the tile where the stabiliser output was (own position, read first)
    for (int pp = tid; pp < (SF_TW / 2) * SF_TH; pp += TS2_THREADS) {
        const int ty = pp / (SF_TW / 2), tx = 2 * (pp - ty * (SF_TW / 2));
        const int gy = y0 + ty, gx = x0 + tx;
        const bool in0 = gy < H && gx < W, in1 = gy < H && gx + 1 < W;
        const int tyc = in0 ? ty : 0, txc = in0 ? tx : 0;  // (out-of-frame pairs compute on a valid position, store nothing)
        const int by = tyc + off, bx0 = txc + off;
        const int bx1 = (in1 ? txc + 1 : txc) + off;
        float t0[C], t1[C];
        if (n3 > 0) {
            const int l = n3 - 1;
            const float *wl = sw3 + l * C * 9 * CP;
#pragma unroll
            for (int co = 0; co < C; co++) t0[co] = t1[co] = sb3[l * CP + co];
#pragma unroll
            for (int ci = 0; ci < C; ci++)
#pragma unroll
                for (int ky = 0; ky < 3; ky++) {
                    const float *row = cur + (ci * chh + by + ky - 1) * cwid;
                    float v0[3], v1[3];
                    v0[0] = row[bx0 - 1]; v0[1] = row[bx0]; v0[2] = row[bx0 + 1];
                    if (bx1 == bx0 + 1) {
                        v1[0] = v0[1]; v1[1] = v0[2]; v1[2] = row[bx0 + 2];
                    } else {
                        v1[0] = row[bx1 - 1]; v1[1] = row[bx1]; v1[2] = row[bx1 + 1];
                    }
#pragma unroll
                    for (int kx = 0; kx < 3; kx++) {
                        float w[CP];
#pragma unroll
                        for (int v = 0; v < CP / 4; v++) {
                            const float4 t = *reinterpret_cast<const float4 *>(wl + ((ci * 3 + ky) * 3 + kx) * CP + 4 * v);
                            w[4 * v] = t.x; w[4 * v + 1] = t.y; w[4 * v + 2] = t.z; w[4 * v + 3] = t.w;
                        }
#pragma unroll
                        for (int co = 0; co < C; co++) {
                            t0[co] = __fmaf_rn(w[co], v0[kx], t0[co]);
                            t1[co] = __fmaf_rn(w[co], v1[kx], t1[co]);
                        }
                    }
                }
#pragma unroll
            for (int co = 0; co < C; co++) {
                if (P.res3[l]) {
                    t0[co] = __fadd_rn(t0[co], cur[(co * chh + by) * cwid + bx0]);
                    t1[co] = __fadd_rn(t1[co], cur[(co * chh + by) * cwid + bx1]);
                }
                if (P.relu3[l]) { t0[co] = fmaxf(t0[co], 0.0f); t1[co] = fmaxf(t1[co], 0.0f); }
            }
        } else {
#pragma unroll
            for (int co = 0; co < C; co++) {
                t0[co] = cur[(co * chh + by) * cwid + bx0];
                t1[co] = cur[(co * chh + by) * cwid + bx1];
            }
        }
        if (P.stab_in) {
#pragma unroll
            for (int co = 0; co < C; co++) {
                t0[co] = __fadd_rn(t0[co], sstab[(co * SF_TH + tyc) * SF_TW + txc]);
                t1[co] = __fadd_rn(t1[co], sstab[(co * SF_TH + tyc) * SF_TW + (in1 ? txc + 1 : txc)]);
            }
        }
        float ov0[C], ov1[C];
#pragma unroll
        for (int co = 0; co < C; co++) {
            float a0 = sbo[co], a1 = sbo[co];
#pragma unroll
            for (int ci = 0; ci < C; ci++) {
                a0 = __fmaf_rn(swo[co * CP + ci], t0[ci], a0);
                a1 = __fmaf_rn(swo[co * CP + ci], t1[ci], a1);
            }
            ov0[co] = a0;
            ov1[co] = a1;
        }
        const size_t oi = (size_t)gy * W + gx;
        if (P.finish != 0) {
#pragma unroll
            for (int co = 0; co < C; co++) {
                ov0[co] = quant(ov0[co], M);
                ov1[co] = quant(ov1[co], M);
            }
        }
        const int n_full = P.finish == 2 ? 1 : C;  // planes stored at full resolution by this loop
#pragma unroll
        for (int co = 0; co < C; co++) {
            if (co < n_full) {
                float a0 = ov0[co], a1 = ov1[co];
                if (P.finish != 0) { a0 = quant(clamp01(a0), M); a1 = quant(clamp01(a1), M); }
                float *dst = P.out[co] + oi;
                if (in1 && (reinterpret_cast<uintptr_t>(dst) & 7) == 0) *reinterpret_cast<float2 *>(dst) = make_float2(a0, a1);
                else {
                    if (in0) P.out[co][oi] = a0;
                    if (in1) P.out[co][oi + 1] = a1;
                }
            }
        }
        if (P.finish == 2) {
            // (rounded U, V of own positions; read above, overwritten now)
            uvq[(0 * SF_TH + ty) * SF_TW + tx] = ov0[1 < C ? 1 : 0];
            uvq[(0 * SF_TH + ty) * SF_TW + tx + 1] = ov1[1 < C ? 1 : 0];
            uvq[(1 * SF_TH + ty) * SF_TW + tx] = ov0[2 < C ? 2 : 0];
            uvq[(1 * SF_TH + ty) * SF_TW + tx + 1] = ov1[2 < C ? 2 : 0];
        }
    }
    if (P.finish == 2) {
        __syncthreads();
        const int h2 = H / 2, w2 = W / 2;
        for (int pp = tid; pp < 2 * (SF_TW / 2) * (SF_TH / 2); pp += TS2_THREADS) {
            const int c = pp / ((SF_TW / 2) * (SF_TH / 2)), r = pp - c * (SF_TW / 2) * (SF_TH / 2);
            const int by = r / (SF_TW / 2), bx = r - by * (SF_TW / 2);
            const int y2 = y0 / 2 + by, x2 = x0 / 2 + bx;
            if (y2 >= h2 || x2 >= w2) continue;
            const float *q = uvq + (c * SF_TH + 2 * by) * SF_TW + 2 * bx;
            float s = 0.0f;
            s = __fadd_rn(s, q[0]);
            s = __fadd_rn(s, q[1]);
            s = __fadd_rn(s, q[SF_TW]);
            s = __fadd_rn(s, q[SF_TW + 1]);
            P.out[1 + c][(size_t)y2 * w2 + x2] = quant(clamp01(__fdiv_rn(s, 4.0f)), M);
        }
    }
}

__global__ void k_add(float *__restrict__ a, const float *__restrict__ b, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) a[i] = __fadd_rn(a[i], b[i]);
}

// legacy "nearest": src = min(floor(dst * (in/out as fp32)), in - 1)
__global__ void k_resize_nearest(const float *__restrict__ in, int h, int w, float *__restrict__ out, int H, int W,
                                 float sy, float sx) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    const int c = blockIdx.z;
    if (x >= W || y >= H) return;
    int yy = (int)floorf(__fmul_rn((float)y, sy));
    int xx = (int)floorf(__fmul_rn((float)x, sx));
    yy = yy > h - 1 ? h - 1 : yy;
    xx = xx > w - 1 ? w - 1 : xx;
    out[((size_t)c * H + y) * W + x] = in[((size_t)c * h + yy) * w + xx];
}

// F.interpolate(mode = bilinear | bicubic, align_corners=False, antialias=False), same operation order as
// oracle/ccoracle.c::resize_torch (PyTorch's separable CPU kernel): per axis src = fma(scale, dst + 0.5, -0.5),
// taps clamped to the grid, A = -0.75 cubic coefficients; value = sum_i wy[i] * (sum_j wx[j] * v[i][j]) as fma chains.
__device__ __forceinline__ float cubic_near(float x) {
    const float a = __fsub_rn(__fmul_rn(1.25f, x), 2.25f);
    return __fmaf_rn(__fmul_rn(a, x), x, 1.0f);
}
__device__ __forceinline__ float cubic_far(float x) {
    const float a = __fadd_rn(__fmul_rn(-0.75f, x), 3.75f);
    const float b = __fadd_rn(__fmul_rn(a, x), -6.0f);
    return __fadd_rn(__fmul_rn(b, x), 3.0f);
}
template <int MODE>  // 1 bilinear (2 taps), 2 bicubic (4 taps)
__device__ __forceinline__ void resize_taps(int n_in, int i, float scale, int (&idx)[4], float (&wt)[4]) {
    float src = __fmaf_rn(scale, __fadd_rn((float)i, 0.5f), -0.5f);
    if (MODE == 1 && src < 0.0f) src = 0.0f;
    int i0 = (int)floorf(src);
    if (i0 > n_in - 1) i0 = n_in - 1;
    float lam = __fsub_rn(src, (float)i0);
    lam = lam < 0.0f ? 0.0f : (lam > 1.0f ? 1.0f : lam);
    if (MODE == 1) {
        idx[0] = i0;
        idx[1] = i0 + (i0 < n_in - 1 ? 1 : 0);
        wt[0] = __fsub_rn(1.0f, lam);
        wt[1] = lam;
    } else {
#pragma unroll
        for (int j = 0; j < 4; j++) idx[j] = clampi(i0 + j - 1, 0, n_in - 1);
        const float x2 = __fsub_rn(1.0f, lam);
        wt[0] = cubic_far(__fadd_rn(lam, 1.0f));
        wt[1] = cubic_near(lam);
        wt[2] = cubic_near(x2);
        wt[3] = cubic_far(__fadd_rn(x2, 1.0f));
    }
}
template <int MODE>
__global__ void k_resize_torch(const float *__restrict__ in, int h, int w, float *__restrict__ out, int H, int W,
                               float sy, float sx) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    const int c = blockIdx.z;
    if (x >= W || y >= H) return;
    constexpr int N = MODE == 1 ? 2 : 4;
    int iy[4], ix[4];
    float wy[4], wx[4];
    resize_taps<MODE>(h, y, sy, iy, wy);
    resize_taps<MODE>(w, x, sx, ix, wx);
    const float *p = in + (size_t)c * h * w;
    float acc = 0.0f;
#pragma unroll
    for (int i = 0; i < N; i++) {
        const float *row = p + (size_t)iy[i] * w;
        float r = __fmul_rn(wx[0], __ldg(row + ix[0]));
#pragma unroll
        for (int j = 1; j < N; j++) r = __fmaf_rn(wx[j], __ldg(row + ix[j]), r);
        acc = (i == 0) ? __fmul_rn(wy[0], r) : __fmaf_rn(wy[i], r, acc);
    }
    out[((size_t)c * H + y) * W + x] = acc;
}

// Common randomness (core/noise.py:18-55): sample k of the Park-Miller sequence, Box-Muller in f64.
// seed_j = a^j * seed_0 mod m is evaluated directly (square-and-multiply) instead of serially.
__device__ __forceinline__ uint64_t lcg_pow(uint64_t e) {
    const uint64_t m = 2147483647ULL;
    uint64_t r = 1, b = 16807ULL;
    while (e) {
        if (e & 1) r = (r * b) % m;
        b = (b * b) % m;
        e >>= 1;
    }
    return r;
}
__global__ void k_cr_noise(float *__restrict__ out, size_t first, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t m = 2147483647ULL;
    const size_t k = first + i;
    const uint64_t s1 = (lcg_pow(2 * k + 1) * 18101995ULL) % m;
    const uint64_t s2 = (s1 * 16807ULL) % m;
    const double u1 = (double)s1 / (double)m, u2 = (double)s2 / (double)m;
    // Box-Muller (noise.py:28-34) with the canonical log / cos of ccd_detmath.h: bit-identical to the oracle
    out[i] = (float)__dmul_rn(__dsqrt_rn(__dmul_rn(-2.0, ccdm_log(u1))), ccdm_cos(__dmul_rn(2 * 3.14159265359, u2)));
}

__device__ __forceinline__ float quant(float v, float M) { return __fdiv_rn(rintf(__fmul_rn(M, v)), M); }
__device__ __forceinline__ float clamp01(float v) { return v < 0.0f ? 0.0f : (v > 1.0f ? 1.0f : v); }

__global__ void k_finish_444(const float *__restrict__ in, size_t n, float M, float *__restrict__ out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = quant(clamp01(quant(in[i], M)), M);
}

__global__ void k_finish_420_uv(const float *__restrict__ in, int h, int w, float M, float *__restrict__ ou,
                                float *__restrict__ ov) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    const int c = blockIdx.z;  // 0: u, 1: v
    const int h2 = h / 2, w2 = w / 2;
    if (x >= w2 || y >= h2) return;
    const float *p = in + (size_t)(c + 1) * h * w;
    float s = 0.0f;
#pragma unroll
    for (int dy = 0; dy < 2; dy++)
#pragma unroll
        for (int dx = 0; dx < 2; dx++) s = __fadd_rn(s, quant(p[(size_t)(2 * y + dy) * w + 2 * x + dx], M));
    float v = __fdiv_rn(s, 4.0f);
    (c == 0 ? ou : ov)[(size_t)y * w2 + x] = quant(clamp01(v), M);
}

inline dim3 grid2(int w, int h, int z = 1) { return dim3((w + 31) / 32, (h + 7) / 8, z); }
const dim3 kBlock2(32, 8, 1);

K1d make_k1d(const float *w1d, int k) {
    K1d r;
    for (int i = 0; i < 16; i++) r.w[i] = i < k ? w1d[i] : 0.0f;
    return r;
}

}  // namespace

int ccd_ups_first(const int8_t *d_lat, int h, int w, float *d_out, cudaStream_t st) {
    size_t n = (size_t)h * w;
    k_ups_first<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_lat, n, d_out);
    g_ccd_launches++;
    return (int)cudaGetLastError();
}

int ccd_ups_pre(const int8_t *d_lat, int h, int w, const float *w1d, int k, float *d_out, cudaStream_t st) {
    k_ups_pre<<<grid2(w, h), kBlock2, 0, st>>>(d_lat, h, w, make_k1d(w1d, k), k, d_out);
    g_ccd_launches++;
    return (int)cudaGetLastError();
}

int ccd_ups_convt(const float *d_in, int c, int h, int w, const float *w1d, int k, float *d_out, int ht,
                  int wt, cudaStream_t st) {
    k_ups_convt<<<grid2(wt, ht, c), kBlock2, 0, st>>>(d_in, h, w, make_k1d(w1d, k), k, d_out, ht, wt);
    g_ccd_launches++;
    return (int)cudaGetLastError();
}

int ccd_ups_level(const int8_t *d_lat, int th, int tw, const float *d_in, int cc, int ch, int cw, const float *wt1d,
                  const float *wc1d, float *d_out, cudaStream_t st) {
    UpsLevelParams P;
    P.lat = d_lat; P.in = d_in; P.out = d_out; P.cc = cc; P.ch = ch; P.cw = cw; P.th = th; P.tw = tw;
    for (int a = 0; a < 8; a++)
        for (int b = 0; b < 8; b++) {
            volatile float k = wt1d[a] * wt1d[b];  // one rounded fp32 product, no contraction
            P.kt[a][b] = k;
        }
    for (int a = 0; a < 7; a++)
        for (int b = 0; b < 7; b++) {
            volatile float k = wc1d[a] * wc1d[b];
            P.kc[a][b] = k;
        }
    k_ups_level<<<grid2(tw, th, cc + 1), kBlock2, 0, st>>>(P);
    g_ccd_launches++;
    return (int)cudaGetLastError();
}

int ccd_syn_layer(const float *d_in, int h, int w, const SynLayerDev &L, float *d_out, cudaStream_t st) {
    k_syn_layer<<<grid2(w, h), kBlock2, 0, st>>>(d_in, h, w, L.cin, L.cout, L.k, L.residual, L.relu, L.w, L.b,
                                                 d_out);
    g_ccd_launches++;
    return (int)cudaGetLastError();
}

int ccd_syn_pointwise2(const float *d_in, int h, int w, const SynLayerDev &L0, const SynLayerDev &L1,
                       float *d_out, cudaStream_t st) {
    // preconditions checked by the caller: k == 1, no residual, cin <= 16, cout(L1) <= 8
    size_t plane = (size_t)h * w;
    size_t smem = ((size_t)L0.cout * L0.cin + L0.cout + (size_t)L1.cout * L0.cout + L1.cout) * sizeof(float);
    k_syn_pw2<16, 8><<<(unsigned)((plane + 255) / 256), 256, smem, st>>>(
        d_in, plane, L0.cin, L0.cout, L1.cout, L0.relu, L1.relu, L0.w, L0.b, L1.w, L1.b, d_out);
    g_ccd_launches++;
    return (int)cudaGetLastError();
}

template <int CINP, int C>
static int launch_syn_fused(const SynFusedParams &P, cudaStream_t st) {
    constexpr int CP = (C + 3) & ~3;
    const int RW = SF_TW + 2 * P.n3, RH = SF_TH + 2 * P.n3;
    size_t fl = (size_t)P.hid * CINP + P.hid + (size_t)P.hid * CP + CP + 2 * C * C * 9 + 2 * CP + C * CINP + CP + C * CP + CP;
    fl += (size_t)C * RH * RW + (P.n3 == 2 ? (size_t)C * (RH - 2) * (RW - 2) : 0) + (size_t)C * SF_TH * SF_TW;
    const size_t smem = fl * sizeof(float);
    auto kern = k_syn_fused<CINP, C>;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
    }
    const dim3 grid((P.w + SF_TW - 1) / SF_TW, (P.h + SF_TH - 1) / SF_TH, 1);
    kern<<<grid, SF_THREADS, smem, st>>>(P);
    g_ccd_launches++;
    return (int)cudaGetLastError();
}

// returns -1 when the architecture is outside the fused family (caller falls back to the layer kernels)
int ccd_syn_fused(const float *d_in, int h, int w, int cin, const SynLayerDev *layers, int n_layers,
                  const SynLayerDev *stab, const SynLayerDev &ot, float *d_out, cudaStream_t st) {
    if (n_layers < 2 || n_layers > 4) return -1;
    const SynLayerDev &L0 = layers[0], &L1 = layers[1];
    const int C = L1.cout;
    if (L0.k != 1 || L1.k != 1 || L0.residual || L1.residual || cin > 16 || L0.cout > 256 || C < 2 || C > 5) return -1;
    if (ot.cin != C || ot.cout != C) return -1;
    for (int l = 2; l < n_layers; l++)
        if (layers[l].k != 3 || layers[l].cin != C || layers[l].cout != C) return -1;
    if (stab && (stab->cin > cin || stab->cout != C)) return -1;
    SynFusedParams P;
    P.in = d_in; P.out = d_out; P.h = h; P.w = w; P.cin = cin; P.hid = L0.cout; P.n3 = n_layers - 2;
    P.relu0 = L0.relu; P.relu1 = L1.relu;
    for (int l = 0; l < 2; l++) {
        const bool on = l < P.n3;
        P.res3[l] = on ? layers[2 + l].residual : 0;
        P.relu3[l] = on ? layers[2 + l].relu : 0;
        P.w3[l] = on ? layers[2 + l].w : nullptr;
        P.b3[l] = on ? layers[2 + l].b : nullptr;
    }
    P.stab_in = stab ? stab->cin : 0;
    P.w0 = L0.w; P.b0 = L0.b; P.w1 = L1.w; P.b1 = L1.b;
    P.ws = stab ? stab->w : nullptr; P.bs = stab ? stab->b : nullptr;
    P.wo = ot.w; P.bo = ot.b;
    const int cinp = cin <= 4 ? 4 : (cin <= 8 ? 8 : 16);
#define SF_CASE(CI, CC) if (cinp == CI && C == CC) return launch_syn_fused<CI, CC>(P, st)
    SF_CASE(4, 2); SF_CASE(4, 3); SF_CASE(4, 4); SF_CASE(4, 5);
    SF_CASE(8, 2); SF_CASE(8, 3); SF_CASE(8, 4); SF_CASE(8, 5);
    SF_CASE(16, 2); SF_CASE(16, 3); SF_CASE(16, 4); SF_CASE(16, 5);
#undef SF_CASE
    return -1;
}

// ---- batched float tail: host side -----------------------------------------------------------------------
size_t ccd_tail_job_bytes(void) { return sizeof(TailSynJob); }
size_t ccd_tail_level_job_bytes(void) { return sizeof(UpsLevelJob); }

void ccd_tail_fill_level(void *dst, const int8_t *lat, const float *in, const int8_t *in8, float *out, int cc, int ch,
                         int cw, int th, int tw, const float *wt1d, const float *wc1d) {
    UpsLevelJob J;
    memset(&J, 0, sizeof(J));
    J.lat = lat; J.in = in; J.in8 = in8; J.out = out; J.cc = cc; J.ch = ch; J.cw = cw; J.th = th; J.tw = tw;
    for (int a = 0; a < 8; a++)
        for (int b = 0; b < 8; b++) {
            volatile float k = wt1d[a] * wt1d[b];  // one rounded fp32 product, no contraction
            J.kt[a][b] = k;
        }
    for (int a = 0; a < 7; a++)
        for (int b = 0; b < 7; b++) {
            volatile float k = wc1d[a] * wc1d[b];
            J.kc[a][b] = k;
        }
    memcpy(dst, &J, sizeof(J));
}

int ccd_tail_launch_level(const void *d_jobs, int n_jobs, int planes, int max_tw, int max_th, cudaStream_t st) {
    const dim3 grid((max_tw + 31) / 32, (max_th + 7) / 8, (unsigned)(n_jobs * planes));
    k_ups_level_b<<<grid, kBlock2, 0, st>>>(reinterpret_cast<const UpsLevelJob *>(d_jobs), planes);
    g_ccd_launches++;
    return (int)cudaGetLastError();
}

namespace {
typedef int (*PFN_encodeTiled)(void *tensorMap, int dataType, unsigned rank, void *globalAddress, const uint64_t *globalDim,
                               const uint64_t *globalStrides, const uint32_t *boxDim, const uint32_t *elementStrides,
                               int interleave, int swizzle, int l2Promotion, int oobFill);
PFN_encodeTiled get_encode_tiled() {
    static PFN_encodeTiled fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_encodeTiled>(p);
        cudaGetLastError();
    }
    return fn;
}
}  // namespace

// Fills one TailSynJob (host memory).  Returns 3 when the tiles are staged with TMA, 0 when with plain loads
// (pitches / addresses that cuTensorMapEncodeTiled does not take), < 0 when the architecture is outside the family.
int ccd_tail_fill_syn(void *dst, const CcdTailSynDesc &T) {
    const int n_layers = T.n_layers;
    if (n_layers < 2 || n_layers > 4) return -1;
    const SynLayerDev &L0 = T.layers[0], &L1 = T.layers[1];
    const int C = L1.cout;
    if (L0.k != 1 || L1.k != 1 || L0.residual || L1.residual || T.cin > 16 || T.cin < 2 || L0.cout > 256 || C < 2 || C > 5) return -1;
    if (T.ot.cin != C || T.ot.cout != C) return -1;
    for (int l = 2; l < n_layers; l++)
        if (T.layers[l].k != 3 || T.layers[l].cin != C || T.layers[l].cout != C) return -1;
    if (T.stab && (T.stab->cin > T.cin || T.stab->cout != C)) return -1;
    TailSynJob J;
    memset(&J, 0, sizeof(J));
    J.lat = T.lat; J.stk = T.stk; J.stk8 = T.stk8;
    for (int c = 0; c < 5; c++) J.out[c] = T.out[c];
    J.h = T.h; J.w = T.w; J.ch = T.ch; J.cw = T.cw; J.cin = T.cin; J.hid = L0.cout; J.n3 = n_layers - 2;
    J.relu0 = L0.relu; J.relu1 = L1.relu;
    for (int l = 0; l < 2; l++) {
        const bool on = l < J.n3;
        J.res3[l] = on ? T.layers[2 + l].residual : 0;
        J.relu3[l] = on ? T.layers[2 + l].relu : 0;
        J.w3[l] = on ? T.layers[2 + l].w : nullptr;
        J.b3[l] = on ? T.layers[2 + l].b : nullptr;
    }
    J.stab_in = T.stab ? T.stab->cin : 0;
    J.w0 = L0.w; J.b0 = L0.b; J.w1 = L1.w; J.b1 = L1.b;
    J.ws = T.stab ? T.stab->w : nullptr; J.bs = T.stab ? T.stab->b : nullptr;
    J.wo = T.ot.w; J.bo = T.ot.b;
    J.finish = T.finish;
    J.M = T.M;
    for (int a = 0; a < 8; a++)
        for (int b = 0; b < 8; b++) {
            volatile float k = T.wt1d[a] * T.wt1d[b];
            J.kt[a][b] = k;
        }
    for (int a = 0; a < 7; a++)
        for (int b = 0; b < 7; b++) {
            volatile float k = T.wc1d[a] * T.wc1d[b];
            J.kc[a][b] = k;
        }
    // TMA descriptors (CU_TENSOR_MAP_DATA_TYPE_UINT8 = 0, FLOAT32 = 7; no interleave, no swizzle, L2 promotion 128 B,
    // out-of-bounds elements read as zero)
    J.use_tma = 0;
    PFN_encodeTiled enc = get_encode_tiled();
    const int cc = T.cin - 1;
    if (enc && T.allow_tma && !T.stk8 && (T.w % 16) == 0 && (T.cw % 4) == 0 && (reinterpret_cast<uintptr_t>(T.lat) % 16) == 0 &&
        (reinterpret_cast<uintptr_t>(T.stk) % 16) == 0) {
        const uint64_t gd0[2] = {(uint64_t)T.w, (uint64_t)T.h};
        const uint64_t gs0[1] = {(uint64_t)T.w};
        const int n3t = ts2_n3e(J.n3);  // halo of the staged tiles
        const uint32_t bx0[2] = {(uint32_t)ts_lw(n3t), (uint32_t)ts_lh(n3t)};
        const uint32_t es[3] = {1, 1, 1};
        const uint64_t gd1[3] = {(uint64_t)T.cw, (uint64_t)T.ch, (uint64_t)cc};
        const uint64_t gs1[2] = {(uint64_t)T.cw * 4, (uint64_t)T.cw * 4 * (uint64_t)T.ch};
        const uint32_t bx1[3] = {(uint32_t)ts_sw(n3t), (uint32_t)ts_sh(n3t), (uint32_t)cc};
        const int r0 = enc(J.tmap_lat, 0, 2, const_cast<int8_t *>(T.lat), gd0, gs0, bx0, es, 0, 0, 1, 0);
        const int r1 = enc(J.tmap_stk, 7, 3, const_cast<float *>(T.stk), gd1, gs1, bx1, es, 0, 0, 1, 0);
        J.use_tma = (r0 == 0 && r1 == 0) ? 3 : 0;  // bit 0: TMA staging, bit 1: descriptor fence before the first use
    }
    memcpy(dst, &J, sizeof(J));
    return J.use_tma;
}

template <int CINP, int C>
static int launch_tail_syn(const void *d_jobs, int n_jobs, int n3_max, int hid_max, int max_w, int max_h, cudaStream_t st) {
    constexpr int CP = (C + 3) & ~3;
    const int n3t = ts2_n3e(n3_max);
    const int RW = SF_TW + 2 * n3t, RH = SF_TH + 2 * n3t;
    size_t bytes = 128 + (((size_t)ts_lw(n3t) * ts_lh(n3t) + 127) & ~(size_t)127);
    size_t fl = (((size_t)(CINP - 1) * ts_sh(n3t) * ts_sw(n3t) + 31) & ~(size_t)31);
    fl += (size_t)ts_lw(n3t) * ts_lh(n3t);
    fl += (size_t)hid_max * CINP + ((hid_max + 3) & ~3) + (size_t)hid_max * CP + CP + 2 * C * 9 * CP + 2 * CP + C * CINP + CP + C * CP + CP + 64 + 56;
    fl += (size_t)C * RH * RW + (n3_max == 2 ? (size_t)C * (RH - 2) * (RW - 2) : 0) + (size_t)C * SF_TH * SF_TW;
    const size_t smem = bytes + fl * sizeof(float);
    auto kern = k_tail_syn2<CINP, C>;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
    }
    const dim3 grid((max_w + SF_TW - 1) / SF_TW, (max_h + SF_TH - 1) / SF_TH, (unsigned)n_jobs);
    kern<<<grid, TS2_THREADS, smem, st>>>(reinterpret_cast<const TailSynJob *>(d_jobs));
    g_ccd_launches++;
    return (int)cudaGetLastError();
}

// all jobs of one launch share (cinp, C); n3 / hid / sizes may differ (shared memory sized for the maxima)
int ccd_tail_launch_syn(const void *d_jobs, int n_jobs, int cinp, int C, int n3_max, int hid_max, int max_w, int max_h,
                        cudaStream_t st) {
#define TS_CASE(CI, CC) if (cinp == CI && C == CC) return launch_tail_syn<CI, CC>(d_jobs, n_jobs, n3_max, hid_max, max_w, max_h, st)
    TS_CASE(4, 2); TS_CASE(4, 3); TS_CASE(4, 4); TS_CASE(4, 5);
    TS_CASE(8, 2); TS_CASE(8, 3); TS_CASE(8, 4); TS_CASE(8, 5);
    TS_CASE(16, 2); TS_CASE(16, 3); TS_CASE(16, 4); TS_CASE(16, 5);
#undef TS_CASE
    return -1;
}

int ccd_syn_add(float *d_a, const float *d_b, size_t n, cudaStream_t st) {
    k_add<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_a, d_b, n);
    g_ccd_launches++;
    return (int)cudaGetLastError();
}

int ccd_resize_nearest(const float *d_in, int c, int h, int w, float *d_out, int H, int W, cudaStream_t st) {
    k_resize_nearest<<<grid2(W, H, c), kBlock2, 0, st>>>(d_in, h, w, d_out, H, W, (float)h / (float)H,
                                                         (float)w / (float)W);
    g_ccd_launches++;
    return (int)cudaGetLastError();
}

int ccd_resize_torch(const float *d_in, int c, int h, int w, float *d_out, int H, int W, int mode, float sy, float sx,
                     cudaStream_t st) {
    if (mode == 1)
        k_resize_torch<1><<<grid2(W, H, c), kBlock2, 0, st>>>(d_in, h, w, d_out, H, W, sy, sx);
    else
        k_resize_torch<2><<<grid2(W, H, c), kBlock2, 0, st>>>(d_in, h, w, d_out, H, W, sy, sx);
    g_ccd_launches++;
    return (int)cudaGetLastError();
}

int ccd_cr_noise(float *d_out, size_t first, size_t n, cudaStream_t st) {
    k_cr_noise<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_out, first, n);
    g_ccd_launches++;
    return (int)cudaGetLastError();
}

// ---- output packing (io/format/yuv.py:150-162, ppm.py:160-203): finished planes -> integer samples.
// Planar: thread = 4 consecutive samples of one plane (one float4 load, one 4- or 8-byte store).
template <typename T>
__global__ void k_pack_planar(const float *__restrict__ p0, const float *__restrict__ p1, const float *__restrict__ p2,
                              size_t n0, size_t n1, float M, T *__restrict__ out) {
    const size_t total4 = (n0 + 3) / 4 + 2 * ((n1 + 3) / 4);
    for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < total4; q += (size_t)gridDim.x * blockDim.x) {
        const size_t q0 = (n0 + 3) / 4, q1 = (n1 + 3) / 4;
        const float *src;
        size_t base, n, off;
        if (q < q0) { src = p0; base = 0; n = n0; off = q * 4; }
        else if (q < q0 + q1) { src = p1; base = n0; n = n1; off = (q - q0) * 4; }
        else { src = p2; base = n0 + n1; n = n1; off = (q - q0 - q1) * 4; }
        T v[4];
        if (off + 4 <= n && ((reinterpret_cast<uintptr_t>(src + off) & 15) == 0)) {
            const float4 f = __ldg(reinterpret_cast<const float4 *>(src + off));
            v[0] = (T)rintf(__fmul_rn(f.x, M)); v[1] = (T)rintf(__fmul_rn(f.y, M));
            v[2] = (T)rintf(__fmul_rn(f.z, M)); v[3] = (T)rintf(__fmul_rn(f.w, M));
        } else {
#pragma unroll
            for (int k = 0; k < 4; k++) v[k] = (off + k < n) ? (T)rintf(__fmul_rn(__ldg(src + off + k), M)) : (T)0;
        }
        T *dst = out + base + off;
        if (off + 4 <= n && ((reinterpret_cast<uintptr_t>(dst) & (4 * sizeof(T) - 1)) == 0)) {
            if (sizeof(T) == 1) *reinterpret_cast<uchar4 *>(dst) = make_uchar4(v[0], v[1], v[2], v[3]);
            else *reinterpret_cast<ushort4 *>(dst) = make_ushort4(v[0], v[1], v[2], v[3]);
        } else {
#pragma unroll
            for (int k = 0; k < 4; k++)
                if (off + k < n) dst[k] = v[k];
        }
    }
}
// Interleaved [H][W][3]: thread = 4 pixels = 12 samples (three float4 loads, 12 or 24 contiguous bytes out).
template <typename T>
__global__ void k_pack_hwc(const float *__restrict__ p0, const float *__restrict__ p1, const float *__restrict__ p2, size_t n,
                           float M, T *__restrict__ out) {
    const size_t nq = (n + 3) / 4;
    for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += (size_t)gridDim.x * blockDim.x) {
        const size_t off = q * 4;
        T v[12];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const size_t i = off + k < n ? off + k : n - 1;
            v[3 * k] = (T)rintf(__fmul_rn(__ldg(p0 + i), M));
            v[3 * k + 1] = (T)rintf(__fmul_rn(__ldg(p1 + i), M));
            v[3 * k + 2] = (T)rintf(__fmul_rn(__ldg(p2 + i), M));
        }
        T *dst = out + off * 3;
        if (off + 4 <= n) {
            if (sizeof(T) == 1) {
                uint32_t *d32 = reinterpret_cast<uint32_t *>(dst);  // off * 3 is a multiple of 12: 4-byte aligned
#pragma unroll
                for (int k = 0; k < 3; k++)
                    d32[k] = (uint32_t)v[4 * k] | ((uint32_t)v[4 * k + 1] << 8) | ((uint32_t)v[4 * k + 2] << 16) |
                             ((uint32_t)v[4 * k + 3] << 24);
            } else {
                uint2 *d64 = reinterpret_cast<uint2 *>(dst);        // 24 bytes: 8-byte aligned
#pragma unroll
                for (int k = 0; k < 3; k++)
                    d64[k] = make_uint2((uint32_t)v[4 * k] | ((uint32_t)v[4 * k + 1] << 16),
                                        (uint32_t)v[4 * k + 2] | ((uint32_t)v[4 * k + 3] << 16));
            }
        } else {
            for (int k = 0; k < 12; k++)
                if (off * 3 + k < n * 3) dst[k] = v[k];
        }
    }
}

int ccd_pack(const float *const planes[3], int h, int w, int cs, int bitdepth, int sample_bytes, int interleaved,
             void *d_out, cudaStream_t st) {
    const float M = (float)((1 << bitdepth) - 1);
    const size_t n0 = (size_t)h * w, n1 = (size_t)(h >> cs) * (w >> cs);
    const unsigned blocks = 148 * 8;
    if (interleaved) {
        if (sample_bytes == 1) k_pack_hwc<uint8_t><<<blocks, 256, 0, st>>>(planes[0], planes[1], planes[2], n0, M, (uint8_t *)d_out);
        else k_pack_hwc<uint16_t><<<blocks, 256, 0, st>>>(planes[0], planes[1], planes[2], n0, M, (uint16_t *)d_out);
    } else {
        if (sample_bytes == 1) k_pack_planar<uint8_t><<<blocks, 256, 0, st>>>(planes[0], planes[1], planes[2], n0, n1, M, (uint8_t *)d_out);
        else k_pack_planar<uint16_t><<<blocks, 256, 0, st>>>(planes[0], planes[1], planes[2], n0, n1, M, (uint16_t *)d_out);
    }
    g_ccd_launches++;
    return (int)cudaGetLastError();
}

// n samples that already lie in output order (the planes of a batch of finished frames, one after the other)
int ccd_pack_flat(const float *d_in, size_t n, int bitdepth, int sample_bytes, void *d_out, cudaStream_t st) {
    const float M = (float)((1 << bitdepth) - 1);
    const unsigned blocks = 148 * 8;
    if (sample_bytes == 1) k_pack_planar<uint8_t><<<blocks, 256, 0, st>>>(d_in, d_in, d_in, n, 0, M, (uint8_t *)d_out);
    else k_pack_planar<uint16_t><<<blocks, 256, 0, st>>>(d_in, d_in, d_in, n, 0, M, (uint16_t *)d_out);
    g_ccd_launches++;
    return (int)cudaGetLastError();
}

int ccd_finish(const float *d_in, int h, int w, int bitdepth, int data_type, float *a, float *b, float *c,
               cudaStream_t st) {
    const float M = (float)((1 << bitdepth) - 1);
    const size_t n = (size_t)h * w;
    if (data_type != 1) {
        k_finish_444<<<(unsigned)((3 * n + 255) / 256), 256, 0, st>>>(d_in, 3 * n, M, a);
    } else {
        k_finish_444<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_in, n, M, a);
        if (h / 2 > 0 && w / 2 > 0) {
            k_finish_420_uv<<<grid2(w / 2, h / 2, 2), kBlock2, 0, st>>>(d_in, h, w, M, b, c);
            g_ccd_launches++;
        }
    }
    g_ccd_launches++;
    return (int)cudaGetLastError();
}
