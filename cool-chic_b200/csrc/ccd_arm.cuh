// ccd_arm.cuh -- device code shared by the entropy decoder (ccd_entropy.cu) and the data-parallel encoder
// (ccd_encode.cu): the causal context pattern, the fixed-point ARM / IFCE evaluation (fast quad layout and generic
// int64 path, blob layouts in ccd_internal.h) and the quantised-Laplace cumulatives (SURVEY Appendix C.1).
// Everything here is file-local (anonymous namespace) in each translation unit that includes it.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "ccd_internal.h"

namespace {

// context pattern: core/arm.py:496-562 (priority order over the 9x9 causal mask)
__constant__ int8_t c_ctx_dy[40] = {0,  -1, -1, -1, 0,  -2, -3, 0,  -1, -2, -2, -1, -2, -1,
                                    -2, -3, 0,  -1, -2, -2, -3, -3, -3, -4, -1, -4, -1, -2,
                                    -3, -3, -4, -4, -2, -3, -3, -4, -4, -4, -4, -4};
__constant__ int8_t c_ctx_dx[40] = {-1, 0,  -1, 1, -2, 0,  0,  -3, -2, 1,  -1, 2,  -2, -3,
                                    2,  1,  -4, 3, -3, 3,  -1, -2, 2,  0,  -4, -1, 4,  4,
                                    -3, 3,  -2, 1, -4, -4, 4,  -3, 2,  3,  -4, 4};

constexpr double kFreeWeight = 16777215.0 - 127.0;  // (2^24 - 1) - (max - min)
constexpr int kSymMin = -64, kSymMax = 63;

// trunc(FW * cdf(d / b)) with cdf the Laplace CDF of constriction's QuantizedLaplace
// (SURVEY Appendix C.1); d = (s - 0.5) - mu is exact in f64.
__device__ __forceinline__ uint32_t laplace_nonleaky(double d, double b) {
    double c;
    if (d <= 0.0)
        c = __dmul_rn(0.5, exp(__ddiv_rn(d, b)));
    else
        c = __dsub_rn(1.0, __dmul_rn(0.5, exp(__ddiv_rn(-d, b))));
    return (uint32_t)__double2ll_rz(__dmul_rn(kFreeWeight, c));
}

__device__ __forceinline__ uint32_t laplace_left_exact(int s, double mu, double b) {
    if (s <= kSymMin) return 0u;
    if (s > kSymMax) return 1u << 24;
    return laplace_nonleaky(((double)s - 0.5) - mu, b) + (uint32_t)(s - kSymMin);
}

__device__ __forceinline__ uint64_t shfl_xor_u64(uint64_t v, int mask) {
    uint32_t lo = __shfl_xor_sync(0xffffffffu, (uint32_t)v, mask);
    uint32_t hi = __shfl_xor_sync(0xffffffffu, (uint32_t)(v >> 32), mask);
    return ((uint64_t)hi << 32) | lo;
}

__device__ __forceinline__ int lds_s8(uint32_t a) {
    int v;
    asm volatile("ld.volatile.shared.s8 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
    return v;
}

// ---------------------------------------------------------------------------------------
// ARM / IFCE evaluation (armint.py:180-203).
// FAST path: int32 operands (proven safe by the host), int64 accumulators (IMAD.WIDE), and
// each symbol is spread over a QUAD of lanes: member m owns activations [m*OPM, m*OPM+OPM).
// One warp = 8 symbols.  This cuts the ARM latency ~8x w.r.t. one thread per symbol, which
// is what bounds the short diagonals (the next diagonal cannot start before its ARM is done).
template <int NCTX, int CF>
struct QuadArm {
    static constexpr int DIM = NCTX + CF;
    static constexpr int OPM = (DIM + 3) / 4;                       // activations per member
    static constexpr int OPMP = OPM <= 2 ? 2 : (OPM <= 4 ? 4 : 8);  // padded for vector LDS
    static constexpr int DIMP = 4 * OPM;
    static constexpr int CFP = (CF + 3) & ~3;
    static_assert(OPM <= 8, "ARM too wide for the quad layout");

    static __device__ __forceinline__ void ld_w(const int32_t *p, int32_t (&w)[8]) {
        if constexpr (OPMP == 2) {
            int2 a = *reinterpret_cast<const int2 *>(p);
            w[0] = a.x; w[1] = a.y;
        } else if constexpr (OPMP == 4) {
            int4 a = *reinterpret_cast<const int4 *>(p);
            w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w;
        } else {
            int4 a = *reinterpret_cast<const int4 *>(p);
            int4 b = *reinterpret_cast<const int4 *>(p + 4);
            w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w;
            w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
        }
    }

    // IFCE inputs of the pixel (y, x): the already decoded coarser grids at (y>>1 >> sh, x>>1 >> sh)
    // (component/coolchic.py:95-100, core/upsampling.py:575-593).  All loads are issued back to back,
    // BEFORE the producer waits for its dependencies: their L2 latency is hidden by that wait.
    static __device__ __forceinline__ void ifce_prefetch(const EntGrid *g, const int8_t *lat, int y, int x, int m,
                                                         int (&ifv)[CCD_IFCE_FAST_MAX]) {
#pragma unroll
        for (int c = 0; c < CCD_IFCE_FAST_MAX; c++) ifv[c] = 0;
        if constexpr (CF > 0) {
            const int n_in = g->ifce_in;
            if (n_in > 0 && (m + 1) * OPM > NCTX) {
                const int yy = y >> 1, xx = x >> 1;
#pragma unroll
                for (int c = 0; c < CCD_IFCE_FAST_MAX; c++) {
                    if (c < n_in) {
                        const int sh = g->ch_sh[c];
                        if (sh >= 0) ifv[c] = lat[g->ch_off[c] + (long long)(yy >> sh) * g->ch_w[c] + (xx >> sh)];
                    }
                }
            }
        }
    }

    // returns (mu, log-scale) in 1/256 units, identical on the 4 lanes of the quad
    static __device__ __forceinline__ void run(const EntGrid *g, const unsigned char *arm_blob,
                                               const unsigned char *ifce_blob, const int (&ifv)[CCD_IFCE_FAST_MAX],
                                               uint32_t rows, uint32_t row_mask, int n_hidden, int y, int x,
                                               int m, long long &o0, long long &o1) {
        const int w = g->w;
        int32_t x0[OPM];
        // ---- my share of the context: causal neighbours (latent.py:148-153) ...
#pragma unroll
        for (int o = 0; o < OPM; o++) {
            const int i = m * OPM + o;
            int v = 0;
            if (i < NCTX) {
                const int yy = y + c_ctx_dy[i], xx = x + c_ctx_dx[i];
                if (yy >= 0 && xx >= 0 && xx < w)
                    v = lds_s8(rows + ((((uint32_t)yy & row_mask) << 6) | ((uint32_t)xx & (CCD_ROW_COLS - 1))));
            }
            x0[o] = v;
        }
        // ---- ... and IFCE features (component/coolchic.py:105-146) from the prefetched inputs
        if constexpr (CF > 0) {
            const int n_in = g->ifce_in;
            if (n_in > 0 && (m + 1) * OPM > NCTX) {
                const int32_t *W = reinterpret_cast<const int32_t *>(ifce_blob);
                const long long *B =
                    reinterpret_cast<const long long *>(ifce_blob + (((size_t)n_in * CFP * 4 + 7) & ~(size_t)7));
                long long acc[OPM];
#pragma unroll
                for (int o = 0; o < OPM; o++) {
                    const int f = m * OPM + o - NCTX;
                    acc[o] = (f >= 0 && f < CF) ? B[f] : 0;
                }
#pragma unroll
                for (int c = 0; c < CCD_IFCE_FAST_MAX; c++) {
                    if (c < n_in) {
                        const int xi = ifv[c] << 16;
#pragma unroll
                        for (int o = 0; o < OPM; o++) {
                            const int f = m * OPM + o - NCTX;
                            if (f >= 0 && f < CF) acc[o] += (long long)W[c * CFP + f] * xi;
                        }
                    }
                }
#pragma unroll
                for (int o = 0; o < OPM; o++) {
                    const int f = m * OPM + o - NCTX;
                    if (f >= 0 && f < CF) {
                        // F.interpolate(ctx.to(torch.float)).to(int64): fp32 round trip (coolchic.py:142-144)
                        x0[o] = (int32_t)__float2ll_rz(__ll2float_rn(acc[o] >> 24));
                    }
                }
            }
        }
        // ---- MLP
        const int32_t *Wh = reinterpret_cast<const int32_t *>(arm_blob);
        const int32_t *Wl = Wh + (size_t)n_hidden * DIM * 4 * OPMP;
        const int32_t *Ws = Wl + DIMP * 2;
        const size_t wbytes = ((size_t)(n_hidden * DIM * 4 * OPMP + DIMP * 4) * 4 + 7) & ~(size_t)7;
        const long long *Bh = reinterpret_cast<const long long *>(arm_blob + wbytes);
        const long long *Bl = Bh + (size_t)n_hidden * DIMP;
        int32_t xo[OPM];
#pragma unroll
        for (int o = 0; o < OPM; o++) {
            x0[o] <<= 16;
            xo[o] = x0[o];
        }
        for (int l = 0; l < n_hidden; l++) {
            long long acc[OPM];
            const long long *B = Bh + (size_t)l * DIMP + m * OPM;
#pragma unroll
            for (int o = 0; o < OPM; o++) acc[o] = B[o];
            const int32_t *W = Wh + ((size_t)l * DIM * 4 + m) * OPMP;
#pragma unroll
            for (int i = 0; i < DIM; i++) {
                const int xi = __shfl_sync(0xffffffffu, xo[i % OPM], i / OPM, 4);
                int32_t wv[8];
                ld_w(W + (size_t)i * 4 * OPMP, wv);
#pragma unroll
                for (int o = 0; o < OPM; o++) acc[o] += (long long)wv[o] * xi;
            }
#pragma unroll
            for (int o = 0; o < OPM; o++) {
                long long a = acc[o];
                a = a < 0 ? 0 : a;
                xo[o] = (int32_t)(a >> 16);
            }
        }
        // last layer (on the hidden state) + stabiliser (on the input): partial sums over my inputs
        long long t0 = 0, t1 = 0;
#pragma unroll
        for (int o = 0; o < OPM; o++) {
            const int i = m * OPM + o;
            const int2 wl = *reinterpret_cast<const int2 *>(Wl + 2 * i);
            const int2 ws = *reinterpret_cast<const int2 *>(Ws + 2 * i);
            t0 += (long long)wl.x * xo[o] + (long long)ws.x * x0[o];
            t1 += (long long)wl.y * xo[o] + (long long)ws.y * x0[o];
        }
#pragma unroll
        for (int d = 1; d < 4; d <<= 1) {
            t0 += (long long)shfl_xor_u64((uint64_t)t0, d);
            t1 += (long long)shfl_xor_u64((uint64_t)t1, d);
        }
        o0 = (t0 + Bl[0] + Bl[2]) >> 24;
        o1 = (t1 + Bl[1] + Bl[3]) >> 24;
    }
};

// GENERIC: everything int64, runtime sizes, arrays in local memory.  Always correct, slow.
struct GenericArm {
    static __device__ void ifce(const EntGrid *g, const unsigned char *blob, const int8_t *lat, int cf,
                                int yy, int xx, long long *xf) {
        const int n_in = g->ifce_in;
        if (n_in == 0) {
            for (int f = 0; f < cf; f++) xf[f] = 0;
            return;
        }
        const long long *W = reinterpret_cast<const long long *>(blob);
        const long long *B = W + (size_t)n_in * cf;
        for (int f = 0; f < cf; f++) xf[f] = B[f];
        for (int c = 0; c < n_in; c++) {
            int sh = g->ch_sh[c];
            long long v = 0;
            if (sh >= 0) v = lat[g->ch_off[c] + (long long)(yy >> sh) * g->ch_w[c] + (xx >> sh)];
            long long xi = v << 16;
            for (int f = 0; f < cf; f++) xf[f] += W[(size_t)c * cf + f] * xi;
        }
        for (int f = 0; f < cf; f++) xf[f] = __float2ll_rz(__ll2float_rn(xf[f] >> 24));
    }
    static __device__ void arm(const unsigned char *blob, int dim, int n_hidden, long long *x, long long &o0,
                               long long &o1) {
        const long long *Wh = reinterpret_cast<const long long *>(blob);
        const long long *Wl = Wh + (size_t)n_hidden * dim * dim;
        const long long *Ws = Wl + (size_t)dim * 2;
        const long long *Bh = Ws + (size_t)dim * 2;
        const long long *Bl = Bh + (size_t)n_hidden * dim;
        const long long *Bs = Bl + 2;
        long long y[CCD_MAX_DIM];
        for (int i = 0; i < dim; i++) x[i] <<= 16;
        long long s0 = Bs[0], s1 = Bs[1];
        for (int i = 0; i < dim; i++) {
            s0 += Ws[2 * i] * x[i];
            s1 += Ws[2 * i + 1] * x[i];
        }
        for (int l = 0; l < n_hidden; l++) {
            const long long *W = Wh + (size_t)l * dim * dim;
            for (int o = 0; o < dim; o++) y[o] = Bh[(size_t)l * dim + o];
            for (int i = 0; i < dim; i++) {
                long long xi = x[i];
                for (int o = 0; o < dim; o++) y[o] += W[(size_t)i * dim + o] * xi;
            }
            for (int o = 0; o < dim; o++) {
                long long a = y[o] < 0 ? 0 : y[o];
                x[o] = a >> 16;
            }
        }
        long long a0 = Bl[0], a1 = Bl[1];
        for (int i = 0; i < dim; i++) {
            a0 += Wl[2 * i] * x[i];
            a1 += Wl[2 * i + 1] * x[i];
        }
        o0 = (a0 + s0) >> 24;
        o1 = (a1 + s1) >> 24;
    }
};

// cumulative of symbol s from its table entry: leak term + clamps (SURVEY Appendix C.1)
__device__ __forceinline__ uint32_t fix_left(uint32_t nl, int s) {
    uint32_t l = nl + (uint32_t)(s - kSymMin);
    l = (s <= kSymMin) ? 0u : l;
    l = (s > kSymMax) ? (1u << 24) : l;
    return l;
}

__device__ __noinline__ uint2 exact_bounds(int sym, int mu_idx, int sc_idx, const float *scale_tab) {
    const double mu = (double)(mu_idx - 16384) * (1.0 / 256.0);
    const double b = (double)scale_tab[sc_idx];
    return make_uint2(laplace_left_exact(sym, mu, b), laplace_left_exact(sym + 1, mu, b));
}

}  // namespace
