// ccd_encode.cu -- data-parallel range ENcoder of known latents on sm_100a.
//
// The mode="encode" branch of the reference operator (component/coolchic.py:89-170, latent.py:142-173 with
// range_coder.encode, rangecoder.py:46-78 -> constriction RangeEncoder) when every latent is given.  Decoding is a
// serial wavefront because a symbol's context holds symbols not yet decoded; encoding is not: all contexts are known
// up front.  So the work splits in two kernels:
//
//   * k_enc_arm: ONE data-parallel pass over every symbol of every job of a launch group.  Per symbol: causal
//     context from the caller's latents, IFCE inputs from the coarser grids, the fixed-point ARM (the decoder's own
//     QuadArm / GenericArm code and blob layouts, ccd_arm.cuh), then the symbol's interval (left(s), left(s + 1))
//     from the cumulative table (leak term + clamps, fix_left) or, outside the 31-symbol window, from the exact f64
//     model (exact_bounds).  The interval is stored at the symbol's CODING-order position (diagonals k = x + 10 y,
//     y ascending inside a diagonal; raster when w <= 9, SURVEY Appendix A).
//   * k_enc_range: one warp per job, the range-encoder recursion of encoder_emit (SURVEY Appendix C.4) over the
//     interval array.  R is the only loop-carried dependency; interval loads (a batch of 32 ahead, one per lane),
//     the D update, carries and word stores stay off it.
#include <cuda_runtime.h>
#include <stdint.h>

#include "ccd_internal.h"
#include "ccd_arm.cuh"

namespace {

constexpr int kEncWarps = CCD_ENC_THREADS / 32;
__host__ __device__ inline size_t align16_enc(size_t v) { return (v + 15) & ~(size_t)15; }
constexpr int kStageRows = 8;  // per-warp context stage: int8 [8][CCD_ROW_COLS], the decoder's row-ring addressing

__device__ __forceinline__ void st_shared_u8(uint32_t a, int v) {
    asm volatile("st.shared.u8 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}

// Rank of pixel (y, x) in the coding order of its grid.  Wavefront: the pixels of the diagonals before k = x + 10 y,
// sum over rows y' of clamp(k - 10 y', 0, w), then the pixels of diagonal k above y.  Rows y' < a lie entirely
// before diagonal k (10 y' <= k - w); rows a .. min(h - 1, k / 10) contribute k - 10 y'.
__device__ __forceinline__ int64_t coding_rank(const EntGrid &g, int y, int x) {
    const int h = g.h, w = g.w;
    if (g.raster) return (int64_t)y * w + x;
    const int k = x + CCD_MASK_STRIDE * y;
    const int a = (k < w) ? 0 : min(h, (k - w) / CCD_MASK_STRIDE + 1);
    const int y_hi = min(h - 1, k / CCD_MASK_STRIDE);
    int64_t r = (int64_t)a * w;
    const int n = y_hi - a + 1;
    if (n > 0) r += (int64_t)n * k - (int64_t)CCD_MASK_STRIDE * (((int64_t)(a + y_hi) * n) >> 1);
    return r + (y - a);
}

// One CTA = one tile: chunks [c0, c0 + n) of one grid of one job (a chunk = CHUNK consecutive pixels of one row).
template <int NCTX, int CF, bool FAST>
__global__ void __launch_bounds__(CCD_ENC_THREADS)
    k_enc_arm(const EntStream *__restrict__ streams, const EncTile *__restrict__ tiles, const uint32_t *__restrict__ cdf,
              const float *__restrict__ scale_tab) {
    constexpr int CHUNK = FAST ? CCD_ENC_CHUNK_FAST : CCD_ENC_CHUNK_GENERIC;
    constexpr int NCOL = CHUNK + 8;  // the context reaches 4 columns left and right of the chunk
    static_assert(NCOL <= CCD_ROW_COLS, "chunk too wide for the row stage");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const EncTile T = tiles[blockIdx.x];
    const EntStream &G = streams[T.stream];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    EntGrid *g = reinterpret_cast<EntGrid *>(smem_raw);
    unsigned char *arm = smem_raw + align16_enc(sizeof(EntGrid));
    unsigned char *ifce = arm + align16_enc((size_t)G.arm_blob_bytes);
    unsigned char *stage = ifce + align16_enc((size_t)G.ifce_blob_max);
    const uint32_t rows = (uint32_t)__cvta_generic_to_shared(stage) + (uint32_t)warp * (kStageRows * CCD_ROW_COLS);
    {
        const EntGrid &Gg = G.grid[T.grid];
        const uint32_t *src = reinterpret_cast<const uint32_t *>(&Gg);
        for (int i = tid; i < (int)(sizeof(EntGrid) / 4); i += CCD_ENC_THREADS) reinterpret_cast<uint32_t *>(g)[i] = src[i];
        for (int i = tid * 4; i < G.arm_blob_bytes; i += CCD_ENC_THREADS * 4)
            *reinterpret_cast<uint32_t *>(arm + i) = *reinterpret_cast<const uint32_t *>(G.blob + i);
        for (int i = tid * 4; i < Gg.ifce_blob_bytes; i += CCD_ENC_THREADS * 4)
            *reinterpret_cast<uint32_t *>(ifce + i) = *reinterpret_cast<const uint32_t *>(G.blob + Gg.ifce_blob_off + i);
    }
    __syncthreads();

    const int8_t *__restrict__ lat = G.latents;
    // mode 3: the interval array takes the place of the compressed words (EntStream.words)
    uint2 *__restrict__ iv_out = reinterpret_cast<uint2 *>(const_cast<uint32_t *>(G.words));
    const int w = g->w;
    const int64_t lat_off = g->lat_off;
    const int cpr = (w + CHUNK - 1) / CHUNK;
    const int member = FAST ? (lane & 3) : 0;
    const int i = FAST ? (lane >> 2) : lane;
    uint32_t slow = 0;
    bool bad = false;
    for (int c = T.chunk0 + warp; c < T.chunk0 + T.n_chunks; c += kEncWarps) {
        const int y = c / cpr;
        const int x0 = (c - y * cpr) * CHUNK;
        // stage rows y-4 .. y, columns x0-4 .. x0+CHUNK+3 of this grid (only the causal ones are read)
        __syncwarp();
        for (int t = lane; t < 5 * NCOL; t += 32) {
            const int dy = t / NCOL, dx = t - dy * NCOL;
            const int yy = y - 4 + dy, xx = x0 - 4 + dx;
            if (yy >= 0 && xx >= 0 && xx < w)
                st_shared_u8(rows + ((((uint32_t)yy & (kStageRows - 1)) << 6) | ((uint32_t)xx & (CCD_ROW_COLS - 1))),
                             lat[lat_off + (int64_t)yy * w + xx]);
        }
        __syncwarp();
        const int x = x0 + i;
        const bool valid = x < w;
        long long o0 = 0, o1 = 0;
        if constexpr (FAST) {
            // all 32 lanes take part (quad shuffles); out-of-range symbols compute on clamped coordinates
            const int xc = valid ? x : x0;
            int ifv[CCD_IFCE_FAST_MAX];
            QuadArm<NCTX, CF>::ifce_prefetch(g, lat, y, xc, member, ifv);
            QuadArm<NCTX, CF>::run(g, arm, ifce, ifv, rows, kStageRows - 1, G.n_hidden, y, xc, member, o0, o1);
        } else {
            if (valid) {
                const int n_ctx = G.n_ctx, cf = G.cf;
                long long xin[CCD_MAX_DIM];
                for (int t = 0; t < n_ctx; t++) {
                    const int yy = y + c_ctx_dy[t], xx = x + c_ctx_dx[t];
                    int v = 0;
                    if (yy >= 0 && xx >= 0 && xx < w)
                        v = lds_s8(rows + ((((uint32_t)yy & (kStageRows - 1)) << 6) | ((uint32_t)xx & (CCD_ROW_COLS - 1))));
                    xin[t] = v;
                }
                if (cf > 0) GenericArm::ifce(g, ifce, lat, cf, y >> 1, x >> 1, xin + n_ctx);
                GenericArm::arm(arm, n_ctx + cf, G.n_hidden, xin, o0, o1);
            }
        }
        if (valid && member == 0) {
            // latent.py:165 + rangecoder.py:89-91, exactly as the decoder's producer
            long long im = o0 + 16384, is = o1 + 1280;
            im = im < 0 ? 0 : (im > 32767 ? 32767 : im);
            is = is < 0 ? 0 : (is > 2560 ? 2560 : is);
            const int mu_idx = (int)im, sc_idx = (int)is;
            const int mu_int = ((mu_idx + 128) >> 8) - 64;
            const int fr = (mu_idx + 128) & 255;
            const int s_lo = mu_int - CCD_WIN_HALF;
            const int sym = lat[lat_off + (int64_t)y * w + x];
            uint2 iv;
            if (sym < kSymMin || sym > kSymMax) {  // AC_MAX_VAL (constants.py:9-11): an error, never clamped
                bad = true;
                iv = make_uint2(0u, 1u << 24);
            } else if (sym >= s_lo && sym < s_lo + 31) {
                const uint32_t *row = cdf + (((size_t)sc_idx << 8 | (size_t)fr) << 5) + (sym - s_lo);
                iv = make_uint2(fix_left(__ldg(row), sym), fix_left(__ldg(row + 1), sym + 1));
            } else {
                slow++;
                iv = exact_bounds(sym, mu_idx, sc_idx, scale_tab);
            }
            iv_out[lat_off + coding_rank(*g, y, x)] = iv;
        }
    }
    const uint32_t n_slow = __reduce_add_sync(0xffffffffu, slow);
    const bool any_bad = __any_sync(0xffffffffu, bad);
    if (lane == 0) {
        if (n_slow) atomicAdd(&G.status[2], (int)n_slow);
        if (any_bad) atomicExch(&G.status[0], CCD_ERR_ARG);
    }
}

// Carry into the words already stored below index i (SURVEY Appendix C.4); the newest word is still in a register.
__device__ __noinline__ void carry_into_stored(uint32_t *out, int64_t cap, int64_t i) {
    while (i > 0) {
        i--;
        if (i < cap) {
            const uint32_t v = out[i] + 1u;
            out[i] = v;
            if (v != 0u) break;
        }
    }
}

// One warp per job.  All lanes run the recursion (the interval of symbol j is one shuffle away); lane 0 stores.  The
// newest emitted word (index nout - 1) stays in `pend` until the next one is emitted, so a carry is a register add.
// (A branch-free step -- carry and renormalisation as selects, predicated store -- measured slower: DESIGN.md 4.4.)
__global__ void __launch_bounds__(32) k_enc_range(const EntStream *__restrict__ streams) {
    const EntStream &G = streams[blockIdx.x];
    const int lane = threadIdx.x;
    const uint2 *__restrict__ iv = reinterpret_cast<const uint2 *>(G.words);
    const int64_t n = G.n_symbols;
    uint32_t *__restrict__ out = G.out_words;
    const int64_t cap = G.out_cap;
    uint64_t D = 0, R = ~0ull;
    int64_t nout = 0;
    uint32_t pend = 0;
    auto carry = [&]() {
        if (nout == 0) return;
        pend += 1u;
        if (pend == 0u && lane == 0) carry_into_stored(out, cap, nout - 1);
    };
    auto emit = [&](uint32_t word) {
        if (lane == 0 && nout >= 1 && nout - 1 < cap) out[nout - 1] = pend;
        pend = word;
        nout++;
    };
    auto step = [&](uint32_t L0, uint32_t L1) {
        const uint64_t scale = R >> 24;
        const uint64_t nl = D + scale * L0;
        if (nl < D) carry();
        D = nl;
        R = scale * (uint64_t)(L1 - L0);
        if ((uint32_t)(R >> 32) == 0u) {
            emit((uint32_t)(D >> 32));
            D <<= 32;
            R <<= 32;
        }
    };
    uint2 cur = (lane < n) ? __ldg(iv + lane) : make_uint2(0u, 0u);
    int64_t base = 0;
    for (; base + 32 <= n; base += 32) {
        const uint2 nxt = (base + 32 + lane < n) ? __ldg(iv + base + 32 + lane) : make_uint2(0u, 0u);
#pragma unroll 8
        for (int j = 0; j < 32; j++) step(__shfl_sync(0xffffffffu, cur.x, j), __shfl_sync(0xffffffffu, cur.y, j));
        cur = nxt;
    }
    for (int j = 0; base + j < n; j++) step(__shfl_sync(0xffffffffu, cur.x, j), __shfl_sync(0xffffffffu, cur.y, j));
    if (n > 0) {
        // seal (SURVEY Appendix C.4): point = lower + 2^32 - 1, emit its high word
        const uint64_t point = D + ((1ull << 32) - 1);
        if (point < D) carry();
        emit((uint32_t)(point >> 32));
    }
    if (lane == 0) {
        if (nout >= 1 && nout - 1 < cap) out[nout - 1] = pend;
        G.status[3] = (int32_t)nout;
    }
}

template <int NCTX, int CF, bool FAST>
int enc_arm_t(const EntStream *d_streams, const EncTile *d_tiles, int n_tiles, size_t smem, const uint32_t *cdf,
              const float *scale, cudaStream_t st) {
    auto kern = k_enc_arm<NCTX, CF, FAST>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    kern<<<n_tiles, CCD_ENC_THREADS, smem, st>>>(d_streams, d_tiles, cdf, scale);
    g_ccd_launches++;
    return (int)cudaGetLastError();
}

}  // namespace

size_t ccd_encode_smem_bytes(int arm_blob_bytes, int ifce_blob_max) {
    return align16_enc(sizeof(EntGrid)) + align16_enc((size_t)arm_blob_bytes) + align16_enc((size_t)ifce_blob_max) +
           (size_t)kEncWarps * kStageRows * CCD_ROW_COLS;
}

int ccd_enc_arm_launch(const EntStream *d_streams, const EncTile *d_tiles, int n_tiles, const EntLaunchCfg &cfg,
                       const uint32_t *d_cdf, const float *d_scale, cudaStream_t st) {
    if (n_tiles <= 0) return 0;
    const size_t s = cfg.smem_bytes;
    if (cfg.fast) {
        if (cfg.n_ctx == 6 && cfg.cf == 2) return enc_arm_t<6, 2, true>(d_streams, d_tiles, n_tiles, s, d_cdf, d_scale, st);
        if (cfg.n_ctx == 10 && cfg.cf == 2) return enc_arm_t<10, 2, true>(d_streams, d_tiles, n_tiles, s, d_cdf, d_scale, st);
        if (cfg.n_ctx == 10 && cfg.cf == 4) return enc_arm_t<10, 4, true>(d_streams, d_tiles, n_tiles, s, d_cdf, d_scale, st);
        if (cfg.n_ctx == 14 && cfg.cf == 6) return enc_arm_t<14, 6, true>(d_streams, d_tiles, n_tiles, s, d_cdf, d_scale, st);
        if (cfg.n_ctx == 20 && cfg.cf == 6) return enc_arm_t<20, 6, true>(d_streams, d_tiles, n_tiles, s, d_cdf, d_scale, st);
    }
    return enc_arm_t<0, 0, false>(d_streams, d_tiles, n_tiles, s, d_cdf, d_scale, st);
}

int ccd_enc_range_launch(const EntStream *d_streams, int n_streams, cudaStream_t st) {
    if (n_streams <= 0) return 0;
    k_enc_range<<<n_streams, 32, 0, st>>>(d_streams);
    g_ccd_launches++;
    return (int)cudaGetLastError();
}
