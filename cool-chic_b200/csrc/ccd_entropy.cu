// ccd_entropy.cu -- entropy stage of the Cool-chic decoder on sm_100a.
//
// Replaces, for one Cool-chic stream, the reference's hot loops A/B/C
//   component/coolchic.py:89-166   per-grid loop, IFCE context (coarse -> fine)
//   latent.py:142-173              wavefront loop: gather context, ARM, range decode, scatter
//   armint.py:180-203              int64 fixed-point ARM MLP
//   rangecoder.py:87-94            (mu, scale) table lookup + constriction RangeDecoder.decode
// with ONE persistent CTA per stream (a stream is a strict serial chain, SURVEY F8):
//
//   * producer warps, a QUAD of lanes per symbol (8 symbols per warp): wait until the
//     symbol's left neighbour is decoded (shared-memory progress counter), gather the causal
//     neighbourhood from a shared-memory row ring, evaluate IFCE + ARM in integer arithmetic
//     (IMAD.WIDE, int32 operands proven safe by the host, int64 accumulators, activations
//     exchanged with quad shuffles), then fetch the symbol's 32-entry cumulative window from
//     the device-resident quantised-Laplace table and publish it in a shared-memory ring.
//   * 1 range-coder warp: each lane owns one candidate symbol of the window; the lane whose
//     [scale*left, scale*left') interval contains (point - lower) wins (no division), the
//     new state is broadcast with shuffles.  ~1 ballot + 4 shuffles per symbol.
//
// The same kernel runs in "encode" / "sample" mode (range ENcoder, rangecoder.py:46-78) to
// fabricate self-consistent synthetic streams on the device.  (The data-parallel encoder of known
// latents is ccd_encode.cu; the ARM / Laplace code both use is in ccd_arm.cuh.)
#include <cuda_runtime.h>
#include <stdint.h>

#include "ccd_internal.h"
#include "ccd_arm.cuh"

#ifdef CCD_PROFILE
#define PROF_T(var) long long var = clock64()
#define PROF_ADD(acc, t0) acc += clock64() - (t0)
#else
#define PROF_T(var)
#define PROF_ADD(acc, t0)
#endif

namespace {

struct ProfCounters {
    long long wait = 0, arm = 0, win = 0, total = 0;
    long long seg[6] = {0, 0, 0, 0, 0, 0};  // coder: per-segment cycles of the decode step
};

// Table: NL[sc][f][t] = trunc(FW*cdf((t - CCD_WIN_HALF - 0.5) - (f-128)/256)), sc < 2561, f < 256, t < 32.
__global__ void k_cdf_table(uint32_t *__restrict__ tab, const float *__restrict__ scale) {
    size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t total = (size_t)CCD_N_SCALE * 256 * CCD_WIN;
    if (idx >= total) return;
    int t = (int)(idx & 31);
    int f = (int)((idx >> 5) & 255);
    int sc = (int)(idx >> 13);
    double b = (double)scale[sc];
    double d = ((double)t - ((double)CCD_WIN_HALF + 0.5)) - (double)(f - 128) * (1.0 / 256.0);
    tab[idx] = laplace_nonleaky(d, b);
}

__global__ void k_laplace_domain(const float *__restrict__ scale, int sc_lo, int sc_hi, uint32_t *lo,
                                 uint32_t *hi) {
    const int ND = 32641;
    size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t total = (size_t)(sc_hi - sc_lo) * ND;
    if (idx >= total) return;
    int n = (int)(idx % ND);
    int sc = sc_lo + (int)(idx / ND);
    double b = (double)scale[sc];
    double d = (double)n * (1.0 / 256.0);
    lo[idx] = laplace_nonleaky(-d, b);
    hi[idx] = (n == 0) ? laplace_nonleaky(0.0, b) : laplace_nonleaky(d, b);
}

__device__ __forceinline__ uint64_t splitmix64(uint64_t &s) {
    uint64_t z = (s += 0x9E3779B97F4A7C15ull);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

// per-stream scalars, copied to registers once (EntStream lives in global memory)
struct SLoc {
    int ring, rows, n_hidden, n_ctx, cf, mode;
    int8_t *latents;
    const uint32_t *words;
    int64_t n_words;
    uint32_t *out_words;
    int64_t out_cap;
    int32_t *status;
    int64_t n_symbols;
};

// Shared-memory accessors by 32-bit shared-space address (explicit LDS/STS, never generic).
__device__ __forceinline__ void sts_v4(uint32_t a, uint4 v) {
    asm volatile("st.volatile.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w)
                 : "memory");
}
__device__ __forceinline__ void sts_v2(uint32_t a, uint2 v) {
    asm volatile("st.volatile.shared.v2.u32 [%0], {%1, %2};" ::"r"(a), "r"(v.x), "r"(v.y) : "memory");
}
__device__ __forceinline__ uint4 lds_v4(uint32_t a) {
    uint4 v;
    asm volatile("ld.volatile.shared.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
                 : "r"(a)
                 : "memory");
    return v;
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) {
    uint32_t v;
    asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ void sts_u32(uint32_t a, uint32_t v) {
    asm volatile("st.volatile.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}
// Flag words of the hand-offs (progress, ready, done, the meta tags) are written with release and read with acquire
// semantics at CTA scope: what a flag announces (window / hot entries, result words, decoded symbols) is visible to
// the thread that saw the flag.  One exception, measured (tools/ab.sh): the coder's `done` store stays a plain volatile
// store -- a release there is a fence in front of it on the serial chain's warp; it is ordered after the coder's own
// result-word stores because shared-memory stores of one warp are performed in program order, and the helper reads
// `done` with acquire.  (-DCCD_RELEASE_DONE makes it a release store.)
__device__ __forceinline__ uint32_t lds_acq_u32(uint32_t a) {
    uint32_t v;
#ifdef CCD_RELAXED_FLAGS
    asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
#else
    asm volatile("ld.acquire.cta.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
#endif
    return v;
}
__device__ __forceinline__ void sts_rel_u32(uint32_t a, uint32_t v) {
#ifdef CCD_RELAXED_FLAGS
    asm volatile("st.volatile.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
#else
    asm volatile("st.release.cta.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
#endif
}
__device__ __forceinline__ void sts_done(uint32_t a, uint32_t v) {
#ifdef CCD_RELEASE_DONE
    sts_rel_u32(a, v);
#else
    asm volatile("st.volatile.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
#endif
}
__device__ __forceinline__ void sts_u8(uint32_t a, int v) {
    asm volatile("st.volatile.shared.u8 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}

// shared memory carve-up -----------------------------------------------------------------
struct SmemLayout {
    uint32_t ctrl;         // shared address: [0] progress (symbols decoded)
    EntGrid *grid;         // current grid
    unsigned char *arm;    // ARM blob
    unsigned char *ifce;   // IFCE blob of the current grid
    uint32_t meta;         // shared address: uint4 [ring]
    uint32_t win;          // shared address: u32 [ring][32]: left(s_lo + t), t = 0..31 (mode at t = 15)
    uint32_t hot;          // shared address: uint4 [ring]: left(M), left(M+1)-left(M), left(M-1), left(M+2), M = mode
    uint32_t res;          // shared address: u32 [ring]: result word of each symbol that is NOT the mode (coder -> helper)
    uint32_t rows;         // shared address: int8 [rows][64]
};

__host__ __device__ inline size_t align16(size_t v) { return (v + 15) & ~(size_t)15; }

__device__ __forceinline__ SmemLayout carve(unsigned char *base, int ring, int rows, int arm_bytes,
                                            int ifce_bytes) {
    SmemLayout L;
    uint32_t base_a = (uint32_t)__cvta_generic_to_shared(base);
    asm volatile("" : "+r"(base_a));  // opaque: keep it in a register instead of re-deriving it
    size_t p = 0;
    L.ctrl = base_a + (uint32_t)p;
    p += 64;
    L.grid = reinterpret_cast<EntGrid *>(base + p);
    p += align16(sizeof(EntGrid));
    L.arm = base + p;
    p += align16((size_t)arm_bytes);
    L.ifce = base + p;
    p += align16((size_t)ifce_bytes);
    p += 16;  // (spare line)
    L.meta = base_a + (uint32_t)p;
    p += (size_t)ring * 16;
    L.win = base_a + (uint32_t)p;
    p += (size_t)ring * CCD_WIN * 4;
    L.hot = base_a + (uint32_t)p;
    p += (size_t)(ring + CCD_HOT_MIRROR) * 16;  // entries 0..7 are mirrored after the end: +32 B never wraps
    L.res = base_a + (uint32_t)p;
    p += (size_t)(ring + 4) * 4;  // (+ CCD_RES_MIRROR slots)
    L.rows = base_a + (uint32_t)p;
    (void)rows;
    return L;
}

// ---------------------------------------------------------------------------------------
// Producer: symbols [c0, c0 + CHUNK) of diagonal k.  FAST: CHUNK = 8 (quad per symbol),
// GENERIC: CHUNK = 32 (thread per symbol).
template <int NCTX, int CF, bool FAST>
__device__ __forceinline__ void produce_chunk(const SLoc &S, const SmemLayout &sm,
                                              const uint32_t *__restrict__ cdf, int lane, int y0, int x0,
                                              int n_k, int c0, uint32_t ord_diag, uint32_t ord_prev,
                                              int y0_prev, ProfCounters &pc) {
    const EntGrid *g = sm.grid;
    const int member = FAST ? (lane & 3) : 0;
    const int i = c0 + (FAST ? (lane >> 2) : lane);
    const bool valid = i < n_k;
    const int w = g->w;
    const int y = y0 + i;
    const int x = g->raster ? x0 : x0 - CCD_MASK_STRIDE * i;
    const uint32_t ord = ord_diag + (uint32_t)i;
    const uint32_t ring_mask = (uint32_t)S.ring - 1u;
    const uint32_t row_mask = (uint32_t)S.rows - 1u;

    // ---- dependencies: left neighbour decoded (and everything older), ring slot free
    uint32_t need;
    if (g->raster) need = ord;                                      // everything before me
    else if (x > 0) need = ord_prev + (uint32_t)(y - y0_prev) + 1u; // (y, x-1) sits on diagonal k-1
    else need = ord_prev;                                            // first pixel of a row
    const uint32_t need_ring = ord + 1u - (uint32_t)S.ring;          // slot reuse: ord - ring consumed
    if ((int32_t)(need_ring - need) > 0) need = need_ring;
    int ifv[CCD_IFCE_FAST_MAX];
    if constexpr (FAST) QuadArm<NCTX, CF>::ifce_prefetch(g, S.latents, valid ? y : y0, valid ? x : x0, member, ifv);
    // needs grow with the lane: one warp-wide wait on the maximum
    int32_t rel = valid ? (int32_t)(need - ord_diag) : INT32_MIN;
    rel = __reduce_max_sync(0xffffffffu, rel);
    need = ord_diag + (uint32_t)rel;
    PROF_T(t0);
    while ((int32_t)(lds_acq_u32(sm.ctrl) - need) < 0) {
#ifdef CCD_SPIN_SLEEP
        __nanosleep(CCD_SPIN_SLEEP);
#endif
    }
    PROF_ADD(pc.wait, t0);
    PROF_T(t1);
    long long o0 = 0, o1 = 0;
    if constexpr (FAST) {
        // all 32 lanes take part (quad shuffles); out-of-range symbols compute on clamped coordinates
        const int yc = valid ? y : y0, xc = valid ? x : x0;
        QuadArm<NCTX, CF>::run(g, sm.arm, sm.ifce, ifv, sm.rows, row_mask, S.n_hidden, yc, xc, member, o0, o1);
    } else {
        if (valid) {
            const int n_ctx = S.n_ctx, cf = S.cf;
            long long xin[CCD_MAX_DIM];
            for (int t = 0; t < n_ctx; t++) {
                const int yy = y + c_ctx_dy[t], xx = x + c_ctx_dx[t];
                int v = 0;
                if (yy >= 0 && xx >= 0 && xx < w)
                    v = lds_s8(sm.rows + ((((uint32_t)yy & row_mask) << 6) | ((uint32_t)xx & (CCD_ROW_COLS - 1))));
                xin[t] = v;
            }
            if (cf > 0) GenericArm::ifce(g, sm.ifce, S.latents, cf, y >> 1, x >> 1, xin + n_ctx);
            GenericArm::arm(sm.arm, n_ctx + cf, S.n_hidden, xin, o0, o1);
        }
    }
    PROF_ADD(pc.arm, t1);
    PROF_T(t2);
    // latent.py:165 + rangecoder.py:89-91 (np.take(..., mode="clip"))
    long long im = o0 + 16384, is = o1 + 1280;
    im = im < 0 ? 0 : (im > 32767 ? 32767 : im);
    is = is < 0 ? 0 : (is > 2560 ? 2560 : is);
    const int mu_idx = (int)im, sc_idx = (int)is;
    const int mu_int = ((mu_idx + 128) >> 8) - 64;
    const int fr = (mu_idx + 128) & 255;
    const int s_lo = mu_int - CCD_WIN_HALF;
    // ---- cumulative window: table row -> leak term + clamps -> shared ring
    const uint4 *row = reinterpret_cast<const uint4 *>(cdf + (((size_t)sc_idx << 8 | (size_t)fr) << 5));
    const uint32_t slot = ord & ring_mask;
    const uint32_t wdst = sm.win + slot * (CCD_WIN * 4);
    if constexpr (FAST) {
        if (valid) {
            // member m owns entries [8m, 8m+8)
            const uint4 va = __ldg(row + 2 * member), vb = __ldg(row + 2 * member + 1);
            const int s0 = s_lo + 8 * member;
            sts_v4(wdst + 32u * member, make_uint4(fix_left(va.x, s0), fix_left(va.y, s0 + 1), fix_left(va.z, s0 + 2),
                                                   fix_left(va.w, s0 + 3)));
            const uint4 fb = make_uint4(fix_left(vb.x, s0 + 4), fix_left(vb.y, s0 + 5), fix_left(vb.z, s0 + 6),
                                        fix_left(vb.w, s0 + 7));
            sts_v4(wdst + 32u * member + 16u, fb);
            // hot entry (the coder's steady state reads nothing else): window entries 13 .. 16 =
            // left(M-1), left(M), left(M+1), left(M+2); the ring's first entries are mirrored behind its end so that
            // a group of consecutive entries is read from one base address
            static_assert(CCD_WIN_HALF == 14, "hot entry layout");
            const uint32_t hdst = sm.hot + slot * 16u;
            const bool mirror = slot < CCD_HOT_MIRROR;
            const uint32_t hmir = hdst + (uint32_t)S.ring * 16u;
            if (member == 1) {
                sts_v2(hdst, make_uint2(fb.y, fb.z));
                sts_u32(hdst + 8u, fb.w);
                if (mirror) {
                    sts_v2(hmir, make_uint2(fb.y, fb.z));
                    sts_u32(hmir + 8u, fb.w);
                }
            } else if (member == 2) {
                const uint32_t l16 = fix_left(va.x, s0);
                sts_u32(hdst + 12u, l16);
                if (mirror) sts_u32(hmir + 12u, l16);
            }
        }
        __threadfence_block();
        __syncwarp();
    } else {
        if (valid) {
            uint4 v[8];
#pragma unroll
            for (int c = 0; c < 8; c++) v[c] = __ldg(row + c);
#pragma unroll
            for (int c = 0; c < 8; c++)
                sts_v4(wdst + 16u * c, make_uint4(fix_left(v[c].x, s_lo + 4 * c), fix_left(v[c].y, s_lo + 4 * c + 1),
                                                  fix_left(v[c].z, s_lo + 4 * c + 2), fix_left(v[c].w, s_lo + 4 * c + 3)));
            {
                const uint32_t l13 = fix_left(v[3].y, s_lo + 13), l14 = fix_left(v[3].z, s_lo + 14);
                const uint32_t l15 = fix_left(v[3].w, s_lo + 15), l16 = fix_left(v[4].x, s_lo + 16);
                sts_v4(sm.hot + slot * 16u, make_uint4(l13, l14, l15, l16));
                if (slot < CCD_HOT_MIRROR) sts_v4(sm.hot + (slot + (uint32_t)S.ring) * 16u, make_uint4(l13, l14, l15, l16));
            }
            __threadfence_block();
        }
    }
    if (valid && member == 0) {
        const uint32_t out_off = (uint32_t)(g->lat_off + (long long)y * w + x);
        const uint32_t row_idx = (((uint32_t)y & row_mask) << 6) | ((uint32_t)x & (CCD_ROW_COLS - 1));
        // meta: x = output offset, y = row-ring index | (s_lo + 128) << 16, z = mu_idx | sc_idx << 16, w = tag
        const uint32_t ma = sm.meta + slot * 16u;
        sts_v2(ma, make_uint2(out_off, row_idx | ((uint32_t)(s_lo + 128) << 16)));
        sts_u32(ma + 8u, (uint32_t)mu_idx | ((uint32_t)sc_idx << 16));
        sts_rel_u32(ma + 12u, ord + 1u);  // the tag: everything this quad / thread stored for the symbol is visible before it
    }
    PROF_ADD(pc.win, t2);
#ifdef CCD_PROFILE
    pc.seg[5]++;
#endif
}

template <int NCTX, int CF, bool FAST>
__device__ __forceinline__ void producer_grid(const SLoc &S, const SmemLayout &sm, const uint32_t *__restrict__ cdf,
                                           int prank, int n_prod, int lane, uint32_t ord_grid, int &chunk_ctr,
                                           ProfCounters &pc) {
    constexpr int CHUNK = FAST ? 8 : 32;
    const EntGrid *g = sm.grid;
    const int h = g->h, w = g->w, n_diag = g->n_diag, raster = g->raster;
    uint32_t ord = ord_grid, ord_prev = ord_grid;
    int y0_prev = 0;
    for (int k = 0; k < n_diag; k++) {
        int y0, x0, n_k;
        if (raster) {
            y0 = k / w;
            x0 = k - y0 * w;
            n_k = 1;
        } else if (k < w) {
            y0 = 0;
            x0 = k;
            n_k = min(h, x0 / CCD_MASK_STRIDE + 1);
        } else {
            const int r = k - w;
            y0 = r / CCD_MASK_STRIDE + 1;
            x0 = w - CCD_MASK_STRIDE + (r - (y0 - 1) * CCD_MASK_STRIDE);
            n_k = min(h - y0, x0 / CCD_MASK_STRIDE + 1);
        }
        for (int c0 = 0; c0 < n_k; c0 += CHUNK) {
            if (chunk_ctr == prank)
                produce_chunk<NCTX, CF, FAST>(S, sm, cdf, lane, y0, x0, n_k, c0, ord, ord_prev, y0_prev, pc);
            chunk_ctr = (chunk_ctr + 1 == n_prod) ? 0 : chunk_ctr + 1;
        }
        ord_prev = ord;
        y0_prev = y0;
        ord += (uint32_t)n_k;
    }
}

// ---------------------------------------------------------------------------------------
// Range-coder warp.  State (SURVEY Appendix C.2): D = point - lower (mod 2^64), R = range.
// (lower and point only ever appear through their difference, so one u64 replaces two.)
struct Coder {          // range ENcoder state (SURVEY Appendix C.4)
    uint64_t D, R;       // D = lower, R = range
    uint64_t prng;
    int64_t nout;        // words emitted
    uint32_t slow;       // symbols outside the window
};

// Exhaustive search with the exact f64 model for a symbol outside the 31-symbol window.
// q: quantile (uniform).  Returns {l0, l1, src, sym}: per-lane cumulatives of the lane's
// candidate in the winning round, the winning lane and the symbol.  (Returned in registers:
// reference outputs would force the hot loop's variables into local memory.)
__device__ __noinline__ uint4 slow_search(uint32_t q, int mu_idx, int sc_idx, const float *scale_tab, int lane) {
    const double mu = (double)(mu_idx - 16384) * (1.0 / 256.0);
    const double b = (double)scale_tab[sc_idx];
    uint32_t ballot = 0, l0 = 0, l1 = 0;
    int s = 0;
    for (int r = 0; r < 4; r++) {
        s = kSymMin + r * 32 + lane;
        l0 = laplace_left_exact(s, mu, b);
        l1 = laplace_left_exact(s + 1, mu, b);
        ballot = __ballot_sync(0xffffffffu, l0 <= q && q < l1);
        if (ballot) break;
    }
    if (ballot == 0u) ballot = 1u;  // unreachable: left(-64) = 0 <= q < 2^24 = left(64)
    const int src = __ffs(ballot) - 1;
    const int sym = __shfl_sync(0xffffffffu, s, src);
    return make_uint4(l0, l1, (uint32_t)src, (uint32_t)sym);
}

__device__ __noinline__ void encoder_emit(const SLoc &S, Coder &c, uint32_t L0, uint32_t L1, int lane) {
    const uint64_t scale = c.R >> 24;
    const uint64_t nl = c.D + scale * L0;
    const bool carry = nl < c.D;
    c.D = nl;
    c.R = scale * (uint64_t)(L1 - L0);
    if (lane == 0 && carry) {
        int64_t i = c.nout;
        while (i > 0) {
            i--;
            if (i < S.out_cap) {
                uint32_t v = S.out_words[i] + 1u;
                S.out_words[i] = v;
                if (v != 0u) break;
            }
        }
    }
    if (c.R < (1ull << 32)) {
        if (lane == 0 && c.nout < S.out_cap) S.out_words[c.nout] = (uint32_t)(c.D >> 32);
        c.nout++;
        c.D <<= 32;
        c.R <<= 32;
    }
}

// =======================================================================================
// Range DEcoder = two warps.
//   coder  (warp 15): only the (D, R) recursion.  Its lanes enumerate SEQUENCES of the next three symbols and run
//          the exact recursion each on its own hypothesis; one shared-memory record round trip per three symbols
//          hands the matching lane's state to all of them (coder_grid_spec below; the design it replaced -- all
//          lanes executing one scalar chain, blocks of four "is it the mode?" steps -- is kept behind
//          -DCCD_CODER_BLOCKS for A/B measurements).  Measured on B200: a vote / shuffle / shared-memory round trip
//          costs this warp 27-35 cycles, a dependent ALU op 4-5, a taken branch 10-45.
//   helper (warp 14): everything that is not on that recursion, 32 symbols at a time:
//          finds how far the producers have got (contiguous valid tags -> `ready`), turns the
//          coder's result words into symbols, writes the row ring / latent array and
//          advances `progress` for the producers.
// ctrl words: [0] progress (symbols published), [1] ready (symbols whose window is in the ring)
// =======================================================================================
struct DecState {
    uint64_t D, R;        // D = point - lower (mod 2^64), R = range   (SURVEY Appendix C.2)
    uint32_t w0;          // word[wpos]: the next unread word of the stream
    uint32_t wpos;        // index of the next unread word
    uint32_t wcur, wnxt;  // lane l holds words wbase + l and wbase + 32 + l
    uint32_t wbase;
    uint32_t slow;        // symbols decoded with the exact f64 model (outside the 31-symbol window)
    uint32_t n_far;       // symbols outside {M-1, M, M+1} (instrumented build)
    uint32_t n_redo;      // fast groups decoded again one symbol at a time (instrumented build)
    int err;
};

// word i of the stream; the host pads the payload with zero words (missing words read as 0 like
// constriction does), the index is clamped so that a corrupt stream cannot run away
__device__ __forceinline__ uint32_t coder_word(const uint32_t *__restrict__ words, uint32_t wmax, uint32_t i) {
    return __ldg(words + (i < wmax ? i : wmax));
}

// The compressed words reach the coder through REGISTERS: lane l of the coder warp keeps words wbase + l and
// wbase + 32 + l; word[wpos] is one shuffle away (requested right after a symbol, consumed by the next one: no
// memory instruction, hence no scoreboard wait, on the serial chain).  wbase advances at group boundaries.
__device__ __forceinline__ uint32_t word_at(uint32_t wcur, uint32_t wnxt, uint32_t wbase, uint32_t i) {
    const uint32_t idx = i - wbase;  // 0 .. 63
    return __shfl_sync(0xffffffffu, (idx & 32u) ? wnxt : wcur, (int)idx);
}

// Result word of a symbol j that is NOT the mode (coder -> helper): [31:10] tag = (j + 1) mod 2^22, [9] valid (an
// all-zero word never matches), [8] the value is the symbol itself (else the window index t), [7:0] value.  The word of
// symbol j + i is (j << 10) + a constant: one instruction in the coder.  The ring has CCD_RES_MIRROR slots behind its
// end: the coder writes the words of consecutive symbols at consecutive addresses (no wrap test), the helper looks
// at both places for the first slots of the ring.  Mode symbols leave no trace: the helper infers them from `done`
// and the absence of a tagged word.
#define CCD_RES_MIRROR 4u
__device__ __forceinline__ uint32_t res_tag(uint32_t j) { return ((j + 1u) << 10) | 0x200u; }

// ---------------------------------------------------------------------------------------------------------------
// The scalar recursion, two tiers (cycle figures: tools/ubench/steps.cu on a B200, one warp).  TIER 2 and the far
// path serve both coders (the symbol no sequence matched / short diagonals); the blocks of TIER 1 only the block coder.
//
// TIER 1 -- "is it the mode?", branch-free, K symbols per branch.  h = (left(M-1), left(M), left(M+1), left(M+2))
//   of the most probable symbol M.  With scale = R >> 24, lo = scale * left(M), rn = scale * p(M), Dn = D - lo:
//   hi32(Dn) < hi32(rn) implies both Dn < rn (the symbol is M) and rn >= 2^32 (no renormalisation); then D = Dn,
//   R = rn and NOTHING is written.  The loop-carried chain is shift -> multiply -> R (~30 cycles / symbol for a group
//   of four, against ~86 for a step that decides three candidates with selects and ~52 for one branch per symbol).
//   The K flags are tested together; when one fails the state BEFORE the first failing symbol is taken from the
//   registers of the group (selects) and that symbol goes through tier 2.
// TIER 2 -- one symbol, any case: M-1 / M / M+1 decided with selects (a branch on fresh data costs this warp ~30
//   cycles, a select ~5), renormalisation with selects, the word from a register; anything else (`far`: ~1 % of the
//   symbols of a natural image) searches the 32-entry window lane-parallel, then the exact f64 model.
// ---------------------------------------------------------------------------------------------------------------
struct FastOut {
    uint32_t t;    // window index of the decoded symbol (CCD_WIN_HALF - 1 .. CCD_WIN_HALF + 1)
    uint32_t far;  // != 0: not one of the three candidates (everything this step produced is to be discarded)
};
__device__ __forceinline__ FastOut fast_step(uint64_t &D, uint64_t &R, uint32_t &w0, uint32_t &wpos, const uint32_t wcur,
                                             const uint32_t wnxt, const uint32_t wbase, const uint4 h) {
    const uint64_t scale = R >> 24;
    const uint64_t P0 = scale * h.x, P1 = scale * h.y, P2 = scale * h.z, P3 = scale * h.w;
    const bool c1 = D >= P1, c2 = D >= P2;
    FastOut o;
    const uint64_t nlo = c2 ? P2 : (c1 ? P1 : P0);
    const uint64_t nhi = c2 ? P3 : (c1 ? P2 : P1);
    const uint64_t Dn = D - nlo, Rn = nhi - nlo;
    // none of the three candidates <=> Dn >= Rn: D < P0 wraps Dn above any Rn (Rn <= R < 2^64 - (P0 - D) would need
    // 2^64 + D < P1), D >= P3 leaves Dn >= P3 - P2 = Rn; an empty candidate interval (left(M-1) == left(M) at the
    // lower end of the alphabet) wraps as well
    o.far = (uint32_t)(Dn >= Rn);
    const bool renorm = (uint32_t)(Rn >> 32) == 0u;
    D = renorm ? ((Dn << 32) | w0) : Dn;
    R = renorm ? (Rn << 32) : Rn;
    wpos += renorm ? 1u : 0u;
    w0 = word_at(wcur, wnxt, wbase, wpos);
    o.t = c2 ? (CCD_WIN_HALF + 1u) : (c1 ? (uint32_t)CCD_WIN_HALF : (CCD_WIN_HALF - 1u));
    return o;
}

// Exact path of one symbol that is not M-1 / M / M+1: the whole 32-entry window at once (lane per entry:
// one conflict-free LDS, one product, one vote -- the cost does not depend on how far from the mode the
// symbol is), then the exact f64 model (warp-cooperative) outside the window.  Out of line, by value.
struct FarOut {
    uint64_t lo, hi;  // scale * left(sym), scale * left(sym + 1)
    uint32_t rw;      // result word (without the tag)
    uint32_t flags;   // 2: outside the window (exact search), 4: desynchronised
};
__device__ __noinline__ FarOut coder_far(uint32_t wrow, uint32_t meta_slot, const float *__restrict__ scale_tab, int lane,
                                         uint64_t scale, uint64_t D) {
    FarOut o;
    o.flags = 0;
    const uint32_t Lt = lds_u32(wrow + 4u * (uint32_t)lane);
    const uint32_t b = __ballot_sync(0xffffffffu, scale * Lt <= D);  // lefts are non-decreasing: bits 0..t
    if (b != 0u && b != 0xffffffffu) {
        const int t = 31 - __clz((int)b);
        o.lo = scale * (uint64_t)__shfl_sync(0xffffffffu, Lt, t);
        o.hi = scale * (uint64_t)__shfl_sync(0xffffffffu, Lt, t + 1);
        o.rw = (uint32_t)t;
        return o;
    }
    // outside the window, or corrupt stream
    o.flags = 2;
    uint64_t q = D / scale;
    if (q >= (1ull << 24)) {
        o.flags |= 4;
        q = (1ull << 24) - 1;
    }
    const uint4 m = lds_v4(meta_slot);
    const uint4 r = slow_search((uint32_t)q, (int)(m.z & 0xffffu), (int)(m.z >> 16), scale_tab, lane);
    o.lo = scale * (uint64_t)__shfl_sync(0xffffffffu, r.x, (int)r.z);
    o.hi = scale * (uint64_t)__shfl_sync(0xffffffffu, r.y, (int)r.z);
    o.rw = 0x100u | (r.w & 0xffu);
    return o;
}

// TIER 2 as a function: symbol j, state and word queue by value in, by value out (registers; a reference into the
// kernel's state would put it in local memory).  A taken branch costs the coder warp ~40 cycles (instruction
// refetch: no other warp on its scheduler hides it), so the steady loop below is straight-line code whose only
// taken branches are this call / return and one back-edge per 2 K symbols.
struct T2Out {
    uint32_t d_lo, d_hi, r_lo, r_hi, w0, wpos;
    uint32_t flags;  // 2: outside the window (exact search), 4: desynchronised, 8: far (instrumented build)
};
#ifdef CCD_CODER_BLOCKS
__device__ __noinline__ T2Out coder_tier2(uint32_t res_a, uint32_t win_a, uint32_t meta_a, const float *__restrict__ scale_tab,
                                          uint32_t ring_mask, int lane, uint32_t j, const uint4 h, uint64_t D, uint64_t R,
                                          uint32_t w0, uint32_t wpos, const uint32_t wcur, const uint32_t wnxt,
                                          const uint32_t wbase) {
    const uint64_t D0 = D, R0 = R;
    const uint32_t w00 = w0, wp0 = wpos;
#ifdef CCD_T2_WINDOW
    // variant: no select tree, straight to the lane-parallel window search (compact code)
    FastOut f;
    f.far = 1u;
    f.t = 0u;
    (void)h;
#else
    const FastOut f = fast_step(D, R, w0, wpos, wcur, wnxt, wbase, h);
#endif
    uint32_t rw = f.t, flags = 0u;
    if (f.far) {
        const uint32_t slot = j & ring_mask;
        const uint64_t scale = R0 >> 24;
        const FarOut o = coder_far(win_a + slot * (CCD_WIN * 4), meta_a + slot * 16u, scale_tab, lane, scale, D0);
        uint64_t Dn = D0 - o.lo, Rn = o.hi - o.lo;
        w0 = w00;
        wpos = wp0;
        if ((Rn >> 32) == 0) {
            Dn = (Dn << 32) | w0;
            Rn <<= 32;
            wpos++;
            w0 = word_at(wcur, wnxt, wbase, wpos);
        }
        D = Dn;
        R = Rn;
        rw = o.rw;
#ifdef CCD_T2_WINDOW
        flags = o.flags;
#else
        flags = o.flags | 8u;
#endif
    }
    // shared-memory stores of one warp are performed in program order: this word is visible before the `done`
    // store that follows it
    if (rw != (uint32_t)CCD_WIN_HALF) sts_u32(res_a + (j & ring_mask) * 4u, res_tag(j) | rw);
    T2Out r;
    r.d_lo = (uint32_t)D;
    r.d_hi = (uint32_t)(D >> 32);
    r.r_lo = (uint32_t)R;
    r.r_hi = (uint32_t)(R >> 32);
    r.w0 = w0;
    r.wpos = wpos;
    r.flags = flags;
    return r;
}

__device__ __forceinline__ void coder_grid(const SLoc &S, const SmemLayout &sm, const float *__restrict__ scale_tab,
                                           int lane, uint32_t ord_begin, uint32_t ord_end, DecState &c,
                                           ProfCounters &pc) {
#ifdef CCD_ONE_BLOCK
#define CCD_STEADY_MIN 2u
#else
#define CCD_STEADY_MIN 3u
#endif
    constexpr uint32_t K = 4;  // symbols per straight-line block
    static_assert(K <= CCD_HOT_MIRROR, "block size");
    const uint32_t ring_mask = (uint32_t)S.ring - 1u;
    const uint32_t ready_a = sm.ctrl + 4u, done_a = sm.ctrl + 8u;
    const uint32_t *__restrict__ words = S.words;
    const uint32_t wmax = (uint32_t)S.n_words + 1u;  // words[n_words .. n_words + 3] are zero (host padding)
    uint64_t D = c.D, R = c.R;
    uint32_t w0 = c.w0, wpos = c.wpos, wcur = c.wcur, wnxt = c.wnxt, wbase = c.wbase;
    uint32_t j = ord_begin;
    uint32_t limit = ord_begin;  // symbols < limit have their window in the ring
    uint32_t o;
    uint4 a0, a1, a2, a3, b0, b1, b2, b3;
    auto refresh = [&]() {
        const uint32_t r = lds_acq_u32(ready_a);
        limit = ((int32_t)(r - ord_end) > 0) ? ord_end : r;
    };
    auto advance_words = [&]() {  // the lane-held words move on (at most K words are consumed between two calls)
        wcur = wnxt;
        wbase += 32u;
        wnxt = coder_word(words, wmax, wbase + 32u + (uint32_t)lane);
    };
    auto note_flags = [&](uint32_t fl) {  // rare: touches the (local-memory) decoder state
        if (fl & 2u) c.slow++;
        if (fl & 4u) c.err = CCD_ERR_DESYNC;
#ifdef CCD_PROFILE
        c.n_far++;
#endif
    };
// tier 2 through the function (two more taken branches: used off the steady path only)
#define CCD_TIER2(JJ, H)                                                                                              \
    do {                                                                                                              \
        const T2Out r_ = coder_tier2(sm.res, sm.win, sm.meta, scale_tab, ring_mask, lane, (JJ), (H), D, R, w0, wpos, wcur, \
                                     wnxt, wbase);                                                                    \
        D = ((uint64_t)r_.d_hi << 32) | r_.d_lo;                                                                      \
        R = ((uint64_t)r_.r_hi << 32) | r_.r_lo;                                                                      \
        w0 = r_.w0;                                                                                                   \
        wpos = r_.wpos;                                                                                               \
        if (__builtin_expect(r_.flags != 0u, 0)) note_flags(r_.flags);                                                \
    } while (0)
// tier 2 inline (the first failing symbol of a block): three candidates + renormalisation by selects, far by call
#define CCD_T2_INLINE(JJ, H)                                                                                          \
    {                                                                                                                 \
        const uint64_t D0_ = D, R0_ = R;                                                                              \
        const uint32_t w00_ = w0, wp0_ = wpos;                                                                        \
        const FastOut f_ = fast_step(D, R, w0, wpos, wcur, wnxt, wbase, (H));                                         \
        uint32_t rw_ = f_.t;                                                                                          \
        if (__builtin_expect(f_.far != 0u, 0)) {                                                                      \
            const uint32_t slot_ = (JJ) & ring_mask;                                                                  \
            const FarOut o_ = coder_far(sm.win + slot_ * (CCD_WIN * 4), sm.meta + slot_ * 16u, scale_tab, lane, R0_ >> 24, D0_); \
            uint64_t Dn_ = D0_ - o_.lo, Rn_ = o_.hi - o_.lo;                                                          \
            w0 = w00_;                                                                                                \
            wpos = wp0_;                                                                                              \
            if ((Rn_ >> 32) == 0) {                                                                                   \
                Dn_ = (Dn_ << 32) | w0;                                                                               \
                Rn_ <<= 32;                                                                                           \
                wpos++;                                                                                               \
                w0 = word_at(wcur, wnxt, wbase, wpos);                                                                \
            }                                                                                                         \
            D = Dn_;                                                                                                  \
            R = Rn_;                                                                                                  \
            rw_ = o_.rw;                                                                                              \
            note_flags(o_.flags | 8u);                                                                                \
        }                                                                                                             \
        if (rw_ != (uint32_t)CCD_WIN_HALF) sts_u32(sm.res + ((JJ) & ring_mask) * 4u, res_tag(JJ) | rw_);              \
    }
// K tier-1 steps on entries H0..H3; bad_i != 0 when symbol i is not "the mode, no renormalisation"
#define CCD_BLOCK(H0, H1, H2, H3)                                                                                     \
    uint64_t Ds1, Rs1, Ds2, Rs2, Ds3, Rs3, Ds4, Rs4;                                                                  \
    uint32_t bad0, bad1, bad2, bad3;                                                                                  \
    {                                                                                                                 \
        uint64_t sc_ = R >> 24;                                                                                       \
        Rs1 = sc_ * ((H0).z - (H0).y);                                                                                \
        Ds1 = D - sc_ * (H0).y;                                                                                       \
        bad0 = (uint32_t)(Ds1 >> 32) >= (uint32_t)(Rs1 >> 32);                                                        \
        sc_ = Rs1 >> 24;                                                                                              \
        Rs2 = sc_ * ((H1).z - (H1).y);                                                                                \
        Ds2 = Ds1 - sc_ * (H1).y;                                                                                     \
        bad1 = (uint32_t)(Ds2 >> 32) >= (uint32_t)(Rs2 >> 32);                                                        \
        sc_ = Rs2 >> 24;                                                                                              \
        Rs3 = sc_ * ((H2).z - (H2).y);                                                                                \
        Ds3 = Ds2 - sc_ * (H2).y;                                                                                     \
        bad2 = (uint32_t)(Ds3 >> 32) >= (uint32_t)(Rs3 >> 32);                                                        \
        sc_ = Rs3 >> 24;                                                                                              \
        Rs4 = sc_ * ((H3).z - (H3).y);                                                                                \
        Ds4 = Ds3 - sc_ * (H3).y;                                                                                     \
        bad3 = (uint32_t)(Ds4 >> 32) >= (uint32_t)(Rs4 >> 32);                                                        \
    }
// first failing symbol f of the block: state before it by selects, the hot entries of the K symbols after it are
// requested (their latency hides behind tier 2), tier 2 through the function, back to the top
#define CCD_RECOVER(H0, H1, H2, H3)                                                                                   \
    {                                                                                                                 \
        uint32_t f_ = 3u;                                                                                             \
        uint4 hf_ = (H3);                                                                                             \
        uint64_t Df_ = Ds3, Rf_ = Rs3;                                                                                \
        if (bad2) { f_ = 2u; hf_ = (H2); Df_ = Ds2; Rf_ = Rs2; }                                                      \
        if (bad1) { f_ = 1u; hf_ = (H1); Df_ = Ds1; Rf_ = Rs1; }                                                      \
        if (bad0) { f_ = 0u; hf_ = (H0); Df_ = D; Rf_ = R; }                                                          \
        D = Df_;                                                                                                      \
        R = Rf_;                                                                                                      \
        j += f_;                                                                                                      \
        o = sm.hot + ((j + 1u) & ring_mask) * 16u;                                                                    \
        a0 = lds_v4(o);                                                                                               \
        a1 = lds_v4(o + 16u);                                                                                         \
        a2 = lds_v4(o + 32u);                                                                                         \
        a3 = lds_v4(o + 48u);                                                                                         \
        CCD_T2_INLINE(j, hf_)                                                                                         \
        j++;                                                                                                          \
        sts_done(done_a, j);                                                                                           \
        PROF_COUNT_RECOVER(f_);                                                                                       \
    }
#ifdef CCD_PROFILE
#define PROF_COUNT_RECOVER(F) do { pc.seg[3] += (F); c.n_redo++; } while (0)
#else
#define PROF_COUNT_RECOVER(F)
#endif
    while (j != ord_end) {
        if ((int32_t)(limit - j) <= 0) {
            PROF_T(t0);
            do {
                refresh();
            } while ((int32_t)(limit - j) <= 0);
            PROF_ADD(pc.wait, t0);
        }
        if (wpos - wbase >= 32u) advance_words();
        if ((int32_t)(limit - j) < (int32_t)(CCD_STEADY_MIN * K) && (int32_t)(limit - j) >= (int32_t)K) {
            // fewer symbols ready than the steady loop wants (short diagonals): one block, entries requested now
            o = sm.hot + (j & ring_mask) * 16u;
            a0 = lds_v4(o);
            a1 = lds_v4(o + 16u);
            a2 = lds_v4(o + 32u);
            a3 = lds_v4(o + 48u);
            CCD_BLOCK(a0, a1, a2, a3)
            if ((bad0 | bad1 | bad2 | bad3) != 0u) {
                CCD_RECOVER(a0, a1, a2, a3)
            } else {
                D = Ds4;
                R = Rs4;
                j += K;
                sts_done(done_a, j);
#ifdef CCD_PROFILE
                pc.seg[3] += K;
#endif
            }
            continue;
        }
        if ((int32_t)(limit - j) < (int32_t)(CCD_STEADY_MIN * K)) {
            // the coder is close behind the producers (small grids, where the ARM latency bounds the stream);
            // (same bound as the steady loop's: between the two nothing would be decoded)
            const uint4 hh = lds_v4(sm.hot + (j & ring_mask) * 16u);
            {
                const uint64_t scale_ = R >> 24;
                const uint64_t lo_ = scale_ * hh.y, rn_ = scale_ * (hh.z - hh.y);
                const uint64_t dn_ = D - lo_;
                if ((uint32_t)(dn_ >> 32) < (uint32_t)(rn_ >> 32)) {  // tier 1
                    D = dn_;
                    R = rn_;
                } else {
                    CCD_TIER2(j, hh);
                }
            }
            j++;
            sts_done(done_a, j);
#ifdef CCD_PROFILE
            pc.seg[4]++;
#endif
            continue;
        }
        // ---- steady state: blocks of K symbols, branch-free (tier 1 on every symbol, flags and intermediate states
        // kept in registers), ONE branch per block; two blocks per iteration with the roles of the two sets of hot
        // entries swapped (no copies).  A far taken branch costs this warp ~40 cycles (instruction refetch; nothing
        // else runs on its scheduler), a short forward skip ~11.
        o = sm.hot + (j & ring_mask) * 16u;  // (the ring's first entries are mirrored behind its end)
        a0 = lds_v4(o);
        a1 = lds_v4(o + 16u);
        a2 = lds_v4(o + 32u);
        a3 = lds_v4(o + 48u);
        while (true) {
            // (K entries in a0..a3 valid for j; 2 K more must be ready for the two prefetches of this iteration)
            // (the two rare maintenance cases behind ONE test: every skipped block is a taken branch for this warp)
            if (((int32_t)(limit - j) < (int32_t)(CCD_STEADY_MIN * K)) | (wpos - wbase >= 32u)) {
                if (wpos - wbase >= 32u) advance_words();
                if ((int32_t)(limit - j) < (int32_t)(CCD_STEADY_MIN * K)) {
                    refresh();
                    if ((int32_t)(limit - j) < (int32_t)(CCD_STEADY_MIN * K)) break;
                }
            }
            o = sm.hot + ((j + K) & ring_mask) * 16u;
            b0 = lds_v4(o);
            b1 = lds_v4(o + 16u);
            b2 = lds_v4(o + 32u);
            b3 = lds_v4(o + 48u);
            {
                CCD_BLOCK(a0, a1, a2, a3)
                if ((bad0 | bad1 | bad2 | bad3) != 0u) {
                    CCD_RECOVER(a0, a1, a2, a3)
                    continue;
                }
                D = Ds4;
                R = Rs4;
            }
#ifdef CCD_ONE_BLOCK
            // variant: one block per iteration (the steady loop needs 2 K ready symbols instead of 3 K), entries copied
            j += K;
            sts_done(done_a, j);
            a0 = b0;
            a1 = b1;
            a2 = b2;
            a3 = b3;
            continue;
#endif
            sts_done(done_a, j + K);  // every lane stores the same word: no predicate on the hot path
            o = sm.hot + ((j + 2u * K) & ring_mask) * 16u;
            a0 = lds_v4(o);
            a1 = lds_v4(o + 16u);
            a2 = lds_v4(o + 32u);
            a3 = lds_v4(o + 48u);
            {
                CCD_BLOCK(b0, b1, b2, b3)
                if ((bad0 | bad1 | bad2 | bad3) != 0u) {
                    j += K;
                    CCD_RECOVER(b0, b1, b2, b3)
                    continue;
                }
                D = Ds4;
                R = Rs4;
            }
            j += 2u * K;
            sts_done(done_a, j);
#ifdef CCD_PROFILE
            pc.seg[3] += 2 * K;
#endif
        }
    }
#undef CCD_BLOCK
#undef CCD_RECOVER
#undef CCD_T2_INLINE
#undef CCD_TIER2
    c.D = D;
    c.R = R;
    c.w0 = w0;
    c.wpos = wpos;
    c.wcur = wcur;
    c.wnxt = wnxt;
    c.wbase = wbase;
}

#endif  // CCD_CODER_BLOCKS

// ---------------------------------------------------------------------------------------------------------------
// SPECULATIVE coder (default): the lanes of the coder warp enumerate SYMBOL SEQUENCES.
//   Lane l = c1 + 3 c2 + 9 c3 (27 lanes) assumes that the next three symbols are M1-1+c1, M2-1+c2, M3-1+c3 (Mi = the
//   most probable symbol of symbol i) and runs the exact recursion -- interval test, update, renormalisation by
//   selects -- on its OWN copy of (D, R): no branch, no vote, no shuffle inside the three steps (a vote / shuffle /
//   shared-memory round trip costs this warp 27-35 cycles, which is why one round trip per SYMBOL loses against the
//   scalar chain).  The candidate intervals of a symbol are disjoint, so at most one lane passes all three tests:
//   it writes the result words of its non-mode symbols and its state into a 24-byte record; every lane reads the
//   record back (ONE shared-memory round trip per three symbols).  A record without this round's tag means that one
//   of the three symbols is outside {M-1, M, M+1} (0.8 ... 3 % of the symbols of a natural image): the prefix
//   records tell how many symbols were decided, the next one goes through tier 2 / the window search.
//   The words a renormalisation shifts in are uniform: W0, W1, W2 = word[wpos ...], a lane that has renormalised k
//   times so far takes W_k (selects).
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void sts_v4_if(uint32_t pred, uint32_t a, uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %0, 0;\n\t@p st.volatile.shared.v4.u32 [%1], {%2, %3, %4, %5};\n\t}" ::"r"(pred),
        "r"(a), "r"(x), "r"(y), "r"(z), "r"(w)
        : "memory");
}
__device__ __forceinline__ void sts_v2_if(uint32_t pred, uint32_t a, uint32_t x, uint32_t y) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %0, 0;\n\t@p st.volatile.shared.v2.u32 [%1], {%2, %3};\n\t}" ::"r"(pred),
                 "r"(a), "r"(x), "r"(y)
                 : "memory");
}
__device__ __forceinline__ void sts_u32_if(uint32_t pred, uint32_t a, uint32_t x) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %0, 0;\n\t@p st.volatile.shared.u32 [%1], %2;\n\t}" ::"r"(pred), "r"(a),
                 "r"(x)
                 : "memory");
}
__device__ __forceinline__ uint2 lds_v2(uint32_t a) {
    uint2 v;
    asm volatile("ld.volatile.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a) : "memory");
    return v;
}

// TIER 2 of the speculative coder (one symbol, any case; out of line, rare): as coder_tier2, the words from memory.
__device__ __noinline__ T2Out coder_tier2_g(uint32_t res_a, uint32_t win_a, uint32_t meta_a, const float *__restrict__ scale_tab,
                                            uint32_t ring_mask, int lane, uint32_t j, const uint4 h, uint64_t D, uint64_t R,
                                            uint32_t w0, uint32_t wpos, const uint32_t *__restrict__ words, uint32_t wmax) {
    const uint64_t scale = R >> 24;
    const uint64_t P0 = scale * h.x, P1 = scale * h.y, P2 = scale * h.z, P3 = scale * h.w;
    const bool c1 = D >= P1, c2 = D >= P2;
    const uint64_t nlo = c2 ? P2 : (c1 ? P1 : P0);
    const uint64_t nhi = c2 ? P3 : (c1 ? P2 : P1);
    uint64_t Dn = D - nlo, Rn = nhi - nlo;  // (none of the three <=> Dn >= Rn: see fast_step)
    uint32_t rw = c2 ? (CCD_WIN_HALF + 1u) : (c1 ? (uint32_t)CCD_WIN_HALF : (CCD_WIN_HALF - 1u));
    uint32_t flags = 0u;
    if (Dn >= Rn) {
        const uint32_t slot = j & ring_mask;
        const FarOut o = coder_far(win_a + slot * (CCD_WIN * 4), meta_a + slot * 16u, scale_tab, lane, scale, D);
        Dn = D - o.lo;
        Rn = o.hi - o.lo;
        rw = o.rw;
        flags = o.flags | 8u;
    }
    if ((Rn >> 32) == 0) {
        Dn = (Dn << 32) | w0;
        Rn <<= 32;
        wpos++;
        w0 = coder_word(words, wmax, wpos);
    }
    if (rw != (uint32_t)CCD_WIN_HALF) sts_u32(res_a + (j & ring_mask) * 4u, res_tag(j) | rw);
    T2Out r;
    r.d_lo = (uint32_t)Dn;
    r.d_hi = (uint32_t)(Dn >> 32);
    r.r_lo = (uint32_t)Rn;
    r.r_hi = (uint32_t)(Rn >> 32);
    r.w0 = w0;
    r.wpos = wpos;
    r.flags = flags;
    return r;
}

// A round none of whose sequences matched: the longest decided prefix (0, 1 or 2 symbols) is taken from a lane that
// matched it -- its state after that prefix, its result words -- and the next symbol goes through tier 2.
struct PrefixOut {
    uint32_t d_lo, d_hi, r_lo, r_hi, k, n;
};
__device__ __noinline__ PrefixOut spec_prefix(uint32_t res_a, uint32_t ring_mask, int lane, uint32_t j, uint32_t ok1,
                                              uint32_t ok12, uint64_t d1, uint64_t r1, uint32_t k1, uint64_t d2,
                                              uint64_t r2, uint32_t k2) {
    PrefixOut o;
    const uint32_t b1 = __ballot_sync(0xffffffffu, ok1 != 0u), b2 = __ballot_sync(0xffffffffu, ok12 != 0u);
    o.n = b2 ? 2u : (b1 ? 1u : 0u);
    o.d_lo = o.d_hi = o.r_lo = o.r_hi = o.k = 0u;
    if (o.n) {
        const int src = __ffs((int)(b2 ? b2 : b1)) - 1;
        const uint64_t ds = b2 ? d2 : d1, rs = b2 ? r2 : r1;
        o.d_lo = __shfl_sync(0xffffffffu, (uint32_t)ds, src);
        o.d_hi = __shfl_sync(0xffffffffu, (uint32_t)(ds >> 32), src);
        o.r_lo = __shfl_sync(0xffffffffu, (uint32_t)rs, src);
        o.r_hi = __shfl_sync(0xffffffffu, (uint32_t)(rs >> 32), src);
        o.k = __shfl_sync(0xffffffffu, b2 ? k2 : k1, src);
        const uint32_t q1 = (uint32_t)src % 3u, q2 = ((uint32_t)src / 3u) % 3u;
        if (lane == 0) {
            if (q1 != 1u) sts_u32(res_a + (j & ring_mask) * 4u, res_tag(j) | (CCD_WIN_HALF - 1u + q1));
            if (o.n == 2u && q2 != 1u)
                sts_u32(res_a + ((j + 1u) & ring_mask) * 4u, res_tag(j + 1u) | (CCD_WIN_HALF - 1u + q2));
        }
        __syncwarp();
    }
    return o;
}

__device__ __forceinline__ void coder_grid_spec(const SLoc &S, const SmemLayout &sm, const float *__restrict__ scale_tab,
                                                int lane, uint32_t ord_begin, uint32_t ord_end, DecState &c,
                                                ProfCounters &pc) {
    constexpr uint32_t NS = 3;  // symbols per round
    const uint32_t ring_mask = (uint32_t)S.ring - 1u;
    const uint32_t ready_a = sm.ctrl + 4u, done_a = sm.ctrl + 8u;
    const uint32_t rec_a = sm.ctrl + 32u;  // record: D lo, D hi, R lo, R hi | words consumed, tag
    const uint32_t *__restrict__ words = S.words;
    const uint32_t wmax = (uint32_t)S.n_words + 1u;  // words[n_words .. n_words + 3] are zero (host padding)
    uint64_t D = c.D, R = c.R;
    uint32_t w0 = c.w0, wpos = c.wpos, w1 = 0u, w2 = 0u;
    uint32_t j = ord_begin, limit = ord_begin;
    // this lane's sequence: digits, the addresses of its candidates in a hot entry, its result words
    const uint32_t c1 = (uint32_t)lane % 3u, c2 = ((uint32_t)lane / 3u) % 3u, c3 = (uint32_t)lane / 9u;
    const uint32_t live = (uint32_t)lane < 27u ? 1u : 0u;
    const uint32_t hb1 = sm.hot + c1 * 4u, hb2 = sm.hot + 16u + c2 * 4u, hb3 = sm.hot + 32u + (c3 < 3u ? c3 : 2u) * 4u;
    // result word of a round, written by the matching lane at the slot of the round's FIRST symbol unless all three are
    // the mode: value = 0x40 | the lane's number (its three digits)
    const uint32_t CR = (1u << 10) | 0x200u | 0x40u | (uint32_t)lane;
    const uint32_t ner = (live != 0u && lane != 13) ? 1u : 0u;
    auto refresh = [&]() {
        const uint32_t r = lds_acq_u32(ready_a);
        limit = ((int32_t)(r - ord_end) > 0) ? ord_end : r;
    };
    // the words a round may shift in come from REGISTERS: lane l holds word[wbase + l]; the window moves (one global
    // load per lane) when fewer than 8 words are left in it -- two rounds take at most 6 and look 2 ahead
    uint32_t wcur = c.wcur, wbase = c.wbase;
    auto move_window = [&]() {
        wbase = wpos;
        wcur = coder_word(words, wmax, wbase + (uint32_t)lane);
    };
    auto load_words = [&]() {
        const uint32_t t = wpos - wbase;
        w0 = __shfl_sync(0xffffffffu, wcur, (int)t);
        w1 = __shfl_sync(0xffffffffu, wcur, (int)(t + 1u));
        w2 = __shfl_sync(0xffffffffu, wcur, (int)(t + 2u));
    };
    auto note_flags = [&](uint32_t fl) {
        if (fl & 2u) c.slow++;
        if (fl & 4u) c.err = CCD_ERR_DESYNC;
#ifdef CCD_PROFILE
        c.n_far++;
#endif
    };
    if (lane == 0) sts_v2(rec_a + 16u, make_uint2(0u, 0xffffffffu));
    __syncwarp();
// one step of this lane's hypothesis: [LA, LB) = its candidate's interval, WK = the word a renormalisation shifts in
// given the renormalisations of the lane so far
#define CCD_SSTEP(LA, LB, WK)                                                                                         \
    {                                                                                                                 \
        const uint32_t sl_ = __funnelshift_r(rl, rh, 24), sh_ = rh >> 24; /* scale = R >> 24 (40 bits) */             \
        const uint32_t p_ = (LB) - (LA);                                                                              \
        const uint64_t t_ = (uint64_t)sl_ * p_, u_ = (uint64_t)sl_ * (LA);                                            \
        const uint32_t nl_ = (uint32_t)t_, nh_ = (uint32_t)(t_ >> 32) + sh_ * p_;           /* scale * prob */       \
        const uint64_t lo_ = ((uint64_t)((uint32_t)(u_ >> 32) + sh_ * (LA)) << 32) | (uint32_t)u_; /* scale * left */ \
        const uint64_t dn_ = (((uint64_t)dh << 32) | dl) - lo_;                                                       \
        ok &= (dn_ < (((uint64_t)nh_ << 32) | nl_)) ? 1u : 0u;                                                        \
        const bool small_ = nh_ == 0u;                                                                                \
        dh = small_ ? (uint32_t)dn_ : (uint32_t)(dn_ >> 32);                                                          \
        dl = small_ ? (WK) : (uint32_t)dn_;                                                                           \
        rh = small_ ? nl_ : nh_;                                                                                      \
        rl = small_ ? 0u : nl_;                                                                                       \
        k += small_ ? 1u : 0u;                                                                                        \
    }
// entries of the round that starts at symbol JJ, into set X
#define CCD_SLOAD(X, JJ)                                                                                              \
    {                                                                                                                 \
        const uint32_t so_ = ((JJ) & ring_mask) << 4; /* (the ring's first entries are mirrored behind its end) */     \
        X##a1 = lds_u32(hb1 + so_), X##b1 = lds_u32(hb1 + so_ + 4u);                                                  \
        X##a2 = lds_u32(hb2 + so_), X##b2 = lds_u32(hb2 + so_ + 4u);                                                  \
        X##a3 = lds_u32(hb3 + so_), X##b3 = lds_u32(hb3 + so_ + 4u);                                                  \
    }
// one round on set X; failed != 0 afterwards when no sequence matched (state advanced over the decided prefix)
// (shared-memory accesses of one warp are performed in program order: the record is read back without a barrier)
#ifdef CCD_SPEC_SYNCWARP
#define CCD_SPEC_SYNC() __syncwarp()
#else
#define CCD_SPEC_SYNC()
#endif
#define CCD_RSTEPS(X)                                                                                                 \
        uint32_t dl = (uint32_t)D, dh = (uint32_t)(D >> 32), rl = (uint32_t)R, rh = (uint32_t)(R >> 32);              \
        uint32_t ok = live, k = 0u;                                                                                   \
        CCD_SSTEP(X##a1, X##b1, w0)                                                                                   \
        const uint32_t dl1_ = dl, dh1_ = dh, rl1_ = rl, rh1_ = rh, k1_ = k, ok1_ = ok;                                \
        const uint32_t wk2_ = k ? w1 : w0;                                                                            \
        CCD_SSTEP(X##a2, X##b2, wk2_)                                                                                 \
        const uint32_t dl2_ = dl, dh2_ = dh, rl2_ = rl, rh2_ = rh, k2_ = k, ok12_ = ok;                               \
        const uint32_t wk3_ = (k & 2u) ? w2 : ((k & 1u) ? w1 : w0);                                                   \
        CCD_SSTEP(X##a3, X##b3, wk3_)                                                                                 \
        const uint32_t tag_ = j + NS;                                                                                 \
        /* the matching lane: the result word of the round, then the record (program order) */                       \
        sts_u32_if(ok & ner, sm.res + ((j & ring_mask) << 2), (j << 10) + CR);                                        \
        sts_v4_if(ok, rec_a, dl, dh, rl, rh);                                                                         \
        sts_v2_if(ok, rec_a + 16u, k, tag_);                                                                          \
        CCD_SPEC_SYNC();                                                                                              \
        const uint4 rv_ = lds_v4(rec_a);                                                                              \
        const uint2 rt_ = lds_v2(rec_a + 16u);
// (the three macros share the names the steps define)
#define CCD_MATCHED() (rt_.y == tag_)
#define CCD_ACCEPT()                                                                                                  \
    {                                                                                                                 \
        D = ((uint64_t)rv_.y << 32) | rv_.x;                                                                          \
        R = ((uint64_t)rv_.w << 32) | rv_.z;                                                                          \
        wpos += rt_.x;                                                                                                \
        j = tag_;                                                                                                     \
        sts_done(done_a, j);                                                                                          \
        load_words();                                                                                                 \
        PROF_COUNT_OK();                                                                                              \
    }
// no sequence matched: the decided prefix, then the symbol outside {M-1, M, M+1} through tier 2
#define CCD_FAILED()                                                                                                  \
    {                                                                                                                 \
        const PrefixOut po_ = spec_prefix(sm.res, ring_mask, lane, j, ok1_, ok12_, ((uint64_t)dh1_ << 32) | dl1_,     \
                                          ((uint64_t)rh1_ << 32) | rl1_, k1_, ((uint64_t)dh2_ << 32) | dl2_,          \
                                          ((uint64_t)rh2_ << 32) | rl2_, k2_);                                        \
        if (po_.n) {                                                                                                  \
            D = ((uint64_t)po_.d_hi << 32) | po_.d_lo;                                                                \
            R = ((uint64_t)po_.r_hi << 32) | po_.r_lo;                                                                \
            wpos += po_.k;                                                                                            \
            j += po_.n;                                                                                               \
        }                                                                                                             \
        {                                                                                                             \
            const uint4 hh_ = lds_v4(sm.hot + (j & ring_mask) * 16u);                                                 \
            const uint32_t wj_ = __shfl_sync(0xffffffffu, wcur, (int)(wpos - wbase));                                 \
            const T2Out t2_ = coder_tier2_g(sm.res, sm.win, sm.meta, scale_tab, ring_mask, lane, j, hh_, D, R, wj_, wpos, \
                                            words, wmax);                                                             \
            D = ((uint64_t)t2_.d_hi << 32) | t2_.d_lo;                                                                \
            R = ((uint64_t)t2_.r_hi << 32) | t2_.r_lo;                                                                \
            wpos = t2_.wpos;                                                                                          \
            if (t2_.flags != 0u) note_flags(t2_.flags);                                                               \
        }                                                                                                             \
        j++;                                                                                                          \
        sts_done(done_a, j);                                                                                          \
        if (wpos - wbase >= 24u) move_window();                                                                       \
        load_words();                                                                                                 \
        PROF_COUNT_FAIL(po_.n);                                                                                       \
    }
#ifdef CCD_PROFILE
#define PROF_COUNT_FAIL(N) do { pc.seg[3] += (N); c.n_redo++; } while (0)
#define PROF_COUNT_OK() do { pc.seg[3] += NS; } while (0)
#else
#define PROF_COUNT_FAIL(N)
#define PROF_COUNT_OK()
#endif
    uint32_t pa1, pb1, pa2, pb2, pa3, pb3, qa1, qb1, qa2, qb2, qa3, qb3;  // two sets of candidate intervals
    while (j != ord_end) {
        if ((int32_t)(limit - j) <= 0) {
            PROF_T(t0);
            do {
                refresh();
            } while ((int32_t)(limit - j) <= 0);
            PROF_ADD(pc.wait, t0);
        }
        if ((int32_t)(limit - j) < (int32_t)NS) {
            // one symbol: tier-1 test, tier 2 through the function (short diagonals)
            const uint4 hh = lds_v4(sm.hot + (j & ring_mask) * 16u);
            {
                const uint64_t scale_ = R >> 24;
                const uint64_t lo_ = scale_ * hh.y, rn_ = scale_ * (hh.z - hh.y);
                const uint64_t dn_ = D - lo_;
                if ((uint32_t)(dn_ >> 32) < (uint32_t)(rn_ >> 32)) {
                    D = dn_;
                    R = rn_;
                } else {
                    const T2Out r_ = coder_tier2_g(sm.res, sm.win, sm.meta, scale_tab, ring_mask, lane, j, hh, D, R, w0, wpos,
                                                   words, wmax);
                    D = ((uint64_t)r_.d_hi << 32) | r_.d_lo;
                    R = ((uint64_t)r_.r_hi << 32) | r_.r_lo;
                    w0 = r_.w0;
                    wpos = r_.wpos;
                    if (__builtin_expect(r_.flags != 0u, 0)) note_flags(r_.flags);
                }
            }
            j++;
            sts_done(done_a, j);
#ifdef CCD_PROFILE
            pc.seg[4]++;
#endif
            continue;
        }
        if (wpos - wbase >= 24u) move_window();
        load_words();
        CCD_SLOAD(p, j)
        if ((int32_t)(limit - j) < (int32_t)(3u * NS)) {
            // fewer symbols ready than the steady loop wants: one round
            CCD_RSTEPS(p)
            if (CCD_MATCHED()) CCD_ACCEPT() else CCD_FAILED()
            continue;
        }
        // ---- steady state: two rounds per iteration, the two sets of intervals swapping roles (no copies); the
        // intervals of the next round are requested before the steps of the current one.  The common path is the
        // fall-through all the way to the back-edge (a taken branch costs this warp 10 ... 40 cycles).
        while (true) {
            if (((int32_t)(limit - j) < (int32_t)(3u * NS)) | (wpos - wbase >= 24u)) {  // (two rare cases, one test)
                if (wpos - wbase >= 24u) {
                    move_window();
                    load_words();
                }
                if ((int32_t)(limit - j) < (int32_t)(3u * NS)) {
                    refresh();
                    if ((int32_t)(limit - j) < (int32_t)(3u * NS)) break;
                }
            }
            CCD_SLOAD(q, j + NS)
            {
                CCD_RSTEPS(p)
                if (__builtin_expect(CCD_MATCHED(), 1)) {
                    CCD_ACCEPT()
                    CCD_SLOAD(p, j + NS)
                    {
                        CCD_RSTEPS(q)
                        if (__builtin_expect(CCD_MATCHED(), 1)) {
                            CCD_ACCEPT()
                            continue;
                        }
                        CCD_FAILED()
                        CCD_SLOAD(p, j)
                        continue;
                    }
                }
                CCD_FAILED()
                CCD_SLOAD(p, j)
            }
        }
    }
#undef CCD_SSTEP
#undef CCD_SLOAD
#undef CCD_RSTEPS
#undef CCD_MATCHED
#undef CCD_ACCEPT
#undef CCD_FAILED
    c.D = D;
    c.R = R;
    c.w0 = w0;
    c.wpos = wpos;
    c.wcur = wcur;
    c.wbase = wbase;
}

// Helper warp: readiness scan + publication, 32 symbols per round (lane = symbol).
__device__ __forceinline__ void helper_grid(const SLoc &S, const SmemLayout &sm, int lane, uint32_t ord_begin,
                                            uint32_t ord_end, ProfCounters &pc) {
    const uint32_t ring_mask = (uint32_t)S.ring - 1u;
    uint32_t r = ord_begin, p = ord_begin;
    while (p != ord_end) {
        if (r != ord_end) {
            const uint32_t jj = r + (uint32_t)lane;
            bool ok = false;
            if ((int32_t)(ord_end - jj) > 0) ok = lds_acq_u32(sm.meta + (jj & ring_mask) * 16u + 12u) == jj + 1u;
            const uint32_t b = __ballot_sync(0xffffffffu, ok);
            const uint32_t cnt = (b == 0xffffffffu) ? 32u : (uint32_t)(__ffs(~b) - 1);
            if (cnt) {
                r += cnt;
                if (lane == 0) sts_rel_u32(sm.ctrl + 4u, r);
            }
        }
        {
            // symbols [p, done) are decoded: mode symbols left no trace, the others a tagged result word
            const uint32_t d = lds_acq_u32(sm.ctrl + 8u);
            const int32_t avail = (int32_t)(d - p);
            const uint32_t cnt = avail <= 0 ? 0u : (avail > 32 ? 32u : (uint32_t)avail);
            if ((uint32_t)lane < cnt) {
                const uint32_t jj = p + (uint32_t)lane;
                const uint32_t slot = jj & ring_mask;
                const uint32_t ra = sm.res + slot * 4u;
                const uint32_t w = lds_u32(ra);
                const uint4 m = lds_v4(sm.meta + slot * 16u);
                const int base = (int)(m.y >> 16) - 128;  // s_lo
                int sym = base + CCD_WIN_HALF;
                if ((w & 0xfffffe00u) == res_tag(jj)) {
                    const uint32_t v = w & 0x1ffu;
                    if (v & 0x100u) sym = (int)(int8_t)(v & 0xffu);                                    // the symbol itself
                    else if ((v & 0xc0u) == 0x40u) sym = base + (int)(CCD_WIN_HALF - 1u + (v & 0x3fu) % 3u);  // first of a round
                    else sym = base + (int)v;                                                          // window index
                    if ((v & 0x1c0u) != 0x40u) sts_u32(ra, 0u);  // no stale word survives a trip around the ring
                } else {
                    // second or third symbol of a round whose word sits one or two slots back?
                    const uint32_t ra1 = sm.res + ((jj - 1u) & ring_mask) * 4u, ra2 = sm.res + ((jj - 2u) & ring_mask) * 4u;
                    const uint32_t w1 = lds_u32(ra1), w2 = lds_u32(ra2);
                    if ((w1 & 0xffffffc0u) == (res_tag(jj - 1u) | 0x40u))
                        sym = base + (int)(CCD_WIN_HALF - 1u + ((w1 & 0x3fu) / 3u) % 3u);
                    else if ((w2 & 0xffffffc0u) == (res_tag(jj - 2u) | 0x40u)) {
                        sym = base + (int)(CCD_WIN_HALF - 1u + (w2 & 0x3fu) / 9u);
                        sts_u32(ra2, 0u);  // (the last reader of the round's word)
                    }
                }
                sts_u8(sm.rows + (m.y & 0xffffu), sym);
                S.latents[m.x] = (int8_t)sym;
            }
            __syncwarp();
            if (cnt) {
                p += cnt;
                if (lane == 0) sts_rel_u32(sm.ctrl, p);
            }
        }
    }
}

// ---- encode (MODE 1: the latents given in S.latents; MODE 2: draw them from the model).
// Not performance critical: used to fabricate synthetic streams.  Runs in the coder warp and
// publishes by itself (the helper warp idles).
template <int MODE>
__device__ __noinline__ void encode_grid(const SLoc &S, const SmemLayout &sm, const float *__restrict__ scale_tab,
                                         int lane, uint32_t ord_begin, uint32_t ord_end, Coder &c) {
    const uint32_t ring_mask = (uint32_t)S.ring - 1u;
    for (uint32_t j = ord_begin; j != ord_end; j++) {
        const uint32_t slot = j & ring_mask;
        while (!__all_sync(0xffffffffu, lds_acq_u32(sm.meta + slot * 16u + 12u) == j + 1u)) {
        }
        const uint4 m = lds_v4(sm.meta + slot * 16u);
        const uint32_t L0 = lds_u32(sm.win + slot * (CCD_WIN * 4) + (uint32_t)lane * 4u);
        const uint32_t L1 = __shfl_down_sync(0xffffffffu, L0, 1);  // lane 31 keeps L0: empty interval
        const int mu_idx = (int)(m.z & 0xffffu), sc_idx = (int)(m.z >> 16);
        const int s_lo = (int)(m.y >> 16) - 128;
        uint32_t l0, l1;
        int src = -1, sym;
        if constexpr (MODE == 2) {
            const uint32_t q = (uint32_t)(splitmix64(c.prng) >> 40);
            const uint32_t ballot = __ballot_sync(0xffffffffu, L0 <= q && q < L1);
            if (ballot) {
                src = __ffs(ballot) - 1;
                sym = s_lo + src;
                l0 = __shfl_sync(0xffffffffu, L0, src);
                l1 = __shfl_sync(0xffffffffu, L1, src);
            } else {
                c.slow++;
                const uint4 r = slow_search(q, mu_idx, sc_idx, scale_tab, lane);
                src = (int)r.z;
                sym = (int)r.w;
                l0 = __shfl_sync(0xffffffffu, r.x, src);
                l1 = __shfl_sync(0xffffffffu, r.y, src);
            }
        } else {
            sym = S.latents[m.x];
            if (sym >= s_lo && sym < s_lo + 31) {
                src = sym - s_lo;
                l0 = __shfl_sync(0xffffffffu, L0, src);
                l1 = __shfl_sync(0xffffffffu, L1, src);
            } else {
                c.slow++;
                const uint2 r = exact_bounds(sym, mu_idx, sc_idx, scale_tab);
                l0 = r.x;
                l1 = r.y;
            }
        }
        encoder_emit(S, c, l0, l1, lane);
        if (lane == 0) {
            sts_u8(sm.rows + (m.y & 0xffffu), sym);
            S.latents[m.x] = (int8_t)sym;
            sts_rel_u32(sm.ctrl, j + 1u);
        }
        __syncwarp();
    }
}

__device__ __forceinline__ void named_barrier(int nthreads) {
    asm volatile("bar.sync 1, %0;" ::"r"(nthreads) : "memory");
}

// ---------------------------------------------------------------------------------------
template <int NCTX, int CF, bool FAST>
__global__ void __launch_bounds__(CCD_ENT_THREADS, 1)
    k_entropy(const EntStream *__restrict__ streams, const uint32_t *__restrict__ cdf,
              const float *__restrict__ scale_tab) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const EntStream &G = streams[blockIdx.x];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // role assignment: the last warp = range coder (recursion), the one before = its helper; producer warps are those
    // enabled in prod_mask (by default the coder keeps its scheduler partition for itself: warps 3, 7, 11 idle).  The
    // CTA has 16 warps, or 8 when the call holds more streams than the GPU has SMs (two CTAs per SM then: the two coder
    // warps share the scheduler the idle warps leave to them, each issuing ~40 % of the time)
    const int nw = (int)(blockDim.x >> 5);
    const uint32_t prod_mask = G.prod_mask & ((1u << (nw - 2)) - 1u);
    const bool is_coder = (warp == nw - 1);
    const bool is_helper = (warp == nw - 2);
    const bool is_prod = !is_coder && !is_helper && ((prod_mask >> warp) & 1u);
    if (!is_coder && !is_helper && !is_prod) return;
    const int n_prod = __popc(prod_mask);
    const int prank = __popc(prod_mask & ((1u << warp) - 1u));
    const int n_active = (n_prod + 2) * 32;
    // dense index among active threads
    const int atid = is_coder ? (n_prod + 1) * 32 + lane : (is_helper ? n_prod * 32 + lane : prank * 32 + lane);

    SmemLayout sm = carve(smem_raw, G.ring, G.rows, G.arm_blob_bytes, G.ifce_blob_max);
    SLoc S;
    S.ring = G.ring;
    S.rows = G.rows;
    S.n_hidden = G.n_hidden;
    S.n_ctx = G.n_ctx;
    S.cf = G.cf;
    S.mode = G.mode;
    S.latents = G.latents;
    S.words = G.words;
    S.n_words = G.n_words;
    S.out_words = G.out_words;
    S.out_cap = G.out_cap;
    S.status = G.status;
    S.n_symbols = G.n_symbols;

    // one-time: control words, meta tags, ARM parameters
    if (atid < 16) sts_u32(sm.ctrl + 4u * atid, 0u);
    for (int i = atid; i < S.ring; i += n_active) {
        sts_v4(sm.meta + 16u * i, make_uint4(0, 0, 0, 0));
        sts_u32(sm.res + 4u * i, 0u);
    }
    if (atid < (int)CCD_RES_MIRROR) sts_u32(sm.res + 4u * (uint32_t)(S.ring + atid), 0u);
    for (int i = atid * 4; i < G.arm_blob_bytes; i += n_active * 4)
        *reinterpret_cast<uint32_t *>(sm.arm + i) = *reinterpret_cast<const uint32_t *>(G.blob + i);

    Coder cd;
    cd.slow = 0;
    cd.nout = 0;
    cd.prng = G.seed;
    cd.D = 0;
    cd.R = ~0ull;
    DecState ds;
    ds.err = 0;
    ds.slow = 0;
    ds.n_far = 0;
    ds.n_redo = 0;
    ds.wpos = 2;
    ds.w0 = ds.wcur = ds.wnxt = ds.wbase = 0;
    ds.D = 0;
    ds.R = ~0ull;
    if (is_coder && S.mode == 0) {
        const uint32_t wmax = (uint32_t)S.n_words + 1u;
        ds.wcur = coder_word(S.words, wmax, (uint32_t)lane);
        ds.wnxt = coder_word(S.words, wmax, 32u + (uint32_t)lane);
        ds.D = ((uint64_t)word_at(ds.wcur, ds.wnxt, 0u, 0u) << 32) | word_at(ds.wcur, ds.wnxt, 0u, 1u);
        ds.w0 = word_at(ds.wcur, ds.wnxt, 0u, 2u);
    }
    uint32_t ord = 0;
    int chunk_ctr = 0;
    ProfCounters pc;
    const int n_grids = G.n_grids;
    for (int gi = 0; gi < n_grids; gi++) {
        named_barrier(n_active);  // previous grid fully decoded, its latents visible CTA-wide
        {
            const uint32_t *src = reinterpret_cast<const uint32_t *>(&G.grid[gi]);
            uint32_t *dst = reinterpret_cast<uint32_t *>(sm.grid);
            for (int i = atid; i < (int)(sizeof(EntGrid) / 4); i += n_active) dst[i] = src[i];
            const EntGrid &Gg = G.grid[gi];
            for (int i = atid * 4; i < Gg.ifce_blob_bytes; i += n_active * 4)
                *reinterpret_cast<uint32_t *>(sm.ifce + i) =
                    *reinterpret_cast<const uint32_t *>(G.blob + Gg.ifce_blob_off + i);
        }
        named_barrier(n_active);
        const uint32_t n_sym = (uint32_t)sm.grid->h * (uint32_t)sm.grid->w;
        PROF_T(tg);
        if (is_coder) {
#ifdef CCD_CODER_BLOCKS
            if (S.mode == 0) coder_grid(S, sm, scale_tab, lane, ord, ord + n_sym, ds, pc);
#else
            if (S.mode == 0) coder_grid_spec(S, sm, scale_tab, lane, ord, ord + n_sym, ds, pc);
#endif
            else if (S.mode == 1) encode_grid<1>(S, sm, scale_tab, lane, ord, ord + n_sym, cd);
            else encode_grid<2>(S, sm, scale_tab, lane, ord, ord + n_sym, cd);
        } else if (is_helper) {
            if (S.mode == 0) helper_grid(S, sm, lane, ord, ord + n_sym, pc);
        } else {
            producer_grid<NCTX, CF, FAST>(S, sm, cdf, prank, n_prod, lane, ord, chunk_ctr, pc);
        }
        PROF_ADD(pc.total, tg);
        ord += n_sym;
    }
#ifdef CCD_PROFILE
    // status words of the instrumented build (kilo-cycles unless stated): [4] coder wait, [5] coder total,
    // [6..9] producers (summed over the warps): wait, ARM, window fetch + publication, total, [10] symbols outside
    // {M-1, M, M+1}, [11] fast groups decoded again, [12] symbols decoded one at a time, [13] symbols decoded in
    // fast groups, [14] chunks produced, [15] helper total
    if (lane == 0) {
        if (is_helper) {
            G.status[15] = (int)(pc.total >> 10);
        } else if (is_coder) {
            G.status[4] = (int)(pc.wait >> 10);
            G.status[5] = (int)(pc.total >> 10);
            G.status[10] = (int)ds.n_far;
            G.status[11] = (int)ds.n_redo;
            G.status[12] = (int)pc.seg[4];
            G.status[13] = (int)pc.seg[3];
        } else {
            atomicAdd(&G.status[6], (int)(pc.wait >> 10));
            atomicAdd(&G.status[7], (int)(pc.arm >> 10));
            atomicAdd(&G.status[8], (int)(pc.win >> 10));
            atomicAdd(&G.status[9], (int)(pc.total >> 10));
            atomicAdd(&G.status[14], (int)pc.seg[5]);
        }
    }
#endif
    if (is_coder) {
        if (S.mode != 0 && ord > 0) {
            // seal (SURVEY Appendix C.4): point = lower + 2^32 - 1, emit its high word
            const uint64_t point = cd.D + ((1ull << 32) - 1);
            if (lane == 0) {
                if (point < cd.D) {
                    int64_t i = cd.nout;
                    while (i > 0) {
                        i--;
                        if (i < S.out_cap) {
                            uint32_t v = S.out_words[i] + 1u;
                            S.out_words[i] = v;
                            if (v != 0u) break;
                        }
                    }
                }
                if (cd.nout < S.out_cap) S.out_words[cd.nout] = (uint32_t)(point >> 32);
            }
            cd.nout++;
        }
        if (lane == 0) {
            G.status[0] = ds.err;
            G.status[1] = (int32_t)ds.wpos;
            G.status[2] = (int32_t)(ds.slow + cd.slow);
            G.status[3] = (int32_t)cd.nout;
        }
    }
}

template <int NCTX, int CF, bool FAST>
int launch_t(const EntStream *d_streams, int n, size_t smem, int threads, const uint32_t *cdf, const float *scale,
             cudaStream_t st) {
    auto kern = k_entropy<NCTX, CF, FAST>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    e = cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return (int)e;
    kern<<<n, threads, smem, st>>>(d_streams, cdf, scale);
    g_ccd_launches++;
    return (int)cudaGetLastError();
}

}  // namespace

unsigned long long g_ccd_launches = 0;

size_t ccd_entropy_smem_bytes(int ring, int rows, int arm_blob_bytes, int ifce_blob_max) {
    size_t p = 64 + align16(sizeof(EntGrid)) + align16((size_t)arm_blob_bytes) + align16((size_t)ifce_blob_max);
    p += 16 + (size_t)ring * 16 + (size_t)ring * CCD_WIN * 4 + (size_t)(ring + CCD_HOT_MIRROR) * 16 + (size_t)(ring + 4) * 4 +
         (size_t)rows * CCD_ROW_COLS;
    return p;
}

bool ccd_entropy_has_fast(int n_ctx, int cf) {
    return (n_ctx == 6 && cf == 2) || (n_ctx == 10 && cf == 2) || (n_ctx == 10 && cf == 4) ||
           (n_ctx == 14 && cf == 6) || (n_ctx == 20 && cf == 6);
}

int ccd_entropy_launch(const EntStream *d_streams, int n_streams, const EntLaunchCfg &cfg,
                       const uint32_t *d_cdf, const float *d_scale, cudaStream_t st) {
    if (cfg.fast) {
        if (cfg.n_ctx == 6 && cfg.cf == 2) return launch_t<6, 2, true>(d_streams, n_streams, cfg.smem_bytes, cfg.threads, d_cdf, d_scale, st);
        if (cfg.n_ctx == 10 && cfg.cf == 2) return launch_t<10, 2, true>(d_streams, n_streams, cfg.smem_bytes, cfg.threads, d_cdf, d_scale, st);
        if (cfg.n_ctx == 10 && cfg.cf == 4) return launch_t<10, 4, true>(d_streams, n_streams, cfg.smem_bytes, cfg.threads, d_cdf, d_scale, st);
        if (cfg.n_ctx == 14 && cfg.cf == 6) return launch_t<14, 6, true>(d_streams, n_streams, cfg.smem_bytes, cfg.threads, d_cdf, d_scale, st);
        if (cfg.n_ctx == 20 && cfg.cf == 6) return launch_t<20, 6, true>(d_streams, n_streams, cfg.smem_bytes, cfg.threads, d_cdf, d_scale, st);
    }
    return launch_t<0, 0, false>(d_streams, n_streams, cfg.smem_bytes, cfg.threads, d_cdf, d_scale, st);
}

int ccd_cdf_table_build(uint32_t *d_cdf, const float *d_scale, cudaStream_t st) {
    size_t total = (size_t)CCD_N_SCALE * 256 * CCD_WIN;
    k_cdf_table<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(d_cdf, d_scale);
    return (int)cudaGetLastError();
}

int ccd_laplace_domain(const float *d_scale, int sc_lo, int sc_hi, uint32_t *d_lo, uint32_t *d_hi,
                       cudaStream_t st) {
    size_t total = (size_t)(sc_hi - sc_lo) * 32641;
    k_laplace_domain<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(d_scale, sc_lo, sc_hi, d_lo, d_hi);
    return (int)cudaGetLastError();
}
