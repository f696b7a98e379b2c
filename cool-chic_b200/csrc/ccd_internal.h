// ccd_internal.h -- structures shared between the host API and the sm_100a kernels.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/ccdec.h"

// --------------------------------------------------------------------------------------
// Entropy stage (ccd_entropy.cu): one persistent CTA per Cool-chic stream.
// --------------------------------------------------------------------------------------
#define CCD_ENT_THREADS 512          // <= 14 producer warps + helper warp + range-coder warp
#define CCD_ENT_THREADS_NARROW 256   // 5 producer warps + helper + coder: two streams per SM when a call holds more streams than SMs
#define CCD_ENT_WARPS (CCD_ENT_THREADS / 32)
#define CCD_ENT_PRODUCERS (CCD_ENT_WARPS - 2)
#define CCD_WIN 32                   // cumulative-window entries per symbol (31 decodable symbols)
#define CCD_WIN_HALF 14              // window = symbols mu_int-14 .. mu_int+16; the mode sits at the EVEN index 14
                                     // so that (left(mode), left(mode+1)) is one aligned LDS.64
#define CCD_HOT_MIRROR 8            // hot-ring entries duplicated behind the end of the ring
#define CCD_ROW_COLS 64              // row ring: columns kept per row (power of 2)
#define CCD_IFCE_FAST_MAX 12         // IFCE inputs handled by the fast (quad) kernel; more -> generic kernel
#define CCD_MAX_DIM 72               // n_ctx (<=40) + n_ifce_out (<=31)
#define CCD_N_SCALE 2561
#define CCD_MASK_STRIDE 10           // wavefront stride = ARM mask size 9 + 1 (latent.py:63,72)

// One latent grid, in DECODE order (index 0 = coarsest = first decoded).
struct EntGrid {
    int32_t h, w;
    int32_t n_diag;        // w + 10*(h-1), or h*w in raster mode
    int32_t raster;        // w <= 9: plain raster scan (latent.py:113-122)
    int64_t lat_off;       // offset of this grid in the latent array (decode order)
    int32_t ifce_in;       // number of IFCE inputs (0: features are zero)
    int32_t ifce_blob_off; // byte offset of this grid's IFCE parameters in the blob
    int32_t ifce_blob_bytes;
    int32_t n_dec;         // grids decoded before this one
    // IFCE input channel c reads grid (this-1-c) at (yy >> sh, xx >> sh); sh < 0: constant 0
    int32_t ch_w[31];
    int32_t ch_sh[31];
    int64_t ch_off[31];
};

struct EntStream {
    int32_t n_grids;
    int32_t n_ctx, cf, n_hidden, has_ifce;
    int32_t ring;          // window ring entries (power of two)
    int32_t rows;          // row ring rows (power of two)
    int32_t mode;          // 0 decode, 1 encode given latents, 2 sample + encode, 3 data-parallel encode (ccd_encode.cu)
    uint32_t prod_mask;    // which of warps 0..13 produce (14 = coder helper, 15 = range coder)
    const uint32_t *words; // compressed words (device); mode 3: the symbols' intervals, uint2 [n_symbols] in coding order
    int64_t n_words;
    int8_t *latents;       // device, decode order
    int64_t n_symbols;
    const unsigned char *blob; // device: ARM parameters followed by IFCE parameters
    int32_t arm_blob_bytes;
    int32_t ifce_blob_max;     // largest per-grid IFCE blob
    int32_t *status;           // device: [0] error code, [1] words consumed, [2] slow-path count
    uint64_t seed;
    uint32_t *out_words;       // encode modes: output words (device)
    int64_t out_cap;
    EntGrid grid[CCD_MAX_GRIDS];
};

// Blob layouts ---------------------------------------------------------------------------
// FAST (int32 operands, proven not to overflow by the host-side bound analysis); a symbol is
// evaluated by a quad of lanes, member m owning activations [m*opm, (m+1)*opm):
//   opm = ceil(dim/4), opmp = 2|4|8 (opm padded for vector loads), dimp = 4*opm
//   int32 Wh[n_hidden][dim][4][opmp]   weight of input i for the outputs of member m
//   int32 Wl[dimp][2]                  last layer   (rows >= dim are zero)
//   int32 Ws[dimp][2]                  stabiliser   (zeros if absent)
//   (pad to 8 bytes)
//   int64 Bh[n_hidden][dimp], Bl[2], Bs[2]
// IFCE arm (FAST): int32 W[n_in][cfp] (cfp = cf rounded up to 4), pad8, int64 B[cf]
// GENERIC (all int64): W64h[n_hidden][dim][dim], Wl[dim][2], Ws[dim][2], Bh, Bl, Bs;
//   IFCE: int64 W[n_in][cf], B[cf]

// number of kernels launched by this library since load (bench.py reports it)
extern unsigned long long g_ccd_launches;

struct EntLaunchCfg {
    int n_ctx, cf;   // template selection
    bool fast;
    size_t smem_bytes;
    int threads;     // CCD_ENT_THREADS, or CCD_ENT_THREADS_NARROW for two CTAs per SM
};

int ccd_entropy_launch(const EntStream *d_streams, int n_streams, const EntLaunchCfg &cfg,
                       const uint32_t *d_cdf, const float *d_scale, cudaStream_t st);
size_t ccd_entropy_smem_bytes(int ring, int rows, int arm_blob_bytes, int ifce_blob_max);
bool ccd_entropy_has_fast(int n_ctx, int cf);
int ccd_cdf_table_build(uint32_t *d_cdf, const float *d_scale, cudaStream_t st);
int ccd_laplace_domain(const float *d_scale, int sc_lo, int sc_hi, uint32_t *d_lo, uint32_t *d_hi,
                       cudaStream_t st);

// --------------------------------------------------------------------------------------
// Data-parallel encoder of known latents (ccd_encode.cu): k_enc_arm over tiles of every job of a launch group
// (intervals in coding order into EntStream.words), then k_enc_range, one warp per job (words into out_words,
// status [0] error, [2] slow-path symbols, [3] words emitted).
// --------------------------------------------------------------------------------------
#define CCD_ENC_THREADS 256
#define CCD_ENC_CHUNK_FAST 8       // pixels of one row per warp step: a quad of lanes per symbol
#define CCD_ENC_CHUNK_GENERIC 32   // one lane per symbol
#define CCD_ENC_TILE_CHUNKS 256    // chunks per CTA
struct EncTile {
    int32_t stream;    // index into the launch's EntStream array
    int32_t grid;      // decode-order grid index
    int32_t chunk0, n_chunks;
};
size_t ccd_encode_smem_bytes(int arm_blob_bytes, int ifce_blob_max);
int ccd_enc_arm_launch(const EntStream *d_streams, const EncTile *d_tiles, int n_tiles, const EntLaunchCfg &cfg,
                       const uint32_t *d_cdf, const float *d_scale, cudaStream_t st);
int ccd_enc_range_launch(const EntStream *d_streams, int n_streams, cudaStream_t st);

// --------------------------------------------------------------------------------------
// Synthesis stage (ccd_synth.cu)
// --------------------------------------------------------------------------------------
struct SynLayerDev {
    int cin, cout, k, residual, relu;
    const float *w; // [cout][cin][k][k]
    const float *b; // [cout]
};

int ccd_ups_pre(const int8_t *d_lat, int h, int w, const float *w1d, int k, float *d_out, cudaStream_t st);
int ccd_ups_first(const int8_t *d_lat, int h, int w, float *d_out, cudaStream_t st);
int ccd_ups_convt(const float *d_in, int c, int h, int w, const float *w1d, int k, float *d_out, int ht,
                  int wt, cudaStream_t st);
// one cascade level in one launch (ups_k == 8, ups_pre_k == 7 only): out[0] = pre-concat conv of the target latent,
// out[1 + c] = transposed conv of in[c]
int ccd_ups_level(const int8_t *d_lat, int th, int tw, const float *d_in, int cc, int ch, int cw, const float *wt1d,
                  const float *wc1d, float *d_out, cudaStream_t st);
int ccd_syn_layer(const float *d_in, int h, int w, const SynLayerDev &L, float *d_out, cudaStream_t st);
int ccd_syn_pointwise2(const float *d_in, int h, int w, const SynLayerDev &L0, const SynLayerDev &L1,
                       float *d_out, cudaStream_t st);
// whole synthesis in one kernel when the architecture allows it (returns -1 otherwise: use the layer kernels)
int ccd_syn_fused(const float *d_in, int h, int w, int cin, const SynLayerDev *layers, int n_layers,
                  const SynLayerDev *stab, const SynLayerDev &ot, float *d_out, cudaStream_t st);
int ccd_syn_add(float *d_a, const float *d_b, size_t n, cudaStream_t st);

// ---- batched float tail (ccd_synth.cu): device-resident job arrays, one launch per cascade level and one for
// the last level + synthesis + frame tail of ALL streams of a group
struct CcdTailSynDesc {
    const int8_t *lat;        // finest latent grid [h][w]
    const float *stk;         // coarser stack [cin - 1][ch][cw] (fp32), or ...
    const int8_t *stk8;       // ... the coarsest latent itself when the stream has two grids
    float *out[5];            // output planes
    int h, w, ch, cw, cin;
    const SynLayerDev *layers;
    int n_layers;
    const SynLayerDev *stab;  // may be null
    SynLayerDev ot;
    int finish;               // 0 raw, 1 frame tail (full planes), 2 frame tail 4:2:0
    float M;
    const float *wt1d, *wc1d; // 8 / 7 taps of the last cascade level
    int allow_tma;
};
size_t ccd_tail_job_bytes(void);
size_t ccd_tail_level_job_bytes(void);
void ccd_tail_fill_level(void *dst, const int8_t *lat, const float *in, const int8_t *in8, float *out, int cc, int ch,
                         int cw, int th, int tw, const float *wt1d, const float *wc1d);
int ccd_tail_launch_level(const void *d_jobs, int n_jobs, int planes, int max_tw, int max_th, cudaStream_t st);
int ccd_tail_fill_syn(void *dst, const CcdTailSynDesc &T);
int ccd_tail_launch_syn(const void *d_jobs, int n_jobs, int cinp, int C, int n3_max, int hid_max, int max_w, int max_h,
                        cudaStream_t st);
int ccd_resize_nearest(const float *d_in, int c, int h, int w, float *d_out, int H, int W, cudaStream_t st);
// F.interpolate bilinear (mode 1) / bicubic (mode 2), align_corners=False; sy/sx = 0.5 (scale_factor 2) or in/out
int ccd_resize_torch(const float *d_in, int c, int h, int w, float *d_out, int H, int W, int mode, float sy, float sx,
                     cudaStream_t st);
// samples [first, first+n) of the common-randomness generator (noise.py)
int ccd_cr_noise(float *d_out, size_t first, size_t n, cudaStream_t st);
int ccd_finish(const float *d_in, int h, int w, int bitdepth, int data_type, float *a, float *b, float *c,
               cudaStream_t st);

int ccd_pack(const float *const planes[3], int h, int w, int cs, int bitdepth, int sample_bytes, int interleaved,
             void *d_out, cudaStream_t st);
int ccd_pack_flat(const float *d_in, size_t n, int bitdepth, int sample_bytes, void *d_out, cudaStream_t st);

// P/B reconstruction (ccd_inter.cu); returns -1 for an unsupported filter size
struct InterLaunch {
    const float *residue, *motion;  // [4|5][h][w], [2|4][h][w]
    const float *ref0[3], *ref1[3]; // planes of the references; ref1 all null for a P frame
    int ref_cs;                     // 1: reference chroma planes are [h/2][w/2] (4:2:0), 0: full size
    int h, w, is_b;
    int32_t gf[4];                  // global flow (x, y) per reference
    int filter_size;
    float M;                        // 0: pre-rounding output; 2^bitdepth - 1: finished frame (decode.py:191-206)
    int out_420;                    // finished output with [h/2][w/2] chroma planes
    float *out[3];
};
int ccd_inter_launch(const InterLaunch &a, cudaStream_t st);
