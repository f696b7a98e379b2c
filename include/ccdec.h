/* ccdec.h -- C-ABI of libccdec.so, the B200-native (sm_100a) Cool-chic 5.0 decoder.
 *
 * Drop-in boundary for the DECODE path of Orange-OpenSource/Cool-Chic.  The reference is
 * pure Python and has no FFI of its own; each entry point below names the reference
 * function it replaces (paths relative to the reference checkout).  Host language above
 * this ABI is Python (ctypes, cool-chic_b200/_native.py), mirroring the reference's
 * decode_video / decode_frame / encode_decode_coolchic operator interface; see
 * INTEGRATION.md for the stub a reference maintainer would add.
 *
 * Conventions: plain pointers and sizes, no torch types.  Every function returns an int
 * status (0 = CCD_OK, negative = error, never throws); ccd_last_error() gives the message.
 * "d_" pointers are DEVICE pointers owned by the caller (e.g. torch.empty(..., device="cuda")
 * .data_ptr()); other pointers are HOST memory borrowed for the duration of the call.
 * One CcdContext per device; calls on one context must be serialised by the caller.
 * There is NO CPU fallback: without a CUDA device ccd_create() fails.
 */
#ifndef CCDEC_H
#define CCDEC_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CCD_VERSION 100 /* 0.1.0 */
#define CCD_MAX_GRIDS 32 /* n_latent_grids: 5-bit header field (bitstream/header/header.py:268) */
#define CCD_MAX_SYN 8    /* n_layer_synthesis: 3-bit header field (header.py:249) */

/* Architecture of one Cool-chic, as parsed from CoolChicHeader (header.py:243-377) and
 * derived like CoolChicEncoderParameter.__post_init__ (component/core/coolchic.py:149-225).
 * Grid index 0 is the finest grid (size_per_latent order). */
typedef struct CcdCoolChicDesc {
    int32_t img_h, img_w;
    int32_t n_grids;
    int32_t grid_h[CCD_MAX_GRIDS];
    int32_t grid_w[CCD_MAX_GRIDS];
    int32_t grid_is_hyper[CCD_MAX_GRIDS];
    int32_t grid_ifce_in[CCD_MAX_GRIDS];
    int32_t latent_res_lo, latent_res_hi;
    int32_t n_ctx;
    int32_t n_ifce_out;
    int32_t arm_hidden;
    int32_t arm_stab;
    int32_t ups_k, ups_pre_k;
    int32_t n_ups;
    int32_t n_syn_layers;
    int32_t syn_out[CCD_MAX_SYN];
    int32_t syn_k[CCD_MAX_SYN];
    int32_t syn_res[CCD_MAX_SYN];
    int32_t syn_relu[CCD_MAX_SYN];
    int32_t syn_stab;
    int32_t syn_in;
    int32_t common_randomness;
    int32_t final_ups; /* 0 nearest, 1 bilinear, 2 bicubic */
    int32_t qshift[8]; /* log2(q_step): arm.w arm.b ifce.w ifce.b ups.w ups.b syn.w syn.b */
    int32_t expgol[8];
    int32_t nn_n_bit_pad;
    int32_t flag_ifce;
} CcdCoolChicDesc;

enum {
    CCD_OK = 0,
    CCD_ERR_ARG = -1,          /* bad argument / inconsistent descriptor */
    CCD_ERR_NN_TRUNCATED = -2, /* NN payload shorter than announced */
    CCD_ERR_DESYNC = -3,       /* range decoder quantile >= 2^24: corrupt latent payload */
    CCD_ERR_UNSUPPORTED = -4,  /* valid syntax the device path does not implement yet */
    CCD_ERR_NOMEM = -5,
    CCD_ERR_CUDA = -6,         /* CUDA runtime error (message in ccd_last_error) */
    CCD_ERR_NO_DEVICE = -7
};

typedef struct CcdContext CcdContext;

int ccd_version(void);
int ccd_sizeof_desc(void);
/* message of the last failing call on this thread (ctx may be NULL) */
const char *ccd_last_error(const CcdContext *ctx);

/* Creates the per-device context: allocates scratch, uploads the normative scale table
 * (bitstream/component/mu_scale.npy, constants.py:24-37) and builds the device-resident
 * quantised-Laplace cumulative table (replaces constriction's per-symbol f64 CDF
 * evaluation, call site rangecoder.py:93). */
int ccd_create(int device_ordinal, CcdContext **out);
void ccd_destroy(CcdContext *ctx);

/* number of transmitted NN integers / latent symbols for a descriptor */
int64_t ccd_nn_count(const CcdCoolChicDesc *desc);
int64_t ccd_latent_count(const CcdCoolChicDesc *desc, int64_t offsets_by_grid[CCD_MAX_GRIDS]);

/* Host-side exp-Golomb decode of the NN payload.
 * Replaces decode_network + decode_exp_golomb (bitstream/neuralnet/neuralnet.py:92-204,
 * bitstream/neuralnet/expgolomb.py:74-130).  Returns the count or a negative status. */
int64_t ccd_decode_nn(const CcdCoolChicDesc *desc, const uint8_t *nn_bytes, size_t nn_nbytes,
                      int64_t *out_ints, size_t cap);

/* One independent Cool-chic to decode.  d_out: float32 [C_out][img_h][img_w] raw synthesis
 * output (un-clamped, un-rounded -- what encode_decode_coolchic returns).  d_latents
 * (optional, may be NULL): int8 decoded latents in decode order (coarsest grid first, each
 * grid row-major).  status (out): per-job status written on completion.
 * Frame tail (optional, the Cool-chic of an I frame): finish_bitdepth != 0 asks for decode_frame's
 * round / (4:2:0 average) / clamp / round (bitstream/decode.py:191-206) fused into the synthesis
 * kernel's epilogue: d_out then receives the FINISHED frame -- [3][H][W] for finish_type 0 (rgb),
 * 2 (yuv444), 3 (flow); for finish_type 1 (yuv420) d_out = y [H][W], d_out_u, d_out_v [H/2][W/2]. */
typedef struct CcdJob {
    const CcdCoolChicDesc *desc;
    const uint8_t *nn_bytes;
    size_t nn_nbytes;
    const uint8_t *latent_bytes;
    size_t latent_nbytes;
    float *d_out;
    int8_t *d_latents;
    int32_t status;
    int32_t finish_bitdepth;
    int32_t finish_type;
    float *d_out_u;
    float *d_out_v;
} CcdJob;

/* Decode n independent Cool-chics concurrently (one persistent CTA per stream for the
 * entropy stage, whole-GPU kernels for upsampling + synthesis).  Synchronous w.r.t. the
 * host: returns once results are in device memory.  Replaces, per job,
 * encode_decode_coolchic(mode="decode") (bitstream/component/coolchic.py:29-207), i.e.
 * arm_to_fixed_point_param (armint.py:30-170), the IFCE + wavefront ARM + range-decode loop
 * (component/coolchic.py:89-166, latent.py:18-187, armint.py:180-203, rangecoder.py:87-94
 * -> constriction RangeDecoder.decode), Upsampling.forward (core/upsampling.py:463-500),
 * Synthesis.forward (core/synthesis.py:272-294) and the final F.interpolate
 * (component/coolchic.py:187-192).  Returns CCD_OK if every job succeeded, else the first
 * failing job's status. */
int ccd_decode_many(CcdContext *ctx, CcdJob *jobs, int n_jobs, void *cuda_stream);

/* Convenience: single job. */
int ccd_decode_coolchic(CcdContext *ctx, const CcdCoolChicDesc *desc, const uint8_t *nn_bytes,
                        size_t nn_nbytes, const uint8_t *latent_bytes, size_t latent_nbytes,
                        float *d_out, int8_t *d_latents, void *cuda_stream);

/* Stage entry points (used by tests / profiling; same semantics as the stages above). */
int ccd_decode_latents(CcdContext *ctx, const CcdCoolChicDesc *desc, const int64_t *nn_ints,
                       const uint8_t *latent_bytes, size_t latent_nbytes, int8_t *d_latents,
                       void *cuda_stream);
int ccd_synthesize(CcdContext *ctx, const CcdCoolChicDesc *desc, const int64_t *nn_ints,
                   const int8_t *d_latents, float *d_out, void *cuda_stream);

/* Range ENcoder on the device: the mode="encode" branch of the same reference functions
 * (component/coolchic.py:152-170,194-195, latent.py:166-170, rangecoder.py:46-78 ->
 * constriction RangeEncoder.encode / get_compressed).  mode 1: encode the latents found in
 * d_latents (decode order);  mode 2: DRAW the latents from the stream's own ARM (seeded
 * splitmix64, one 24-bit quantile per symbol), store them in d_latents and encode them --
 * used to fabricate self-consistent synthetic streams (SURVEY 8d).  Output: little-endian
 * u32 words in d_out_words (device), count in *n_words_out. */
int ccd_encode_latents(CcdContext *ctx, const CcdCoolChicDesc *desc, const int64_t *nn_ints, int mode,
                       uint64_t seed, int8_t *d_latents, uint32_t *d_out_words, int64_t out_cap_words,
                       int64_t *n_words_out, int32_t *slow_path_count_out, void *cuda_stream);

/* One Cool-chic to ENcode from known latents.  desc / nn_bytes as in CcdJob.  d_latents: int8 latents in decode
 * order (coarsest grid first, each grid row-major and compact, offsets as ccd_latent_count gives them), every value
 * in [-64, 63] (AC_MAX_VAL, constants.py:9-11; anything else fails the call with CCD_ERR_ARG, nothing is clamped).
 * d_words / cap_words: device output, little-endian u32 words of the range-coded payload; n_symbols + 1 words always
 * suffice (a symbol renormalises at most once, plus the seal), a smaller capacity that is exceeded fails the call with
 * CCD_ERR_ARG.  d_out (optional, may be NULL): float32 [C_out][img_h][img_w] raw synthesis output of the given
 * latents -- what encode_decode_coolchic(mode="encode") returns as its first value.  Out: n_words, status and slow
 * (symbols outside the 31-symbol window, coded with the exact f64 model). */
typedef struct CcdEncodeJob {
    const CcdCoolChicDesc *desc;
    const uint8_t *nn_bytes;
    size_t nn_nbytes;
    const int8_t *d_latents;
    uint32_t *d_words;
    int64_t cap_words;
    float *d_out;
    int64_t n_words;
    int32_t status;
    int32_t slow;
} CcdEncodeJob;

/* Encode n independent Cool-chics: the latent half of encode_decode_coolchic(mode="encode")
 * (component/coolchic.py:29-207, latent.py:142-173 with range_coder.encode, rangecoder.py:46-78 -> constriction
 * RangeEncoder.encode / get_compressed) plus, for the jobs with a d_out, the same upsampling + synthesis as
 * ccd_decode_many.  Every latent is known, so the ARM of all symbols of all jobs runs as one data-parallel pass over
 * the GPU; only the range recursion is serial (one warp per job).  Byte-identical to ccd_encode_latents mode 1.
 * Synchronous w.r.t. the host.  ccd_last_timing afterwards: ms[0] ARM pass + range coder, ms[1] synthesis, ms[2]
 * host prep + H2D. */
int ccd_encode_many(CcdContext *ctx, CcdEncodeJob *jobs, int n_jobs, void *cuda_stream);

/* Tail of decode_frame for every frame type (bitstream/decode.py:191-206 with
 * io/format/yuv.py:239-256,274-300): round to the 2^b-1 grid -> (444->420 2x2 average of
 * U,V) -> clamp [0,1] -> round again.  data_type: 0 rgb, 1 yuv420, 2 yuv444.
 * d_in [3][H][W];  rgb/444: d_out_a [3][H][W];  420: d_out_a=y [H][W], d_out_b=u, d_out_c=v
 * [H/2][W/2]. */
int ccd_finish_frame(CcdContext *ctx, const float *d_in, int h, int w, int bitdepth, int data_type,
                     float *d_out_a, float *d_out_b, float *d_out_c, void *cuda_stream);

/* P/B-frame prediction + residue (bitstream/decode.py:156-189: apply_global_translation
 * globalmotion.py:151-160, Warper.forward warp.py:294-397 in its training branch, alpha/beta
 * blending).  d_residue [n_res_ch][H][W], d_motion [n_mot_ch][H][W]: raw synthesis outputs; the
 * channel counts are checked against what the path reads (P: 4 / 2, B: 5 / 4; the reference raises a
 * shape error otherwise).  d_ref0/d_ref1 [3][H][W] (444).  global_flow: (x,y) per reference.
 * d_out [3][H][W] pre-rounding frame.  warp_filter_size 2 / 4: grid_sample bilinear / bicubic (border,
 * align_corners); 6, 8, 10, 12, 14: windowed sinc (14 is the largest value of the 4-bit header field,
 * header/header.py:217); odd sizes are an argument error. */
int ccd_inter_predict(CcdContext *ctx, const float *d_residue, int n_res_ch, const float *d_motion,
                      int n_mot_ch, const float *d_ref0, const float *d_ref1, int h, int w, int is_b,
                      const int32_t *global_flow, int warp_filter_size, float *d_out,
                      void *cuda_stream);

/* Whole reconstruction of a P/B frame in ONE kernel: the prediction above + the frame tail of
 * ccd_finish_frame (bitstream/decode.py:156-206).  The references are given as three plane pointers
 * each, in the layout of the frames this function (or ccd_finish_frame) produced: frame_data_type 1
 * (yuv420): y [H][W], u, v [H/2][W/2] -- read through the nearest x2 up-conversion of
 * convert_420_to_444 (io/format/yuv.py:303-316) folded into the gather index; otherwise three [H][W]
 * planes.  out_planes: the finished frame in the same layout.  ref1_planes may be NULL for a P frame. */
int ccd_reconstruct_frame(CcdContext *ctx, const float *d_residue, int n_res_ch, const float *d_motion,
                          int n_mot_ch, const float *const ref0_planes[3],
                          const float *const ref1_planes[3], int frame_data_type, int bitdepth, int h,
                          int w, int is_b, const int32_t *global_flow, int warp_filter_size,
                          float *const out_planes[3], void *cuda_stream);

/* Output packing on the device (io/format/yuv.py:150-162, ppm.py:160-203, png.py:44-62): finished
 * planes (values on the k / (2^b - 1) grid) -> integer samples round(x * (2^b - 1)), uint8 when
 * sample_bytes == 1, little-endian uint16 when 2.  interleaved == 0: the three planes one after the
 * other (planar YUV file order; chroma planes [H >> cs][W >> cs], cs = 1 for yuv420);
 * interleaved == 1 (cs must be 0): pixel-interleaved [H][W][3] (PPM / PNG order).  d_out holds
 * sample_bytes * (H*W + 2 * (H>>cs) * (W>>cs)) bytes. */
int ccd_pack_frame(CcdContext *ctx, const float *const planes[3], int h, int w, int chroma_shift,
                   int bitdepth, int sample_bytes, int interleaved, void *d_out, void *cuda_stream);

/* The same conversion for n samples that already lie in output order -- the planes of a BATCH of finished
 * planar frames stored one after the other (what ccd_decode_many writes when the caller hands it slices
 * of one buffer): one launch and one device-to-host copy for the whole batch instead of one per frame. */
int ccd_pack_samples(CcdContext *ctx, const float *d_samples, size_t n, int bitdepth, int sample_bytes,
                     void *d_out, void *cuda_stream);

/* Device-side evaluation of the quantised-Laplace left cumulative for testing the f64
 * exp() agreement with the host (SURVEY Appendix C.3): for sc in [sc_lo, sc_hi) and every
 * numerator index n in [0, 32641) (|d| = n/256), writes to host arrays
 * out_lo[(sc-sc_lo)*32641+n] = trunc(FW * 0.5*exp(-|d|/b)) and
 * out_hi[...]                = trunc(FW * (1 - 0.5*exp(-|d|/b))). */
int ccd_debug_laplace_domain(CcdContext *ctx, int sc_lo, int sc_hi, uint32_t *out_lo,
                             uint32_t *out_hi);

/* Number of CUDA kernels this library has launched since it was loaded. */
uint64_t ccd_debug_launch_count(void);

/* 1 (default): one fused kernel for the synthesis when the architecture allows it; 0: one kernel per
 * layer.  Both give bit-identical results (tests/test_gpu_decode.py). */
int ccd_debug_set_fused_synthesis(CcdContext *ctx, int on);

/* Entropy-kernel status words of the last job of the last call: [0] error, [1] words consumed,
 * [2] slow-path symbols (outside the 31-symbol window), [3] words emitted (encode modes),
 * [4..15] cycle / event counters when the library is built with -DCCD_PROFILE (else 0; layout in
 * csrc/ccd_entropy.cu). */
int ccd_debug_last_status(const CcdContext *ctx, int32_t st[16]);

/* Timing of the last ccd_decode_many call on this context, measured with CUDA events on the
 * launching stream: ms[0] entropy stage, ms[1] upsampling+synthesis, ms[2] host prep + H2D;
 * ms[3] = bytes uploaded host->device by that call (as a float). */
int ccd_last_timing(const CcdContext *ctx, float ms[4]);

#ifdef __cplusplus
}
#endif
#endif
