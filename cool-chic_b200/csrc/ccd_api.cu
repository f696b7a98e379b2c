// ccd_api.cu -- host side of libccdec.so: the C-ABI of include/ccdec.h.
//
// Host work per Cool-chic (all tiny, <= a few kB): exp-Golomb decode of the NN payload
// (neuralnet.py:92-204, expgolomb.py:74-130), conversion of the ARM / IFCE integers into
// fixed-point parameters (armint.py:30-170) packed for the entropy kernel, a worst-case
// bound analysis that proves the int32-operand fast path safe (otherwise the generic int64
// kernel is used -- still on the GPU), dequantisation of upsampling / synthesis weights.
// Everything per-pixel runs in ccd_entropy.cu / ccd_synth.cu.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "ccd_internal.h"

namespace {

thread_local std::string g_err;

int fail(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CUDA_TRY(expr)                                                                         \
    do {                                                                                       \
        cudaError_t e__ = (expr);                                                              \
        if (e__ != cudaSuccess)                                                                \
            return fail(CCD_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), \
                        __FILE__, __LINE__);                                                   \
    } while (0)

const uint32_t k_scale_bits[CCD_N_SCALE] = {
#include "ccd_scale_table.inc"
};

// ---- NN integer layout (neuralnet.py:120-148; module order arm, ifce, upsampling, synthesis;
// per module all weights then all biases; parameter registration order of each module) --------
struct NNLayout {
    int dim = 0, n_arm_lin = 0;
    int64_t arm_w[9] = {0}, arm_b[9] = {0};  // [n_arm_lin] = stabiliser
    int n_ifce = 0;
    int ifce_grid[CCD_MAX_GRIDS] = {0};
    int64_t ifce_w[CCD_MAX_GRIDS] = {0}, ifce_b[CCD_MAX_GRIDS] = {0};
    int kt_par = 0, kc_par = 0;
    int64_t ups_tw = 0, ups_cw = 0;
    int syn_c = 0, syn_stab_in = 0;
    int64_t syn_ot_w = 0, syn_st_w = 0, syn_w[CCD_MAX_SYN] = {0};
    int64_t syn_ot_b = 0, syn_st_b = 0, syn_b[CCD_MAX_SYN] = {0};
    int64_t counts[8] = {0};
    int64_t total = 0;
};

int validate_desc(const CcdCoolChicDesc *d) {
    if (!d) return fail(CCD_ERR_ARG, "null descriptor");
    if (d->n_grids < 1 || d->n_grids > CCD_MAX_GRIDS) return fail(CCD_ERR_ARG, "n_grids=%d out of range", d->n_grids);
    if (d->n_syn_layers < 1 || d->n_syn_layers > CCD_MAX_SYN)
        return fail(CCD_ERR_ARG, "n_syn_layers=%d out of range", d->n_syn_layers);
    if (d->arm_hidden < 0 || d->arm_hidden > 7) return fail(CCD_ERR_ARG, "arm_hidden=%d out of range", d->arm_hidden);
    if (d->n_ctx < 0 || d->n_ctx > 40) return fail(CCD_ERR_ARG, "n_ctx=%d out of range", d->n_ctx);
    if (d->n_ifce_out < 0 || d->n_ifce_out > 31) return fail(CCD_ERR_ARG, "n_ifce_out=%d out of range", d->n_ifce_out);
    if (d->n_ctx + d->n_ifce_out < 1) return fail(CCD_ERR_ARG, "ARM without any context");
    if (d->img_h < 1 || d->img_w < 1) return fail(CCD_ERR_ARG, "bad image size");
    for (int g = 0; g < d->n_grids; g++) {
        if (d->grid_h[g] < 1 || d->grid_w[g] < 1) return fail(CCD_ERR_ARG, "grid %d has an empty dimension", g);
        if (d->grid_ifce_in[g] < 0 || d->grid_ifce_in[g] > 31) return fail(CCD_ERR_ARG, "grid %d: bad ifce_in", g);
        if (d->flag_ifce && d->grid_ifce_in[g] > 0 && d->grid_ifce_in[g] != std::max(d->n_grids - 1 - g, 1))
            return fail(CCD_ERR_ARG, "grid %d: ifce_in=%d inconsistent", g, d->grid_ifce_in[g]);
    }
    for (int i = 0; i < 8; i++) {
        if (d->expgol[i] < 0 || d->expgol[i] > 12) return fail(CCD_ERR_ARG, "exp-Golomb order out of range");
        if (d->qshift[i] > 0 || d->qshift[i] < -24) return fail(CCD_ERR_ARG, "q_step out of range");
    }
    if (d->qshift[0] < -8 || d->qshift[2] < -8 || d->qshift[1] < -16 || d->qshift[3] < -16)
        return fail(CCD_ERR_ARG, "ARM/IFCE q_step out of range");
    if (d->ups_k < 4 || (d->ups_k & 1) || d->ups_k > 14) return fail(CCD_ERR_ARG, "ups_k=%d unsupported", d->ups_k);
    if (!(d->ups_pre_k & 1) || d->ups_pre_k > 15 || d->ups_pre_k < 1)
        return fail(CCD_ERR_ARG, "ups_pre_k=%d unsupported", d->ups_pre_k);
    for (int l = 0; l < d->n_syn_layers; l++) {
        if (d->syn_out[l] < 1 || d->syn_out[l] > 127 || d->syn_k[l] < 1 || !(d->syn_k[l] & 1))
            return fail(CCD_ERR_ARG, "synthesis layer %d malformed", l);
    }
    return CCD_OK;
}

int nn_layout(const CcdCoolChicDesc *d, NNLayout *L) {
    int rc = validate_desc(d);
    if (rc) return rc;
    int64_t p = 0, q;
    const int dim = d->n_ctx + d->n_ifce_out;
    L->dim = dim;
    L->n_arm_lin = d->arm_hidden + 1;
    for (int l = 0; l < L->n_arm_lin; l++) {
        L->arm_w[l] = p;
        p += (int64_t)((l == d->arm_hidden) ? 2 : dim) * dim;
    }
    if (d->arm_stab) {
        L->arm_w[L->n_arm_lin] = p;
        p += 2 * dim;
    }
    L->counts[0] = p;
    q = p;
    for (int l = 0; l < L->n_arm_lin; l++) {
        L->arm_b[l] = p;
        p += (l == d->arm_hidden) ? 2 : dim;
    }
    if (d->arm_stab) {
        L->arm_b[L->n_arm_lin] = p;
        p += 2;
    }
    L->counts[1] = p - q;
    q = p;
    if (d->flag_ifce)
        for (int g = 0; g < d->n_grids; g++)
            if (d->grid_ifce_in[g] > 0) {
                L->ifce_grid[L->n_ifce] = g;
                L->ifce_w[L->n_ifce++] = p;
                p += (int64_t)d->n_ifce_out * d->grid_ifce_in[g];
            }
    L->counts[2] = p - q;
    q = p;
    for (int j = 0; j < L->n_ifce; j++) {
        L->ifce_b[j] = p;
        p += d->n_ifce_out;
    }
    L->counts[3] = p - q;
    L->kt_par = (d->ups_k + 1) / 2;
    L->kc_par = (d->ups_pre_k + 1) / 2;
    q = p;
    L->ups_tw = p;
    p += (int64_t)d->n_ups * L->kt_par;
    L->ups_cw = p;
    p += (int64_t)d->n_ups * L->kc_par;
    L->counts[4] = p - q;
    L->counts[5] = 2 * (int64_t)d->n_ups;  // one (unused) bias per kernel, upsampling.py:123,243
    p += L->counts[5];
    const int C = d->syn_out[d->n_syn_layers - 1];
    L->syn_c = C;
    L->syn_stab_in = d->common_randomness ? d->syn_in / 2 : d->syn_in;
    q = p;
    L->syn_ot_w = p;
    p += (int64_t)C * C;
    if (d->syn_stab) {
        L->syn_st_w = p;
        p += (int64_t)C * L->syn_stab_in;
    }
    int in_ft = d->syn_in;
    for (int l = 0; l < d->n_syn_layers; l++) {
        L->syn_w[l] = p;
        p += (int64_t)d->syn_out[l] * in_ft * d->syn_k[l] * d->syn_k[l];
        in_ft = d->syn_out[l];
    }
    L->counts[6] = p - q;
    q = p;
    L->syn_ot_b = p;
    p += C;
    if (d->syn_stab) {
        L->syn_st_b = p;
        p += C;
    }
    for (int l = 0; l < d->n_syn_layers; l++) {
        L->syn_b[l] = p;
        p += d->syn_out[l];
    }
    L->counts[7] = p - q;
    L->total = p;
    return CCD_OK;
}

// MSB-first exp-Golomb reader over the NN payload
int64_t decode_nn_host(const CcdCoolChicDesc *d, const NNLayout &L, const uint8_t *bytes, size_t nbytes,
                       int64_t *out) {
    const size_t nbits = nbytes * 8;
    size_t pos = (size_t)d->nn_n_bit_pad;
    auto bit = [&](size_t i) -> int { return (bytes[i >> 3] >> (7 - (i & 7))) & 1; };
    int64_t n = 0;
    for (int m = 0; m < 8; m++) {
        const int k = d->expgol[m];
        for (int64_t i = 0; i < L.counts[m]; i++) {
            int z = 0;
            while (pos < nbits && bit(pos) == 0) {
                z++;
                pos++;
            }
            if (pos + (size_t)z + 1 + (size_t)k > nbits || z > 60)
                return fail(CCD_ERR_NN_TRUNCATED, "NN payload truncated at parameter %lld", (long long)n);
            uint64_t val = 0;
            for (int j = 0; j <= z; j++) val = (val << 1) | (uint64_t)bit(pos++);
            uint64_t rem = 0;
            for (int j = 0; j < k; j++) rem = (rem << 1) | (uint64_t)bit(pos++);
            const int64_t v = (int64_t)(((val - 1) << k) + rem);
            out[n++] = (v & 1) ? (v + 1) / 2 : -(v / 2);
        }
    }
    return n;
}

// ---- fixed-point ARM parameters (armint.py:30-170) ------------------------------------------
struct ArmInts {
    int dim = 0, n_hidden = 0, n_out = 2;
    std::vector<std::vector<int64_t>> W;  // per linear layer, TRANSPOSED: [in][out]
    std::vector<std::vector<int64_t>> B;
    std::vector<int64_t> Ws, Bs;          // stabiliser [in][n_out], [n_out] (zeros if absent)
};

ArmInts build_arm(int dim, int n_hidden, int n_out, const int64_t *const *qw, const int64_t *const *qb,
                  const int64_t *qws, const int64_t *qbs, int s_w, int s_b, bool subtract_last,
                  int n_inter_ft, bool no_residual) {
    ArmInts a;
    a.dim = dim;
    a.n_hidden = n_hidden;
    a.n_out = n_out;
    a.W.resize(n_hidden + 1);
    a.B.resize(n_hidden + 1);
    for (int l = 0; l <= n_hidden; l++) {
        const int out = (l == n_hidden) ? n_out : dim;
        a.W[l].assign((size_t)dim * out, 0);
        a.B[l].assign((size_t)out, 0);
        for (int o = 0; o < out; o++) {
            for (int i = 0; i < dim; i++) {
                const bool ifce_col = n_inter_ft > 0 && l == 0 && i >= dim - n_inter_ft;
                const int shift = 16 + s_w - (ifce_col ? 8 : 0);
                int64_t v = qw[l][(size_t)o * dim + i] * ((int64_t)1 << shift);
                // every square layer is residual: +I folded into the weights (armint.py:114-124)
                if (out == dim && !no_residual && o == i) v += (int64_t)1 << (ifce_col ? 8 : 16);
                a.W[l][(size_t)i * out + o] = v;
            }
            int64_t qv = qb[l][o];
            if (l == n_hidden && subtract_last && o == 1) qv -= (int64_t)4 << (-s_b);  // armint.py:98-100
            a.B[l][o] = qv * ((int64_t)1 << (32 + s_b));
        }
    }
    a.Ws.assign((size_t)dim * n_out, 0);
    a.Bs.assign((size_t)n_out, 0);
    if (qws) {
        for (int o = 0; o < n_out; o++) {
            for (int i = 0; i < dim; i++) {
                const bool ifce_col = n_inter_ft > 0 && i >= dim - n_inter_ft;
                a.Ws[(size_t)i * n_out + o] = qws[(size_t)o * dim + i] * ((int64_t)1 << (16 + s_w - (ifce_col ? 8 : 0)));
            }
            a.Bs[o] = qbs[o] * ((int64_t)1 << (32 + s_b));
        }
    }
    return a;
}

typedef __int128 i128;
inline i128 iabs128(int64_t v) { return v < 0 ? -(i128)v : (i128)v; }

// worst-case |IFCE feature| (8 fractional bits), incl. the fp32 round trip
bool ifce_bound(const ArmInts &a, i128 *bound) {
    i128 best = 0;
    for (int o = 0; o < a.n_out; o++) {
        i128 acc = iabs128(a.B[0][o]);
        for (int i = 0; i < a.dim; i++) {
            if (iabs128(a.W[0][(size_t)i * a.n_out + o]) > INT32_MAX) return false;
            acc += iabs128(a.W[0][(size_t)i * a.n_out + o]) * ((i128)64 << 16);
        }
        if (acc >= ((i128)1 << 62)) return false;
        i128 f = (acc >> 24) + 1;
        f += (f >> 22) + 1;  // float rounding
        best = std::max(best, f);
    }
    *bound = best;
    return true;
}

// Can the ARM run with int32 operands (weights, activations) and int64 accumulators?
bool arm_fits_int32(const ArmInts &a, int n_ctx, i128 ifce_feat_bound) {
    std::vector<i128> X((size_t)a.dim);
    for (int i = 0; i < a.dim; i++) X[i] = (i < n_ctx) ? ((i128)64 << 16) : (ifce_feat_bound << 16);
    for (int i = 0; i < a.dim; i++)
        if (X[i] > INT32_MAX) return false;
    auto layer_ok = [&](const std::vector<int64_t> &W, const std::vector<int64_t> &B, int out,
                        const std::vector<i128> &Xin, std::vector<i128> *acc) {
        acc->assign((size_t)out, 0);
        for (int o = 0; o < out; o++) {
            i128 s = iabs128(B[o]);
            for (int i = 0; i < a.dim; i++) {
                if (iabs128(W[(size_t)i * out + o]) > INT32_MAX) return false;
                s += iabs128(W[(size_t)i * out + o]) * Xin[i];
            }
            if (s >= ((i128)1 << 61)) return false;
            (*acc)[o] = s;
        }
        return true;
    };
    std::vector<i128> acc, stab;
    if (!layer_ok(a.Ws, a.Bs, a.n_out, X, &stab)) return false;
    for (int l = 0; l < a.n_hidden; l++) {
        if (!layer_ok(a.W[l], a.B[l], a.dim, X, &acc)) return false;
        for (int o = 0; o < a.dim; o++) {
            X[o] = acc[o] >> 16;
            if (X[o] > INT32_MAX) return false;
        }
    }
    if (!layer_ok(a.W[a.n_hidden], a.B[a.n_hidden], a.n_out, X, &acc)) return false;
    return true;
}

void put_i32(std::vector<unsigned char> &b, int64_t v) {
    int32_t t = (int32_t)v;
    b.insert(b.end(), (unsigned char *)&t, (unsigned char *)&t + 4);
}
void put_i64(std::vector<unsigned char> &b, int64_t v) { b.insert(b.end(), (unsigned char *)&v, (unsigned char *)&v + 8); }
void pad_to(std::vector<unsigned char> &b, size_t a) {
    while (b.size() % a) b.push_back(0);
}

void pack_arm(const ArmInts &a, bool fast, std::vector<unsigned char> &b) {
    const int dim = a.dim;
    if (fast) {
        const int opm = (dim + 3) / 4, opmp = opm <= 2 ? 2 : (opm <= 4 ? 4 : 8), dimp = 4 * opm;
        for (int l = 0; l < a.n_hidden; l++)
            for (int i = 0; i < dim; i++)
                for (int m = 0; m < 4; m++)
                    for (int o = 0; o < opmp; o++) {
                        const int out = m * opm + o;
                        put_i32(b, (o < opm && out < dim) ? a.W[l][(size_t)i * dim + out] : 0);
                    }
        for (int i = 0; i < dimp; i++)
            for (int o = 0; o < 2; o++) put_i32(b, i < dim ? a.W[a.n_hidden][(size_t)i * 2 + o] : 0);
        for (int i = 0; i < dimp; i++)
            for (int o = 0; o < 2; o++) put_i32(b, i < dim ? a.Ws[(size_t)i * 2 + o] : 0);
        pad_to(b, 8);
        for (int l = 0; l < a.n_hidden; l++)
            for (int o = 0; o < dimp; o++) put_i64(b, o < dim ? a.B[l][o] : 0);
    } else {
        for (int l = 0; l < a.n_hidden; l++)
            for (size_t t = 0; t < (size_t)dim * dim; t++) put_i64(b, a.W[l][t]);
        for (size_t t = 0; t < (size_t)dim * 2; t++) put_i64(b, a.W[a.n_hidden][t]);
        for (size_t t = 0; t < (size_t)dim * 2; t++) put_i64(b, a.Ws[t]);
        for (int l = 0; l < a.n_hidden; l++)
            for (int o = 0; o < dim; o++) put_i64(b, a.B[l][o]);
    }
    put_i64(b, a.B[a.n_hidden][0]);
    put_i64(b, a.B[a.n_hidden][1]);
    put_i64(b, a.Bs[0]);
    put_i64(b, a.Bs[1]);
    pad_to(b, 16);
}

void pack_ifce(const ArmInts &a, bool fast, std::vector<unsigned char> &b) {
    const int n_in = a.dim, cf = a.n_out, cfp = (cf + 3) & ~3;
    if (fast) {
        for (int i = 0; i < n_in; i++)
            for (int o = 0; o < cfp; o++) put_i32(b, o < cf ? a.W[0][(size_t)i * cf + o] : 0);
        pad_to(b, 8);
    } else {
        for (size_t t = 0; t < (size_t)n_in * cf; t++) put_i64(b, a.W[0][t]);
    }
    for (int o = 0; o < cf; o++) put_i64(b, a.B[0][o]);
    pad_to(b, 16);
}

int next_pow2(int v) {
    int p = 1;
    while (p < v) p <<= 1;
    return p;
}

struct DeviceBuf {
    unsigned char *p = nullptr;
    size_t cap = 0;
};

struct PreparedJob {
    CcdJob *job = nullptr;
    const CcdCoolChicDesc *d = nullptr;
    NNLayout L;
    std::vector<int64_t> nn;
    std::vector<unsigned char> blob;
    EntStream es;
    bool fast = false;
    size_t smem = 0;
    int64_t n_sym = 0;
    int64_t lat_off_by_grid[CCD_MAX_GRIDS];
    bool pad_lat = false;   // latents owned by the library: every grid starts on a 16-byte boundary (TMA source)
    int64_t lat_bytes = 0;  // bytes of the latent buffer in that layout
    // batched float tail (run_tail_batched)
    bool tail = false;      // goes through the batched path
    int tail_nl = 0, tail_gl[CCD_MAX_GRIDS];
    int tail_cinp = 0, tail_C = 0;
    size_t off_tailP = 0, off_tailQ = 0, off_tailRaw = 0, off_rawtmp = 0;  // inside the synthesis scratch
    // device offsets inside the upload arena
    size_t off_words = 0, off_blob = 0, off_status = 0, off_syn = 0, off_lat = 0;
    size_t off_iv = 0;      // data-parallel encode: the symbols' intervals, inside the scratch
    int n_tiles = 0;        // data-parallel encode: tiles of k_enc_arm
    std::vector<float> syn_f;  // dequantised synthesis weights, packed
    size_t syn_off_ot_w = 0, syn_off_ot_b = 0, syn_off_st_w = 0, syn_off_st_b = 0;
    size_t syn_off_w[CCD_MAX_SYN], syn_off_b[CCD_MAX_SYN];
};

}  // namespace

struct CcdContext {
    int device = 0;
    float *d_scale = nullptr;
    uint32_t *d_cdf = nullptr;
    DeviceBuf upload;   // words / blobs / stream structs / statuses / synthesis weights
    DeviceBuf scratch;  // synthesis intermediates, latents when the caller does not want them
    unsigned char *h_pin = nullptr;
    size_t h_pin_cap = 0;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    float last_ms[4] = {0, 0, 0, 0};
    int32_t last_status[16] = {0};
    uint64_t last_upload_bytes = 0;
    uint32_t prod_mask = 0x3777u;  // warps 3, 7, 11 stay idle: the coder warp (15) owns its scheduler
    int n_sm = 148;
    int narrow_cta = 1;  // (CCD_NARROW_CTA=0 in the environment: always 16-warp CTAs)
    int fused_synthesis = 1;       // 0: layer-by-layer kernels (ccd_debug_set_fused_synthesis, tests compare both)
    // entropy launches of different ARM architectures (e.g. intra / residue / motion streams of a GOP) run
    // side by side on these streams: each launch only fills as many SMs as it has streams
    cudaStream_t aux[3] = {nullptr, nullptr, nullptr};
    cudaEvent_t ev_join[3] = {nullptr, nullptr, nullptr};
};

namespace {

// Entry points run on the context's device and put the caller's current device back on return (the host
// application -- PyTorch -- keeps its own notion of the current device).
struct DeviceGuard {
    int prev = -1;
    bool ok = false;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        ok = (prev == dev) || cudaSetDevice(dev) == cudaSuccess;
        if (prev == dev) prev = -1;  // nothing to restore
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

int ensure_dev(DeviceBuf &b, size_t bytes) {
    if (bytes <= b.cap) return CCD_OK;
    if (b.p) CUDA_TRY(cudaFree(b.p));
    b.p = nullptr;
    b.cap = 0;
    size_t want = bytes + bytes / 4 + (1 << 20);
    CUDA_TRY(cudaMalloc(&b.p, want));
    b.cap = want;
    return CCD_OK;
}

int ensure_pin(CcdContext *c, size_t bytes) {
    if (bytes <= c->h_pin_cap) return CCD_OK;
    if (c->h_pin) CUDA_TRY(cudaFreeHost(c->h_pin));
    c->h_pin = nullptr;
    c->h_pin_cap = 0;
    size_t want = bytes + bytes / 4 + (1 << 16);
    CUDA_TRY(cudaMallocHost(&c->h_pin, want));
    c->h_pin_cap = want;
    return CCD_OK;
}

inline size_t al(size_t v, size_t a = 256) { return (v + a - 1) / a * a; }

// Host preparation of one job: NN decode, ARM/IFCE packing, stream descriptor.
int prepare_job(PreparedJob &P, const int64_t *nn_ints_opt) {
    const CcdCoolChicDesc *d = P.d;
    int rc = nn_layout(d, &P.L);
    if (rc) return rc;
    const NNLayout &L = P.L;
    P.nn.resize((size_t)L.total);
    if (nn_ints_opt) {
        memcpy(P.nn.data(), nn_ints_opt, (size_t)L.total * 8);
    } else {
        int64_t n = decode_nn_host(d, L, P.job->nn_bytes, P.job->nn_nbytes, P.nn.data());
        if (n < 0) return (int)n;
    }
    const int64_t *nn = P.nn.data();
    // ---- latent layout (decode order: coarsest first)
    int64_t off = 0, nsym = 0;
    for (int g = d->n_grids - 1; g >= 0; g--) {
        if (P.pad_lat) off = (off + 15) & ~(int64_t)15;
        P.lat_off_by_grid[g] = off;
        off += (int64_t)d->grid_h[g] * d->grid_w[g];
        nsym += (int64_t)d->grid_h[g] * d->grid_w[g];
    }
    P.n_sym = nsym;
    P.lat_bytes = off;
    if (off >= ((int64_t)1 << 31)) return fail(CCD_ERR_UNSUPPORTED, "more than 2^31 latent symbols");
    // ---- ARM + IFCE integers
    const int dim = L.dim;
    std::vector<const int64_t *> qw, qb;
    for (int l = 0; l < L.n_arm_lin; l++) {
        qw.push_back(nn + L.arm_w[l]);
        qb.push_back(nn + L.arm_b[l]);
    }
    // component/coolchic.py:72-77
    ArmInts arm = build_arm(dim, d->arm_hidden, 2, qw.data(), qb.data(),
                            d->arm_stab ? nn + L.arm_w[L.n_arm_lin] : nullptr,
                            d->arm_stab ? nn + L.arm_b[L.n_arm_lin] : nullptr, d->qshift[0], d->qshift[1], true,
                            d->n_ifce_out, false);
    std::vector<ArmInts> ifce;
    i128 feat_bound = 0;
    bool fast = ccd_entropy_has_fast(d->n_ctx, d->n_ifce_out);
    for (int j = 0; j < L.n_ifce; j++) {
        const int64_t *w1[1] = {nn + L.ifce_w[j]};
        const int64_t *b1[1] = {nn + L.ifce_b[j]};
        // component/coolchic.py:114-123
        ifce.push_back(build_arm(d->grid_ifce_in[L.ifce_grid[j]], 0, d->n_ifce_out, w1, b1, nullptr, nullptr,
                                 d->qshift[2], d->qshift[3], false, 0, true));
        i128 bnd = 0;
        if (!ifce_bound(ifce.back(), &bnd)) fast = false;
        if (d->grid_ifce_in[L.ifce_grid[j]] > CCD_IFCE_FAST_MAX) fast = false;
        feat_bound = std::max(feat_bound, bnd);
    }
    if (fast) fast = arm_fits_int32(arm, d->n_ctx, feat_bound);
    P.fast = fast;
    P.blob.clear();
    pack_arm(arm, fast, P.blob);
    const int arm_bytes = (int)P.blob.size();

    EntStream &S = P.es;
    memset(&S, 0, sizeof(S));
    S.n_grids = d->n_grids;
    S.n_ctx = d->n_ctx;
    S.cf = d->flag_ifce ? d->n_ifce_out : 0;
    if (!d->flag_ifce && d->n_ifce_out != 0) return fail(CCD_ERR_ARG, "n_ifce_out without flag_ifce");
    S.n_hidden = d->arm_hidden;
    S.has_ifce = d->flag_ifce;
    S.arm_blob_bytes = arm_bytes;
    S.n_symbols = P.n_sym;
    int n_max = 1, rows_need = 8, ifce_max = 0;
    for (int gi = 0; gi < d->n_grids; gi++) {
        const int g = d->n_grids - 1 - gi;  // fine-first index
        EntGrid &G = S.grid[gi];
        G.h = d->grid_h[g];
        G.w = d->grid_w[g];
        G.raster = G.w <= 9;
        G.n_diag = G.raster ? G.h * G.w : G.w + CCD_MASK_STRIDE * (G.h - 1);
        G.lat_off = P.lat_off_by_grid[g];
        G.n_dec = gi;
        G.ifce_in = d->flag_ifce ? d->grid_ifce_in[g] : 0;
        G.ifce_blob_off = 0;
        G.ifce_blob_bytes = 0;
        if (G.ifce_in > 0) {
            int j = -1;
            for (int t = 0; t < L.n_ifce; t++)
                if (L.ifce_grid[t] == g) j = t;
            G.ifce_blob_off = (int)P.blob.size();
            pack_ifce(ifce[(size_t)j], fast, P.blob);
            G.ifce_blob_bytes = (int)P.blob.size() - G.ifce_blob_off;
            ifce_max = std::max(ifce_max, G.ifce_blob_bytes);
            // channel c <- grid g+1+c, nearest-upsampled to grid g+1's size
            // (core/upsampling.py:575-593: x2 + crop only when consecutive shapes differ)
            const int n_ch = G.ifce_in;
            int sh = 0;
            for (int c = 0; c < n_ch; c++) {
                if (gi == 0) {  // nothing decoded yet: a single all-zero channel (coolchic.py:95-96)
                    G.ch_sh[c] = -1;
                    G.ch_w[c] = 1;
                    G.ch_off[c] = 0;
                    continue;
                }
                const int gc = g + 1 + c;
                if (c > 0) {
                    const int ga = g + c;
                    if (d->grid_h[ga] != d->grid_h[gc] || d->grid_w[ga] != d->grid_w[gc]) sh++;
                }
                G.ch_sh[c] = sh;
                G.ch_w[c] = d->grid_w[gc];
                G.ch_off[c] = P.lat_off_by_grid[gc];
            }
        }
        const int nk = G.raster ? 1 : std::min(G.h, (G.w + CCD_MASK_STRIDE - 1) / CCD_MASK_STRIDE);
        n_max = std::max(n_max, nk);
        rows_need = std::max(rows_need, G.raster ? 8 : (G.w - 1) / CCD_MASK_STRIDE + 6);
    }
    S.ifce_blob_max = ifce_max;
    S.ring = std::min(1024, std::max(64, next_pow2(2 * n_max + 64)));  // 148 B of shared memory per slot
    S.rows = next_pow2(rows_need);
    P.smem = ccd_entropy_smem_bytes(S.ring, S.rows, S.arm_blob_bytes, S.ifce_blob_max);
    if (P.smem > 227 * 1024)
        return fail(CCD_ERR_UNSUPPORTED, "stream needs %zu bytes of shared memory (grid too wide)", P.smem);

    // ---- synthesis weights, dequantised (neuralnet.py:185-190: float32(int) * q_step)
    const float qs_w = ldexpf(1.0f, d->qshift[6]), qs_b = ldexpf(1.0f, d->qshift[7]);
    std::vector<float> &F = P.syn_f;
    F.clear();
    auto push = [&](int64_t off0, int64_t n, float qs) {
        size_t at = F.size();
        for (int64_t i = 0; i < n; i++) F.push_back((float)nn[off0 + i] * qs);
        while (F.size() % 4) F.push_back(0.0f);
        return at;
    };
    const int C = L.syn_c;
    P.syn_off_ot_w = push(L.syn_ot_w, (int64_t)C * C, qs_w);
    P.syn_off_ot_b = push(L.syn_ot_b, C, qs_b);
    if (d->syn_stab) {
        P.syn_off_st_w = push(L.syn_st_w, (int64_t)C * L.syn_stab_in, qs_w);
        P.syn_off_st_b = push(L.syn_st_b, C, qs_b);
    }
    int in_ft = d->syn_in;
    for (int l = 0; l < d->n_syn_layers; l++) {
        P.syn_off_w[l] = push(L.syn_w[l], (int64_t)d->syn_out[l] * in_ft * d->syn_k[l] * d->syn_k[l], qs_w);
        P.syn_off_b[l] = push(L.syn_b[l], d->syn_out[l], qs_b);
        if (d->syn_res[l] && d->syn_out[l] != in_ft) return fail(CCD_ERR_ARG, "residual layer %d changes width", l);
        in_ft = d->syn_out[l];
    }
    return CCD_OK;
}

// Device scratch of the float tail of one job.
struct SynScratch {
    size_t off_nxt = 0, off_a = 0, off_b = 0, off_stab = 0, off_noise_raw = 0, off_noise_a = 0, off_noise_b = 0, total = 0;
    std::vector<int> fused;  // layer l is evaluated together with l + 1 (two 1x1 layers)
};
SynScratch syn_scratch_plan(const CcdCoolChicDesc *d) {
    SynScratch S;
    int nl = 0, g0 = -1;
    for (int g = 0; g < d->n_grids; g++)
        if (!d->grid_is_hyper[g]) {
            if (g0 < 0) g0 = g;
            nl++;
        }
    S.fused.assign((size_t)std::max(d->n_syn_layers, 1), 0);
    if (g0 < 0 || d->n_syn_layers < 1) return S;
    const size_t plane = (size_t)d->grid_h[g0] * d->grid_w[g0];
    const int C = d->syn_out[d->n_syn_layers - 1];
    int maxc = std::max(d->syn_in, C);
    int in_ft = d->syn_in;
    for (int l = 0; l < d->n_syn_layers; l++) {
        const bool can = l + 1 < d->n_syn_layers && d->syn_k[l] == 1 && d->syn_k[l + 1] == 1 && !d->syn_res[l] &&
                         !d->syn_res[l + 1] && in_ft <= 16 && d->syn_out[l + 1] <= 8;
        if (can) {
            S.fused[(size_t)l] = 1;
            maxc = std::max(maxc, d->syn_out[l + 1]);
            in_ft = d->syn_out[l + 1];
            l++;
        } else {
            maxc = std::max(maxc, d->syn_out[l]);
            in_ft = d->syn_out[l];
        }
    }
    const size_t dense = al(plane * (size_t)(std::max(nl, d->syn_in) + 1) * 4);
    const size_t trunk = al(plane * (size_t)maxc * 4);
    size_t p = dense;
    S.off_nxt = p; p += dense;
    S.off_a = p; p += trunk;
    S.off_b = p; p += trunk;
    S.off_stab = p; p += al(plane * (size_t)C * 4);
    if (d->common_randomness) {
        S.off_noise_raw = p; p += al(plane * 2 * 4 + (size_t)nl * 64);  // sum of ceil(H/2^i) ceil(W/2^i) <= 2 plane
        S.off_noise_a = p; p += al(plane * (size_t)nl * 4);
        S.off_noise_b = p; p += al(plane * (size_t)nl * 4);
    }
    S.total = p;
    return S;
}

void expand_sym(const float *par, int k, float *full) {
    // _Parameterization_Symmetric_1d (core/upsampling.py:42-64): a b c d -> a b c d [d] c b a
    const int np = (k + 1) / 2;
    for (int i = 0; i < np; i++) full[i] = par[i];
    for (int i = 0; i < k - np; i++) full[np + i] = par[np - 1 - (k % 2) - i];
}

// Upsampling cascade + synthesis + final resize for one job (all kernels on `st`).
int run_synthesis(CcdContext *ctx, const PreparedJob &P, const int8_t *d_lat, const float *d_synw, float *d_out,
                  unsigned char *scratch, size_t scratch_bytes, cudaStream_t st) {
    const CcdCoolChicDesc *d = P.d;
    const NNLayout &L = P.L;
    const int cr = d->common_randomness != 0;
    int gl[CCD_MAX_GRIDS], nl = 0;
    for (int g = 0; g < d->n_grids; g++)
        if (!d->grid_is_hyper[g]) gl[nl++] = g;
    if (nl * (cr ? 2 : 1) != d->syn_in || nl < 1)
        return fail(CCD_ERR_ARG, "synthesis input width %d does not match %d latent grids", d->syn_in, nl);
    const int h0 = d->grid_h[gl[0]], w0 = d->grid_w[gl[0]];
    if (cr && (h0 != d->img_h || w0 != d->img_w || nl != d->latent_res_hi - d->latent_res_lo + 1))
        return fail(CCD_ERR_ARG, "common randomness needs a full-resolution finest latent grid");
    const size_t plane = (size_t)h0 * w0;
    const int C = L.syn_c;
    const SynScratch SS = syn_scratch_plan(d);
    if (SS.total > scratch_bytes) return fail(CCD_ERR_NOMEM, "internal: scratch too small (%zu > %zu)", SS.total, scratch_bytes);
    const std::vector<int> &fused = SS.fused;
    float *cur = reinterpret_cast<float *>(scratch);
    float *nxt = reinterpret_cast<float *>(scratch + SS.off_nxt);
    float *bufa = reinterpret_cast<float *>(scratch + SS.off_a);
    float *bufb = reinterpret_cast<float *>(scratch + SS.off_b);
    float *stab = reinterpret_cast<float *>(scratch + SS.off_stab);

    const float qs_uw = ldexpf(1.0f, d->qshift[4]);
    int gc = gl[nl - 1];
    int ch = d->grid_h[gc], cw = d->grid_w[gc], cc = 1;
    int rc;
    if ((rc = ccd_ups_first(d_lat + P.lat_off_by_grid[gc], ch, cw, cur, st))) return fail(CCD_ERR_CUDA, "ups_first launch");
    for (int idx = 0; idx < nl - 1; idx++) {
        const int gt = gl[nl - 2 - idx];
        const int th = d->grid_h[gt], tw = d->grid_w[gt];
        if (th > 2 * ch || tw > 2 * cw) return fail(CCD_ERR_ARG, "grid %d more than twice the size of its parent", gt);
        float par_t[8], par_c[8], full_t[16], full_c[16];
        const int kid = idx % d->n_ups;
        for (int i = 0; i < L.kt_par; i++) par_t[i] = (float)P.nn[(size_t)(L.ups_tw + (int64_t)kid * L.kt_par + i)] * qs_uw;
        for (int i = 0; i < L.kc_par; i++) par_c[i] = (float)P.nn[(size_t)(L.ups_cw + (int64_t)kid * L.kc_par + i)] * qs_uw;
        expand_sym(par_t, d->ups_k, full_t);
        expand_sym(par_c, d->ups_pre_k, full_c);
        if (ctx->fused_synthesis && d->ups_k == 8 && d->ups_pre_k == 7) {
            if ((rc = ccd_ups_level(d_lat + P.lat_off_by_grid[gt], th, tw, cur, cc, ch, cw, full_t, full_c, nxt, st)))
                return fail(CCD_ERR_CUDA, "ups_level launch");
        } else {
            if ((rc = ccd_ups_pre(d_lat + P.lat_off_by_grid[gt], th, tw, full_c, d->ups_pre_k, nxt, st)))
                return fail(CCD_ERR_CUDA, "ups_pre launch");
            if ((rc = ccd_ups_convt(cur, cc, ch, cw, full_t, d->ups_k, nxt + (size_t)th * tw, th, tw, st)))
                return fail(CCD_ERR_CUDA, "ups_convt launch");
        }
        std::swap(cur, nxt);
        ch = th;
        cw = tw;
        cc++;
    }
    if (cr) {
        // bitstream/component/coolchic.py:179-183: noise grids (noise.py) -> fixed_upsampling(bicubic)
        // (upsampling.py:556-595) -> channels nl .. 2 nl - 1 of the synthesis input
        float *raw = reinterpret_cast<float *>(scratch + SS.off_noise_raw);
        float *na = reinterpret_cast<float *>(scratch + SS.off_noise_a);
        float *nb = reinterpret_cast<float *>(scratch + SS.off_noise_b);
        int gh[CCD_MAX_GRIDS], gw[CCD_MAX_GRIDS];
        size_t goff[CCD_MAX_GRIDS], tot = 0;
        for (int i = 0; i < nl; i++) {
            const int sh = d->latent_res_lo + i;
            gh[i] = (int)((d->img_h + (1LL << sh) - 1) >> sh);
            gw[i] = (int)((d->img_w + (1LL << sh) - 1) >> sh);
            goff[i] = tot;
            tot += (size_t)gh[i] * gw[i];
        }
        if (ccd_cr_noise(raw, 0, tot, st)) return fail(CCD_ERR_CUDA, "noise launch");
        int nh = gh[nl - 1], nw = gw[nl - 1], nc = 1;
        const float *ncur = raw + goff[nl - 1];
        for (int i = nl - 2; i >= 0; i--) {
            const int th = gh[i], tw = gw[i];
            float *dstp = (i == 0) ? cur + plane * (size_t)nl : ((ncur == na) ? nb : na);
            if (th > 2 * nh || tw > 2 * nw) return fail(CCD_ERR_ARG, "noise grid %d more than twice its parent", i);
            if (cudaMemcpyAsync(dstp, raw + goff[i], (size_t)th * tw * 4, cudaMemcpyDeviceToDevice, st) != cudaSuccess)
                return fail(CCD_ERR_CUDA, "noise copy");
            if (th != nh || tw != nw) {
                if (ccd_resize_torch(ncur, nc, nh, nw, dstp + (size_t)th * tw, th, tw, 2, 0.5f, 0.5f, st))
                    return fail(CCD_ERR_CUDA, "noise upsampling launch");
            } else if (cudaMemcpyAsync(dstp + (size_t)th * tw, ncur, (size_t)nc * nh * nw * 4, cudaMemcpyDeviceToDevice,
                                       st) != cudaSuccess) {
                return fail(CCD_ERR_CUDA, "noise copy");
            }
            ncur = dstp;
            nh = th;
            nw = tw;
            nc++;
        }
        if (nl == 1 &&
            cudaMemcpyAsync(cur + plane, raw, plane * 4, cudaMemcpyDeviceToDevice, st) != cudaSuccess)
            return fail(CCD_ERR_CUDA, "noise copy");
        // gh[0] x gw[0] == image size here, so the final bicubic interpolate is the identity
    }
    // ---- synthesis (core/synthesis.py:272-294)
    auto layer = [&](int l, int cin) {
        SynLayerDev Ld;
        Ld.cin = cin;
        Ld.cout = d->syn_out[l];
        Ld.k = d->syn_k[l];
        Ld.residual = d->syn_res[l];
        Ld.relu = d->syn_relu[l];
        Ld.w = d_synw + P.syn_off_w[l];
        Ld.b = d_synw + P.syn_off_b[l];
        return Ld;
    };
    const bool same = (h0 == d->img_h && w0 == d->img_w);
    SynLayerDev Lo{C, C, 1, 0, 0, d_synw + P.syn_off_ot_w, d_synw + P.syn_off_ot_b};
    bool fused_done = false;
    if (ctx->fused_synthesis) {
        // one kernel for the whole synthesis when the architecture is in the fused family
        SynLayerDev Ls{L.syn_stab_in, C, 1, 0, 0, d_synw + P.syn_off_st_w, d_synw + P.syn_off_st_b};
        SynLayerDev all[CCD_MAX_SYN];
        int in_ft0 = d->syn_in;
        for (int l = 0; l < d->n_syn_layers; l++) {
            all[l] = layer(l, in_ft0);
            in_ft0 = d->syn_out[l];
        }
        rc = ccd_syn_fused(cur, h0, w0, d->syn_in, all, d->n_syn_layers, d->syn_stab ? &Ls : nullptr, Lo,
                           same ? d_out : bufa, st);
        if (rc > 0) return fail(CCD_ERR_CUDA, "fused synthesis launch");
        fused_done = (rc == 0);
    }
    float *ot_dst = same ? d_out : bufa;
    if (!fused_done) {
    if (d->syn_stab) {
        SynLayerDev Ls{L.syn_stab_in, C, 1, 0, 0, d_synw + P.syn_off_st_w, d_synw + P.syn_off_st_b};
        if ((rc = ccd_syn_layer(cur, h0, w0, Ls, stab, st))) return fail(CCD_ERR_CUDA, "stabiliser launch");
    }
    const float *src = cur;
    float *dst = bufa, *other = bufb;
    int in_ft = d->syn_in;
    for (int l = 0; l < d->n_syn_layers; l++) {
        if (fused[(size_t)l]) {
            SynLayerDev L0 = layer(l, in_ft), L1 = layer(l + 1, d->syn_out[l]);
            if ((rc = ccd_syn_pointwise2(src, h0, w0, L0, L1, dst, st))) return fail(CCD_ERR_CUDA, "pointwise launch");
            in_ft = d->syn_out[l + 1];
            l++;
        } else {
            SynLayerDev L0 = layer(l, in_ft);
            if ((rc = ccd_syn_layer(src, h0, w0, L0, dst, st))) return fail(CCD_ERR_CUDA, "synthesis layer launch");
            in_ft = d->syn_out[l];
        }
        src = dst;
        std::swap(dst, other);
    }
    float *trunk = const_cast<float *>(src);
    if (trunk == cur) return fail(CCD_ERR_ARG, "synthesis without layers");
    if (d->syn_stab)
        if ((rc = ccd_syn_add(trunk, stab, plane * (size_t)C, st))) return fail(CCD_ERR_CUDA, "add launch");
    ot_dst = same ? d_out : dst;
    if ((rc = ccd_syn_layer(trunk, h0, w0, Lo, ot_dst, st))) return fail(CCD_ERR_CUDA, "output transform launch");
    }
    if (!same) {
        // final F.interpolate (component/coolchic.py:187-192)
        if (d->final_ups == 0)
            rc = ccd_resize_nearest(ot_dst, C, h0, w0, d_out, d->img_h, d->img_w, st);
        else
            rc = ccd_resize_torch(ot_dst, C, h0, w0, d_out, d->img_h, d->img_w, d->final_ups == 1 ? 1 : 2,
                                  (float)h0 / (float)d->img_h, (float)w0 / (float)d->img_w, st);
        if (rc) return fail(CCD_ERR_CUDA, "resize launch");
    }
    (void)ctx;
    return CCD_OK;
}

size_t synthesis_scratch_bytes(const CcdCoolChicDesc *d) { return syn_scratch_plan(d).total + 4096; }

// ---- batched float tail ------------------------------------------------------------------------------------
// A job takes the batched path when its upsampling uses the default kernel sizes (8 / 7), it has at least two
// latent grids, no common randomness, and its synthesis is in the fused family.  All such jobs of a call share
//   * one launch per cascade level (all but the last), and
//   * one launch (per (cinp, C) pair) of the kernel that evaluates the last level, the synthesis and -- for I
//     frames that ask for it -- the frame tail.
bool tail_eligible(const CcdCoolChicDesc *d, const NNLayout &L, PreparedJob &P) {
    if (d->ups_k != 8 || d->ups_pre_k != 7 || d->common_randomness) return false;
    int nl = 0;
    for (int g = 0; g < d->n_grids; g++)
        if (!d->grid_is_hyper[g]) P.tail_gl[nl++] = g;
    if (nl < 2 || nl > 16 || nl != d->syn_in) return false;
    const int nlay = d->n_syn_layers;
    if (nlay < 2 || nlay > 4) return false;
    const int C = d->syn_out[1];
    if (d->syn_k[0] != 1 || d->syn_k[1] != 1 || d->syn_res[0] || d->syn_res[1] || d->syn_out[0] > 256 || C < 2 || C > 5) return false;
    if (L.syn_c != C) return false;
    for (int l = 2; l < nlay; l++)
        if (d->syn_k[l] != 3 || d->syn_out[l] != C) return false;
    if (d->syn_stab && L.syn_stab_in > nl) return false;
    for (int i = 0; i + 1 < nl; i++) {
        const int gt = P.tail_gl[i], gc = P.tail_gl[i + 1];
        if (d->grid_h[gt] > 2 * d->grid_h[gc] || d->grid_w[gt] > 2 * d->grid_w[gc]) return false;  // (reported by the generic path)
    }
    P.tail_nl = nl;
    P.tail_cinp = nl <= 4 ? 4 : (nl <= 8 ? 8 : 16);
    P.tail_C = C;
    return true;
}

struct TailScratch {
    size_t p = 0, q = 0, raw = 0, total = 0;
};
TailScratch tail_scratch_plan(const CcdCoolChicDesc *d, const PreparedJob &P) {
    TailScratch T;
    const int nl = P.tail_nl;
    size_t o = 0;
    if (nl >= 3) {
        const int g1 = P.tail_gl[1];
        T.p = o;
        o += al((size_t)(nl - 1) * d->grid_h[g1] * d->grid_w[g1] * 4);
    }
    if (nl >= 4) {
        const int g2 = P.tail_gl[2];
        T.q = o;
        o += al((size_t)(nl - 2) * d->grid_h[g2] * d->grid_w[g2] * 4);
    }
    const int g0 = P.tail_gl[0];
    if (d->grid_h[g0] != d->img_h || d->grid_w[g0] != d->img_w) {
        T.raw = o;
        o += al((size_t)P.tail_C * d->grid_h[g0] * d->grid_w[g0] * 4);
    }
    T.total = o;
    return T;
}

}  // namespace

// =========================================================================================
extern "C" {

int ccd_version(void) { return CCD_VERSION; }
int ccd_sizeof_desc(void) { return (int)sizeof(CcdCoolChicDesc); }
const char *ccd_last_error(const CcdContext *) { return g_err.c_str(); }

int ccd_create(int device_ordinal, CcdContext **out) {
    if (!out) return fail(CCD_ERR_ARG, "null out pointer");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(CCD_ERR_NO_DEVICE, "no CUDA device available (%s): libccdec has no CPU fallback",
                    e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    if (device_ordinal < 0 || device_ordinal >= n) return fail(CCD_ERR_ARG, "device %d out of range [0,%d)", device_ordinal, n);
    CUDA_TRY(cudaSetDevice(device_ordinal));
    CcdContext *c = new CcdContext();
    c->device = device_ordinal;
    {
        int nsm = 0;
        if (cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, device_ordinal) == cudaSuccess && nsm > 0) c->n_sm = nsm;
        const char *env = getenv("CCD_NARROW_CTA");
        if (env && env[0] == '0') c->narrow_cta = 0;
    }
    int rc = CCD_OK;
    do {
        if (cudaMalloc(&c->d_scale, CCD_N_SCALE * 4) != cudaSuccess ||
            cudaMalloc(&c->d_cdf, (size_t)CCD_N_SCALE * 256 * CCD_WIN * 4) != cudaSuccess) {
            rc = fail(CCD_ERR_NOMEM, "cudaMalloc of the cumulative table failed");
            break;
        }
        if (cudaMemcpy(c->d_scale, k_scale_bits, CCD_N_SCALE * 4, cudaMemcpyHostToDevice) != cudaSuccess) {
            rc = fail(CCD_ERR_CUDA, "scale table upload failed");
            break;
        }
        if (ccd_cdf_table_build(c->d_cdf, c->d_scale, 0) != 0 || cudaDeviceSynchronize() != cudaSuccess) {
            rc = fail(CCD_ERR_CUDA, "cumulative table kernel failed: %s", cudaGetErrorString(cudaGetLastError()));
            break;
        }
        for (int i = 0; i < 4; i++)
            if (cudaEventCreate(&c->ev[i]) != cudaSuccess) rc = fail(CCD_ERR_CUDA, "event creation failed");
    } while (0);
    if (rc) {
        ccd_destroy(c);
        return rc;
    }
    *out = c;
    return CCD_OK;
}

void ccd_destroy(CcdContext *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->d_scale) cudaFree(c->d_scale);
    if (c->d_cdf) cudaFree(c->d_cdf);
    if (c->upload.p) cudaFree(c->upload.p);
    if (c->scratch.p) cudaFree(c->scratch.p);
    if (c->h_pin) cudaFreeHost(c->h_pin);
    for (int i = 0; i < 4; i++)
        if (c->ev[i]) cudaEventDestroy(c->ev[i]);
    for (int i = 0; i < 3; i++) {
        if (c->aux[i]) cudaStreamDestroy(c->aux[i]);
        if (c->ev_join[i]) cudaEventDestroy(c->ev_join[i]);
    }
    delete c;
}

int64_t ccd_nn_count(const CcdCoolChicDesc *desc) {
    NNLayout L;
    int rc = nn_layout(desc, &L);
    return rc ? rc : L.total;
}

int64_t ccd_latent_count(const CcdCoolChicDesc *d, int64_t offsets_by_grid[CCD_MAX_GRIDS]) {
    int rc = validate_desc(d);
    if (rc) return rc;
    int64_t off = 0;
    for (int g = d->n_grids - 1; g >= 0; g--) {
        if (offsets_by_grid) offsets_by_grid[g] = off;
        off += (int64_t)d->grid_h[g] * d->grid_w[g];
    }
    return off;
}

int64_t ccd_decode_nn(const CcdCoolChicDesc *desc, const uint8_t *nn_bytes, size_t nn_nbytes, int64_t *out_ints,
                      size_t cap) {
    NNLayout L;
    int rc = nn_layout(desc, &L);
    if (rc) return rc;
    if (!nn_bytes || !out_ints || (size_t)L.total > cap) return fail(CCD_ERR_ARG, "bad buffer");
    return decode_nn_host(desc, L, nn_bytes, nn_nbytes, out_ints);
}

// stages: bit 0 entropy, bit 1 synthesis.  mode: 0 decode, 1 / 2 the wavefront encoder (ccd_encode_latents), 3 the
// data-parallel encoder of the latents in d_lat_in (ccd_encode_many; synthesis only for the jobs with a d_out).
// out_caps (optional): per-job capacity of d_out_words, else out_cap for every job.
static int decode_impl_body(CcdContext *ctx, CcdJob *jobs, int n_jobs, const int64_t *const *nn_ints, int stages,
                            const int8_t *const *d_lat_in, int mode, uint64_t seed, uint32_t *const *d_out_words,
                            int64_t out_cap, const int64_t *out_caps, int32_t (*statuses)[16], cudaStream_t st);

static int decode_impl(CcdContext *ctx, CcdJob *jobs, int n_jobs, const int64_t *const *nn_ints, int stages,
                       const int8_t *const *d_lat_in, int mode, uint64_t seed, uint32_t *const *d_out_words,
                       int64_t out_cap, const int64_t *out_caps, int32_t (*statuses)[16], void *cuda_stream) {
    if (!ctx) return fail(CCD_ERR_ARG, "null context");
    if (n_jobs < 0 || (n_jobs > 0 && !jobs)) return fail(CCD_ERR_ARG, "bad job list");
    if (n_jobs == 0) return CCD_OK;
    if ((stages & 2) && mode != 3)
        for (int i = 0; i < n_jobs; i++)
            if (!jobs[i].d_out) return fail(CCD_ERR_ARG, "job %d: null output pointer", i);
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(CCD_ERR_CUDA, "cudaSetDevice(%d) failed", ctx->device);
    cudaStream_t st = (cudaStream_t)cuda_stream;
    const int rc =
        decode_impl_body(ctx, jobs, n_jobs, nn_ints, stages, d_lat_in, mode, seed, d_out_words, out_cap, out_caps, statuses, st);
    if (rc != CCD_OK) {
        // every exit path leaves the context quiescent: the pinned staging buffer, the upload arena and the scratch
        // may be reused (or re-allocated) by the next call
        const std::string keep = g_err;
        cudaStreamSynchronize(st);
        for (int a = 0; a < 3; a++)
            if (ctx->aux[a]) cudaStreamSynchronize(ctx->aux[a]);
        cudaGetLastError();
        g_err = keep;
    }
    return rc;
}

static int decode_impl_body(CcdContext *ctx, CcdJob *jobs, int n_jobs, const int64_t *const *nn_ints, int stages,
                            const int8_t *const *d_lat_in, int mode, uint64_t seed, uint32_t *const *d_out_words,
                            int64_t out_cap, const int64_t *out_caps, int32_t (*statuses)[16], cudaStream_t st) {
    CUDA_TRY(cudaEventRecord(ctx->ev[0], st));

    std::vector<PreparedJob> P((size_t)n_jobs);
    size_t up = 0, scratch_syn = 0, scratch_lat = 0, scratch_tail = 0, scratch_iv = 0;
    size_t n_tail = 0, n_tail_levels = 0, n_enc_tiles = 0;
    for (int i = 0; i < n_jobs; i++) {
        P[(size_t)i].job = &jobs[i];
        P[(size_t)i].d = jobs[i].desc;
        jobs[i].status = CCD_OK;
        const bool own_lat = !(jobs[i].d_latents || (d_lat_in && d_lat_in[i]));
        P[(size_t)i].pad_lat = own_lat && mode == 0;
        int rc = prepare_job(P[(size_t)i], nn_ints ? nn_ints[i] : nullptr);
        if (rc) {
            jobs[i].status = rc;
            return rc;
        }
        PreparedJob &J = P[(size_t)i];
        if ((stages & 1) && mode == 0 && (!jobs[i].latent_bytes && jobs[i].latent_nbytes))
            return fail(CCD_ERR_ARG, "job %d: null latent bytes", i);
        const size_t nwords = (stages & 1) && mode == 0 ? jobs[i].latent_nbytes / 4 : 0;
        J.off_words = up;
        up += al(nwords * 4 + 16);
        J.off_blob = up;
        up += al(J.blob.size());
        J.off_status = up;
        up += al(64);
        J.off_syn = up;
        up += al(J.syn_f.size() * 4);
        if (mode == 3) {
            J.off_iv = scratch_iv;
            scratch_iv += al((size_t)J.n_sym * 8);
            const int chunk = J.fast ? CCD_ENC_CHUNK_FAST : CCD_ENC_CHUNK_GENERIC;
            for (int g = 0; g < J.d->n_grids; g++) {
                const int64_t n_chunks = (int64_t)J.d->grid_h[g] * ((J.d->grid_w[g] + chunk - 1) / chunk);
                J.n_tiles += (int)((n_chunks + CCD_ENC_TILE_CHUNKS - 1) / CCD_ENC_TILE_CHUNKS);
            }
            n_enc_tiles += (size_t)J.n_tiles;
        }
        if ((stages & 2) && jobs[i].d_out) {
            if (jobs[i].finish_bitdepth != 0) {
                if (jobs[i].finish_bitdepth < 1 || jobs[i].finish_bitdepth > 16 || jobs[i].finish_type < 0 || jobs[i].finish_type > 3)
                    return fail(CCD_ERR_ARG, "job %d: bad frame tail request (bitdepth %d, type %d)", i, jobs[i].finish_bitdepth, jobs[i].finish_type);
                if (J.L.syn_c != 3) return fail(CCD_ERR_ARG, "job %d: the frame tail needs a 3-channel output, found %d", i, J.L.syn_c);
                if (jobs[i].finish_type == 1 && (!jobs[i].d_out_u || !jobs[i].d_out_v))
                    return fail(CCD_ERR_ARG, "job %d: yuv420 frame tail needs u and v outputs", i);
            }
            J.tail = ctx->fused_synthesis && tail_eligible(J.d, J.L, J);
            if (J.tail) {
                const TailScratch T = tail_scratch_plan(J.d, J);
                J.off_tailP = scratch_tail + T.p;
                J.off_tailQ = scratch_tail + T.q;
                J.off_tailRaw = scratch_tail + T.raw;
                scratch_tail += al(T.total);
                n_tail++;
                n_tail_levels += (size_t)(J.tail_nl - 2);
            } else {
                size_t need = synthesis_scratch_bytes(J.d);
                if (jobs[i].finish_bitdepth != 0) {  // raw output first, then the frame tail kernel
                    J.off_rawtmp = al(need);
                    need = J.off_rawtmp + al((size_t)3 * J.d->img_h * J.d->img_w * 4);
                }
                scratch_syn = std::max(scratch_syn, need);
            }
        }
        J.off_lat = scratch_lat;
        if (own_lat) scratch_lat += al((size_t)J.lat_bytes);
    }
    // device-resident job arrays of the batched float tail (filled below, uploaded with everything else)
    const size_t off_tail_syn = up;
    up += al(n_tail * ccd_tail_job_bytes());
    const size_t off_tail_lvl = up;
    up += al(n_tail_levels * ccd_tail_level_job_bytes());
    const size_t off_streams = up;
    up += al(sizeof(EntStream) * (size_t)n_jobs);
    const size_t off_enc_tiles = up;
    up += al(sizeof(EncTile) * n_enc_tiles);
    int rc;
    if ((rc = ensure_pin(ctx, up))) return rc;
    if ((rc = ensure_dev(ctx->upload, up))) return rc;
    if ((rc = ensure_dev(ctx->scratch, scratch_lat + al(scratch_syn) + scratch_tail + scratch_iv + 4096))) return rc;
    unsigned char *h = ctx->h_pin, *dv = ctx->upload.p;
    unsigned char *d_scr_syn = ctx->scratch.p + scratch_lat;
    unsigned char *d_scr_tail = d_scr_syn + al(scratch_syn);
    unsigned char *d_scr_iv = d_scr_tail + scratch_tail;

    // group jobs by kernel configuration so that each group is one launch
    std::vector<int> order((size_t)n_jobs);
    for (int i = 0; i < n_jobs; i++) order[(size_t)i] = i;
    auto key = [&](int i) {
        const PreparedJob &J = P[(size_t)i];
        return J.fast ? (J.d->n_ctx * 64 + J.d->n_ifce_out) : -1;
    };
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return key(a) < key(b); });

    std::vector<int8_t *> d_lat((size_t)n_jobs);
    for (int i = 0; i < n_jobs; i++) {
        PreparedJob &J = P[(size_t)i];
        const size_t nbytes4 = (stages & 1) && mode == 0 ? jobs[i].latent_nbytes / 4 * 4 : 0;
        memset(h + J.off_words, 0, al(nbytes4 + 16));
        if (nbytes4) memcpy(h + J.off_words, jobs[i].latent_bytes, nbytes4);
        memcpy(h + J.off_blob, J.blob.data(), J.blob.size());
        memset(h + J.off_status, 0, 64);
        if (!J.syn_f.empty()) memcpy(h + J.off_syn, J.syn_f.data(), J.syn_f.size() * 4);
        int8_t *lat = jobs[i].d_latents;
        if (!lat && d_lat_in && d_lat_in[i]) lat = const_cast<int8_t *>(d_lat_in[i]);
        if (!lat) lat = reinterpret_cast<int8_t *>(ctx->scratch.p + J.off_lat);
        d_lat[(size_t)i] = lat;
        EntStream &S = J.es;
        S.mode = mode;
        S.prod_mask = ctx->prod_mask;
        S.seed = seed + (uint64_t)i;
        S.words = reinterpret_cast<const uint32_t *>(dv + J.off_words);
        S.n_words = (int64_t)(nbytes4 / 4);
        S.latents = lat;
        S.blob = dv + J.off_blob;
        S.status = reinterpret_cast<int32_t *>(dv + J.off_status);
        S.out_words = d_out_words ? d_out_words[i] : nullptr;
        S.out_cap = d_out_words ? (out_caps ? out_caps[i] : out_cap) : 0;
        if (mode == 3) {
            S.words = reinterpret_cast<const uint32_t *>(d_scr_iv + J.off_iv);
            S.n_words = 2 * J.n_sym;
        }
    }
    for (int t = 0; t < n_jobs; t++)
        memcpy(h + off_streams + sizeof(EntStream) * (size_t)t, &P[(size_t)order[(size_t)t]].es, sizeof(EntStream));
    // data-parallel encode: the tiles of k_enc_arm, launch group after launch group (stream index = position in the
    // sorted EntStream array)
    std::vector<size_t> enc_group_tile0;
    if (mode == 3) {
        EncTile *tiles = reinterpret_cast<EncTile *>(h + off_enc_tiles);
        size_t nt = 0;
        for (int t = 0; t < n_jobs; t++) {
            if (t == 0 || key(order[(size_t)t]) != key(order[(size_t)t - 1])) enc_group_tile0.push_back(nt);
            const PreparedJob &J = P[(size_t)order[(size_t)t]];
            const int chunk = J.fast ? CCD_ENC_CHUNK_FAST : CCD_ENC_CHUNK_GENERIC;
            for (int gi = 0; gi < J.es.n_grids; gi++) {
                const EntGrid &Gg = J.es.grid[gi];
                const int n_chunks = Gg.h * ((Gg.w + chunk - 1) / chunk);
                for (int c0 = 0; c0 < n_chunks; c0 += CCD_ENC_TILE_CHUNKS)
                    tiles[nt++] = EncTile{t, gi, c0, std::min(CCD_ENC_TILE_CHUNKS, n_chunks - c0)};
            }
        }
        enc_group_tile0.push_back(nt);
    }

    // ---- batched float tail: job arrays.  Launch groups: cascade level `idx` of every stream that has one
    // (planes = idx + 2), then one launch per (cinp, C) pair for the last level + synthesis (+ frame tail).
    struct TailGroup { int cinp, C, n3_max, hid_max, max_w, max_h, first, count; };
    std::vector<TailGroup> tail_groups;
    struct TailLevelLaunch { size_t first; int count, planes, max_tw, max_th; };
    std::vector<TailLevelLaunch> tail_levels;
    std::vector<int> tail_order;  // jobs of the batched path, sorted by (cinp, C)
    if (n_tail) {
        for (int i = 0; i < n_jobs; i++)
            if (P[(size_t)i].tail) tail_order.push_back(i);
        std::stable_sort(tail_order.begin(), tail_order.end(), [&](int a, int b) {
            const PreparedJob &A = P[(size_t)a], &B = P[(size_t)b];
            return A.tail_cinp * 8 + A.tail_C < B.tail_cinp * 8 + B.tail_C;
        });
        const size_t jb = ccd_tail_job_bytes(), lb = ccd_tail_level_job_bytes();
        // cascade levels
        int max_levels = 0;
        for (int i : tail_order) max_levels = std::max(max_levels, P[(size_t)i].tail_nl - 2);
        size_t lvl_at = 0;
        for (int idx = 0; idx < max_levels; idx++) {
            TailLevelLaunch LL{lvl_at, 0, idx + 2, 0, 0};
            for (int i : tail_order) {
                const PreparedJob &J = P[(size_t)i];
                const CcdCoolChicDesc *d = J.d;
                const int nl = J.tail_nl;
                if (idx >= nl - 2) continue;
                const int gt = J.tail_gl[nl - 2 - idx], gc = J.tail_gl[nl - 1 - idx];
                float par_t[8], par_c[8], full_t[16], full_c[16];
                const float qs_uw = ldexpf(1.0f, d->qshift[4]);
                const int kid = idx % d->n_ups;
                for (int t = 0; t < J.L.kt_par; t++) par_t[t] = (float)J.nn[(size_t)(J.L.ups_tw + (int64_t)kid * J.L.kt_par + t)] * qs_uw;
                for (int t = 0; t < J.L.kc_par; t++) par_c[t] = (float)J.nn[(size_t)(J.L.ups_cw + (int64_t)kid * J.L.kc_par + t)] * qs_uw;
                expand_sym(par_t, d->ups_k, full_t);
                expand_sym(par_c, d->ups_pre_k, full_c);
                // level idx writes P when (nl - 3 - idx) is even (the last one, idx = nl - 3, always writes P)
                const bool to_p = ((nl - 3 - idx) & 1) == 0;
                float *out = reinterpret_cast<float *>(d_scr_tail + (to_p ? J.off_tailP : J.off_tailQ));
                const float *in = reinterpret_cast<const float *>(d_scr_tail + (to_p ? J.off_tailQ : J.off_tailP));
                const int8_t *in8 = idx == 0 ? d_lat[(size_t)i] + J.lat_off_by_grid[gc] : nullptr;
                ccd_tail_fill_level(h + off_tail_lvl + (lvl_at + (size_t)LL.count) * lb, d_lat[(size_t)i] + J.lat_off_by_grid[gt],
                                    idx == 0 ? nullptr : in, in8, out, idx + 1, d->grid_h[gc], d->grid_w[gc], d->grid_h[gt],
                                    d->grid_w[gt], full_t, full_c);
                LL.count++;
                LL.max_tw = std::max(LL.max_tw, d->grid_w[gt]);
                LL.max_th = std::max(LL.max_th, d->grid_h[gt]);
            }
            lvl_at += (size_t)LL.count;
            if (LL.count) tail_levels.push_back(LL);
        }
        // last level + synthesis
        const float *d_synw_base = reinterpret_cast<const float *>(dv);
        for (size_t t = 0; t < tail_order.size(); t++) {
            const int i = tail_order[t];
            PreparedJob &J = P[(size_t)i];
            const CcdCoolChicDesc *d = J.d;
            const NNLayout &L = J.L;
            const int nl = J.tail_nl, g0 = J.tail_gl[0], g1 = J.tail_gl[1];
            const float *d_synw = reinterpret_cast<const float *>(dv + J.off_syn);
            (void)d_synw_base;
            SynLayerDev all[CCD_MAX_SYN];
            int in_ft = d->syn_in;
            for (int l = 0; l < d->n_syn_layers; l++) {
                all[l] = SynLayerDev{in_ft, d->syn_out[l], d->syn_k[l], d->syn_res[l], d->syn_relu[l], d_synw + J.syn_off_w[l],
                                     d_synw + J.syn_off_b[l]};
                in_ft = d->syn_out[l];
            }
            const int C = J.tail_C;
            SynLayerDev Ls{L.syn_stab_in, C, 1, 0, 0, d_synw + J.syn_off_st_w, d_synw + J.syn_off_st_b};
            CcdTailSynDesc T;
            memset(&T, 0, sizeof(T));
            T.lat = d_lat[(size_t)i] + J.lat_off_by_grid[g0];
            if (nl == 2) T.stk8 = d_lat[(size_t)i] + J.lat_off_by_grid[g1];
            else T.stk = reinterpret_cast<const float *>(d_scr_tail + J.off_tailP);
            T.h = d->grid_h[g0]; T.w = d->grid_w[g0]; T.ch = d->grid_h[g1]; T.cw = d->grid_w[g1]; T.cin = nl;
            T.layers = all; T.n_layers = d->n_syn_layers; T.stab = d->syn_stab ? &Ls : nullptr;
            T.ot = SynLayerDev{C, C, 1, 0, 0, d_synw + J.syn_off_ot_w, d_synw + J.syn_off_ot_b};
            const bool same = (T.h == d->img_h && T.w == d->img_w);
            const size_t plane = (size_t)T.h * T.w;
            const CcdJob &job = jobs[i];
            if (!same) {
                float *raw = reinterpret_cast<float *>(d_scr_tail + J.off_tailRaw);
                for (int c = 0; c < C; c++) T.out[c] = raw + (size_t)c * plane;
            } else if (job.finish_bitdepth != 0 && job.finish_type == 1) {
                T.out[0] = job.d_out; T.out[1] = job.d_out_u; T.out[2] = job.d_out_v;
                T.finish = 2;
            } else {
                for (int c = 0; c < C; c++) T.out[c] = job.d_out + (size_t)c * plane;
                T.finish = job.finish_bitdepth != 0 ? 1 : 0;
            }
            T.M = job.finish_bitdepth != 0 ? (float)((1 << job.finish_bitdepth) - 1) : 0.0f;
            float par_t[8], par_c[8], full_t[16], full_c[16];
            const float qs_uw = ldexpf(1.0f, d->qshift[4]);
            const int kid = (nl - 2) % d->n_ups;
            for (int k = 0; k < L.kt_par; k++) par_t[k] = (float)J.nn[(size_t)(L.ups_tw + (int64_t)kid * L.kt_par + k)] * qs_uw;
            for (int k = 0; k < L.kc_par; k++) par_c[k] = (float)J.nn[(size_t)(L.ups_cw + (int64_t)kid * L.kc_par + k)] * qs_uw;
            expand_sym(par_t, d->ups_k, full_t);
            expand_sym(par_c, d->ups_pre_k, full_c);
            T.wt1d = full_t; T.wc1d = full_c;
            T.allow_tma = J.pad_lat ? 1 : 0;
            const int tr = ccd_tail_fill_syn(h + off_tail_syn + t * jb, T);
            if (tr < 0) return fail(CCD_ERR_ARG, "internal: job %d is not in the fused synthesis family", i);
            if (tail_groups.empty() || tail_groups.back().cinp != J.tail_cinp || tail_groups.back().C != C)
                tail_groups.push_back(TailGroup{J.tail_cinp, C, 0, 0, 0, 0, (int)t, 0});
            TailGroup &G = tail_groups.back();
            G.count++;
            G.n3_max = std::max(G.n3_max, d->n_syn_layers - 2);
            G.hid_max = std::max(G.hid_max, d->syn_out[0]);
            G.max_w = std::max(G.max_w, T.w);
            G.max_h = std::max(G.max_h, T.h);
        }
    }
    CUDA_TRY(cudaMemcpyAsync(dv, h, up, cudaMemcpyHostToDevice, st));
    ctx->last_upload_bytes = up;
    CUDA_TRY(cudaEventRecord(ctx->ev[1], st));

    if ((stages & 1) && mode == 3) {
        // one data-parallel ARM pass per launch group, then the range coder of every job in one launch
        int t = 0, g = 0;
        while (t < n_jobs) {
            int u = t;
            size_t smem = 0;
            while (u < n_jobs && key(order[(size_t)u]) == key(order[(size_t)t])) {
                const PreparedJob &J = P[(size_t)order[(size_t)u]];
                smem = std::max(smem, ccd_encode_smem_bytes(J.es.arm_blob_bytes, J.es.ifce_blob_max));
                u++;
            }
            const PreparedJob &J0 = P[(size_t)order[(size_t)t]];
            EntLaunchCfg cfg{J0.d->n_ctx, J0.d->flag_ifce ? J0.d->n_ifce_out : 0, J0.fast, smem, CCD_ENC_THREADS};
            const size_t t0 = enc_group_tile0[(size_t)g], t1 = enc_group_tile0[(size_t)g + 1];
            const int e = ccd_enc_arm_launch(reinterpret_cast<const EntStream *>(dv + off_streams),
                                             reinterpret_cast<const EncTile *>(dv + off_enc_tiles) + t0, (int)(t1 - t0), cfg,
                                             ctx->d_cdf, ctx->d_scale, st);
            if (e != 0) return fail(CCD_ERR_CUDA, "encoder ARM launch failed: %s", cudaGetErrorString((cudaError_t)e));
            t = u;
            g++;
        }
        const int e = ccd_enc_range_launch(reinterpret_cast<const EntStream *>(dv + off_streams), n_jobs, st);
        if (e != 0) return fail(CCD_ERR_CUDA, "range encoder launch failed: %s", cudaGetErrorString((cudaError_t)e));
    } else if (stages & 1) {
        int t = 0, g = 0;
        while (t < n_jobs) {
            int u = t;
            size_t smem = 0;
            while (u < n_jobs && key(order[(size_t)u]) == key(order[(size_t)t])) {
                smem = std::max(smem, P[(size_t)order[(size_t)u]].smem);
                u++;
            }
            const PreparedJob &J0 = P[(size_t)order[(size_t)t]];
            // more streams than SMs: 8-warp CTAs, two per SM (registers: 2 x 256 x 128; shared memory permitting)
            const bool narrow = mode == 0 && ctx->narrow_cta != 0 && (u - t) > ctx->n_sm &&
                                2 * (smem + 1024) <= (size_t)227 * 1024;
            EntLaunchCfg cfg{J0.d->n_ctx, J0.d->flag_ifce ? J0.d->n_ifce_out : 0, J0.fast, smem,
                             narrow ? CCD_ENT_THREADS_NARROW : CCD_ENT_THREADS};
            // group 0 on the caller's stream, the next ones on auxiliary streams forked after the upload
            cudaStream_t sg = st;
            if (g > 0) {
                const int a = (g - 1) % 3;
                if (!ctx->aux[a]) {
                    CUDA_TRY(cudaStreamCreateWithFlags(&ctx->aux[a], cudaStreamNonBlocking));
                    CUDA_TRY(cudaEventCreateWithFlags(&ctx->ev_join[a], cudaEventDisableTiming));
                }
                sg = ctx->aux[a];
                CUDA_TRY(cudaStreamWaitEvent(sg, ctx->ev[1], 0));  // the upload (recorded on st before any launch)
            }
            int e = ccd_entropy_launch(reinterpret_cast<const EntStream *>(dv + off_streams) + t, u - t, cfg, ctx->d_cdf,
                                       ctx->d_scale, sg);
            if (e != 0) return fail(CCD_ERR_CUDA, "entropy kernel launch failed: %s", cudaGetErrorString((cudaError_t)e));
            if (g > 0) {
                const int a = (g - 1) % 3;
                CUDA_TRY(cudaEventRecord(ctx->ev_join[a], sg));
                CUDA_TRY(cudaStreamWaitEvent(st, ctx->ev_join[a], 0));
            }
            t = u;
            g++;
        }
    }
    CUDA_TRY(cudaEventRecord(ctx->ev[2], st));
    if (stages & 2) {
        // batched path: all cascade levels, then the fused last level + synthesis (+ frame tail)
        const size_t jb = ccd_tail_job_bytes(), lb = ccd_tail_level_job_bytes();
        for (const TailLevelLaunch &LL : tail_levels)
            if (ccd_tail_launch_level(dv + off_tail_lvl + LL.first * lb, LL.count, LL.planes, LL.max_tw, LL.max_th, st))
                return fail(CCD_ERR_CUDA, "cascade level launch failed");
        for (const TailGroup &G : tail_groups) {
            const int e = ccd_tail_launch_syn(dv + off_tail_syn + (size_t)G.first * jb, G.count, G.cinp, G.C, G.n3_max, G.hid_max,
                                              G.max_w, G.max_h, st);
            if (e != 0) return fail(CCD_ERR_CUDA, "fused tail launch failed (%d)", e);
        }
        for (int i : tail_order) {
            // grids smaller than the image (motion fields): final F.interpolate (component/coolchic.py:187-192)
            const PreparedJob &J = P[(size_t)i];
            const CcdCoolChicDesc *d = J.d;
            const int g0 = J.tail_gl[0], h0 = d->grid_h[g0], w0 = d->grid_w[g0];
            if (h0 == d->img_h && w0 == d->img_w) continue;
            const float *raw = reinterpret_cast<const float *>(d_scr_tail + J.off_tailRaw);
            float *dst = jobs[i].d_out;
            unsigned char *tmp = nullptr;
            if (jobs[i].finish_bitdepth != 0) return fail(CCD_ERR_UNSUPPORTED, "job %d: frame tail on a resized output", i);
            (void)tmp;
            if (d->final_ups == 0)
                rc = ccd_resize_nearest(raw, J.tail_C, h0, w0, dst, d->img_h, d->img_w, st);
            else
                rc = ccd_resize_torch(raw, J.tail_C, h0, w0, dst, d->img_h, d->img_w, d->final_ups == 1 ? 1 : 2,
                                      (float)h0 / (float)d->img_h, (float)w0 / (float)d->img_w, st);
            if (rc) return fail(CCD_ERR_CUDA, "resize launch");
        }
        // everything else: one stream after the other through the general kernels
        for (int i = 0; i < n_jobs; i++) {
            if (P[(size_t)i].tail || !jobs[i].d_out) continue;
            const bool fin = jobs[i].finish_bitdepth != 0;
            float *raw_dst = fin ? reinterpret_cast<float *>(d_scr_syn + P[(size_t)i].off_rawtmp) : jobs[i].d_out;
            rc = run_synthesis(ctx, P[(size_t)i], d_lat[(size_t)i], reinterpret_cast<const float *>(dv + P[(size_t)i].off_syn),
                               raw_dst, d_scr_syn, scratch_syn, st);
            if (rc) {
                jobs[i].status = rc;
                return rc;
            }
            if (fin) {
                const int ft = jobs[i].finish_type == 3 ? 2 : jobs[i].finish_type;
                if (ccd_finish(raw_dst, P[(size_t)i].d->img_h, P[(size_t)i].d->img_w, jobs[i].finish_bitdepth, ft, jobs[i].d_out,
                               jobs[i].d_out_u, jobs[i].d_out_v, st))
                    return fail(CCD_ERR_CUDA, "finish_frame launch failed");
            }
        }
    }
    CUDA_TRY(cudaEventRecord(ctx->ev[3], st));
    // statuses back
    for (int i = 0; i < n_jobs; i++)
        CUDA_TRY(cudaMemcpyAsync(h + P[(size_t)i].off_status, dv + P[(size_t)i].off_status, 64, cudaMemcpyDeviceToHost, st));
    cudaError_t se = cudaStreamSynchronize(st);
    if (se != cudaSuccess) return fail(CCD_ERR_CUDA, "kernel execution failed: %s", cudaGetErrorString(se));
    cudaEventElapsedTime(&ctx->last_ms[2], ctx->ev[0], ctx->ev[1]);
    cudaEventElapsedTime(&ctx->last_ms[0], ctx->ev[1], ctx->ev[2]);
    cudaEventElapsedTime(&ctx->last_ms[1], ctx->ev[2], ctx->ev[3]);
    int first = CCD_OK;
    for (int i = 0; i < n_jobs; i++) {
        const int32_t *s = reinterpret_cast<const int32_t *>(h + P[(size_t)i].off_status);
        if (statuses) memcpy(statuses[i], s, 64);
        memcpy(ctx->last_status, s, 64);
        if ((stages & 1) && s[0] != 0) {
            jobs[i].status = s[0];
            if (!first)
                first = mode == 3 ? fail(s[0], "job %d: latent value outside [-64, 63]", i)
                                  : fail(s[0], "job %d: corrupt latent payload (range decoder desynchronised)", i);
        }
    }
    return first;
}

int ccd_decode_many(CcdContext *ctx, CcdJob *jobs, int n_jobs, void *cuda_stream) {
    return decode_impl(ctx, jobs, n_jobs, nullptr, 3, nullptr, 0, 0, nullptr, 0, nullptr, nullptr, cuda_stream);
}

int ccd_decode_coolchic(CcdContext *ctx, const CcdCoolChicDesc *desc, const uint8_t *nn_bytes, size_t nn_nbytes,
                        const uint8_t *latent_bytes, size_t latent_nbytes, float *d_out, int8_t *d_latents,
                        void *cuda_stream) {
    CcdJob j{desc, nn_bytes, nn_nbytes, latent_bytes, latent_nbytes, d_out, d_latents, 0, 0, 0, nullptr, nullptr};
    return ccd_decode_many(ctx, &j, 1, cuda_stream);
}

int ccd_decode_latents(CcdContext *ctx, const CcdCoolChicDesc *desc, const int64_t *nn_ints, const uint8_t *latent_bytes,
                       size_t latent_nbytes, int8_t *d_latents, void *cuda_stream) {
    if (!d_latents || !nn_ints) return fail(CCD_ERR_ARG, "null pointer");
    CcdJob j{desc, nullptr, 0, latent_bytes, latent_nbytes, nullptr, d_latents, 0, 0, 0, nullptr, nullptr};
    const int64_t *nn[1] = {nn_ints};
    return decode_impl(ctx, &j, 1, nn, 1, nullptr, 0, 0, nullptr, 0, nullptr, nullptr, cuda_stream);
}

int ccd_synthesize(CcdContext *ctx, const CcdCoolChicDesc *desc, const int64_t *nn_ints, const int8_t *d_latents,
                   float *d_out, void *cuda_stream) {
    if (!d_latents || !nn_ints || !d_out) return fail(CCD_ERR_ARG, "null pointer");
    CcdJob j{desc, nullptr, 0, nullptr, 0, d_out, nullptr, 0, 0, 0, nullptr, nullptr};
    const int64_t *nn[1] = {nn_ints};
    const int8_t *lat[1] = {d_latents};
    return decode_impl(ctx, &j, 1, nn, 2, lat, 0, 0, nullptr, 0, nullptr, nullptr, cuda_stream);
}

int ccd_encode_latents(CcdContext *ctx, const CcdCoolChicDesc *desc, const int64_t *nn_ints, int mode, uint64_t seed,
                       int8_t *d_latents, uint32_t *d_out_words, int64_t out_cap_words, int64_t *n_words_out,
                       int32_t *slow_out, void *cuda_stream) {
    if (!d_latents || !nn_ints || !d_out_words || (mode != 1 && mode != 2)) return fail(CCD_ERR_ARG, "bad argument");
    CcdJob j{desc, nullptr, 0, nullptr, 0, nullptr, d_latents, 0, 0, 0, nullptr, nullptr};
    const int64_t *nn[1] = {nn_ints};
    uint32_t *ow[1] = {d_out_words};
    int32_t stt[1][16];
    int rc = decode_impl(ctx, &j, 1, nn, 1, nullptr, mode, seed, ow, out_cap_words, nullptr, stt, cuda_stream);
    if (rc) return rc;
    if (n_words_out) *n_words_out = stt[0][3];
    if (slow_out) *slow_out = stt[0][2];
    if (stt[0][3] > out_cap_words) return fail(CCD_ERR_ARG, "output buffer too small (%d words needed)", stt[0][3]);
    return CCD_OK;
}

int ccd_encode_many(CcdContext *ctx, CcdEncodeJob *jobs, int n_jobs, void *cuda_stream) {
    if (!ctx) return fail(CCD_ERR_ARG, "null context");
    if (n_jobs < 0 || (n_jobs > 0 && !jobs)) return fail(CCD_ERR_ARG, "bad job list");
    std::vector<CcdJob> J((size_t)n_jobs);
    std::vector<const int8_t *> lat((size_t)n_jobs);
    std::vector<uint32_t *> ow((size_t)n_jobs);
    std::vector<int64_t> caps((size_t)n_jobs);
    std::vector<int32_t> stt((size_t)n_jobs * 16, 0);
    bool any_out = false;
    for (int i = 0; i < n_jobs; i++) {
        CcdEncodeJob &e = jobs[i];
        e.n_words = 0;
        e.status = CCD_OK;
        e.slow = 0;
        if (!e.d_latents || !e.d_words || e.cap_words < 1 || (!e.nn_bytes && e.nn_nbytes))
            return fail(CCD_ERR_ARG, "job %d: null latents / output words or capacity < 1", i);
        J[(size_t)i] = CcdJob{e.desc, e.nn_bytes, e.nn_nbytes, nullptr, 0, e.d_out, nullptr, 0, 0, 0, nullptr, nullptr};
        lat[(size_t)i] = e.d_latents;
        ow[(size_t)i] = e.d_words;
        caps[(size_t)i] = e.cap_words;
        any_out = any_out || e.d_out;
    }
    const int rc = decode_impl(ctx, J.data(), n_jobs, nullptr, any_out ? 3 : 1, lat.data(), 3, 0, ow.data(), 0, caps.data(),
                               reinterpret_cast<int32_t(*)[16]>(stt.data()), cuda_stream);
    for (int i = 0; i < n_jobs; i++) {
        jobs[i].status = J[(size_t)i].status;
        jobs[i].n_words = stt[(size_t)i * 16 + 3];
        jobs[i].slow = stt[(size_t)i * 16 + 2];
    }
    if (rc) return rc;
    for (int i = 0; i < n_jobs; i++)
        if (jobs[i].n_words > jobs[i].cap_words) {
            jobs[i].status = CCD_ERR_ARG;
            return fail(CCD_ERR_ARG, "job %d: output buffer too small (%lld words needed, capacity %lld)", i,
                        (long long)jobs[i].n_words, (long long)jobs[i].cap_words);
        }
    return CCD_OK;
}

int ccd_finish_frame(CcdContext *ctx, const float *d_in, int h, int w, int bitdepth, int data_type, float *d_out_a,
                     float *d_out_b, float *d_out_c, void *cuda_stream) {
    if (!ctx || !d_in || !d_out_a || h < 1 || w < 1 || bitdepth < 8 || bitdepth > 16 || data_type < 0 || data_type > 2)
        return fail(CCD_ERR_ARG, "bad argument");
    if (data_type == 1 && (!d_out_b || !d_out_c)) return fail(CCD_ERR_ARG, "yuv420 needs u and v outputs");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(CCD_ERR_CUDA, "cudaSetDevice failed");
    if (ccd_finish(d_in, h, w, bitdepth, data_type, d_out_a, d_out_b, d_out_c, (cudaStream_t)cuda_stream))
        return fail(CCD_ERR_CUDA, "finish_frame launch failed");
    return CCD_OK;
}

namespace {
int inter_common(CcdContext *ctx, InterLaunch &L, int n_res_ch, int n_mot_ch, void *cuda_stream) {
    if (!ctx || !L.residue || !L.motion || !L.ref0[0] || !L.ref0[1] || !L.ref0[2] || !L.out[0] || !L.out[1] || !L.out[2] ||
        L.h < 1 || L.w < 1)
        return fail(CCD_ERR_ARG, "bad argument");
    if (L.is_b && (!L.ref1[0] || !L.ref1[1] || !L.ref1[2])) return fail(CCD_ERR_ARG, "B frame without a second reference");
    // decode.py:171-189 reads residue channels 0..3 (P) / 0..4 (B) and motion channels 0..1 (P) / 0..3 (B)
    if (n_res_ch != (L.is_b ? 5 : 4))
        return fail(CCD_ERR_ARG, "%s-frame residue has %d channels, expected %d", L.is_b ? "B" : "P", n_res_ch, L.is_b ? 5 : 4);
    if (n_mot_ch != (L.is_b ? 4 : 2))
        return fail(CCD_ERR_ARG, "%s-frame motion has %d channels, expected %d", L.is_b ? "B" : "P", n_mot_ch, L.is_b ? 4 : 2);
    if ((L.ref_cs || L.out_420) && ((L.h | L.w) & 1)) return fail(CCD_ERR_ARG, "4:2:0 needs even frame sizes, got %dx%d", L.h, L.w);
    if (L.filter_size < 2 || (L.filter_size & 1)) return fail(CCD_ERR_ARG, "bad warp filter size %d", L.filter_size);
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(CCD_ERR_CUDA, "cudaSetDevice failed");
    if (!L.is_b) L.gf[2] = L.gf[3] = 0;
    int rc = ccd_inter_launch(L, (cudaStream_t)cuda_stream);
    if (rc == -1)
        return fail(CCD_ERR_UNSUPPORTED, "warp filter size %d is not supported (2, 4: frames of at least 2x2; 6 .. 14)", L.filter_size);
    if (rc) return fail(CCD_ERR_CUDA, "inter_predict launch failed: %s", cudaGetErrorString((cudaError_t)rc));
    return CCD_OK;
}
}  // namespace

int ccd_inter_predict(CcdContext *ctx, const float *d_residue, int n_res_ch, const float *d_motion, int n_mot_ch,
                      const float *d_ref0, const float *d_ref1, int h, int w, int is_b, const int32_t *global_flow,
                      int warp_filter_size, float *d_out, void *cuda_stream) {
    if (!global_flow || !d_ref0 || !d_out) return fail(CCD_ERR_ARG, "bad argument");
    const size_t plane = (size_t)h * w;
    InterLaunch L{};
    L.residue = d_residue;
    L.motion = d_motion;
    for (int c = 0; c < 3; c++) {
        L.ref0[c] = d_ref0 + c * plane;
        L.ref1[c] = d_ref1 ? d_ref1 + c * plane : nullptr;
        L.out[c] = d_out + c * plane;
    }
    L.h = h; L.w = w; L.is_b = is_b;
    for (int i = 0; i < 4; i++) L.gf[i] = (i < 2 || is_b) ? global_flow[i] : 0;
    L.filter_size = warp_filter_size;
    return inter_common(ctx, L, n_res_ch, n_mot_ch, cuda_stream);
}

int ccd_reconstruct_frame(CcdContext *ctx, const float *d_residue, int n_res_ch, const float *d_motion, int n_mot_ch,
                          const float *const ref0_planes[3], const float *const ref1_planes[3], int frame_data_type,
                          int bitdepth, int h, int w, int is_b, const int32_t *global_flow, int warp_filter_size,
                          float *const out_planes[3], void *cuda_stream) {
    if (!global_flow || !ref0_planes || !out_planes) return fail(CCD_ERR_ARG, "bad argument");
    if (bitdepth < 1 || bitdepth > 16) return fail(CCD_ERR_ARG, "bad bitdepth %d", bitdepth);
    if (frame_data_type < 0 || frame_data_type > 3) return fail(CCD_ERR_ARG, "bad frame_data_type %d", frame_data_type);
    InterLaunch L{};
    L.residue = d_residue;
    L.motion = d_motion;
    for (int c = 0; c < 3; c++) {
        L.ref0[c] = ref0_planes[c];
        L.ref1[c] = (is_b && ref1_planes) ? ref1_planes[c] : nullptr;
        L.out[c] = out_planes[c];
    }
    L.ref_cs = L.out_420 = (frame_data_type == 1);
    L.h = h; L.w = w; L.is_b = is_b;
    for (int i = 0; i < 4; i++) L.gf[i] = (i < 2 || is_b) ? global_flow[i] : 0;
    L.filter_size = warp_filter_size;
    L.M = (float)((1 << bitdepth) - 1);
    return inter_common(ctx, L, n_res_ch, n_mot_ch, cuda_stream);
}

int ccd_pack_frame(CcdContext *ctx, const float *const planes[3], int h, int w, int chroma_shift, int bitdepth,
                   int sample_bytes, int interleaved, void *d_out, void *cuda_stream) {
    if (!ctx || !planes || !planes[0] || !planes[1] || !planes[2] || !d_out || h < 1 || w < 1) return fail(CCD_ERR_ARG, "bad argument");
    if (bitdepth < 1 || bitdepth > 16 || (sample_bytes != 1 && sample_bytes != 2) || (sample_bytes == 1 && bitdepth > 8))
        return fail(CCD_ERR_ARG, "bitdepth %d does not fit %d-byte samples", bitdepth, sample_bytes);
    if (chroma_shift < 0 || chroma_shift > 1 || (interleaved && chroma_shift)) return fail(CCD_ERR_ARG, "bad layout");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(CCD_ERR_CUDA, "cudaSetDevice failed");
    if (ccd_pack(planes, h, w, chroma_shift, bitdepth, sample_bytes, interleaved, d_out, (cudaStream_t)cuda_stream))
        return fail(CCD_ERR_CUDA, "pack_frame launch failed");
    return CCD_OK;
}

int ccd_pack_samples(CcdContext *ctx, const float *d_samples, size_t n, int bitdepth, int sample_bytes, void *d_out,
                     void *cuda_stream) {
    if (!ctx || !d_samples || !d_out || n == 0) return fail(CCD_ERR_ARG, "bad argument");
    if (bitdepth < 1 || bitdepth > 16 || (sample_bytes != 1 && sample_bytes != 2) || (sample_bytes == 1 && bitdepth > 8))
        return fail(CCD_ERR_ARG, "bitdepth %d does not fit %d-byte samples", bitdepth, sample_bytes);
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(CCD_ERR_CUDA, "cudaSetDevice failed");
    if (ccd_pack_flat(d_samples, n, bitdepth, sample_bytes, d_out, (cudaStream_t)cuda_stream))
        return fail(CCD_ERR_CUDA, "pack_samples launch failed");
    return CCD_OK;
}

int ccd_debug_laplace_domain(CcdContext *ctx, int sc_lo, int sc_hi, uint32_t *out_lo, uint32_t *out_hi) {
    if (!ctx || sc_lo < 0 || sc_hi > CCD_N_SCALE || sc_lo >= sc_hi || !out_lo || !out_hi) return fail(CCD_ERR_ARG, "bad argument");
    DeviceGuard guard(ctx->device);
    if (!guard.ok) return fail(CCD_ERR_CUDA, "cudaSetDevice failed");
    const size_t n = (size_t)(sc_hi - sc_lo) * 32641;
    int rc;
    if ((rc = ensure_dev(ctx->scratch, n * 8))) return rc;
    uint32_t *lo = reinterpret_cast<uint32_t *>(ctx->scratch.p), *hi = lo + n;
    if (ccd_laplace_domain(ctx->d_scale, sc_lo, sc_hi, lo, hi, 0)) return fail(CCD_ERR_CUDA, "launch failed");
    CUDA_TRY(cudaMemcpy(out_lo, lo, n * 4, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(out_hi, hi, n * 4, cudaMemcpyDeviceToHost));
    return CCD_OK;
}

uint64_t ccd_debug_launch_count(void) { return g_ccd_launches; }

int ccd_debug_set_fused_synthesis(CcdContext *ctx, int on) {
    if (!ctx) return fail(CCD_ERR_ARG, "null context");
    ctx->fused_synthesis = on ? 1 : 0;
    return CCD_OK;
}

int ccd_debug_set_producer_mask(CcdContext *ctx, uint32_t mask) {
    if (!ctx || (mask & 0x3fffu) == 0) return fail(CCD_ERR_ARG, "bad producer mask");
    ctx->prod_mask = mask & 0x3fffu;
    return CCD_OK;
}

int ccd_debug_last_status(const CcdContext *ctx, int32_t st[16]) {
    if (!ctx || !st) return fail(CCD_ERR_ARG, "null pointer");
    memcpy(st, ctx->last_status, 64);
    return CCD_OK;
}

int ccd_last_timing(const CcdContext *ctx, float ms[4]) {
    if (!ctx || !ms) return fail(CCD_ERR_ARG, "null pointer");
    memcpy(ms, ctx->last_ms, sizeof(float) * 4);
    ms[3] = (float)ctx->last_upload_bytes;
    return CCD_OK;
}

}  // extern "C"
