// Context, weight packing and the forward sequences of the TTS tail + the C-ABI (include/infernos_b200.h).
//
// Reference call sites this file stands in for:
//   HelloSippyTTSRT/HelloSippyRTPipe.py:155-189  (engine construction: vocoder, chunker, resampler)
//   HelloSippyTTSRT/HelloSippyRTPipe.py:231-240  (window builder -> vocoder -> chunker -> re-assembly -> resample)
//   Core/Codecs/G711.py:25-32                    (encode)
#include "common.cuh"
#include "ctx.cuh"
#include "conv_simt.cuh"
#include "conv_umma.cuh"
#include "gemm_tc.cuh"
#include "../../include/infernos_b200.h"

#include <stdarg.h>
#include <string.h>
#include <algorithm>
#include <mutex>

namespace b2 {

thread_local std::string g_last_error;
std::atomic<uint64_t> g_launches{0};

int set_error(const char *fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_last_error = buf;
    return 1;
}

bool pdl_enabled() {
    static const bool on = !(getenv("B2_PDL") && atoi(getenv("B2_PDL")) == 0);
    return on;
}

int sm_count() {
    static int cached[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (dev < 64 && cached[dev]) return cached[dev];
    int n = 148;
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (dev < 64) cached[dev] = n;
    return n;
}

int launch_resample_2to1(const float *d_in, size_t rows, size_t L, int law, uint8_t *d_u8, float *d_f32, cudaStream_t st);

static const int RES_K[3] = {3, 7, 11};
static const int RES_D[3] = {1, 3, 5};
static const int STAGE_C[4] = {256, 128, 64, 32};

template <typename T>
static int dev_alloc(b2_ctx *c, T **p, size_t n) {
    void *q = nullptr;
    size_t bytes = std::max<size_t>(n * sizeof(T), 16);
    cudaError_t e = cudaMalloc(&q, bytes);
    if (e != cudaSuccess) return set_error("cudaMalloc of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
    c->allocs.push_back(q);
    c->device_bytes += bytes;
    *p = reinterpret_cast<T *>(q);
    return 0;
}

static int upload(b2_ctx *c, float **dst, const std::vector<float> &v) {
    if (dev_alloc(c, dst, v.size())) return 1;
    B2_CUDA_OK(cudaMemcpy(*dst, v.data(), v.size() * sizeof(float), cudaMemcpyHostToDevice));
    return 0;
}

static int upload_bf16(b2_ctx *c, __nv_bfloat16 **dst, const std::vector<float> &v) {
    std::vector<__nv_bfloat16> h(v.size());
    for (size_t i = 0; i < v.size(); i++) h[i] = __float2bfloat16_rn(v[i]);
    if (dev_alloc(c, dst, h.size())) return 1;
    B2_CUDA_OK(cudaMemcpy(*dst, h.data(), h.size() * sizeof(__nv_bfloat16), cudaMemcpyHostToDevice));
    return 0;
}

static const HostTensor *find(const std::map<std::string, HostTensor> &m, const std::string &k, std::initializer_list<int64_t> shape) {
    auto it = m.find(k);
    if (it == m.end()) { set_error("weight '%s' was not loaded", k.c_str()); return nullptr; }
    if (it->second.shape != std::vector<int64_t>(shape)) {
        std::string got;
        for (auto s : it->second.shape) got += std::to_string(s) + ",";
        set_error("weight '%s' has shape (%s), expected a different one", k.c_str(), got.c_str());
        return nullptr;
    }
    return &it->second;
}

// torch Conv1d weight [Cout][Cin][k] -> [k][Cin][Cout] fp32 and (optionally) [k][Cout][Cin] bf16
static int pack_conv(b2_ctx *c, Layer &l, const HostTensor &w, const HostTensor &b, int dil, int pad, int stride, bool want_bf16) {
    const int Cout = (int)w.shape[0], Cin = (int)w.shape[1], k = (int)w.shape[2];
    l.Cin = Cin; l.Cout = Cout; l.taps = k; l.dil = dil; l.pad = pad; l.stride = stride;
    std::vector<float> p((size_t)k * Cin * Cout);
    for (int co = 0; co < Cout; co++)
        for (int ci = 0; ci < Cin; ci++)
            for (int j = 0; j < k; j++) p[((size_t)j * Cin + ci) * Cout + co] = w.data[((size_t)co * Cin + ci) * k + j];
    if (upload(c, &l.w32, p)) return 1;
    if (upload(c, &l.bias, b.data)) return 1;
    if (want_bf16) {
        std::vector<float> q((size_t)k * Cout * Cin);
        for (int co = 0; co < Cout; co++)
            for (int ci = 0; ci < Cin; ci++)
                for (int j = 0; j < k; j++) q[((size_t)j * Cout + co) * Cin + ci] = w.data[((size_t)co * Cin + ci) * k + j];
        if (upload_bf16(c, &l.wbf, q)) return 1;
        if (umma_prepare_layer(l)) return 1;
    }
    return 0;
}

// torch ConvTranspose1d(k8, s4, p2) weight [Cin][Cout][8] -> a 3-tap stride-1 conv over the INPUT grid with 4*Cout
// output channels: column ph*Cout + co of output row t is output time 4t + ph.  out[4t+ph] takes
//   x[t]   * w[ph+2]          (tap 1)
//   x[t-1] * w[ph+6], ph < 2  (tap 0)
//   x[t+1] * w[ph-2], ph >= 2 (tap 2)
static int pack_convT(b2_ctx *c, Layer &l, const HostTensor &w, const HostTensor &b, bool want_bf16) {
    const int Cin = (int)w.shape[0], Cout = (int)w.shape[1];
    const int N = 4 * Cout;
    l.Cin = Cin; l.Cout = N; l.taps = 3; l.dil = 1; l.pad = 1; l.stride = 1;
    std::vector<float> p((size_t)3 * Cin * N, 0.0f), q;
    if (want_bf16) q.assign((size_t)3 * N * Cin, 0.0f);
    for (int ci = 0; ci < Cin; ci++)
        for (int co = 0; co < Cout; co++)
            for (int ph = 0; ph < 4; ph++)
                for (int tap = 0; tap < 3; tap++) {
                    int k = (tap == 1) ? ph + 2 : (tap == 0 ? ph + 6 : ph - 2);
                    if (k < 0 || k > 7) continue;
                    float v = w.data[((size_t)ci * Cout + co) * 8 + k];
                    p[((size_t)tap * Cin + ci) * N + ph * Cout + co] = v;
                    if (want_bf16) q[((size_t)tap * N + ph * Cout + co) * Cin + ci] = v;
                }
    std::vector<float> bb((size_t)N);
    for (int ph = 0; ph < 4; ph++)
        for (int co = 0; co < Cout; co++) bb[ph * Cout + co] = b.data[co];
    l.h_bias = bb;
    if (upload(c, &l.w32, p)) return 1;
    if (upload(c, &l.bias, bb)) return 1;
    if (want_bf16) {
        if (upload_bf16(c, &l.wbf, q)) return 1;
        if (umma_prepare_layer(l)) return 1;
    }
    return 0;
}

static int load_tensor(std::map<std::string, HostTensor> &m, const char *key, const float *h, const int64_t *shape, int ndim) {
    if (!key || !h || !shape || ndim < 1 || ndim > 4) return set_error("load tensor: bad arguments");
    HostTensor t;
    size_t n = 1;
    for (int i = 0; i < ndim; i++) { t.shape.push_back(shape[i]); n *= (size_t)shape[i]; }
    t.data.assign(h, h + n);
    m[key] = std::move(t);
    return 0;
}

static int finalize(b2_ctx *c) {
    const bool bf = c->mode == B2_MODE_BF16;
    if (bf && umma_init()) return 1;
    char k1[96], k2[96];
    const HostTensor *w, *b;
    if (!(w = find(c->voc_raw, "mean", {80}))) return 1;
    if (upload(c, &c->mean, w->data)) return 1;
    if (!(w = find(c->voc_raw, "scale", {80}))) return 1;
    if (upload(c, &c->scale, w->data)) return 1;
    if (!(w = find(c->voc_raw, "conv_pre.weight", {512, 80, 7})) || !(b = find(c->voc_raw, "conv_pre.bias", {512}))) return 1;
    if (!bf) {
        if (pack_conv(c, c->conv_pre, *w, *b, 1, 3, 1, false)) return 1;
    } else {
        // tensor-core conv_pre: K padded from 80 to 128 mel bins (zeros) so that it is two 64-wide K blocks
        HostTensor wp;
        wp.shape = {512, 128, 7};
        wp.data.assign((size_t)512 * 128 * 7, 0.0f);
        for (int co = 0; co < 512; co++)
            for (int ci = 0; ci < 80; ci++)
                for (int j = 0; j < 7; j++) wp.data[((size_t)co * 128 + ci) * 7 + j] = w->data[((size_t)co * 80 + ci) * 7 + j];
        if (pack_conv(c, c->conv_pre, wp, *b, 1, 3, 1, true)) return 1;
    }
    int cin = 512;
    for (int i = 0; i < 4; i++) {
        const int C = STAGE_C[i];
        snprintf(k1, sizeof k1, "upsampler.%d.weight", i);
        snprintf(k2, sizeof k2, "upsampler.%d.bias", i);
        if (!(w = find(c->voc_raw, k1, {cin, C, 8})) || !(b = find(c->voc_raw, k2, {C}))) return 1;
        if (pack_convT(c, c->up[i], *w, *b, bf)) return 1;
        for (int j = 0; j < 3; j++)
            for (int d = 0; d < 3; d++) {
                const int k = RES_K[j], dil = RES_D[d];
                snprintf(k1, sizeof k1, "resblocks.%d.convs1.%d.weight", i * 3 + j, d);
                snprintf(k2, sizeof k2, "resblocks.%d.convs1.%d.bias", i * 3 + j, d);
                if (!(w = find(c->voc_raw, k1, {C, C, k})) || !(b = find(c->voc_raw, k2, {C}))) return 1;
                if (pack_conv(c, c->res1[i][j][d], *w, *b, dil, (k * dil - dil) / 2, 1, bf)) return 1;
                snprintf(k1, sizeof k1, "resblocks.%d.convs2.%d.weight", i * 3 + j, d);
                snprintf(k2, sizeof k2, "resblocks.%d.convs2.%d.bias", i * 3 + j, d);
                if (!(w = find(c->voc_raw, k1, {C, C, k})) || !(b = find(c->voc_raw, k2, {C}))) return 1;
                if (pack_conv(c, c->res2[i][j][d], *w, *b, 1, (k - 1) / 2, 1, bf)) return 1;
            }
        if (bf) {
            for (int j = 0; j < 3; j++) {
                if (!resblock_supported(C, RES_K[j])) continue;
                const Layer *l1[3] = {&c->res1[i][j][0], &c->res1[i][j][1], &c->res1[i][j][2]};
                const Layer *l2[3] = {&c->res2[i][j][0], &c->res2[i][j][1], &c->res2[i][j][2]};
                if (resblock_pack(l1, l2, c->rb[i][j], c->allocs, c->device_bytes)) return 1;
            }
        }
        cin = C;
    }
    if (!(w = find(c->voc_raw, "conv_post.weight", {1, 32, 7})) || !(b = find(c->voc_raw, "conv_post.bias", {1}))) return 1;
    {
        std::vector<float> p(7 * 32);
        for (int ci = 0; ci < 32; ci++)
            for (int j = 0; j < 7; j++) p[j * 32 + ci] = w->data[ci * 7 + j];
        if (upload(c, &c->post_w, p) || upload(c, &c->post_b, b->data)) return 1;
    }
    // chunker (optional: a context without chunker weights serves the vocoder/codec entry points only)
    if (!c->chk_raw.empty()) {
        Layer tmp;
        if (!(w = find(c->chk_raw, "conv_pre_m.weight", {32, 80, 3})) || !(b = find(c->chk_raw, "conv_pre_m.bias", {32}))) return 1;
        if (pack_conv(c, tmp, *w, *b, 1, 1, 1, false)) return 1;
        c->cwm = tmp.w32; c->cbm = tmp.bias;
        if (!(w = find(c->chk_raw, "conv_pre_a.weight", {160, 256, 3})) || !(b = find(c->chk_raw, "conv_pre_a.bias", {160}))) return 1;
        if (pack_conv(c, tmp, *w, *b, 1, 1, 1, false)) return 1;
        c->cwa = tmp.w32; c->cba = tmp.bias;
        if (!(w = find(c->chk_raw, "upsampler.0.weight", {192, 128, 8})) || !(b = find(c->chk_raw, "upsampler.0.bias", {128}))) return 1;
        if (bf) {
            // the prologue's output is padded from 192 to 256 channels (one N = 256 tile), so the first upsampler takes 256 input channels
            HostTensor wp;
            wp.shape = {256, 128, 8};
            wp.data.assign((size_t)256 * 128 * 8, 0.0f);
            std::copy(w->data.begin(), w->data.end(), wp.data.begin());
            if (pack_convT(c, c->c_up[0], wp, *b, bf)) return 1;
        } else if (pack_convT(c, c->c_up[0], *w, *b, bf)) return 1;
        if (!(w = find(c->chk_raw, "upsampler.1.weight", {128, 64, 8})) || !(b = find(c->chk_raw, "upsampler.1.bias", {64}))) return 1;
        if (pack_convT(c, c->c_up[1], *w, *b, bf)) return 1;
        if (!(w = find(c->chk_raw, "resblock.conv1.weight", {64, 64, 3})) || !(b = find(c->chk_raw, "resblock.conv1.bias", {64}))) return 1;
        if (pack_conv(c, c->c_res1, *w, *b, 1, 1, 1, bf)) return 1;
        if (!(w = find(c->chk_raw, "resblock.conv2.weight", {64, 64, 3})) || !(b = find(c->chk_raw, "resblock.conv2.bias", {64}))) return 1;
        if (pack_conv(c, c->c_res2, *w, *b, 3, 3, 1, bf)) return 1;
        if (!(w = find(c->chk_raw, "post_conv.weight", {256, 64, 8})) || !(b = find(c->chk_raw, "post_conv.bias", {256}))) return 1;
        if (pack_conv(c, c->c_post, *w, *b, 1, 0, 24, false)) return 1;
        if (bf) {
            // post_conv as a GEMM: row (window, t) of the operand is the 8 x 64 = 512 contiguous bf16 of z3b rows 24t .. 24t+7
            std::vector<float> q((size_t)256 * 512);
            for (int n = 0; n < 256; n++)
                for (int ci = 0; ci < 64; ci++)
                    for (int j = 0; j < 8; j++) q[(size_t)n * 512 + j * 64 + ci] = w->data[((size_t)n * 64 + ci) * 8 + j];
            if (upload_bf16(c, &c->c_post_wbf, q)) return 1;
            // block-diagonal prologue: out 0..31 = conv_pre_m over in-channels 256..335, out 32..191 = conv_pre_a over in-channels 0..255
            const HostTensor *wm, *bm, *wa, *ba;
            if (!(wm = find(c->chk_raw, "conv_pre_m.weight", {32, 80, 3})) || !(bm = find(c->chk_raw, "conv_pre_m.bias", {32})) ||
                !(wa = find(c->chk_raw, "conv_pre_a.weight", {160, 256, 3})) || !(ba = find(c->chk_raw, "conv_pre_a.bias", {160}))) return 1;
            HostTensor wp, bp;
            wp.shape = {256, 384, 3};
            wp.data.assign((size_t)256 * 384 * 3, 0.0f);
            bp.shape = {256};
            bp.data.assign(256, 0.0f);
            for (int co = 0; co < 32; co++) {
                bp.data[co] = bm->data[co];
                for (int ci = 0; ci < 80; ci++)
                    for (int j = 0; j < 3; j++) wp.data[((size_t)co * 384 + 256 + ci) * 3 + j] = wm->data[((size_t)co * 80 + ci) * 3 + j];
            }
            for (int co = 0; co < 160; co++) {
                bp.data[32 + co] = ba->data[co];
                for (int ci = 0; ci < 256; ci++)
                    for (int j = 0; j < 3; j++) wp.data[((size_t)(32 + co) * 384 + ci) * 3 + j] = wa->data[((size_t)co * 256 + ci) * 3 + j];
            }
            if (pack_conv(c, c->c_pre_tc, wp, bp, 1, 1, 1, true)) return 1;
        }
    }
    // SpeechT5 decoder post-net (optional): Conv1d(k5, pad 2, no bias) -> BatchNorm1d(eval) [-> tanh], x5
    // (modeling_speecht5.py:700-737).  y = (conv(x) - mean) / sqrt(var + eps) * gamma + beta is folded into the conv:
    // w' = w * s, b' = beta - mean * s with s = gamma / sqrt(var + 1e-5).  On the tensor-core path the 80-bin ends are
    // padded to 128 (zero weights) like conv_pre.
    if (!c->pn_raw.empty()) {
        for (int i = 0; i < 5; i++) {
            const int cin = i == 0 ? 80 : 256, cout = i == 4 ? 80 : 256;
            const HostTensor *g, *be, *mu, *var;
            snprintf(k1, sizeof k1, "layers.%d.conv.weight", i);
            if (!(w = find(c->pn_raw, k1, {cout, cin, 5}))) return 1;
            snprintf(k1, sizeof k1, "layers.%d.batch_norm.weight", i);
            if (!(g = find(c->pn_raw, k1, {cout}))) return 1;
            snprintf(k1, sizeof k1, "layers.%d.batch_norm.bias", i);
            if (!(be = find(c->pn_raw, k1, {cout}))) return 1;
            snprintf(k1, sizeof k1, "layers.%d.batch_norm.running_mean", i);
            if (!(mu = find(c->pn_raw, k1, {cout}))) return 1;
            snprintf(k1, sizeof k1, "layers.%d.batch_norm.running_var", i);
            if (!(var = find(c->pn_raw, k1, {cout}))) return 1;
            const int cin_p = (bf && cin == 80) ? 128 : cin, cout_p = (bf && cout == 80) ? 128 : cout;
            HostTensor wf, bfold;
            wf.shape = {cout_p, cin_p, 5};
            wf.data.assign((size_t)cout_p * cin_p * 5, 0.0f);
            bfold.shape = {cout_p};
            bfold.data.assign((size_t)cout_p, 0.0f);
            for (int co = 0; co < cout; co++) {
                const float sc = g->data[co] / sqrtf(var->data[co] + 1e-5f);
                bfold.data[co] = be->data[co] - mu->data[co] * sc;
                for (int ci = 0; ci < cin; ci++)
                    for (int j = 0; j < 5; j++) wf.data[((size_t)co * cin_p + ci) * 5 + j] = w->data[((size_t)co * cin + ci) * 5 + j] * sc;
            }
            if (pack_conv(c, c->pn[i], wf, bfold, 1, 2, 1, bf)) return 1;
        }
        c->has_postnet = true;
    }
    // workspaces
    Workspace &ws = c->ws;
    const size_t F = (size_t)c->max_windows * 12, Wn = (size_t)c->max_windows;
    if (dev_alloc(c, &ws.win_raw, F * 80) || dev_alloc(c, &ws.win_norm, F * 80)) return 1;
    if (dev_alloc(c, &ws.h, F * 8192) || dev_alloc(c, &ws.r, F * 8192) || dev_alloc(c, &ws.s0, F * 8192)) return 1;
    if (bf) {
        if (dev_alloc(c, &ws.win_norm_b, F * 128)) return 1;
        if (!c->chk_raw.empty()) {
            if (dev_alloc(c, &ws.z0b, Wn * 12 * 256) || dev_alloc(c, &ws.z1b, Wn * 48 * 128) || dev_alloc(c, &ws.z2b, Wn * 192 * 64) ||
                dev_alloc(c, &ws.zyb, Wn * 192 * 64) || dev_alloc(c, &ws.cinb, Wn * 12 * 384) || dev_alloc(c, &ws.z3b, Wn * 192 * 64 + 512)) return 1;
            CUtensorMap *ta = new CUtensorMap(), *tb = new CUtensorMap();
            c->c_post_tmA = ta; c->c_post_tmB = tb;
            if (make_tma_2d_bf16(ta, ws.z3b, (long long)Wn * 8, 512, 24 * 64, 128) || make_tma_2d_bf16(tb, c->c_post_wbf, 256, 512, 512, 128)) return 1;
        }
        if (dev_alloc(c, &ws.c0b, F * 512) || dev_alloc(c, &ws.hb, F * 8192) || dev_alloc(c, &ws.yb, F * 8192) ||
            dev_alloc(c, &ws.rb, F * 8192) || dev_alloc(c, &ws.sb, F * 4096)) return 1;
    } else {
        if (dev_alloc(c, &ws.c0, F * 512) || dev_alloc(c, &ws.y, F * 8192) || dev_alloc(c, &ws.s1, F * 8192)) return 1;
    }
    if (dev_alloc(c, &ws.audio, F * 256)) return 1;
    if (!c->chk_raw.empty()) {
        if (bf) {
            if (dev_alloc(c, &ws.z2, Wn * 192 * 64) || dev_alloc(c, &ws.post, Wn * 2048)) return 1;
        } else if (dev_alloc(c, &ws.z0, Wn * 12 * 192) || dev_alloc(c, &ws.z1, Wn * 48 * 128) || dev_alloc(c, &ws.z2, Wn * 192 * 64) ||
                   dev_alloc(c, &ws.zy, Wn * 192 * 64) || dev_alloc(c, &ws.z3, Wn * 192 * 64) || dev_alloc(c, &ws.post, Wn * 2048)) return 1;
    }
    if (dev_alloc(c, &ws.audio16k, Wn * 2048)) return 1;
    if (c->has_postnet) {
        if (dev_alloc(c, &ws.pn_a32, F * 256) || dev_alloc(c, &ws.pn_mel, F * 80)) return 1;
        if (bf) { if (dev_alloc(c, &ws.pn_inb, F * 128) || dev_alloc(c, &ws.pn_b0, F * 256) || dev_alloc(c, &ws.pn_b1, F * 256)) return 1; }
        else { if (dev_alloc(c, &ws.pn_f0, F * 256) || dev_alloc(c, &ws.pn_f1, F * 256)) return 1; }
    }
    if (dev_alloc(c, &c->pre_pool, (size_t)(c->max_sessions + 1) * 320) || dev_alloc(c, &c->claim, (size_t)c->max_sessions + 1)) return 1;
    B2_CUDA_OK(cudaMemset(c->pre_pool, 0, (size_t)(c->max_sessions + 1) * 320 * sizeof(float)));
    B2_CUDA_OK(cudaMemset(c->claim, 0, ((size_t)c->max_sessions + 1) * sizeof(unsigned)));
    B2_CUDA_OK(cudaHostAlloc((void **)&c->err_flag_h, sizeof(int), cudaHostAllocMapped));
    *c->err_flag_h = 0;
    B2_CUDA_OK(cudaHostGetDevicePointer((void **)&c->err_flag_d, c->err_flag_h, 0));
    c->voc_raw.clear();
    c->chk_raw.clear();
    c->pn_raw.clear();
    c->finalized = true;
    return 0;
}

// ---------------------------------------------------------------------------------------------------
// forward sequences
// ---------------------------------------------------------------------------------------------------
static ConvArgs conv_args(const Layer &l, const float *in, float *out, int W, int Tin, int Tout, float pre_slope) {
    ConvArgs a;
    a.in = in; a.wt = l.w32; a.bias = l.bias; a.residual = nullptr; a.out = out; a.out_bf16 = nullptr;
    a.W = W; a.Tin = Tin; a.Tout = Tout; a.Cin = l.Cin; a.Cout = l.Cout; a.taps = l.taps; a.dil = l.dil; a.pad = l.pad; a.stride = l.stride;
    a.pre_slope = pre_slope; a.bf16_slope = 1.0f; a.div = 1.0f; a.accumulate = 0;
    return a;
}

// normalised mel [W][T][80] (ws.win_norm or caller-provided) -> audio [W][256*T]
#define PROF(cls, call)                      \
    do {                                     \
        c->prof.begin(cls, st);              \
        int _rc = (call);                    \
        c->prof.end(st);                     \
        if (_rc) return 1;                   \
    } while (0)

// copies a stage-boundary tensor to the caller's debug buffer when one is set (b2_debug_set_taps); channels-last [W][T][C] fp32
static int tap(b2_ctx *c, int k, const float *src, size_t n, cudaStream_t st) {
    if (!c->taps[k]) return 0;
    B2_CUDA_OK(cudaMemcpyAsync(c->taps[k], src, n * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return 0;
}

static int vocoder_fp32(b2_ctx *c, const float *xn, int W, int T, float *audio, cudaStream_t st) {
    Workspace &ws = c->ws;
    ConvArgs a = conv_args(c->conv_pre, xn, ws.c0, W, T, T, 1.0f);
    PROF(PC_CONV_F32, launch_conv_simt(a, st));
    if (tap(c, 0, ws.c0, (size_t)W * T * 512, st)) return 1;
    const float *stage_in = ws.c0;
    float *sbuf[2] = {ws.s0, ws.s1};
    int Tc = T;
    for (int i = 0; i < 4; i++) {
        // leaky_relu(0.1) -> ConvTranspose1d, as a 3-tap conv over the input grid writing [T][4*C] == [4T][C]
        a = conv_args(c->up[i], stage_in, ws.h, W, Tc, Tc, 0.1f);
        PROF(PC_CONV_F32, launch_conv_simt(a, st));
        Tc *= 4;
        if (tap(c, 1 + 2 * i, ws.h, (size_t)W * Tc * STAGE_C[i], st)) return 1;
        float *S = sbuf[i & 1];
        for (int j = 0; j < 3; j++) {
            for (int d = 0; d < 3; d++) {
                const float *x = (d == 0) ? ws.h : ws.r;
                a = conv_args(c->res1[i][j][d], x, ws.y, W, Tc, Tc, 0.1f);
                PROF(PC_CONV_F32, launch_conv_simt(a, st));
                const bool last = d == 2;
                a = conv_args(c->res2[i][j][d], ws.y, last ? S : ws.r, W, Tc, Tc, 0.1f);
                a.residual = x;
                if (last) { a.accumulate = j > 0; a.div = (j == 2) ? 3.0f : 1.0f; }
                PROF(PC_CONV_F32, launch_conv_simt(a, st));
            }
        }
        if (tap(c, 2 + 2 * i, S, (size_t)W * Tc * STAGE_C[i], st)) return 1;
        stage_in = S;
    }
    PROF(PC_CONV_POST, launch_conv_post(stage_in, c->post_w, c->post_b, audio, W, Tc, st));
    return 0;
}

static int vocoder_bf16(b2_ctx *c, const float *xn, int W, int T, float *audio, cudaStream_t st) {
    Workspace &ws = c->ws;
    // conv_pre on tensor cores as well: the normalised mel is handed over as bf16 rows padded to 128 bins; the epilogue
    // writes the leaky_relu(0.1)'d bf16 operand of the first upsampler
    {
        UmmaConvArgs u;
        u.in = ws.win_norm_b; u.layer = &c->conv_pre; u.outb = ws.c0b; u.outb_slope = 0.1f; u.W = W; u.T = T;
        PROF(PC_CONV_TC, launch_conv_umma(u, st));
    }
    const __nv_bfloat16 *stage_in = ws.c0b;
    int Tc = T;
    for (int i = 0; i < 4; i++) {
        // One launch per ResBlock where the fused kernel covers the stage (conv_resblock.cu: C = 128, 64, 32); stage 0 runs conv by conv.
        const bool fused = c->rb[i][0].tmap && c->rb[i][1].tmap && c->rb[i][2].tmap;
        // Stage 3: the stacked-output ResBlock kernel computes the stage's upsampler itself (conv_resblock_t.cu, UP): no upsampler launch, and
        // x (1.6 GB of fp32 at 4,096 windows, read by three launches) never exists in HBM.  Needs all three ResBlocks on that kernel; not while
        // the stage-boundary taps are being recorded (they want x).
        const bool up_fused = fused && i == 3 && c->up[i].tmap_q && !c->taps[1 + 2 * i] &&
                              c->rb[i][0].tmap_t && c->rb[i][1].tmap_t && c->rb[i][2].tmap_t;
        if (!up_fused) {
            UmmaConvArgs u;
            u.in = stage_in; u.layer = &c->up[i]; u.out32 = ws.h; u.outb = fused ? nullptr : ws.hb; u.outb_slope = 0.1f; u.W = W; u.T = Tc;
            PROF(PC_CONV_TC, launch_conv_umma(u, st));
        }
        Tc *= 4;
        if (!up_fused && tap(c, 1 + 2 * i, ws.h, (size_t)W * Tc * STAGE_C[i], st)) return 1;
        if (fused) {
            // MRF mean (modeling_speecht5.py:3069-3072): s0 = rb0(x); s0 += rb1(x); (s0 + rb2(x)) / 3
            for (int j = 0; j < 3; j++) {
                ResBlockArgs ra;
                ra.x = ws.h; ra.pack = &c->rb[i][j]; ra.W = W; ra.T = Tc; ra.slope = 0.1f; ra.outb_slope = 0.1f;
                if (up_fused) { ra.x = nullptr; ra.up_in = stage_in; ra.up_layer = &c->up[i]; }
                ra.acc_src = (j > 0) ? ws.s0 : nullptr;
                if (j < 2) ra.out32 = ws.s0;
                else {
                    ra.div = 3.0f;
                    if (i < 3) ra.outb = ws.sb;
                    else { ra.post_w = c->post_w; ra.post_b = c->post_b; ra.audio = audio; }   // conv_post + tanh in the same launch
                }
                PROF(PC_RESBLOCK, launch_resblock(ra, st));
            }
            stage_in = ws.sb;
            continue;
        }
        for (int j = 0; j < 3; j++) {
            for (int d = 0; d < 3; d++) {
                const float *x = (d == 0) ? ws.h : ws.r;
                const __nv_bfloat16 *xb = (d == 0) ? ws.hb : ws.rb;
                const bool last = d == 2;
                // epilogue of the pair: next pair's residual + operand, or the MRF mean (modeling_speecht5.py:3069-3072):
                // s0 = x0; s0 += x1; (s0 + x2) / 3 as the operand of the next upsampler
                float *o32 = nullptr; __nv_bfloat16 *ob = nullptr; const float *accs = nullptr; float dv = 1.0f;
                if (!last) { o32 = ws.r; ob = ws.rb; }
                else {
                    accs = (j > 0) ? ws.s0 : nullptr;
                    if (j < 2) o32 = ws.s0;
                    else { dv = 3.0f; ob = ws.sb; }
                }
                UmmaConvArgs u1;
                u1.in = xb; u1.layer = &c->res1[i][j][d]; u1.outb = ws.yb; u1.outb_slope = 0.1f; u1.W = W; u1.T = Tc;
                PROF(PC_CONV_TC, launch_conv_umma(u1, st));
                UmmaConvArgs u2;
                u2.in = ws.yb; u2.layer = &c->res2[i][j][d]; u2.residual = x; u2.W = W; u2.T = Tc;
                u2.acc_src = accs; u2.out32 = o32; u2.outb = ob; u2.outb_slope = 0.1f; u2.div = dv;
                PROF(PC_CONV_TC, launch_conv_umma(u2, st));
            }
        }
        stage_in = ws.sb;
    }
    return 0;
}

static int vocoder_any(b2_ctx *c, const float *xn, int W, int T, float *audio, cudaStream_t st) {
    return c->mode == B2_MODE_BF16 ? vocoder_bf16(c, xn, W, T, audio, st) : vocoder_fp32(c, xn, W, T, audio, st);
}

// raw windows [W][12][80] + vocoder audio [W][3072] -> [W][2048]
static int chunker_fwd(b2_ctx *c, const float *win_raw, const float *audio, int W, float *out, cudaStream_t st) {
    Workspace &ws = c->ws;
    if (!c->cwm) return set_error("chunker weights were not loaded into this context");
    if (c->mode == B2_MODE_BF16) {
        // the whole chunker on tensor cores (bf16 operands, fp32 accumulate, fp32 residual): the prologue, 2 upsamplers, the ResBlock, post_conv
        PROF(PC_OTHER, launch_chunker_in(win_raw, audio, ws.cinb, W, st));
        UmmaConvArgs u;
        u.in = ws.cinb; u.layer = &c->c_pre_tc; u.outb = ws.z0b; u.outb_slope = 0.01f; u.W = W; u.T = 12;
        PROF(PC_CONV_TC, launch_conv_umma(u, st));
        u = UmmaConvArgs();
        u.in = ws.z0b; u.layer = &c->c_up[0]; u.outb = ws.z1b; u.outb_slope = 0.01f; u.W = W; u.T = 12;
        PROF(PC_CONV_TC, launch_conv_umma(u, st));
        u = UmmaConvArgs();
        u.in = ws.z1b; u.layer = &c->c_up[1]; u.out32 = ws.z2; u.outb = ws.z2b; u.outb_slope = 0.01f; u.W = W; u.T = 48;
        PROF(PC_CONV_TC, launch_conv_umma(u, st));
        u = UmmaConvArgs();
        u.in = ws.z2b; u.layer = &c->c_res1; u.outb = ws.zyb; u.outb_slope = 0.01f; u.W = W; u.T = 192;
        PROF(PC_CONV_TC, launch_conv_umma(u, st));
        u = UmmaConvArgs();
        u.in = ws.zyb; u.layer = &c->c_res2; u.residual = ws.z2; u.outb = ws.z3b; u.outb_slope = 0.01f; u.W = W; u.T = 192;
        PROF(PC_CONV_TC, launch_conv_umma(u, st));
        // post_conv (64 -> 256, k8, stride 24, no padding; HelloSippyRT.py:233-234) = [W*8][512] x [512][256]
        GemmTcArgs g;
        g.tmA = reinterpret_cast<const CUtensorMap *>(c->c_post_tmA); g.tmB = reinterpret_cast<const CUtensorMap *>(c->c_post_tmB);
        g.bias = c->c_post.bias; g.out32 = ws.post; g.M = W * 8; g.N = 256; g.K = 512; g.nt = 128; g.pdl = pdl_enabled();
        PROF(PC_CONV_TC, launch_gemm_tc(g, st));
        PROF(PC_OTHER, launch_chunker_final(audio, ws.post, out, W, st));
        return 0;
    }
    PROF(PC_OTHER, launch_chunker_pre(win_raw, audio, c->cwm, c->cbm, c->cwa, c->cba, ws.z0, W, st));
    ConvArgs a = conv_args(c->c_up[0], ws.z0, ws.z1, W, 12, 12, 0.01f);
    PROF(PC_CONV_F32, launch_conv_simt(a, st));
    a = conv_args(c->c_up[1], ws.z1, ws.z2, W, 48, 48, 0.01f);
    PROF(PC_CONV_F32, launch_conv_simt(a, st));
    a = conv_args(c->c_res1, ws.z2, ws.zy, W, 192, 192, 0.01f);
    PROF(PC_CONV_F32, launch_conv_simt(a, st));
    a = conv_args(c->c_res2, ws.zy, ws.z3, W, 192, 192, 0.01f);
    a.residual = ws.z2;
    PROF(PC_CONV_F32, launch_conv_simt(a, st));
    a = conv_args(c->c_post, ws.z3, ws.post, W, 192, 8, 0.01f);
    PROF(PC_CONV_F32, launch_conv_simt(a, st));
    PROF(PC_OTHER, launch_chunker_final(audio, ws.post, out, W, st));
    return 0;
}

// speech_decoder_postnet.postnet (modeling_speecht5.py:758-762; HelloSippyRTPipe.py:230): (B, T, 80) -> (B, T, 80), every
// (session, call) zero-padded on its own like the reference's conv over a (B, 80, T) tensor.  B*T <= 12*max_windows.
static int postnet_fwd(b2_ctx *c, const float *d_in, int B, int T, float *d_out, cudaStream_t st) {
    Workspace &ws = c->ws;
    const size_t rows = (size_t)B * T;
    if (c->mode == B2_MODE_BF16) {
        PROF(PC_OTHER, launch_pn_prep(d_in, ws.pn_inb, rows, st));
        const __nv_bfloat16 *x = ws.pn_inb;
        __nv_bfloat16 *pp[2] = {ws.pn_b0, ws.pn_b1};
        for (int i = 0; i < 5; i++) {
            UmmaConvArgs u;
            u.in = x; u.layer = &c->pn[i]; u.out32 = ws.pn_a32; u.W = B; u.T = T;
            PROF(PC_CONV_TC, launch_conv_umma(u, st));
            if (i < 4) {
                PROF(PC_OTHER, launch_pn_tanh(ws.pn_a32, nullptr, pp[i & 1], rows * 256, st));
                x = pp[i & 1];
            }
        }
        PROF(PC_OTHER, launch_pn_out(d_in, ws.pn_a32, 128, d_out, rows, st));
    } else {
        const float *x = d_in;
        float *pp[2] = {ws.pn_f0, ws.pn_f1};
        for (int i = 0; i < 5; i++) {
            float *o = i < 4 ? pp[i & 1] : ws.pn_a32;
            ConvArgs a = conv_args(c->pn[i], x, o, B, T, T, 1.0f);
            PROF(PC_CONV_F32, launch_conv_simt(a, st));
            if (i < 4) PROF(PC_OTHER, launch_pn_tanh(o, o, nullptr, rows * 256, st));
            x = o;
        }
        PROF(PC_OTHER, launch_pn_out(d_in, ws.pn_a32, 80, d_out, rows, st));
    }
    return 0;
}

// check_dups: duplicate-slot detection through claim[] (needs a fresh epoch per launch, so it is off inside captured graphs, whose
// callers validate on the host); pad_slot_ok: slot id max_sessions (the padding session of a graph bucket) is legal
int tail_device(b2_ctx *c, const int32_t *d_slots, const float *d_mel, int B, int nframes, int law, bool apply_postnet,
                uint8_t *d_g711, float *d_audio, cudaStream_t st, bool check_dups, bool pad_slot_ok) {
    const int nwin = nframes / 8;
    const int sess_per_pass = std::max(1, c->max_windows / nwin);
    const size_t Lout = (size_t)nframes * 128;
    for (int b0 = 0; b0 < B; b0 += sess_per_pass) {
        const int nb = std::min(sess_per_pass, B - b0);
        const int W = nb * nwin;
        Workspace &ws = c->ws;
        const float *mel = d_mel + (size_t)b0 * nframes * 80;
        if (apply_postnet) {
            if (postnet_fwd(c, mel, nb, nframes, ws.pn_mel, st)) return 1;
            mel = ws.pn_mel;
        }
        PROF(PC_OTHER, launch_build_windows(d_slots + b0, mel, c->pre_pool, c->mean, c->scale,
                                            ws.win_raw, ws.win_norm, ws.win_norm_b, nb, nframes,
                                            c->max_sessions + (pad_slot_ok ? 1 : 0), check_dups ? c->claim : nullptr, ++c->epoch, c->err_flag_d, st));
        if (vocoder_any(c, ws.win_norm, W, 12, ws.audio, st)) return 1;
        if (c->cwm) { if (chunker_fwd(c, ws.win_raw, ws.audio, W, ws.audio16k, st)) return 1; }
        else { PROF(PC_OTHER, launch_trim(ws.audio, ws.audio16k, W, 3072, 512, 2048, st)); }
        // windows are session-major, so [W][2048] is already [nb][nwin*2048] (HelloSippyRTPipe.py:238-239)
        PROF(PC_RESAMPLE_G711, launch_resample_2to1(ws.audio16k, (size_t)nb, (size_t)nwin * 2048, law == B2_LAW_ALAW ? B2_LAW_ALAW : B2_LAW_ULAW,
                                                    d_g711 ? d_g711 + (size_t)b0 * Lout : nullptr, d_audio ? d_audio + (size_t)b0 * Lout : nullptr, st));
    }
    return 0;
}

}  // namespace b2

using namespace b2;

#define CTX_GUARD(c)                                                                 \
    if (!(c)) return set_error("null context");                                      \
    {                                                                                \
        cudaError_t _e = cudaSetDevice((c)->device);                                 \
        if (_e != cudaSuccess) return set_error("cudaSetDevice(%d): %s", (c)->device, cudaGetErrorString(_e)); \
    }

extern "C" {

int b2_abi_version(void) { return B2_ABI_VERSION; }

const char *b2_last_error(const b2_ctx *ctx) {
    (void)ctx;
    return g_last_error.c_str();
}

uint64_t b2_kernel_launch_count(void) { return g_launches.load(); }

b2_ctx *b2_ctx_create(int device, int mode, int max_sessions, int max_windows) {
    if (mode != B2_MODE_FP32 && mode != B2_MODE_BF16) { set_error("mode must be B2_MODE_FP32 or B2_MODE_BF16"); return nullptr; }
    if (max_sessions < 1 || max_windows < 1) { set_error("max_sessions and max_windows must be >= 1"); return nullptr; }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) { set_error("no CUDA device: %s (this library has no CPU fallback)", cudaGetErrorString(e)); return nullptr; }
    if (device < 0 || device >= ndev) { set_error("device %d out of range (%d devices)", device, ndev); return nullptr; }
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, device);
    if (prop.major != 10) { set_error("device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major, prop.minor); return nullptr; }
    if (cudaSetDevice(device) != cudaSuccess) { set_error("cudaSetDevice(%d) failed", device); return nullptr; }
    b2_ctx *c = new b2_ctx();
    c->device = device; c->mode = mode; c->max_sessions = max_sessions; c->max_windows = max_windows;
    return c;
}

void b2_ctx_destroy(b2_ctx *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    for (void *p : c->allocs) cudaFree(p);
    if (c->err_flag_h) cudaFreeHost(c->err_flag_h);
    for (int i = 0; i < 4; i++) {
        umma_free_layer(c->up[i]);
        for (int j = 0; j < 3; j++)
            for (int d = 0; d < 3; d++) { umma_free_layer(c->res1[i][j][d]); umma_free_layer(c->res2[i][j][d]); }
        for (int j = 0; j < 3; j++) resblock_free(c->rb[i][j]);
    }
    umma_free_layer(c->conv_pre);
    umma_free_layer(c->c_up[0]); umma_free_layer(c->c_up[1]); umma_free_layer(c->c_res1); umma_free_layer(c->c_res2); umma_free_layer(c->c_pre_tc);
    if (c->c_post_tmA) delete reinterpret_cast<CUtensorMap *>(c->c_post_tmA);
    if (c->c_post_tmB) delete reinterpret_cast<CUtensorMap *>(c->c_post_tmB);
    for (int i = 0; i < 5; i++) umma_free_layer(c->pn[i]);
    delete c;
}

int b2_profile_begin(b2_ctx *c) {
    CTX_GUARD(c);
    for (auto &s : c->prof.spans) { cudaEventDestroy(s.a); cudaEventDestroy(s.b); }
    c->prof.spans.clear();
    c->prof.on = true;
    return 0;
}

int b2_profile_end(b2_ctx *c, double *ms_by_class, uint64_t *launches_by_class) {
    CTX_GUARD(c);
    if (!ms_by_class || !launches_by_class) return set_error("b2_profile_end: null output");
    B2_CUDA_OK(cudaDeviceSynchronize());
    for (int i = 0; i < PC_COUNT; i++) { ms_by_class[i] = 0.0; launches_by_class[i] = 0; }
    for (auto &s : c->prof.spans) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, s.a, s.b);
        ms_by_class[s.cls] += ms;
        launches_by_class[s.cls] += 1;
        cudaEventDestroy(s.a); cudaEventDestroy(s.b);
    }
    c->prof.spans.clear();
    c->prof.on = false;
    return 0;
}

int b2_ctx_mode(const b2_ctx *c) { return c ? c->mode : -1; }
size_t b2_ctx_device_bytes(const b2_ctx *c) { return c ? c->device_bytes : 0; }

int b2_load_vocoder_tensor(b2_ctx *c, const char *key, const float *h, const int64_t *shape, int ndim) {
    if (!c) return set_error("null context");
    if (c->finalized) return set_error("weights are already finalized");
    return load_tensor(c->voc_raw, key, h, shape, ndim);
}

int b2_load_chunker_tensor(b2_ctx *c, const char *key, const float *h, const int64_t *shape, int ndim) {
    if (!c) return set_error("null context");
    if (c->finalized) return set_error("weights are already finalized");
    return load_tensor(c->chk_raw, key, h, shape, ndim);
}

int b2_weights_finalize(b2_ctx *c) {
    CTX_GUARD(c);
    if (c->finalized) return set_error("weights are already finalized");
    return finalize(c);
}

int b2_vocoder_forward(b2_ctx *c, const float *d_mel, int W, int T, float *d_audio, void *stream) {
    CTX_GUARD(c);
    if (!c->finalized) return set_error("b2_weights_finalize has not been called");
    if (W < 0 || T < 1) return set_error("b2_vocoder_forward: bad shape W=%d T=%d", W, T);
    if (W == 0) return 0;
    if (!d_mel || !d_audio) return set_error("b2_vocoder_forward: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    const long long cap = (long long)c->max_windows * 12;
    if (T > cap) return set_error("b2_vocoder_forward: T=%d exceeds the context's workspace (%lld frames)", T, cap);
    const int w_per_pass = (int)std::max<long long>(1, cap / T);
    for (int w0 = 0; w0 < W; w0 += w_per_pass) {
        const int nw = std::min(w_per_pass, W - w0);
        if (launch_normalise(d_mel + (size_t)w0 * T * 80, c->mean, c->scale, c->ws.win_norm, c->ws.win_norm_b, (size_t)nw * T, st)) return 1;
        if (vocoder_any(c, c->ws.win_norm, nw, T, d_audio + (size_t)w0 * T * 256, st)) return 1;
    }
    return 0;
}

int b2_chunker_forward(b2_ctx *c, const float *d_mel, const float *d_audio, int W, float *d_out, void *stream) {
    CTX_GUARD(c);
    if (!c->finalized) return set_error("b2_weights_finalize has not been called");
    if (W < 0) return set_error("b2_chunker_forward: bad W");
    if (W == 0) return 0;
    if (!d_mel || !d_audio || !d_out) return set_error("b2_chunker_forward: null pointer");
    for (int w0 = 0; w0 < W; w0 += c->max_windows) {
        const int nw = std::min(c->max_windows, W - w0);
        if (chunker_fwd(c, d_mel + (size_t)w0 * 960, d_audio + (size_t)w0 * 3072, nw, d_out + (size_t)w0 * 2048, (cudaStream_t)stream)) return 1;
    }
    return 0;
}

int b2_load_postnet_tensor(b2_ctx *c, const char *key, const float *h, const int64_t *shape, int ndim) {
    if (!c) return set_error("null context");
    if (c->finalized) return set_error("weights are already finalized");
    return load_tensor(c->pn_raw, key, h, shape, ndim);
}

int b2_postnet_forward(b2_ctx *c, const float *d_in, int B, int T, float *d_out, void *stream) {
    CTX_GUARD(c);
    if (!c->finalized) return set_error("b2_weights_finalize has not been called");
    if (!c->has_postnet) return set_error("b2_postnet_forward: no post-net weights were loaded into this context");
    if (B < 0 || T < 1) return set_error("b2_postnet_forward: bad shape B=%d T=%d", B, T);
    if (B == 0) return 0;
    if (!d_in || !d_out) return set_error("b2_postnet_forward: null pointer");
    if (d_in == d_out) return set_error("b2_postnet_forward: in-place operation is not supported");
    const long long cap = (long long)c->max_windows * 12;
    if (T > cap) return set_error("b2_postnet_forward: T=%d exceeds the context's workspace (%lld frames)", T, cap);
    const int b_per_pass = (int)std::max<long long>(1, cap / T);
    for (int b0 = 0; b0 < B; b0 += b_per_pass) {
        const int nb = std::min(b_per_pass, B - b0);
        if (postnet_fwd(c, d_in + (size_t)b0 * T * 80, nb, T, d_out + (size_t)b0 * T * 80, (cudaStream_t)stream)) return 1;
    }
    return 0;
}

// Reads (and clears) what k_build_windows has flagged so far.  The flag is host-mapped memory written by the kernel, so it is
// only complete for work the caller has synchronised with; b2_ctx_poll_errors synchronises the stream first.
static int poll_slot_errors(b2_ctx *c, const char *who) {
    if (!c->err_flag_h) return 0;
    const int f = *(volatile int *)c->err_flag_h;
    if (!f) return 0;
    *(volatile int *)c->err_flag_h = 0;
    return set_error("%s: a tail call on this context was given %s%s%s (valid ids: 0 .. %d, each at most once per call); those sessions were computed "
                     "with zero pre_frames and their state was not updated", who, (f & 1) ? "a slot id outside the session pool" : "",
                     (f & 3) == 3 ? " and " : "", (f & 2) ? "the same slot id more than once" : "", c->max_sessions - 1);
}

int b2_ctx_poll_errors(b2_ctx *c, void *stream) {
    CTX_GUARD(c);
    B2_CUDA_OK(cudaStreamSynchronize((cudaStream_t)stream));
    return poll_slot_errors(c, "b2_ctx_poll_errors");
}

int b2_debug_set_taps(b2_ctx *c, float *const *d_taps) {
    if (!c) return set_error("null context");
    for (int i = 0; i < 9; i++) c->taps[i] = d_taps ? d_taps[i] : nullptr;
    return 0;
}

int b2_tts_tail(b2_ctx *c, const int32_t *d_slots, const float *d_mel, int B, int nframes, int law,
                uint8_t *d_g711, float *d_audio, void *stream) {
    return b2_tts_tail2(c, d_slots, d_mel, B, nframes, law, 0, d_g711, d_audio, stream);
}

int b2_tts_tail2(b2_ctx *c, const int32_t *d_slots, const float *d_mel, int B, int nframes, int law, int flags,
                 uint8_t *d_g711, float *d_audio, void *stream) {
    CTX_GUARD(c);
    if (flags & ~B2_TAIL_APPLY_POSTNET) return set_error("b2_tts_tail2: unknown flags 0x%x", flags);
    if ((flags & B2_TAIL_APPLY_POSTNET) && !c->has_postnet) return set_error("b2_tts_tail2: B2_TAIL_APPLY_POSTNET without post-net weights in this context");
    if (!c->finalized) return set_error("b2_weights_finalize has not been called");
    if (B < 0 || nframes < 8 || nframes % 8) return set_error("b2_tts_tail: nframes must be a positive multiple of 8 (got %d), B >= 0", nframes);
    if (nframes / 8 > c->max_windows) return set_error("b2_tts_tail: nframes=%d needs more windows than the context's workspace", nframes);
    if (B == 0) return 0;
    if (!d_slots || !d_mel) return set_error("b2_tts_tail: null input");
    if (d_g711 && law != B2_LAW_ULAW && law != B2_LAW_ALAW) return set_error("b2_tts_tail: bad law %d", law);
    if (!d_g711 && !d_audio) return set_error("b2_tts_tail: no output requested");
    if (poll_slot_errors(c, "b2_tts_tail (reported for an EARLIER asynchronous call)")) return 1;
    return tail_device(c, d_slots, d_mel, B, nframes, law, (flags & B2_TAIL_APPLY_POSTNET) != 0, d_g711, d_audio, (cudaStream_t)stream, true, false);
}

int b2_tts_tail_host(b2_ctx *c, const int32_t *h_slots, const float *h_mel, int B, int nframes, int law,
                     uint8_t *h_g711, float *h_audio, void *stream) {
    return b2_tts_tail_host2(c, h_slots, h_mel, B, nframes, law, 0, h_g711, h_audio, stream);
}

int b2_tts_tail_host2(b2_ctx *c, const int32_t *h_slots, const float *h_mel, int B, int nframes, int law, int flags,
                      uint8_t *h_g711, float *h_audio, void *stream) {
    CTX_GUARD(c);
    if (!c->finalized) return set_error("b2_weights_finalize has not been called");
    if (B < 0 || nframes < 8 || nframes % 8) return set_error("b2_tts_tail_host: nframes must be a positive multiple of 8 (got %d)", nframes);
    if (B == 0) return 0;
    if (!h_slots || !h_mel || (!h_g711 && !h_audio)) return set_error("b2_tts_tail_host: null pointer");
    {
        // the slot ids are in host memory here: reject bad ones before anything is launched
        c->host_seen.assign((size_t)c->max_sessions, 0);
        for (int i = 0; i < B; i++) {
            const int s = h_slots[i];
            if (s < 0 || s >= c->max_sessions) return set_error("b2_tts_tail_host: slot %d (session %d of the call) is outside the pool of %d", s, i, c->max_sessions);
            if (c->host_seen[(size_t)s]++) return set_error("b2_tts_tail_host: slot %d appears more than once in the call", s);
        }
    }
    cudaStream_t st = (cudaStream_t)stream;
    Workspace &ws = c->ws;
    const size_t nout = (size_t)B * nframes * 128;
    if ((size_t)B > c->host_stage_cap_sessions || (size_t)B * nframes > c->host_stage_cap_frames) {
        // grow-only staging buffers (not counted per call: steady state allocates nothing)
        B2_CUDA_OK(cudaStreamSynchronize(st));
        const size_t cs = std::max<size_t>(B, c->host_stage_cap_sessions), cf = std::max<size_t>((size_t)B * nframes, c->host_stage_cap_frames);
        void *old[4] = {ws.slots, ws.mel_in, ws.g711_out, ws.audio8k_out};
        for (void *q : old) {
            if (!q) continue;
            cudaFree(q);
            c->allocs.erase(std::remove(c->allocs.begin(), c->allocs.end(), q), c->allocs.end());
        }
        ws.slots = nullptr; ws.mel_in = nullptr; ws.g711_out = nullptr; ws.audio8k_out = nullptr;
        c->host_stage_cap_sessions = c->host_stage_cap_frames = 0;
        if (dev_alloc(c, &ws.slots, cs) || dev_alloc(c, &ws.mel_in, cf * 80) || dev_alloc(c, &ws.g711_out, cf * 128) ||
            dev_alloc(c, &ws.audio8k_out, cf * 128)) return 1;
        c->host_stage_cap_sessions = cs; c->host_stage_cap_frames = cf;
    }
    B2_CUDA_OK(cudaMemcpyAsync(ws.slots, h_slots, (size_t)B * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    B2_CUDA_OK(cudaMemcpyAsync(ws.mel_in, h_mel, (size_t)B * nframes * 80 * sizeof(float), cudaMemcpyHostToDevice, st));
    if (b2_tts_tail2(c, ws.slots, ws.mel_in, B, nframes, law, flags, h_g711 ? ws.g711_out : nullptr, h_audio ? ws.audio8k_out : nullptr, stream)) return 1;
    if (h_g711) B2_CUDA_OK(cudaMemcpyAsync(h_g711, ws.g711_out, nout, cudaMemcpyDeviceToHost, st));
    if (h_audio) B2_CUDA_OK(cudaMemcpyAsync(h_audio, ws.audio8k_out, nout * sizeof(float), cudaMemcpyDeviceToHost, st));
    B2_CUDA_OK(cudaStreamSynchronize(st));
    return poll_slot_errors(c, "b2_tts_tail_host");
}

static int single_layer(const void *d_in, const float *h_weight, const float *h_bias, int W, int T, int Cin, int Cout, int k, int dil,
                        float pre_slope, const float *d_residual, float *d_out32, void *d_outb, float slope, float div, bool tc, cudaStream_t st) {
    if (!d_in || !h_weight || !h_bias || W < 1 || T < 1 || k < 1 || !(k & 1) || dil < 1) return set_error("conv1d: bad arguments");
    b2_ctx tmp;
    int dev = 0;
    B2_CUDA_OK(cudaGetDevice(&dev));
    tmp.device = dev;
    HostTensor w, b;
    w.shape = {Cout, Cin, k};
    w.data.assign(h_weight, h_weight + (size_t)Cout * Cin * k);
    b.shape = {Cout};
    b.data.assign(h_bias, h_bias + Cout);
    Layer l;
    int rc = pack_conv(&tmp, l, w, b, dil, (k - 1) * dil / 2, 1, tc);
    if (!rc) {
        if (tc) {
            UmmaConvArgs u;
            u.in = reinterpret_cast<const __nv_bfloat16 *>(d_in); u.layer = &l; u.residual = d_residual; u.out32 = d_out32;
            u.outb = reinterpret_cast<__nv_bfloat16 *>(d_outb); u.outb_slope = slope; u.div = div; u.W = W; u.T = T;
            rc = launch_conv_umma(u, st);
        } else {
            ConvArgs a = conv_args(l, reinterpret_cast<const float *>(d_in), d_out32, W, T, T, pre_slope);
            a.residual = d_residual; a.out_bf16 = reinterpret_cast<__nv_bfloat16 *>(d_outb); a.bf16_slope = slope; a.div = div;
            rc = launch_conv_simt(a, st);
        }
    }
    cudaStreamSynchronize(st);
    for (void *q : tmp.allocs) cudaFree(q);
    umma_free_layer(l);
    return rc;
}

int b2_conv1d_tc(const void *d_in_bf16, const float *h_weight, const float *h_bias, int W, int T, int Cin, int Cout, int k, int dil,
                 const float *d_residual, float *d_out32, void *d_outb, float slope, float div, void *stream) {
    return single_layer(d_in_bf16, h_weight, h_bias, W, T, Cin, Cout, k, dil, 1.0f, d_residual, d_out32, d_outb, slope, div, true, (cudaStream_t)stream);
}

int b2_conv1d_f32(const float *d_in, const float *h_weight, const float *h_bias, int W, int T, int Cin, int Cout, int k, int dil,
                  float pre_slope, const float *d_residual, float *d_out32, void *d_outb, float slope, float div, void *stream) {
    return single_layer(d_in, h_weight, h_bias, W, T, Cin, Cout, k, dil, pre_slope, d_residual, d_out32, d_outb, slope, div, false, (cudaStream_t)stream);
}

int b2_resblock_tc(const float *d_x, const float *h_weights, const float *h_biases, int W, int T, int C, int k, int d0, int d1, int d2,
                   const float *d_acc, float *d_out32, void *d_outb, float slope, float outb_slope, float div, void *stream) {
    if (!d_x || !h_weights || !h_biases || W < 1 || T < 1) return set_error("b2_resblock_tc: bad arguments");
    if (!resblock_supported(C, k)) return set_error("b2_resblock_tc: unsupported C=%d k=%d", C, k);
    cudaStream_t st = (cudaStream_t)stream;
    b2_ctx tmp;
    int dev = 0;
    B2_CUDA_OK(cudaGetDevice(&dev));
    tmp.device = dev;
    const int dils[3] = {d0, d1, d2};
    Layer l1[3], l2[3];
    int rc = 0;
    for (int i = 0; i < 3 && !rc; i++)
        for (int cv = 0; cv < 2 && !rc; cv++) {
            HostTensor w, b;
            w.shape = {C, C, k};
            const float *hw = h_weights + (size_t)(2 * i + cv) * C * C * k;
            w.data.assign(hw, hw + (size_t)C * C * k);
            b.shape = {C};
            b.data.assign(h_biases + (size_t)(2 * i + cv) * C, h_biases + (size_t)(2 * i + cv + 1) * C);
            const int dil = cv ? 1 : dils[i];
            rc = pack_conv(&tmp, cv ? l2[i] : l1[i], w, b, dil, (k - 1) * dil / 2, 1, true);
        }
    ResBlockPack pk;
    if (!rc) {
        const Layer *p1[3] = {&l1[0], &l1[1], &l1[2]}, *p2[3] = {&l2[0], &l2[1], &l2[2]};
        rc = resblock_pack(p1, p2, pk, tmp.allocs, tmp.device_bytes);
    }
    if (!rc) {
        ResBlockArgs ra;
        ra.x = d_x; ra.pack = &pk; ra.acc_src = d_acc; ra.out32 = d_out32; ra.outb = reinterpret_cast<__nv_bfloat16 *>(d_outb);
        ra.slope = slope; ra.outb_slope = outb_slope; ra.div = div; ra.W = W; ra.T = T;
        rc = launch_resblock(ra, st);
    }
    cudaError_t e = cudaStreamSynchronize(st);
    if (!rc && e != cudaSuccess) rc = set_error("b2_resblock_tc: %s", cudaGetErrorString(e));
    for (void *q : tmp.allocs) cudaFree(q);
    for (int i = 0; i < 3; i++) { umma_free_layer(l1[i]); umma_free_layer(l2[i]); }
    resblock_free(pk);
    return rc;
}

int b2_debug_set_stacked_min_taps(int k) {
    g_rbt_min_taps = k > 0 ? k : 0;
    return 0;
}

int b2_resblock_t_plan(int k, int d0, int d1, int d2, int T, int post, int *out) {
    if (!out || T < 1) return set_error("b2_resblock_t_plan: bad arguments");
    const int dil[3] = {d0, d1, d2};
    if (!resblock_t_supported(32, k, dil)) return set_error("b2_resblock_t_plan: k=%d dilations %d,%d,%d are not covered by the stacked-output kernel", k, d0, d1, d2);
    int S, H, V, tiles, off[3], lim[3];
    if (resblock_t_plan(k, dil, T, (post & 1) != 0, S, H, V, tiles, off, lim, (post & 2) != 0)) return 1;
    out[0] = S; out[1] = H; out[2] = V; out[3] = tiles;
    for (int i = 0; i < 3; i++) { out[4 + i] = off[i]; out[7 + i] = lim[i]; }
    return 0;
}

int b2_session_reset(b2_ctx *c, const int32_t *h_slots, int n, void *stream) {
    CTX_GUARD(c);
    if (!c->finalized) return set_error("b2_weights_finalize has not been called");
    for (int i = 0; i < n; i++) {
        if (h_slots[i] < 0 || h_slots[i] >= c->max_sessions) return set_error("slot %d out of range", h_slots[i]);
        B2_CUDA_OK(cudaMemsetAsync(c->pre_pool + (size_t)h_slots[i] * 320, 0, 320 * sizeof(float), (cudaStream_t)stream));
    }
    return 0;
}

int b2_session_get_pre_frames(b2_ctx *c, int slot, float *h_out, void *stream) {
    CTX_GUARD(c);
    if (!c->finalized || slot < 0 || slot >= c->max_sessions || !h_out) return set_error("b2_session_get_pre_frames: bad arguments");
    B2_CUDA_OK(cudaMemcpyAsync(h_out, c->pre_pool + (size_t)slot * 320, 320 * sizeof(float), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    B2_CUDA_OK(cudaStreamSynchronize((cudaStream_t)stream));
    return 0;
}

int b2_session_set_pre_frames(b2_ctx *c, int slot, const float *h_in, void *stream) {
    CTX_GUARD(c);
    if (!c->finalized || slot < 0 || slot >= c->max_sessions || !h_in) return set_error("b2_session_set_pre_frames: bad arguments");
    B2_CUDA_OK(cudaMemcpyAsync(c->pre_pool + (size_t)slot * 320, h_in, 320 * sizeof(float), cudaMemcpyHostToDevice, (cudaStream_t)stream));
    B2_CUDA_OK(cudaStreamSynchronize((cudaStream_t)stream));
    return 0;
}

}  // extern "C"
