// Context of the TTS tail: packed weights, workspaces, per-session state pool.
#pragma once
#include "common.cuh"
#include <map>
#include <string>
#include <vector>

namespace b2 {

struct HostTensor {
    std::vector<int64_t> shape;
    std::vector<float> data;
};

// one convolution layer, packed for both kernel families
struct Layer {
    int Cin = 0, Cout = 0, taps = 0, dil = 1, pad = 0, stride = 1;
    float *w32 = nullptr;            // [taps][Cin][Cout] fp32 (CUDA-core path)
    float *bias = nullptr;           // [Cout] fp32
    __nv_bfloat16 *wbf = nullptr;    // [taps][Cout][Cin] bf16, K-major (tensor-core path); nullptr if unused
    void *tmap = nullptr;            // host copy of the CUtensorMap for wbf (tensor-core path)
    void *tmap_half = nullptr;       // same weights, box of half the N tile: each CTA of a 2-CTA cluster fetches one half and multicasts it
    void *tmap_q = nullptr;          // 64 -> 4 x 32 transposed conv only: box {32 ci, 128 rows, 1 tap}, SWIZZLE_64B (the stacked-output ResBlock kernel computes this upsampler itself)
    std::vector<float> h_bias;       // host copy of the bias (transposed convs: per (phase, channel))
};

// the six convolutions of one ResBlock packed for the fused kernel (conv_resblock.cu)
struct ResBlockPack {
    int C = 0, taps = 0, dil[3] = {1, 1, 1};
    __nv_bfloat16 *w = nullptr;      // [6*taps (+pad)][C][C] bf16: pair0.conv1, pair0.conv2, pair1.conv1, ...
    std::vector<float> h_bias1;      // [3][C] conv1 biases (host: passed as kernel parameters)
    std::vector<float> h_cbias;      // [3][C] running sums of the conv2 biases
    void *tmap = nullptr;            // host copy of the CUtensorMap over w
    // stacked-output kernel (conv_resblock_t.cu, C = 32): the same weights with every conv's taps in reverse order, one tap per TMA box
    __nv_bfloat16 *wt = nullptr;     // [6*taps][C][C] bf16: wt[c*taps + q] = tap taps-1-q of conv c
    void *tmap_t = nullptr;
};

struct Workspace {
    // sized for `cap_frames` mel frames in flight (12 per window)
    float *win_raw = nullptr, *win_norm = nullptr;     // [F][80]
    float *c0 = nullptr;                               // [F][512] fp32 (FP32 mode)
    float *h = nullptr, *y = nullptr, *r = nullptr, *s0 = nullptr, *s1 = nullptr;   // [F*8192] fp32
    __nv_bfloat16 *c0b = nullptr;                      // [F][512] bf16 (BF16 mode)
    __nv_bfloat16 *hb = nullptr, *yb = nullptr, *rb = nullptr, *sb = nullptr;       // [F*8192] bf16
    float *audio = nullptr;                            // [F*256]
    // chunker, per window (z0, z1, zy, z3: FP32 mode only)
    float *z0 = nullptr, *z1 = nullptr, *z2 = nullptr, *zy = nullptr, *z3 = nullptr, *post = nullptr;
    __nv_bfloat16 *win_norm_b = nullptr;               // [F][128] bf16, bins 80..127 zero (BF16 mode)
    __nv_bfloat16 *z0b = nullptr, *z1b = nullptr, *z2b = nullptr, *zyb = nullptr;   // chunker operands (BF16 mode)
    __nv_bfloat16 *cinb = nullptr, *z3b = nullptr;     // [W][12][384] prologue operand; [W][192][64] bf16(lrelu(z3, 0.01)) = operand of post_conv
    float *audio16k = nullptr;                         // [W][2048]
    // post-net, sized for 12 frames per window like the rest: conv output, ping-pong operands, the post-net's mel
    float *pn_a32 = nullptr, *pn_f0 = nullptr, *pn_f1 = nullptr, *pn_mel = nullptr;    // [F][256] x3, [F][80]
    __nv_bfloat16 *pn_inb = nullptr, *pn_b0 = nullptr, *pn_b1 = nullptr;               // [F][128], [F][256] x2
    int32_t *slots = nullptr;                          // device copy for the host entry point
    float *mel_in = nullptr;                           // device staging for the host entry point
    uint8_t *g711_out = nullptr;
    float *audio8k_out = nullptr;
};

// optional per-kernel-class timing with CUDA events on the launching stream (used by bench.py's roofline leg)
enum ProfClass { PC_CONV_TC = 0, PC_CONV_F32 = 1, PC_CONV_POST = 2, PC_RESAMPLE_G711 = 3, PC_OTHER = 4, PC_RESBLOCK = 5, PC_COUNT = 8 };
struct ProfSpan { int cls; cudaEvent_t a, b; };
struct Prof {
    bool on = false;
    std::vector<ProfSpan> spans;
    void begin(int cls, cudaStream_t st) {
        if (!on) return;
        ProfSpan s; s.cls = cls;
        cudaEventCreate(&s.a); cudaEventCreate(&s.b);
        cudaEventRecord(s.a, st);
        spans.push_back(s);
    }
    void end(cudaStream_t st) { if (on) cudaEventRecord(spans.back().b, st); }
};

}  // namespace b2

struct b2_ctx {
    int device = 0, mode = 0, max_sessions = 0, max_windows = 0;
    bool finalized = false;
    std::map<std::string, b2::HostTensor> voc_raw, chk_raw, pn_raw;
    std::vector<void *> allocs;
    size_t device_bytes = 0;
    std::string err;
    b2::Prof prof;

    float *mean = nullptr, *scale = nullptr;
    b2::Layer conv_pre, up[4], res1[4][3][3], res2[4][3][3];
    b2::ResBlockPack rb[4][3];                         // fused-ResBlock packs (BF16 mode, stages the fused kernel covers)
    float *post_w = nullptr, *post_b = nullptr;        // conv_post [7][32], [1]
    // chunker
    float *cwm = nullptr, *cbm = nullptr, *cwa = nullptr, *cba = nullptr;
    b2::Layer c_up[2], c_res1, c_res2, c_post;
    // BF16 mode: the prologue (conv_pre_m + conv_pre_a as one block-diagonal 384 -> 256 conv, 192 real outputs) and post_conv (k8 s24 = a
    // K = 512 GEMM over strided rows of z3) on tensor cores
    b2::Layer c_pre_tc;
    __nv_bfloat16 *c_post_wbf = nullptr;               // [256][512] bf16: W[n][j * 64 + ci] = post_conv.weight[n][ci][j]
    void *c_post_tmA = nullptr, *c_post_tmB = nullptr; // CUtensorMap: A over z3b with a 24-row (1536-element) stride, B over c_post_wbf

    // SpeechT5 decoder post-net (optional; SURVEY 8 f3): five k5 convs, batch norm folded in
    bool has_postnet = false;
    b2::Layer pn[5];

    float *pre_pool = nullptr;                         // [max_sessions + 1][4][80]; the extra slot is the padding session of graph buckets
    // device-side validation of caller-supplied slot ids (k_build_windows): claim[slot] = epoch of the last launch that used it
    unsigned *claim = nullptr;                         // [max_sessions + 1]
    unsigned epoch = 0;
    int *err_flag_h = nullptr, *err_flag_d = nullptr;  // one host-mapped int: bit 0 slot out of range, bit 1 duplicate slot in a call
    // debug taps of the vocoder's stage boundaries (b2_debug_set_taps): conv_pre, up0, stage0, up1, stage1, up2, stage2, up3, stage3
    float *taps[9] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    b2::Workspace ws;
    size_t host_stage_cap_sessions = 0, host_stage_cap_frames = 0;
    std::vector<uint8_t> host_seen;                    // scratch of the host-side slot check
};

namespace b2 {
// The fused tail over device buffers (tail.cu); the scheduler (sched.cu) captures it into CUDA graphs.
// check_dups: duplicate-slot detection through claim[] (needs a fresh epoch per launch, so it is off inside captured graphs, whose
// callers validate on the host); pad_slot_ok: slot id max_sessions (the padding session of a graph bucket) is legal.
int tail_device(b2_ctx *c, const int32_t *d_slots, const float *d_mel, int B, int nframes, int law, bool apply_postnet,
                uint8_t *d_g711, float *d_audio, cudaStream_t st, bool check_dups, bool pad_slot_ok);
}  // namespace b2
