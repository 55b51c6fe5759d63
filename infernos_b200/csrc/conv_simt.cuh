// fp32 CUDA-core kernels of the TTS tail: the generic channels-last conv1d (used for every HiFiGAN layer in
// B2_MODE_FP32 and for the chunker in both modes), conv_post+tanh, the window builder and the chunker's
// view-reinterpreting prologue/epilogue.
#pragma once
#include "common.cuh"

namespace b2 {

// out[w][t][co] = epi( bias[co] + sum_{j<taps} sum_{ci<Cin} Wt[j][ci][co] * lrelu(in[w][t*stride + j*dil - pad][ci], pre_slope) )
// epi(v): v += residual[w][t][co] (if residual); v += out[w][t][co] (if accumulate); v /= div (if div != 1);
//         out = v (if out); out_bf16 = bf16(lrelu(v, bf16_slope)) (if out_bf16)
// Activations are channels-last [W][T][C] so that one time step's channels are contiguous; zero padding is
// per window (windows never see their neighbours: HelloSippyRTPipe.py:234-236 stacks them on the batch dim).
struct ConvArgs {
    const float *in;
    const float *wt;      // packed [taps][Cin][Cout]
    const float *bias;    // [Cout] or nullptr
    const float *residual;
    float *out;
    __nv_bfloat16 *out_bf16;
    int W, Tin, Tout, Cin, Cout, taps, dil, pad, stride;
    float pre_slope;      // 1.0f = no activation on the input
    float bf16_slope;     // slope applied to the bf16 copy
    float div;            // 1.0f = none
    int accumulate;
};

int launch_conv_simt(const ConvArgs &a, cudaStream_t st);

// conv_post (32 -> 1, k7, pad 3) with the preceding leaky_relu(0.01) and the following tanh
// (modeling_speecht5.py:3074-3076).  in [W][T][32] fp32, wt [7][32], out [W][T]
int launch_conv_post(const float *in, const float *wt, const float *bias, float *out, int W, int T, cudaStream_t st);

// HelloSippyRTPipe.py:231-235: cat(pre_frames, mel) -> windows of 12 frames with stride 8; saves the last 4
// frames back into the session's slot.  Writes the raw windows (chunker input) and the normalised ones
// ((x - mean) / scale, modeling_speecht5.py:3055-3056), both [B*nwin][12][80], window index = b*nwin + i.
// win_norm_b (optional): the normalised windows again as bf16 rows padded to 128 bins (operand of conv_pre on tensor cores)
// Slot ids are validated on the device: see k_build_windows (claim: [max_sessions] epochs, err_flag: host-mapped int).
int launch_build_windows(const int32_t *slots, const float *mel, float *pre_pool, const float *mean, const float *scale,
                         float *win_raw, float *win_norm, __nv_bfloat16 *win_norm_b, int B, int nframes,
                         int max_sessions, unsigned *claim, unsigned epoch, int *err_flag, cudaStream_t st);
// plain normalisation for the stand-alone vocoder callable: out = (mel - mean) / scale, n rows of 80
int launch_normalise(const float *mel, const float *mean, const float *scale, float *out, __nv_bfloat16 *out_b, size_t rows, cudaStream_t st);

// chunker prologue (HelloSippyRT.py:221-228): conv_pre_m over mel *viewed* as (80,12) and conv_pre_a over audio
// *viewed* as (256,12), concatenated -> z0 [W][12][192] channels-last (no activation applied).
// wm packed [3][80][32], wa packed [3][256][160].  FP32 mode; BF16 mode runs the prologue on tensor cores (launch_chunker_in).
int launch_chunker_pre(const float *mel, const float *audio, const float *wm, const float *bm, const float *wa, const float *ba,
                       float *z0, int W, cudaStream_t st);
// tensor-core form of the prologue: the two `.view`s as ONE bf16 channels-last operand [W][12][384] (audio channels 0..255, mel 256..335, zero pad)
int launch_chunker_in(const float *mel, const float *audio, __nv_bfloat16 *inb, int W, cudaStream_t st);
// chunker epilogue (HelloSippyRT.py:235-237): out[w][i] = tanh(audio[w][512+i] * lrelu(post[w][i%8][i/8], 0.01))
int launch_chunker_final(const float *audio, const float *post, float *out, int W, cudaStream_t st);
// vocoder-only trim for calls that bypass the chunker: out[w][i] = audio[w][512+i]
int launch_trim(const float *audio, float *out, int W, int Lin, int lo, int Lout, cudaStream_t st);

// SpeechT5 decoder post-net helpers (transformers modeling_speecht5.py:700-762; call site HelloSippyRTPipe.py:230).  The five
// Conv1d(k5, "same") + BatchNorm1d(eval) layers run through the conv kernels above with the batch norm folded into weight and
// bias; these are the element-wise steps between them.
//   prep : mel fp32 [rows][80] -> bf16 [rows][128], bins 80..127 zero (tensor-core operand of the first layer)
//   tanh : v = tanh(in[i]) -> out32[i] (may alias in) and/or outb[i] (bf16 operand of the next layer)
//   out  : out[r][b] = mel[r][b] + y[r*ystride + b], b < 80   (the post-net is residual: :762)
int launch_pn_prep(const float *mel, __nv_bfloat16 *outb, size_t rows, cudaStream_t st);
int launch_pn_tanh(const float *in, float *out32, __nv_bfloat16 *outb, size_t n, cudaStream_t st);
int launch_pn_out(const float *mel, const float *y, int ystride, float *out, size_t rows, cudaStream_t st);

}  // namespace b2
