// tcgen05 (UMMA) implicit-GEMM conv1d for the HiFiGAN upsamplers and ResBlocks (B2_MODE_BF16).
#pragma once
#include "common.cuh"
#include "ctx.cuh"

namespace b2 {

// out[w][t][n] = epi( bias[n] + sum_{j<taps} sum_{ci} Wb[j][n][ci] * in[w][t + j*dil - pad][ci] )      (stride 1)
//   in    bf16 channels-last [W][T][Cin], activation already applied by its producer
//   epi(v): v += residual (fp32); v += acc_src (fp32); v /= div; out32 = v; outb = bf16(lrelu(v, outb_slope))
// N = layer.Cout (for a ConvTranspose1d packed as a 3-tap conv, Cout is 4x the module's out channels and the
// output row [t][4*C] is the channels-last image of output times 4t..4t+3).
struct UmmaConvArgs {
    const __nv_bfloat16 *in = nullptr;
    const Layer *layer = nullptr;
    const float *residual = nullptr;
    float *out32 = nullptr;
    __nv_bfloat16 *outb = nullptr;
    float outb_slope = 1.0f;
    const float *acc_src = nullptr;   // may alias out32 (same element read then written by one thread)
    float div = 1.0f;
    int W = 0, T = 0;
};

int launch_conv_umma(const UmmaConvArgs &a, cudaStream_t st);

// One whole ResBlock (three conv pairs, dilations d0..d2) in a single launch (conv_resblock.cu).
//   result = x3, where x_{n+1} = x_n + conv2_n(lrelu(conv1_n(lrelu(x_n, slope)), slope));
//   v = result; v = acc_src + v; v /= div; out32 = v; outb = bf16(lrelu(v, outb_slope))
struct ResBlockArgs {
    const float *x = nullptr;              // fp32 channels-last [W][T][C]
    const ResBlockPack *pack = nullptr;
    const float *acc_src = nullptr;        // may alias out32
    float *out32 = nullptr;
    __nv_bfloat16 *outb = nullptr;
    float slope = 0.1f, outb_slope = 1.0f, div = 1.0f;
    int W = 0, T = 0;
    // C = 32 only: fuse the vocoder's last step, audio[W][T] = tanh(conv_post(lrelu((acc_src + x3) / div, 0.01))); nothing else is written
    const float *post_w = nullptr, *post_b = nullptr;     // device: [7][32], [1]
    float *audio = nullptr;
    // C = 32, stacked-output kernel only: x is not read but computed -- x = up_layer(up_in), the stage's upsampler (ConvTranspose1d k8 s4,
    // 64 -> 32 channels, packed by tail.cu:pack_convT), up_in bf16 [W][T/4][64] already leaky-ReLU'd.  x must then be nullptr.
    const __nv_bfloat16 *up_in = nullptr;
    const Layer *up_layer = nullptr;
};
bool resblock_supported(int C, int taps);
// gathers the six convolutions' bf16 weights into one TMA-addressable buffer (device allocations are appended to `allocs`)
int resblock_pack(const Layer *const conv1[3], const Layer *const conv2[3], ResBlockPack &out, std::vector<void *> &allocs, size_t &bytes);
void resblock_free(ResBlockPack &p);
int launch_resblock(const ResBlockArgs &a, cudaStream_t st);
// C = 32: four output time steps stacked into the MMA's N dimension (conv_resblock_t.cu); launch_resblock dispatches to it
bool resblock_t_supported(int C, int taps, const int dil[3]);
int resblock_t_pack(ResBlockPack &out, std::vector<void *> &allocs, size_t &bytes);
void resblock_t_free(ResBlockPack &p);
int resblock_t_plan(int k, const int dil[3], int T, bool post, int &S, int &H, int &V, int &tiles, int off[3], int lim[3], bool align4 = false);
int launch_resblock_t(const ResBlockArgs &a, cudaStream_t st);
extern int g_rbt_min_taps;          // > 0: smallest tap count launch_resblock hands to the stacked-output kernel (b2_debug_set_stacked_min_taps)
// builds the TMA descriptor of a layer's bf16 weights; called once from b2_weights_finalize
int umma_prepare_layer(Layer &l);
void umma_free_layer(Layer &l);
// one-time, per process: resolves cuTensorMapEncodeTiled and sets kernel attributes
int umma_init();

}  // namespace b2
