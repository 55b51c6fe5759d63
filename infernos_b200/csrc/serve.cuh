// What the two serving loops share: the tail scheduler (sched.cu, mel chunks in) and the sentence server (server.cu, token ids in).
#pragma once
#include "common.cuh"
#include "ctx.cuh"

#include <time.h>
#include <algorithm>

struct b2_dec;
struct b2_enc;

namespace b2 {

inline int64_t now_ns() {
    timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (int64_t)ts.tv_sec * 1000000000ll + ts.tv_nsec;
}

// sessions per tail launch are rounded up to: multiples of 8 up to 64, of 32 up to 512, of 128 beyond (<= 12.5 % padding above 64)
inline int bucket_of(int n, int cap) {
    int b = n <= 64 ? ((n + 7) / 8) * 8 : n <= 512 ? ((n + 31) / 32) * 32 : ((n + 127) / 128) * 128;
    return std::min(b, cap);
}

// Captures the fused tail over fixed device buffers at a padded batch size `nb` on stream `st` and instantiates it (nothing is launched).
// *nk receives the kernel nodes of the graph, which are charged to the launch counter only when the graph runs.
int capture_tail_graph(b2_ctx *c, const int32_t *d_slots, const float *d_mel, int nb, int nframes, int law, bool apply_postnet, uint8_t *d_g711,
                       cudaStream_t st, cudaGraphExec_t *exec, int *nk);
// One eager pass of the tail over `nb` scratch sessions (slot max_sessions), synchronised: every kernel of the path sets its function
// attributes before anything is captured.  d_slots, d_mel and d_g711 are workspaces of at least nb sessions.
int warm_tail(b2_ctx *c, int32_t *d_slots, const float *d_mel, int nb, int nframes, int law, bool apply_postnet, uint8_t *d_g711, cudaStream_t st);

// sizes of the decoder and encoder handles (decoder.cu, encoder.cu)
void dec_limits(const b2_dec *d, int *max_sessions, int *max_steps, int *max_enc_len);
void enc_limits(const b2_enc *e, int *max_tokens, int *max_len, int *vocab);

}  // namespace b2
