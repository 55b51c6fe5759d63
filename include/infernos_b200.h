/*
 * infernos_b200 — C-ABI of the B200-native TTS tail (mel chunks -> HiFiGAN -> chunker -> 16k->8k -> G.711).
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch types.  Every entry point names the
 * reference interface it replaces (paths relative to the sippy/Infernos tree).  All `d_*` pointers are
 * BORROWED device pointers on the context's device; `h_*` are host pointers; `stream` is a cudaStream_t
 * passed as void* (NULL = legacy default stream).  Functions return 0 on success, non-zero on error;
 * b2_last_error() returns the message.  Nothing here falls back to the CPU.
 *
 * Threading: one thread at a time per context (the reference serialises every torch call behind
 * InfernGlobals().torcher, HelloSippyTTSRT/HelloSippyRTPipe.py:156,192,246).  The ctx-less codec calls are
 * stateless and thread-safe (Core/Codecs/G711.py encode is called from per-call RTPOutputWorker threads).
 */
#ifndef INFERNOS_B200_H
#define INFERNOS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2_ABI_VERSION 1

#if defined(__GNUC__)
#define B2_API __attribute__((visibility("default")))
#else
#define B2_API
#endif

/* precision modes of the vocoder (north_star: fp32 max-abs 1e-3, bf16 >= 40 dB SNR) */
#define B2_MODE_FP32 0 /* CUDA-core fp32 convolutions                                  */
#define B2_MODE_BF16 1 /* tcgen05 tensor-core convolutions: bf16 operands, fp32 accumulate + fp32 residual stream */

#define B2_LAW_ULAW 0 /* PCMU, RTP payload type 0 (Core/Codecs/G711.py:22-23) */
#define B2_LAW_ALAW 1 /* PCMA, RTP payload type 8 (extension; audioop.lin2alaw semantics) */
#define B2_LAW_NONE (-1)

typedef struct b2_ctx b2_ctx;

B2_API int b2_abi_version(void);
/* message of the last failed call on this thread (ctx may be NULL for the ctx-less calls) */
B2_API const char *b2_last_error(const b2_ctx *ctx);

/* ---- context: packed weights, workspaces, per-session state pool ------------------------------------
 * Replaces what HelloSippyRTPipe.__init__ builds (HelloSippyRTPipe.py:155-189): vocoder, chunker, resampler.
 * max_sessions sizes the pre_frames pool (state.pre_frames, HelloSippyRTPipe.py:67,77,233), one 4x80 fp32
 * slot per session.  max_windows bounds the number of 12-frame windows one call may process. */
B2_API b2_ctx *b2_ctx_create(int device, int mode, int max_sessions, int max_windows);
B2_API void b2_ctx_destroy(b2_ctx *ctx);
B2_API int b2_ctx_mode(const b2_ctx *ctx);
/* bytes of HBM held by the context (weights + workspaces + state) */
B2_API size_t b2_ctx_device_bytes(const b2_ctx *ctx);

/* Weights, by state_dict key, fp32 host memory, torch layout:
 *   vocoder  keys of transformers SpeechT5HifiGan  (mean, scale, conv_pre.weight, upsampler.0.weight, resblocks.0.convs1.0.weight, ...)
 *   chunker  keys of AmendmentNetwork1             (HelloSippyTTSRT/HelloSippyRT.py:202-217)
 * replacing SpeechT5HifiGan.from_pretrained / AmendmentNetwork1.from_pretrained (HelloSippyRTPipe.py:171-179). */
B2_API int b2_load_vocoder_tensor(b2_ctx *ctx, const char *key, const float *h_data, const int64_t *shape, int ndim);
B2_API int b2_load_chunker_tensor(b2_ctx *ctx, const char *key, const float *h_data, const int64_t *shape, int ndim);
/* optional: the `layers.*` keys of transformers SpeechT5SpeechDecoderPostnet (layers.{0..4}.conv.weight and
 * layers.{0..4}.batch_norm.{weight,bias,running_mean,running_var}; modeling_speecht5.py:700-750), i.e. the weights behind
 * self.model.speech_decoder_postnet.postnet (HelloSippyRTPipe.py:230).  Other keys (feat_out, prob_out, num_batches_tracked)
 * are not used by this library and must not be passed. */
B2_API int b2_load_postnet_tensor(b2_ctx *ctx, const char *key, const float *h_data, const int64_t *shape, int ndim);
/* packs the loaded weights for the kernels; must be called once after all tensors are loaded */
B2_API int b2_weights_finalize(b2_ctx *ctx);
/* 28 taps of torchaudio Resample(16000,8000).kernel and 2x15 taps of Resample(8000,16000).kernel; the library
 * has the same values built in, this lets the host pass torchaudio's own (HelloSippyRTPipe.py:185-186). */
B2_API int b2_set_resample_taps(const float *h_down28, const float *h_up30);

/* ---- the three callables the reference engine holds (HelloSippyRTPipe.py:236,237,240) ---------------- */
/* self.vocoder(spectrogram): d_mel (W,T,80) fp32 -> d_audio (W, 256*T) fp32.   T >= 1, W*T <= 12*max_windows */
B2_API int b2_vocoder_forward(b2_ctx *ctx, const float *d_mel, int W, int T, float *d_audio, void *stream);
/* self.chunker(spectrogram, audio): d_mel (W,12,80), d_audio (W,3072) -> d_out (W,2048) */
B2_API int b2_chunker_forward(b2_ctx *ctx, const float *d_mel, const float *d_audio, int W, float *d_out, void *stream);
/* self.resampler(audio): (rows, L) fp32 @16k -> (rows, ceil(L/2)) fp32 @8k, zero padding per row per call */
B2_API int b2_resample_2to1(const float *d_in, size_t rows, size_t L, float *d_out, void *stream);

/* ---- fused tail: HelloSippyRTPipe.infer() lines 231-240 (+ G711Codec.encode) in one call --------------
 * d_slots (B) int32: pre_frames slot of each session; d_mel (B, nframes, 80) fp32: the post-net mel frames of
 * this call (nframes % 8 == 0; the reference uses 32).  Outputs, either may be NULL:
 *   d_g711  (B, nframes*128) uint8  : G.711 payload bytes of the 8 kHz audio (law = B2_LAW_ULAW/ALAW)
 *   d_audio (B, nframes*128) fp32   : state.audio at 8 kHz (what unbatch_and_dispatch slices)
 * The pre_frames slots are updated in place.  Sessions are independent; B*nframes/8 <= max_windows. */
B2_API int b2_tts_tail(b2_ctx *ctx, const int32_t *d_slots, const float *d_mel, int B, int nframes, int law,
                uint8_t *d_g711, float *d_audio, void *stream);
/* same, with HOST buffers (pinned for full speed): H2D of slots+mel, the tail, D2H of the outputs, and a
 * stream synchronise before returning.  This is the end-to-end entry the e2e benchmark times. */
B2_API int b2_tts_tail_host(b2_ctx *ctx, const int32_t *h_slots, const float *h_mel, int B, int nframes, int law,
                     uint8_t *h_g711, float *h_audio, void *stream);
/* The step before the path (SURVEY 8 f3): self.model.speech_decoder_postnet.postnet(spectrogram), HelloSippyRTPipe.py:230 =
 * transformers SpeechT5SpeechDecoderPostnet.postnet (modeling_speecht5.py:758-762): out = x + BNConv5(tanh(BNConv4(...tanh(BNConv1(x))))),
 * eval-mode batch norm, k5 "same" convolutions zero-padded per (session, call).  d_in, d_out (B, T, 80) fp32, not aliased.
 * B2_MODE_FP32: CUDA-core fp32; B2_MODE_BF16: tcgen05 convolutions with bf16 operands, fp32 accumulate, fp32 tanh. */
B2_API int b2_postnet_forward(b2_ctx *ctx, const float *d_in, int B, int T, float *d_out, void *stream);
/* b2_tts_tail with flags: B2_TAIL_APPLY_POSTNET = d_mel holds the PRE-post-net frames (the feat_out outputs,
 * HelloSippyRTPipe.py:213-216) and the post-net runs on the GPU inside the same call. */
#define B2_TAIL_APPLY_POSTNET 1
B2_API int b2_tts_tail2(b2_ctx *ctx, const int32_t *d_slots, const float *d_mel, int B, int nframes, int law, int flags,
                 uint8_t *d_g711, float *d_audio, void *stream);
B2_API int b2_tts_tail_host2(b2_ctx *ctx, const int32_t *h_slots, const float *h_mel, int B, int nframes, int law, int flags,
                      uint8_t *h_g711, float *h_audio, void *stream);
/* Slot ids handed over in DEVICE memory (b2_tts_tail / b2_tts_tail2) are validated by the window-builder kernel itself: an id outside
 * [0, max_sessions) or the same id twice in one call is computed with zero pre_frames, leaves the pool untouched, and raises a flag that
 * the NEXT call on the context reports, or this call once `stream` has been synchronised (returns non-zero + b2_last_error).  The host
 * entries check their slot ids before launching anything.  (The reference keeps pre_frames inside the batch state, HelloSippyRTPipe.py:67,
 * so it has no such failure mode; a slot pool does.) */
B2_API int b2_ctx_poll_errors(b2_ctx *ctx, void *stream);
/* Debug taps for the parity tests (BASELINE config 2: "every stage boundary"): nine device pointers, any of them NULL, in the order
 * conv_pre, upsampler0, stage0 (MRF mean), upsampler1, stage1, upsampler2, stage2, upsampler3, stage3; each receives the fp32 channels-last
 * tensor [W][T_stage][C_stage] of the next b2_vocoder_forward / b2_tts_tail sub-batch (modeling_speecht5.py:3062-3072).  B2_MODE_FP32 fills all
 * nine; B2_MODE_BF16 only the upsampler outputs (the other boundaries never leave the chip there).  d_taps == NULL clears them. */
B2_API int b2_debug_set_taps(b2_ctx *ctx, float *const *d_taps);
/* zero the pre_frames of the given slots (HelloSippyPipeState.__init__, HelloSippyRTPipe.py:77); h_slots host */
B2_API int b2_session_reset(b2_ctx *ctx, const int32_t *h_slots, int n, void *stream);
/* read / write one session's pre_frames (4x80 fp32, host) — used to migrate or checkpoint a session */
B2_API int b2_session_get_pre_frames(b2_ctx *ctx, int slot, float *h_out, void *stream);
B2_API int b2_session_set_pre_frames(b2_ctx *ctx, int slot, const float *h_in, void *stream);

/* ---- latency-bounded serving loop (SURVEY 7 step 6) ---------------------------------------------------------------------------
 * Replaces the reference's strictly serial worker loop  infer() -> unbatch_and_dispatch()  (Cluster/InfernTTSWorker.py:83-92) and the
 * three executors its own load test overlaps generation and dispatch with (HelloSippyTTSRT/HelloSippyRTPipeTest.py:126-161).
 * Callers submit (slot, mel chunk) pairs from any thread; a native launcher thread forms sub-batches adaptively (whatever has arrived
 * when the pipeline has room), runs each as  pinned H2D -> ONE CUDA-graph launch of the fused tail -> D2H  on three streams with
 * `depth` sub-batches in flight, and a completer thread stamps the time at which a chunk's G.711 bytes are in pinned host memory.
 * The scheduler owns the context's workspaces while it exists: do not call the other b2_* entry points of `ctx` concurrently. */
typedef struct b2_sched b2_sched;
typedef struct b2_completion {
    uint64_t tag;            /* the caller's tag (default: the slot id) */
    int64_t t_enqueue_ns;    /* CLOCK_MONOTONIC: the caller's arrival stamp, or the time of b2_sched_submit */
    int64_t t_launch_ns;     /* the sub-batch was closed and handed to the GPU */
    int64_t t_done_ns;       /* its G.711 bytes were in pinned host memory */
    int64_t g711_offset;     /* offset of this chunk's nbytes in the h_g711 buffer given to b2_sched_poll (-1 if none was given) */
    int32_t slot, nbytes, batch_sessions, reserved_;
} b2_completion;
typedef struct b2_sched_stats {
    uint64_t sub_batches, sessions, padded_sessions, graph_launches, graphs_built, max_sub_batch, capacity, depth;
} b2_sched_stats;
/* nframes: mel frames per chunk (multiple of 8; 8 = one 128 ms chunk, 32 = the reference's infer() call); max_batch: sessions per
 * sub-batch (<= 0: as many as the context's workspace holds in one pass); depth: sub-batches in flight (2 = double buffering);
 * use_graphs: run each sub-batch as one captured CUDA graph (sessions are padded to a bucket size with a scratch session). */
B2_API b2_sched *b2_sched_create(b2_ctx *ctx, int nframes, int law, int flags, int max_batch, int depth, int use_graphs);
B2_API void b2_sched_destroy(b2_sched *s);
/* optional batching policy: a sub-batch with fewer than min_batch sessions waits up to max_wait_us after its first chunk (default 0/0:
 * launch whatever is there as soon as the pipeline has room) */
B2_API int b2_sched_set_policy(b2_sched *s, int min_batch, int max_wait_us);
/* n chunks: h_slots[n], h_mel (n, nframes, 80) fp32, optional arrival stamps and tags.  Copies into pinned staging and returns; blocks
 * only when every staging buffer is in use (back-pressure).  Staging buffers are recycled by b2_sched_poll, so polling must not depend on
 * the submitting thread making progress (poll from another thread; a submit that cannot get a buffer for 20 s returns an error).
 * A session's chunks are processed in submission order; two chunks of one session never share a sub-batch. */
B2_API int b2_sched_submit(b2_sched *s, const int32_t *h_slots, const float *h_mel, int n, const int64_t *t_enqueue_ns, const uint64_t *tags);
/* up to max_out finished chunks, oldest first; their bytes are copied to h_g711 (may be NULL) at out[i].g711_offset.
 * timeout_ms: 0 = do not wait, < 0 = wait.  Returns the count, or a negative value on error. */
B2_API int b2_sched_poll(b2_sched *s, b2_completion *out, int max_out, uint8_t *h_g711, size_t g711_capacity, int timeout_ms);
/* returns when everything submitted so far has completed (its completions may still be waiting for b2_sched_poll) */
B2_API int b2_sched_flush(b2_sched *s, int timeout_ms);
B2_API int b2_sched_get_stats(b2_sched *s, b2_sched_stats *out);
/* Captures and instantiates, ahead of time, the CUDA graph of every sub-batch bucket up to `max_sessions` sessions (<= 0: up to max_batch) for
 * every staging buffer, so that no graph is ever built on the serving path: a backlog after a host hiccup makes sub-batches of sizes that were
 * never seen before, and building their graphs right then (a few ms each) turns one hiccup into a latency tail.  Call while the scheduler is
 * idle (before the first submit, or after b2_sched_flush); nothing is launched. */
B2_API int b2_sched_prebuild(b2_sched *s, int max_sessions);

/* ---- the step before the path (SURVEY 8 f3): the autoregressive SpeechT5 speech decoder, HelloSippyRTPipe.py:195-229 ----------------------
 * prenet -> wrapped_decoder (six layers, KV cache) -> feat_out / prob_out, batched over sessions whose state (self-attention KV cache,
 * cross-attention keys / values of the sentence, normalised speaker vector, last frame, step counter) lives in slots on the device.
 * Weights by state_dict key of transformers SpeechT5ForTextToSpeech: `speecht5.decoder.prenet.*`, `speecht5.decoder.wrapped_decoder.layers.*`,
 * `speech_decoder_postnet.feat_out.*`, `speech_decoder_postnet.prob_out.*`, plus key `pe` = the (max_steps, 768) position table
 * (SpeechT5ScaledPositionalEncoding.pe, modeling_speecht5.py:405-412; passed in so that it is torch's own).  Default SpeechT5Config sizes.
 * The text encoder's output (b2_enc_forward below, or any other encoder) is an input here.
 * B2_MODE_FP32: CUDA-core fp32 Linears, fp32 caches.  B2_MODE_BF16: tcgen05 GEMMs fed by TMA, bf16 caches, fp32 residual stream / LayerNorm. */
typedef struct b2_dec b2_dec;
/* max_rows: sessions per internal pass (workspace); max_steps: decoder steps a sentence may run (KV cache depth = positions of `pe`);
 * max_enc_len: encoder positions per sentence */
B2_API b2_dec *b2_dec_create(int device, int mode, int max_sessions, int max_rows, int max_steps, int max_enc_len);
B2_API void b2_dec_destroy(b2_dec *dec);
B2_API size_t b2_dec_device_bytes(const b2_dec *dec);
B2_API int b2_dec_load_tensor(b2_dec *dec, const char *key, const float *h_data, const int64_t *shape, int ndim);
B2_API int b2_dec_finalize(b2_dec *dec);
/* HelloSippyPipeStateBatched.merge (HelloSippyRTPipe.py:97-118) for n new sentences: d_enc (n, L, 768) fp32 = encoder_last_hidden_state,
 * d_enc_len (n) int32 = number of unmasked encoder positions (NULL: all L), d_speaker (n, 512) fp32 (normalised here, :696).  Projects the
 * cross-attention keys / values of all six layers into the slots, zeroes the first frame and the step counter. */
B2_API int b2_dec_start(b2_dec *dec, const int32_t *d_slots, const float *d_enc, const int32_t *d_enc_len, const float *d_speaker, int n, int L, void *stream);
/* nsteps trips of the reference's while loop (:195-223) for n sessions: d_mel (n, 2*nsteps, 80) = the feat_out frames (BEFORE the post-net:
 * feed them to b2_tts_tail2 with B2_TAIL_APPLY_POSTNET), d_prob (n, nsteps, 2) = sigmoid(prob_out).  d_masks (nsteps, 2, 256) fp32 0/1 =
 * the prenet's dropout keep-masks (always on, even in eval: modeling_speecht5.py:671-691), shared by the batch like the reference's; NULL
 * draws them on the device from (seed, call counter).  Asynchronous on `stream`. */
B2_API int b2_dec_steps(b2_dec *dec, const int32_t *d_slots, int n, int nsteps, const float *d_masks, uint64_t seed, float *d_mel, float *d_prob, void *stream);
/* synchronises `stream` and reports what the kernels flagged (slot outside the pool, step past max_steps, bad encoder length) */
B2_API int b2_dec_poll_errors(b2_dec *dec, void *stream);
B2_API int b2_dec_get_step(b2_dec *dec, int slot, int32_t *h_step, void *stream);
/* b2_dec_steps runs as ONE CUDA graph launch per call (cached per padded batch size and step count; a call is ~74 kernels per step).
 * on = 0 launches the kernels one by one instead (default: 1). */
B2_API int b2_dec_set_graphs(b2_dec *dec, int on);

/* ---- the text encoder (HelloSippyRTPipe.py:111-116, once per sentence): SpeechT5EncoderWithTextPrenet, token ids -> encoder_last_hidden_state ----
 * prenet (embedding + alpha * scaled sinusoidal positions) -> LayerNorm -> twelve post-LN layers (self-attention with the relative-position
 * term of SpeechT5RelativePositionalEncoding, GELU feed-forward), modeling_speecht5.py:765-781, :1013-1066, :1230-1320.
 * Weights by state_dict key of transformers SpeechT5ForTextToSpeech: `speecht5.encoder.prenet.{embed_tokens.weight, encode_positions.alpha}`,
 * `speecht5.encoder.wrapped_encoder.{layer_norm.*, embed_positions.pe_k.weight, layers.*}`, plus key `pe` = the (max_len, 768) position table
 * (SpeechT5ScaledPositionalEncoding.pe, a non-persistent buffer: passed in so that it is torch's own).  Default SpeechT5Config sizes.
 * Ragged: only valid tokens are computed; the sentences of a call are packed into passes of <= max_tokens rows (a sentence is never split),
 * and a sentence's output does not depend on its companions or on the packing.
 * B2_MODE_FP32: CUDA-core fp32 Linears.  B2_MODE_BF16: tcgen05 GEMMs fed by TMA; fp32 residual stream, LayerNorm and attention. */
typedef struct b2_enc b2_enc;
/* max_tokens: rows of one internal pass (workspace); max_len: positions per sentence, <= 450 (the scaled positional table) */
B2_API b2_enc *b2_enc_create(int device, int mode, int max_tokens, int max_len);
B2_API void b2_enc_destroy(b2_enc *enc);
B2_API size_t b2_enc_device_bytes(const b2_enc *enc);
B2_API int b2_enc_load_tensor(b2_enc *enc, const char *key, const float *h_data, const int64_t *shape, int ndim);  /* + key "pe" (max_len, 768) */
B2_API int b2_enc_finalize(b2_enc *enc);
/* d_ids (n, L) int32 device, right-padded; h_len (n) HOST valid lengths in [1, L] (NULL: all L); d_out (n, L, 768) fp32 device =
 * encoder_last_hidden_state at valid positions, zeros elsewhere.  Only valid tokens are computed; sessions are packed into passes of
 * <= max_tokens rows (a session is never split).  Asynchronous on `stream`.  Calls on one handle must be ordered (one stream). */
B2_API int b2_enc_forward(b2_enc *enc, const int32_t *d_ids, const int32_t *h_len, int n, int L, float *d_out, void *stream);
/* token ids outside [0, 81) are embedded as zeros and flagged; reported here (stream synchronised) or by the next call */
B2_API int b2_enc_poll_errors(b2_enc *enc, void *stream);

/* ---- sentence server: token ids in, G.711 chunks out ---------------------------------------------------------------------------------
 * Replaces the reference's worker loop  infer() -> unbatch_and_dispatch()  (Cluster/InfernTTSWorker.py:83-92) together with the engine call it
 * drives (HelloSippyTTSRT/HelloSippyRTPipe.py:195-259), for whole sentences.  A native driver thread runs engine calls back to back; each call
 *   admits pending sentences into free slots (one encoder pass + b2_dec_start for all of them), runs ONE b2_dec_steps(16) over every live
 *   slot whatever call admitted it, applies the reference's stop rule on the device (:225-228), runs the fused tail with the post-net
 *   (b2_tts_tail2, B2_TAIL_APPLY_POSTNET) and copies the bytes and the per-sentence slice [startoff, endoff) to pinned host memory,
 * with no host synchronisation between those parts and `depth` calls in flight.  A completer thread turns each finished call into records and
 * returns the slots of ended sentences to the pool.  Semantics are HelloSippyRTPipe's: 16 decoder steps = 32 frames = 4,096 bytes per sentence
 * and call, starts_at = 1, a sentence ends 2 steps after the stop fires, minlen / maxlen from the padded token length of the sentence's
 * admission round (maxlen capped at max_steps - 20), prenet dropout masks drawn on the device from (seed, decoder call counter).
 * Cancel (b2_tts_server_cancel, barge-in): a pending sentence leaves the queue at once and gets one record with call = admit_call = -1,
 * nbytes = 0, ended = 2.  An admitted one is retired on the device at the start of the next engine call built: from that call on it takes no
 * decoder step, and that call's record for it has nbytes = 0, ended = 2.  Records of calls built before the cancel (at most `depth`) still
 * arrive with their bytes.  If one of those calls ends the sentence on its own, that record (ended = 1) stays its last one and the cancel
 * does nothing: every sentence gets exactly one last record either way.
 * The server owns ctx, enc and dec while it exists: do not call other b2_* entry points on them concurrently, and destroy it first. */
typedef struct b2_tts_server b2_tts_server;
typedef struct b2_tts_chunk {
    uint64_t tag;            /* the caller's tag */
    int64_t call;            /* engine call that produced this record (0, 1, ...; -1: cancelled before admission) */
    int64_t admit_call;      /* engine call at which the sentence was admitted (-1: never admitted) */
    int64_t t_submit_ns;     /* CLOCK_MONOTONIC: entry into b2_tts_server_submit */
    int64_t t_done_ns;       /* CLOCK_MONOTONIC: the call's bytes were in pinned host memory */
    int64_t g711_offset;     /* offset of this record's nbytes in the h_g711 buffer given to b2_tts_server_poll (-1 if none was given) */
    int32_t nbytes;          /* G.711 bytes of this sentence in this call (may be 0 on the ended record) */
    int32_t ended;           /* non-zero: the sentence's last record, nothing follows it; 2: ended by b2_tts_server_cancel */
} b2_tts_chunk;
typedef struct b2_tts_server_stats {
    uint64_t calls;          /* engine calls completed */
    uint64_t submitted, admitted, ended;
    uint64_t admission_rounds;
    uint64_t rows;           /* sum over calls of the rows handed to the decoder (live + retired) */
    uint64_t live_rows;      /* sum over calls of the rows that were still live on the device */
    uint64_t padded_rows;    /* scratch sessions added to tail launches to reach a graph bucket */
    uint64_t graph_launches, graphs_built, max_rows;
    uint64_t capacity;       /* sentences in flight at most (slots) */
    uint64_t depth;
} b2_tts_server_stats;
/* ctx needs post-net weights; law B2_LAW_ULAW / ALAW; depth: engine calls in flight (1..4); use_graphs: each call's tail is one CUDA graph
 * launch (rows padded to a bucket with the scratch session).  Reference defaults: threshold 0.5, minlenratio 0, maxlenratio 20. */
B2_API b2_tts_server *b2_tts_server_create(b2_ctx *ctx, b2_enc *enc, b2_dec *dec, int law, int depth, int use_graphs, float threshold,
                                           float minlenratio, float maxlenratio, uint64_t seed);
/* stops the threads (work in flight is abandoned), waits for the device and frees the server; ctx, enc and dec stay valid */
B2_API void b2_tts_server_destroy(b2_tts_server *s);
/* n sentences: h_lens[n] token counts, h_ids[sum(h_lens)] int32 host token ids in [0, vocab) back to back, h_speakers (n, 512) fp32 host
 * (normalised on the device as b2_dec_start does), tags[n] the caller's ids.  Rejected with nothing enqueued: NULL pointers, a sentence of
 * no token, more tokens than the encoder's max_len / max_tokens or the decoder's max_enc_len, a token id outside the vocabulary.  Blocks
 * while every slot is taken by a sentence that has not ended (back-pressure) and fails after 20 s of that.  Sentences enqueued together
 * (all of them when the slots allow) are admitted in one round. */
B2_API int b2_tts_server_submit(b2_tts_server *s, const int32_t *h_ids, const int32_t *h_lens, int n, const float *h_speakers, const uint64_t *tags);
/* Cancels every sentence submitted with one of tags[0..n) whose last record has not been made yet.  Any thread; never waits for the GPU.
 * Tags need not be unique: every matching sentence is cancelled.  Returns the number of sentences found (pending, or admitted and not yet
 * known on the host to have ended); an unknown tag, a sentence that has ended and a second cancel of the same sentence count 0.  Negative
 * on a NULL server, n < 0, tags == NULL with n > 0, or a stopped server. */
B2_API int b2_tts_server_cancel(b2_tts_server *s, const uint64_t *tags, int n);
/* up to max_out records, oldest call first; their bytes are copied to h_g711 (may be NULL) at out[i].g711_offset (a record whose bytes
 * do not fit waits for the next poll).  timeout_ms: 0 = do not wait, < 0 = wait.  Returns the count, or a negative value on error. */
B2_API int b2_tts_server_poll(b2_tts_server *s, b2_tts_chunk *out, int max_out, uint8_t *h_g711, size_t g711_capacity, int timeout_ms);
/* returns when every sentence submitted so far has ended (its records may still be waiting for b2_tts_server_poll) */
B2_API int b2_tts_server_flush(b2_tts_server *s, int timeout_ms);
B2_API int b2_tts_server_get_stats(b2_tts_server *s, b2_tts_server_stats *out);

/* ---- Core/Codecs (G711.py:25-47), ctx-less, stateless ----------------------------------------------- */
/* G711Codec.encode: clamp(x*32767,-32768,32767) -> int16 (trunc toward zero) -> G.711 code.  n samples. */
B2_API int b2_g711_encode_f32(const float *d_in, size_t n, int law, uint8_t *d_out, void *stream);
B2_API int b2_g711_encode_i16(const int16_t *d_in, size_t n, int law, uint8_t *d_out, void *stream);
/* the float -> int16 step on its own (G711.py:27) */
B2_API int b2_f32_to_pcm16(const float *d_in, size_t n, int16_t *d_out, void *stream);
/* G711Codec.decode without resampling: code -> int16 -> float / 32767.0 */
B2_API int b2_g711_decode_f32(const uint8_t *d_in, size_t n, int law, float *d_out, void *stream);
B2_API int b2_g711_decode_i16(const uint8_t *d_in, size_t n, int law, int16_t *d_out, void *stream);
/* fused resampler + encoder: (rows, L) fp32 @16k -> (rows, ceil(L/2)) G.711 bytes @8k */
B2_API int b2_resample_g711_encode(const float *d_in, size_t rows, size_t L, int law, uint8_t *d_out, void *stream);
/* G711Codec.decode(resample=True, sample_rate=16000): (rows, L) bytes @8k -> (rows, 2L) fp32 @16k
 * (G711.py:44-46 -> Core/AudioChunk.py:19-24 -> config/InfernGlobals.py:23-26) */
B2_API int b2_g711_decode_upsample(const uint8_t *d_in, size_t rows, size_t L, int law, float *d_out, void *stream);
/* AudioChunk.resample 8k -> 16k on its own: (rows, L) -> (rows, 2L) */
B2_API int b2_resample_1to2(const float *d_in, size_t rows, size_t L, float *d_out, void *stream);
/* Batched inbound decode (SURVEY 8 f4; RTP/InfernRTPIngest.py:63-100 decodes per packet group, feeding Core/VAD/SileroVAD.py:27-35 and
 * Cluster/STTSession.py:93-94): `rows` packets of ANY lengths in one launch.  Row r = bytes [offsets[r], offsets[r+1]) of d_in; output row r
 * starts at float offsets[r] (x2 when upsample != 0: 8k -> 16k with the per-call zero padding of Core/AudioChunk.py:19-24 at each row's ends). */
B2_API int b2_g711_decode_ragged(const uint8_t *d_in, const unsigned long long *d_offsets, size_t rows, int law, int upsample, float *d_out, void *stream);
/* same from HOST memory: one H2D, one launch (the flat kernels when all rows have one length), one D2H, stream synchronised on return */
B2_API int b2_g711_decode_many_host(const uint8_t *h_in, const unsigned long long *h_offsets, size_t rows, int law, int upsample, float *h_out, void *stream);

/* ---- single-layer entry points (unit tests of the two convolution kernel families) -----------------
 * One Conv1d(Cin, Cout, k, dilation=dil, padding=(k-1)*dil/2) over channels-last activations [W][T][C]:
 *   h_weight torch layout [Cout][Cin][k] fp32 host, h_bias [Cout] host; d_residual / d_out32 fp32 [W][T][Cout] (may be NULL);
 *   d_outb bf16 [W][T][Cout] = bf16(leaky_relu(out, slope)) (may be NULL); out is divided by `div` first.
 * b2_conv1d_tc : tcgen05 kernel, d_in bf16 (already activated).   b2_conv1d_f32 : CUDA-core kernel, d_in fp32,
 * leaky_relu(pre_slope) applied to the input. */
B2_API int b2_conv1d_tc(const void *d_in_bf16, const float *h_weight, const float *h_bias, int W, int T, int Cin, int Cout, int k, int dil,
                        const float *d_residual, float *d_out32, void *d_outb, float slope, float div, void *stream);
B2_API int b2_conv1d_f32(const float *d_in, const float *h_weight, const float *h_bias, int W, int T, int Cin, int Cout, int k, int dil,
                         float pre_slope, const float *d_residual, float *d_out32, void *d_outb, float slope, float div, void *stream);
/* One Linear of the text encoder / speech decoder, C = act(A W^T + b) * colscale, through the same packing and launch (tile choice included)
 * their passes use.  mode B2_MODE_BF16: d_in bf16 [a_rows][K], tcgen05 GEMM, d_out32 fp32 [M][N] and/or d_outb bf16 [M][N];
 * B2_MODE_FP32: d_in fp32 [M][K], CUDA-core kernel, d_out32 only.  h_weight [N][K] and h_bias [N] host fp32 (torch layout); d_colscale [N]
 * or NULL; act 0/1/2 = none / ReLU / GELU (erf).  a_rows >= M: rows the A tensor map spans (the encoder's and decoder's maps span their
 * workspace, not the pass).  h_launched (may be NULL) receives {tile N, ring stages} of the launch ({0, 0} in fp32 mode).
 * K and N multiples of 64; M = 0 does nothing.  Synchronous on `stream`. */
B2_API int b2_linear(int device, int mode, const void *d_in, int M, int a_rows, const float *h_weight, const float *h_bias, int N, int K,
                     int act, const float *d_colscale, float *d_out32, void *d_outb, int *h_launched, void *stream);

/* One whole HiFiGAN ResBlock (modeling_speecht5.py:2903-2962) in a single fused tcgen05 launch:
 *   for d in (d0, d1, d2): x = x + conv2(lrelu(conv1_dil_d(lrelu(x, slope)), slope));   v = (d_acc + x) / div
 * d_x fp32 [W][T][C]; h_weights [6][C][C][k] torch layout in the order pair0.conv1, pair0.conv2, pair1.conv1, ...; h_biases [6][C];
 * d_acc optional fp32 [W][T][C]; d_out32 fp32 / d_outb bf16(lrelu(v, outb_slope)) [W][T][C], either may be NULL.  C in {32, 64, 128}. */
B2_API int b2_resblock_tc(const float *d_x, const float *h_weights, const float *h_biases, int W, int T, int C, int k, int d0, int d1, int d2,
                          const float *d_acc, float *d_out32, void *d_outb, float slope, float outb_slope, float div, void *stream);

/* Slab geometry of the stacked-output C = 32 ResBlock kernel (csrc/conv_resblock_t.cu) for a window of T time steps, k taps, dilations
 * d0..d2 (`post` bit 0: conv_post fused, three more halo rows; bit 1: the stage's upsampler fused, tiles start on a multiple of four rows).
 * Host arithmetic only -- no device is touched; exported so that the CPU tests
 * can run the index-exact numpy model of the kernel (tools/resblock_t_model.py) on the library's own plan.
 * out[10] = {S rows per slab, H halo, V output rows per tile, tiles per window, off[0..2], lim[0..2]}: conv1 of pair i reads slab rows
 * [off[i], off[i] + lim[i]) through the operand mapping of dilation d_i.  Returns non-zero (b2_last_error) when the kernel does not cover the shape. */
B2_API int b2_resblock_t_plan(int k, int d0, int d1, int d2, int T, int post, int *out);
/* Test hook: C = 32 ResBlocks with at least k taps run the stacked-output kernel (default 5; measured: three-tap blocks are
 * faster on the time-as-M kernel).  k <= 0 restores the default.  Process-wide; not for concurrent use with running launches. */
B2_API int b2_debug_set_stacked_min_taps(int k);

/* ---- bookkeeping the benchmark reports ------------------------------------------------------------- */
/* number of kernels this library has launched in this process since load (all contexts) */
B2_API uint64_t b2_kernel_launch_count(void);
/* Per-kernel-class device timing (CUDA events on the launching stream around every launch of this context)
 * between b2_profile_begin and b2_profile_end.  Classes: 0 tcgen05 convs, 1 CUDA-core convs, 2 conv_post+tanh,
 * 3 resample+G.711, 4 other (window builder, chunker prologue/epilogue), 5 fused tcgen05 ResBlock kernel.  Arrays of 8. */
B2_API int b2_profile_begin(b2_ctx *ctx);
B2_API int b2_profile_end(b2_ctx *ctx, double *ms_by_class, uint64_t *launches_by_class);

#ifdef __cplusplus
}
#endif
#endif /* INFERNOS_B200_H */
