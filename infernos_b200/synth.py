"""Seeded synthetic weights and inputs for the TTS tail.

There is no network on the build or GPU boxes, so the HuggingFace checkpoints the
reference loads (``microsoft/speecht5_hifigan``, ``sobomax/speecht5-rt.post_vocoder.v2``,
/root/reference/HelloSippyTTSRT/HelloSippyRTPipe.py:171-176) are replaced by random
weights with the same state_dict keys and shapes.  transformers' default init
(std 0.01) gives |audio| ~ 2e-5 and makes every tolerance vacuous, so the weights are
drawn at ~1/sqrt(fan_in) instead, which yields O(1) audio (SURVEY.md section 8d).

State-dict layouts follow the reference modules exactly:
  * HiFiGAN : transformers SpeechT5HifiGan (modeling_speecht5.py:2974-3010)
  * chunker : AmendmentNetwork1 (/root/reference/HelloSippyTTSRT/HelloSippyRT.py:202-217)
  * post-net: transformers SpeechT5SpeechDecoderPostnet.layers (modeling_speecht5.py:700-750)
"""
from __future__ import annotations

import math
from typing import Dict

import torch

HIFIGAN_SEED = 1234
CHUNKER_SEED = 4321
MEL_SEED = 7
POSTNET_SEED = 2468

UPSAMPLE_INITIAL_CHANNEL = 512
UPSAMPLE_RATES = (4, 4, 4, 4)
UPSAMPLE_KERNELS = (8, 8, 8, 8)
RESBLOCK_KERNELS = (3, 7, 11)
RESBLOCK_DILATIONS = (1, 3, 5)
NUM_MELS = 80


def _conv_w(g, cout, cin, k, fan_in=None):
    fan_in = cin * k if fan_in is None else fan_in
    return torch.randn(cout, cin, k, generator=g) / math.sqrt(fan_in)


def _bias(g, n):
    return torch.randn(n, generator=g) * 0.01


def hifigan_state_dict(seed: int = HIFIGAN_SEED) -> Dict[str, torch.Tensor]:
    """Random SpeechT5HifiGan weights (default SpeechT5HifiGanConfig), fp32, CPU."""
    g = torch.Generator().manual_seed(seed)
    sd: Dict[str, torch.Tensor] = {}
    sd["mean"] = torch.randn(NUM_MELS, generator=g) * 0.5 - 4.0
    sd["scale"] = torch.rand(NUM_MELS, generator=g) * 1.5 + 1.0
    sd["conv_pre.weight"] = _conv_w(g, UPSAMPLE_INITIAL_CHANNEL, NUM_MELS, 7)
    sd["conv_pre.bias"] = _bias(g, UPSAMPLE_INITIAL_CHANNEL)
    ch = UPSAMPLE_INITIAL_CHANNEL
    for i, (r, k) in enumerate(zip(UPSAMPLE_RATES, UPSAMPLE_KERNELS)):
        cin, cout = ch, ch // 2
        # ConvTranspose1d weight is (in, out, k); each output sees k/stride taps per input channel
        w = torch.randn(cin, cout, k, generator=g) / math.sqrt(cin * k / r)
        sd[f"upsampler.{i}.weight"] = w
        sd[f"upsampler.{i}.bias"] = _bias(g, cout)
        for j, rk in enumerate(RESBLOCK_KERNELS):
            n = i * len(RESBLOCK_KERNELS) + j
            for d in range(len(RESBLOCK_DILATIONS)):
                # He gain on conv1 so the residual branches carry about as much energy as the trunk
                sd[f"resblocks.{n}.convs1.{d}.weight"] = _conv_w(g, cout, cout, rk) * math.sqrt(2.0)
                sd[f"resblocks.{n}.convs1.{d}.bias"] = _bias(g, cout)
                sd[f"resblocks.{n}.convs2.{d}.weight"] = _conv_w(g, cout, cout, rk)
                sd[f"resblocks.{n}.convs2.{d}.bias"] = _bias(g, cout)
        ch = cout
    sd["conv_post.weight"] = _conv_w(g, 1, ch, 7) * 0.5
    sd["conv_post.bias"] = _bias(g, 1)
    return sd


def chunker_state_dict(seed: int = CHUNKER_SEED) -> Dict[str, torch.Tensor]:
    """Random AmendmentNetwork1 weights, fp32, CPU."""
    g = torch.Generator().manual_seed(seed)
    sd: Dict[str, torch.Tensor] = {}
    sd["conv_pre_m.weight"] = _conv_w(g, 32, 80, 3)
    sd["conv_pre_m.bias"] = _bias(g, 32)
    sd["conv_pre_a.weight"] = _conv_w(g, 160, 256, 3, fan_in=256 * 3 * 0.05)  # audio is ~0.2 rms
    sd["conv_pre_a.bias"] = _bias(g, 160)
    sd["upsampler.0.weight"] = torch.randn(192, 128, 8, generator=g) / math.sqrt(192 * 2)
    sd["upsampler.0.bias"] = _bias(g, 128)
    sd["upsampler.1.weight"] = torch.randn(128, 64, 8, generator=g) / math.sqrt(128 * 2)
    sd["upsampler.1.bias"] = _bias(g, 64)
    sd["resblock.conv1.weight"] = _conv_w(g, 64, 64, 3)
    sd["resblock.conv1.bias"] = _bias(g, 64)
    sd["resblock.conv2.weight"] = _conv_w(g, 64, 64, 3)
    sd["resblock.conv2.bias"] = _bias(g, 64)
    sd["post_conv.weight"] = _conv_w(g, 256, 64, 8)
    sd["post_conv.bias"] = _bias(g, 256) + 1.0  # gains centred near 1 like a trained seam-smoother
    return sd


def postnet_state_dict(seed: int = POSTNET_SEED) -> Dict[str, torch.Tensor]:
    """Random weights with the `layers.*` keys of transformers SpeechT5SpeechDecoderPostnet (default SpeechT5Config: 5 layers,
    256 units, kernel 5; modeling_speecht5.py:700-750), fp32, CPU.  Scaled so that the tanh layers work in their curved range
    on synth_mel-like inputs (pre-activations ~ N(0, 1)), with non-trivial batch-norm statistics."""
    g = torch.Generator().manual_seed(seed)
    sd: Dict[str, torch.Tensor] = {}
    for i in range(5):
        cin = NUM_MELS if i == 0 else 256
        cout = NUM_MELS if i == 4 else 256
        gain = 1.0 / 4.5 if i == 0 else 1.6          # layer 0 sees mel ~ N(-4, 2^2); the others see tanh outputs (rms ~0.6)
        sd[f"layers.{i}.conv.weight"] = _conv_w(g, cout, cin, 5) * gain
        sd[f"layers.{i}.batch_norm.weight"] = torch.rand(cout, generator=g) * 0.6 + 0.7
        sd[f"layers.{i}.batch_norm.bias"] = torch.randn(cout, generator=g) * 0.1
        sd[f"layers.{i}.batch_norm.running_mean"] = torch.randn(cout, generator=g) * 0.2
        sd[f"layers.{i}.batch_norm.running_var"] = torch.rand(cout, generator=g) * 1.0 + 0.5
    return sd


def synth_mel(batch: int, nframes: int, seed: int = MEL_SEED) -> torch.Tensor:
    """Log-mel-like input: randn*2-4, shape (batch, nframes, 80), fp32, CPU."""
    g = torch.Generator().manual_seed(seed)
    return torch.randn(batch, nframes, NUM_MELS, generator=g) * 2.0 - 4.0


def synth_audio(batch: int, nsamples: int, seed: int = 20240101) -> torch.Tensor:
    """U(-0.9, 0.9) audio used by the codec sweeps (SURVEY.md App. A.4, vector G2)."""
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(batch, nsamples, generator=g) * 2 - 1) * 0.9


DECODER_SEED = 1357
# Gains of the random decoder.  With larger ones (He-style 1.4, sharper attention) the autoregressive loop is chaotic: a 1e-5 perturbation of
# the first frame grows to O(1) within ~10 steps, so no two summation orders (let alone bf16) agree and a parity test means nothing.  With
# these the loop is neutral (the same perturbation stays ~5e-6 over 48 steps) while every frame still depends on the previous one.
G_PRE0, G_PRE1, G_FINAL, G_SPK, G_QK, G_FFN, G_FEAT = 0.3, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0
DEC_HIDDEN, DEC_LAYERS, DEC_HEADS, DEC_FFN, DEC_PRENET_UNITS, DEC_SPK_DIM, DEC_REDUCTION = 768, 6, 12, 3072, 256, 512, 2


def decoder_state_dict(seed: int = DECODER_SEED) -> Dict[str, torch.Tensor]:
    """Random weights with the state_dict keys of the SpeechT5 speech decoder as the reference uses it (HelloSippyRTPipe.py:195-216):
    `speecht5.decoder.prenet.*`, `speecht5.decoder.wrapped_decoder.layers.{0..5}.*` and `speech_decoder_postnet.{feat_out,prob_out}.*`
    (default SpeechT5Config: hidden 768, 6 layers, 12 heads, FFN 3072, prenet 2 x 256, speaker 512, reduction factor 2;
    modeling_speecht5.py:648-697, 1070-1160, 740-750), fp32, CPU.  Scaled so that activations stay O(1), feat_out emits
    log-mel-like frames (~N(-4, 1)) and the stop probability stays low."""
    g = torch.Generator().manual_seed(seed)

    def lin(cout, cin, gain=1.0):
        return torch.randn(cout, cin, generator=g) * (gain / math.sqrt(cin))

    sd: Dict[str, torch.Tensor] = {}
    P = "speecht5.decoder.prenet."
    sd[P + "layers.0.weight"] = lin(DEC_PRENET_UNITS, NUM_MELS, G_PRE0)          # inputs are mel frames ~N(-4, 1): keep pre-activations O(1)
    sd[P + "layers.0.bias"] = _bias(g, DEC_PRENET_UNITS) + 0.5
    sd[P + "layers.1.weight"] = lin(DEC_PRENET_UNITS, DEC_PRENET_UNITS, G_PRE1)
    sd[P + "layers.1.bias"] = _bias(g, DEC_PRENET_UNITS) + 0.2
    sd[P + "final_layer.weight"] = lin(DEC_HIDDEN, DEC_PRENET_UNITS, G_FINAL)
    sd[P + "final_layer.bias"] = _bias(g, DEC_HIDDEN)
    sd[P + "encode_positions.alpha"] = torch.tensor(0.7)
    sd[P + "speaker_embeds_layer.weight"] = lin(DEC_HIDDEN, DEC_HIDDEN + DEC_SPK_DIM, G_SPK)
    sd[P + "speaker_embeds_layer.bias"] = _bias(g, DEC_HIDDEN)
    for i in range(DEC_LAYERS):
        L = f"speecht5.decoder.wrapped_decoder.layers.{i}."
        for att in ("self_attn", "encoder_attn"):
            for pj in ("k_proj", "v_proj", "q_proj", "out_proj"):
                sd[L + f"{att}.{pj}.weight"] = lin(DEC_HIDDEN, DEC_HIDDEN, G_QK if pj in ("q_proj", "k_proj") else 1.0)
                sd[L + f"{att}.{pj}.bias"] = _bias(g, DEC_HIDDEN)
            sd[L + f"{att}_layer_norm.weight"] = torch.rand(DEC_HIDDEN, generator=g) * 0.4 + 0.8
            sd[L + f"{att}_layer_norm.bias"] = _bias(g, DEC_HIDDEN) * 5
        sd[L + "feed_forward.intermediate_dense.weight"] = lin(DEC_FFN, DEC_HIDDEN, 1.0)
        sd[L + "feed_forward.intermediate_dense.bias"] = _bias(g, DEC_FFN)
        sd[L + "feed_forward.output_dense.weight"] = lin(DEC_HIDDEN, DEC_FFN, G_FFN)
        sd[L + "feed_forward.output_dense.bias"] = _bias(g, DEC_HIDDEN)
        sd[L + "final_layer_norm.weight"] = torch.rand(DEC_HIDDEN, generator=g) * 0.4 + 0.8
        sd[L + "final_layer_norm.bias"] = _bias(g, DEC_HIDDEN) * 5
    sd["speech_decoder_postnet.feat_out.weight"] = lin(NUM_MELS * DEC_REDUCTION, DEC_HIDDEN, G_FEAT)
    sd["speech_decoder_postnet.feat_out.bias"] = _bias(g, NUM_MELS * DEC_REDUCTION) - 4.0
    sd["speech_decoder_postnet.prob_out.weight"] = lin(DEC_REDUCTION, DEC_HIDDEN, 1.0)
    sd["speech_decoder_postnet.prob_out.bias"] = torch.full((DEC_REDUCTION,), -3.0)
    return sd


def synth_encoder_states(batch: int, length: int, seed: int = 99) -> torch.Tensor:
    """Stand-in for `encoder_last_hidden_state` (B, L, 768): the text encoder is context glue outside the path (HelloSippyRTPipe.py:111-116)."""
    g = torch.Generator().manual_seed(seed)
    return torch.randn(batch, length, DEC_HIDDEN, generator=g)


def synth_speakers(batch: int, seed: int = 98) -> torch.Tensor:
    g = torch.Generator().manual_seed(seed)
    return torch.randn(batch, DEC_SPK_DIM, generator=g) * 3.0


ENCODER_SEED = 2029
ENC_LAYERS, ENC_VOCAB, ENC_MAX_REL = 12, 81, 160
# Gains of the random text encoder.  q / k at 1.4 / sqrt(fan_in) and pe_k rows at std 1.4 put both terms of the attention score (q.k and the
# relative-position term q.pe_k, each with the 1/8-scaled q) at a spread of about 2: the softmax is far from uniform, and a sign or clamp error
# in the relative positions changes the output at O(1).  The post-LN layers keep the residual stream at unit scale whatever the gains.
G_ENC_QK, G_ENC_PEK, G_ENC_FFN1 = 1.4, 1.4, 1.4


def encoder_state_dict(seed: int = ENCODER_SEED) -> Dict[str, torch.Tensor]:
    """Random weights with the `speecht5.encoder.*` state_dict keys of transformers SpeechT5ForTextToSpeech (SpeechT5EncoderWithTextPrenet,
    default SpeechT5Config: vocab 81, hidden 768, 12 layers, 12 heads, FFN 3072, relative positions +-160; modeling_speecht5.py:765-781,
    1013-1066, 1230-1320), fp32, CPU.  The sinusoidal table `prenet.encode_positions.pe` is a non-persistent buffer and is not included."""
    g = torch.Generator().manual_seed(seed)

    def lin(cout, cin, gain=1.0):
        return torch.randn(cout, cin, generator=g) * (gain / math.sqrt(cin))

    sd: Dict[str, torch.Tensor] = {}
    P, W = "speecht5.encoder.prenet.", "speecht5.encoder.wrapped_encoder."
    sd[P + "embed_tokens.weight"] = torch.randn(ENC_VOCAB, DEC_HIDDEN, generator=g)
    sd[P + "encode_positions.alpha"] = torch.tensor(0.8)
    sd[W + "layer_norm.weight"] = torch.rand(DEC_HIDDEN, generator=g) * 0.4 + 0.8
    sd[W + "layer_norm.bias"] = _bias(g, DEC_HIDDEN) * 5
    sd[W + "embed_positions.pe_k.weight"] = torch.randn(2 * ENC_MAX_REL, DEC_HIDDEN // DEC_HEADS, generator=g) * G_ENC_PEK
    for i in range(ENC_LAYERS):
        L = W + f"layers.{i}."
        for pj in ("k_proj", "v_proj", "q_proj", "out_proj"):
            sd[L + f"attention.{pj}.weight"] = lin(DEC_HIDDEN, DEC_HIDDEN, G_ENC_QK if pj in ("q_proj", "k_proj") else 1.0)
            sd[L + f"attention.{pj}.bias"] = _bias(g, DEC_HIDDEN)
        sd[L + "layer_norm.weight"] = torch.rand(DEC_HIDDEN, generator=g) * 0.4 + 0.8
        sd[L + "layer_norm.bias"] = _bias(g, DEC_HIDDEN) * 5
        sd[L + "feed_forward.intermediate_dense.weight"] = lin(DEC_FFN, DEC_HIDDEN, G_ENC_FFN1)
        sd[L + "feed_forward.intermediate_dense.bias"] = _bias(g, DEC_FFN)
        sd[L + "feed_forward.output_dense.weight"] = lin(DEC_HIDDEN, DEC_FFN, 1.0)
        sd[L + "feed_forward.output_dense.bias"] = _bias(g, DEC_HIDDEN)
        sd[L + "final_layer_norm.weight"] = torch.rand(DEC_HIDDEN, generator=g) * 0.4 + 0.8
        sd[L + "final_layer_norm.bias"] = _bias(g, DEC_HIDDEN) * 5
    return sd


def synth_token_ids(lengths, seed: int = 97) -> tuple:
    """Right-padded token ids (B, max(lengths)) int64 in [4, 81) (0..3 are the tokenizer's special ids) and the matching 0/1 attention mask."""
    g = torch.Generator().manual_seed(seed)
    L = max(lengths)
    ids = torch.randint(4, ENC_VOCAB, (len(lengths), L), generator=g)
    mask = (torch.arange(L)[None] < torch.tensor(list(lengths))[:, None]).to(torch.int)
    return ids * mask + (1 - mask), mask               # padding id 1 (SpeechT5's pad_token_id)
