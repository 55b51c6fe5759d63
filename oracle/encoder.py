"""ORACLE (test infrastructure, never shipped, never on the product path).

CPU restatement, in plain torch functional ops, of the SpeechT5 text encoder the reference runs once per sentence
(/root/reference/HelloSippyTTSRT/HelloSippyRTPipe.py:111-116): transformers SpeechT5EncoderWithTextPrenet in eval mode

    prenet            x = embed_tokens[id] + alpha * pe[pos]                      modeling_speecht5.py:765-781, :400-422
    layer_norm        before the layers; no final norm                            :1292
    twelve layers     h = LN1(x + out_proj(attn(x))); x = LN2(h + FFN(h))          :1013-1066 (FFN :989-1010, erf GELU)
    attention         q scaled by 1/8; score = q.k + q.pe_k[clamp(i - j, -160, 159) + 160], padded keys masked   :837-1000, :425-442

[third-party, transformers 5.5.0 in this image]

Pinned by tests/test_oracle_encoder.py to the LIVE module (oracle/make_golden_encoder.py builds it) and to tests/golden/encoder_golden.npz.
Only tests/, smoke() and bench.py's CPU legs may import this module.
"""
from __future__ import annotations

from typing import Dict, Optional

import torch
import torch.nn.functional as F

from oracle.decoder import position_table

HIDDEN, LAYERS, HEADS, HEAD_DIM, MAX_REL, MAX_TEXT_POSITIONS = 768, 12, 12, 64, 160, 450
P = "speecht5.encoder.prenet."
W = "speecht5.encoder.wrapped_encoder."


def rel_index(L: int, rel: str = "clamp") -> torch.Tensor:
    """(L, L) rows of pe_k used by score[i][j] (SpeechT5RelativePositionalEncoding.forward, :434-442).  rel="flip" (j - i) and rel="wrap"
    (no clamp: the index wraps around the 320-row table) are the two mistakes tests/test_oracle_encoder.py shows the weights can tell apart."""
    i = torch.arange(L)
    d = i[:, None] - i[None, :]
    if rel == "flip":
        d = -d
    if rel == "wrap":
        return (d + MAX_REL) % (2 * MAX_REL)
    return d.clamp(-MAX_REL, MAX_REL - 1) + MAX_REL


def _heads(x):                                                                                  # (B, T, 768) -> (B, 12, T, 64)
    B, T, _ = x.shape
    return x.view(B, T, HEADS, HEAD_DIM).transpose(1, 2)


def encoder_forward(sd: Dict[str, torch.Tensor], ids: torch.Tensor, mask: Optional[torch.Tensor] = None, pe: Optional[torch.Tensor] = None,
                    rel: str = "clamp") -> torch.Tensor:
    """ids (B, L) int, mask (B, L) 0/1 (None: all valid) -> last_hidden_state (B, L, 768) fp32.  Rows at padded positions are computed like the
    module computes them (their keys are masked like everyone else's); only valid positions are compared anywhere."""
    B, L = ids.shape
    pe = position_table(L) if pe is None else pe
    x = F.embedding(ids.long(), sd[P + "embed_tokens.weight"]) + sd[P + "encode_positions.alpha"] * pe[:L]          # :779-780, :420
    x = F.layer_norm(x, (HIDDEN,), sd[W + "layer_norm.weight"], sd[W + "layer_norm.bias"], 1e-5)                    # :1292
    pk = sd[W + "embed_positions.pe_k.weight"][rel_index(L, rel)]                                                    # (L, L, 64)
    keep = torch.ones(B, L, dtype=torch.bool) if mask is None else mask.bool()
    for i in range(LAYERS):
        Lp = W + f"layers.{i}."
        a = Lp + "attention."
        q = _heads(F.linear(x, sd[a + "q_proj.weight"], sd[a + "q_proj.bias"]) * (HEAD_DIM ** -0.5))               # :891
        k = _heads(F.linear(x, sd[a + "k_proj.weight"], sd[a + "k_proj.bias"]))
        v = _heads(F.linear(x, sd[a + "v_proj.weight"], sd[a + "v_proj.bias"]))
        s = torch.matmul(q, k.transpose(2, 3)) + torch.einsum("bhid,ijd->bhij", q, pk)                              # :925, :939-945
        s = s.masked_fill(~keep[:, None, None, :], torch.finfo(s.dtype).min)                                        # additive min == excluded
        o = torch.matmul(F.softmax(s, dim=-1), v).transpose(1, 2).reshape(B, L, HIDDEN)
        o = F.linear(o, sd[a + "out_proj.weight"], sd[a + "out_proj.bias"])
        x = F.layer_norm(x + o, (HIDDEN,), sd[Lp + "layer_norm.weight"], sd[Lp + "layer_norm.bias"], 1e-5)          # :1052-1055
        f = F.gelu(F.linear(x, sd[Lp + "feed_forward.intermediate_dense.weight"], sd[Lp + "feed_forward.intermediate_dense.bias"]))
        f = F.linear(f, sd[Lp + "feed_forward.output_dense.weight"], sd[Lp + "feed_forward.output_dense.bias"])
        x = F.layer_norm(x + f, (HIDDEN,), sd[Lp + "final_layer_norm.weight"], sd[Lp + "final_layer_norm.bias"], 1e-5)   # :1056-1057
    return x
