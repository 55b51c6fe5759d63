"""Pins oracle/encoder.py (the CPU restatement of the SpeechT5 text encoder) to the LIVE transformers SpeechT5EncoderWithTextPrenet on the
synthetic weights (infernos_b200.synth.encoder_state_dict) and to the committed golden (tests/golden/encoder_golden.npz, made by
oracle/make_golden_encoder.py), and checks that those weights can tell a wrong relative-position term from the right one."""
import os

import numpy as np
import pytest
import torch

from infernos_b200 import synth
from oracle import encoder as oenc

tr = pytest.importorskip("transformers")
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

from oracle.make_golden_encoder import live_run  # noqa: E402  (the real module)


@pytest.fixture(scope="module")
def sd():
    return synth.encoder_state_dict()


def _valid_max_abs(a, b, mask):
    m = mask.bool()
    return float((a[m] - b[m]).abs().max())


def test_oracle_matches_the_live_module_on_a_padded_ragged_batch(sd):
    ids, mask = synth.synth_token_ids((23, 8, 1, 17), seed=11)
    ref = live_run(sd, ids, mask)
    with torch.no_grad():
        got = oenc.encoder_forward(sd, ids, mask)
    err = _valid_max_abs(ref, got, mask)
    print(f"oracle vs live encoder, ragged batch: max |d| {err:.2e}, output rms {float(ref[mask.bool()].std()):.2f}")
    assert err <= 1e-5


def test_oracle_matches_the_live_module_past_the_relative_position_clamp(sd):
    ids, mask = synth.synth_token_ids((300,), seed=12)
    ref = live_run(sd, ids, mask)
    with torch.no_grad():
        got = oenc.encoder_forward(sd, ids, mask)
    err = _valid_max_abs(ref, got, mask)
    print(f"oracle vs live encoder, L = 300: max |d| {err:.2e}")
    assert err <= 1e-5


def test_oracle_reproduces_the_committed_golden(sd):
    d = np.load(os.path.join(G, "encoder_golden.npz"))
    ids, mask = torch.from_numpy(d["ids"]), torch.from_numpy(d["mask"])
    assert int(mask.sum(1).max()) > 160 and mask.size(0) == 3
    with torch.no_grad():
        got = oenc.encoder_forward(sd, ids, mask)[mask.bool()]
    assert float(np.abs(got.numpy() - d["out_valid"]).max()) <= 1e-5


def test_synthetic_weights_are_sensitive_to_the_relative_position_term(sd):
    """j - i instead of i - j, or no clamp at +-160, must move the outputs far more than the 1e-3 parity bar; the attention is not uniform."""
    ids, mask = synth.synth_token_ids((200,), seed=13)
    with torch.no_grad():
        ref = oenc.encoder_forward(sd, ids, mask)
        flip = oenc.encoder_forward(sd, ids, mask, rel="flip")
        wrap = oenc.encoder_forward(sd, ids, mask, rel="wrap")
    d_flip, d_wrap = float((ref - flip).abs().max()), float((ref - wrap).abs().max())
    print(f"max |d| with j - i: {d_flip:.3f}; without the clamp: {d_wrap:.3f}")
    assert d_flip > 0.1 and d_wrap > 0.1
    # the first layer's attention: the largest weight of a row is far above uniform (1 / L)
    x = torch.nn.functional.layer_norm(torch.nn.functional.embedding(ids, sd[oenc.P + "embed_tokens.weight"]) +
                                       sd[oenc.P + "encode_positions.alpha"] * oenc.position_table(200),
                                       (768,), sd[oenc.W + "layer_norm.weight"], sd[oenc.W + "layer_norm.bias"], 1e-5)
    a = oenc.W + "layers.0.attention."
    q = oenc._heads(torch.nn.functional.linear(x, sd[a + "q_proj.weight"], sd[a + "q_proj.bias"]) / 8)
    k = oenc._heads(torch.nn.functional.linear(x, sd[a + "k_proj.weight"], sd[a + "k_proj.bias"]))
    pk = sd[oenc.W + "embed_positions.pe_k.weight"][oenc.rel_index(200)]
    qk, rel = q @ k.transpose(2, 3), torch.einsum("bhid,ijd->bhij", q, pk)
    assert 0.5 < float(rel.std() / qk.std()) < 2.0                          # the two terms are comparable
    assert float(torch.softmax(qk + rel, -1).max(-1).values.median()) > 10.0 / 200


def test_encoder_weights_have_the_module_keys_and_shapes(sd):
    from oracle.make_golden_encoder import live_encoder
    real = live_encoder(sd).state_dict()
    assert set("speecht5.encoder." + k for k in real) == set(sd)
    assert len(sd) == 197
