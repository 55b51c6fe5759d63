"""Freezes tests/golden/encoder_golden.npz from the LIVE transformers SpeechT5EncoderWithTextPrenet (eval mode) on
infernos_b200.synth.encoder_state_dict(): three right-padded sentences, the longest past the +-160 clamp of the relative positions.  Only the
valid positions are stored (packed, in sentence order) to keep the file small.  Run in the build container:  python -m oracle.make_golden_encoder

ORACLE / test infrastructure: nothing under infernos_b200/ imports this."""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

LENGTHS = (171, 37, 9)


def live_encoder(sd):
    """SpeechT5EncoderWithTextPrenet with `sd`'s `speecht5.encoder.*` tensors; the non-persistent sinusoidal buffer is rebuilt after to_empty."""
    import transformers as tr
    from oracle.decoder import position_table
    cfg = tr.SpeechT5Config()
    with torch.device("meta"):
        enc = tr.models.speecht5.modeling_speecht5.SpeechT5EncoderWithTextPrenet(cfg)
    enc = enc.to_empty(device="cpu")
    missing, unexpected = enc.load_state_dict({k[len("speecht5.encoder."):]: v for k, v in sd.items() if k.startswith("speecht5.encoder.")}, strict=False)
    assert not unexpected and set(missing) <= {"prenet.encode_positions.pe"}, (missing, unexpected)
    enc.prenet.encode_positions.pe = position_table(cfg.max_text_positions)[None]
    return enc.eval()


def live_run(sd, ids, mask):
    with torch.no_grad():
        return live_encoder(sd)(input_values=ids, attention_mask=mask, return_dict=True).last_hidden_state


def main():
    from infernos_b200 import synth
    ids, mask = synth.synth_token_ids(LENGTHS, seed=5)
    out = live_run(synth.encoder_state_dict(), ids, mask)
    valid = out[mask.bool()]                                   # (sum(LENGTHS), 768), sentence by sentence
    path = os.path.join(ROOT, "tests", "golden", "encoder_golden.npz")
    np.savez_compressed(path, ids=ids.numpy().astype(np.int32), mask=mask.numpy().astype(np.int32), out_valid=valid.numpy())
    print(path, tuple(valid.shape), float(valid.std()), os.path.getsize(path))


if __name__ == "__main__":
    main()
