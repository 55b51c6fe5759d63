"""GPU parity of the text encoder (b2_enc_*, engine.TTSEncoder) against oracle/encoder.py (pinned to the live transformers module by
tests/test_oracle_encoder.py) and against the golden produced by the REAL module (tests/golden/encoder_golden.npz).  fp32 mode: max-abs
<= 1e-3 at valid positions; bf16 mode: >= 40 dB SNR per sentence.  Plus the ragged-packing contract (a sentence's output is bitwise the same
alone, in a cohort or split over passes; padded rows are zero), the loud failures, and the whole chain token ids -> G.711."""
import os

import numpy as np
import pytest
import torch

from infernos_b200 import synth

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def sd():
    return synth.encoder_state_dict()


def _snr(ref, x):
    from oracle.tail import snr_db
    return snr_db(torch.as_tensor(ref), torch.as_tensor(x))


def _oracle(sd, ids, mask):
    from oracle import encoder as oenc
    with torch.no_grad():
        return oenc.encoder_forward(sd, ids, mask)


def _check(mode, ref_valid, got, mask, what):
    """ref_valid: (sum(len), 768) packed valid rows; got (B, L, 768) from the GPU."""
    m = mask.bool()
    if (~m).any():
        assert float(got[~m].abs().max()) == 0.0, "padded rows must be zero"
    lens = mask.sum(1).tolist()
    gv = got[m]
    err = float((gv - ref_valid).abs().max())
    snrs, o = [], 0
    for n in lens:
        snrs.append(_snr(ref_valid[o:o + n], gv[o:o + n]))
        o += n
    snr_all = _snr(ref_valid, gv)
    print(f"encoder {mode} {what}: max |d| {err:.2e}, SNR {snr_all:.1f} dB over the cohort, per sentence {', '.join(f'{s:.1f}' for s in snrs)} dB "
          f"(lengths {lens})")
    if mode == "fp32":
        assert err <= 1e-3
    else:
        # 40 dB over the cohort.  Per sentence the floor is lower: rounding the 48 Linears' weights to bf16 alone costs a 12-layer encoder 41-42 dB,
        # bf16 operands on top 38.8 dB for a one-token sentence (no attention averaging), 41 dB for longer ones -- measured by restating the oracle
        # with exactly those roundings (DESIGN.md section 4e); this kernel's figures match that restatement.
        assert snr_all >= 40.0 and min(snrs) >= 37.0


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_encoder_replays_the_real_modules_golden(sd, mode):
    """Three right-padded sentences (171, 37, 9 tokens: the longest past the +-160 clamp) against the live module's output and the oracle."""
    from infernos_b200.engine import TTSEncoder
    d = np.load(os.path.join(G, "encoder_golden.npz"))
    ids, mask = torch.from_numpy(d["ids"]), torch.from_numpy(d["mask"])
    enc = TTSEncoder("cuda:0", sd, mode=mode, max_tokens=512, max_len=256)
    try:
        out = enc(ids, mask)
        enc.poll_errors()
        got = out.cpu()
    finally:
        enc.close()
    assert got.shape == (3, ids.size(1), 768)
    _check(mode, torch.from_numpy(d["out_valid"]), got, mask, "vs the live module's golden")
    _check(mode, _oracle(sd, ids, mask)[mask.bool()], got, mask, "vs the oracle")


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_encoder_lengths_one_past_the_clamp_and_max_len(sd, mode):
    from infernos_b200.engine import TTSEncoder
    lengths = (1, 161, 200, 57)
    ids, mask = synth.synth_token_ids(lengths, seed=21)
    enc = TTSEncoder("cuda:0", sd, mode=mode, max_tokens=1024, max_len=200)
    try:
        got = enc(ids.cuda(), mask.cuda()).cpu()
        enc.poll_errors()
    finally:
        enc.close()
    _check(mode, _oracle(sd, ids, mask)[mask.bool()], got, mask, "lengths 1 / 161 / max_len 200 / 57")


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_encoder_output_is_bitwise_independent_of_companions_and_passes(sd, mode):
    """Sentence by sentence: alone (its own L), inside a padded cohort, and with max_tokens = 130 so that the cohort runs as three passes."""
    from infernos_b200.engine import TTSEncoder
    lengths = (70, 50, 100, 20, 90)
    ids, mask = synth.synth_token_ids(lengths, seed=22)
    big = TTSEncoder("cuda:0", sd, mode=mode, max_tokens=4096, max_len=128)
    small = TTSEncoder("cuda:0", sd, mode=mode, max_tokens=130, max_len=128)
    try:
        cohort = big(ids, mask).cpu()
        passes = small(ids, mask).cpu()
        alone = [big(ids[i:i + 1, :n], None).cpu()[0] for i, n in enumerate(lengths)]
        big.poll_errors(); small.poll_errors()
    finally:
        big.close(); small.close()
    for i, n in enumerate(lengths):
        assert torch.equal(cohort[i, :n], alone[i]), f"sentence {i}: cohort != alone"
        assert torch.equal(passes[i, :n], alone[i]), f"sentence {i}: three passes != alone"
    assert torch.equal(cohort, passes)


def test_encoder_fails_loudly_and_keeps_working(sd):
    from infernos_b200.engine import TTSEncoder
    enc = TTSEncoder("cuda:0", sd, mode="bf16", max_tokens=64, max_len=80)
    try:
        ids, mask = synth.synth_token_ids((30, 12), seed=23)
        ref = enc(ids, mask).cpu()
        with pytest.raises(RuntimeError, match="max_len"):
            enc(torch.full((1, 81), 5), None)
        with pytest.raises(RuntimeError, match="max_tokens"):
            enc(torch.full((1, 65), 5), None)
        bad_mask = mask.clone()
        bad_mask[0, 3] = 0
        with pytest.raises(RuntimeError, match="prefix"):
            enc(ids, bad_mask)
        bad = ids.clone()
        bad[1, 4] = 81
        enc(bad, mask)
        with pytest.raises(RuntimeError, match="token ids"):
            enc.poll_errors()
        again = enc(ids, mask).cpu()
        enc.poll_errors()
        assert torch.equal(again, ref)
    finally:
        enc.close()


def _char_tokenizer(text):
    return torch.tensor([[4 + (ord(c) % 77) for c in text]], dtype=torch.long)


def test_pipeline_from_state_dict_matches_the_oracle_chain():
    """HelloSippyRTPipe with B200Frontend.from_state_dict in fp32: token ids -> GPU encoder -> GPU decoder -> GPU post-net + tail ->
    unbatch_and_dispatch, against oracle encoder -> oracle decoder -> oracle post-net / tail with the same dropout masks."""
    import uuid
    from infernos_b200.HelloSippyTTSRT.HelloSippyRTPipe import (B200Frontend, HelloSippyPipeState, HelloSippyPipeStateBatched, HelloSippyPlayRequest,
                                                                 HelloSippyRTPipe)
    from oracle import decoder as odec
    from oracle import encoder as oenc
    from oracle import tail as otail
    esd, dsd = synth.encoder_state_dict(), synth.decoder_state_dict()
    vsd, csd, psd = synth.hifigan_state_dict(), synth.chunker_state_dict(), synth.postnet_state_dict()
    texts = ["first sentence", "the second one is longer"]
    g = torch.Generator().manual_seed(8)
    masks = [(torch.rand(16, 2, 256, generator=g) < 0.5).float() for _ in range(4)]
    fe = B200Frontend.from_state_dict({**esd, **dsd}, _char_tokenizer, "cuda:0", mode="fp32", max_sessions=4, max_steps=64, max_enc_len=32,
                                      max_tokens=256, mask_fn=lambda c: masks[c])
    pp = HelloSippyRTPipe("cuda:0", output_sr=8000, frontend=fe, vocoder_state_dict=vsd, chunker_state_dict=csd, postnet_state_dict=psd,
                          mode="fp32", max_sessions=4, speaker_embeddings=[synth.synth_speakers(1, seed=33)])
    pp.maxlenratio = 2.0                                    # maxlen = int(24 * 2 / 2) = 24 decoder steps: both sentences end in call 2
    got, ended = [[], []], [0, 0]

    def cb(i):
        def f(chunk):
            if chunk is None:
                ended[i] += 1
            else:
                got[i].append(chunk.clone())
        return f
    reqs = [HelloSippyPlayRequest(uuid.uuid4(), t, pp.get_voice(0), cb(i)) for i, t in enumerate(texts)]
    state = HelloSippyPipeStateBatched([HelloSippyPipeState(pp, r) for r in reqs], pp)
    assert (state.minlen, state.maxlen) == (0, 24)
    ncalls = 0
    while True:
        pp.infer(state)
        ncalls += 1
        if not pp.unbatch_and_dispatch(state):
            break
    fe.close()
    # oracle chain
    toks = [_char_tokenizer(t)[0] for t in texts]
    L = max(t.numel() for t in toks)
    ids = torch.stack([torch.nn.functional.pad(t, (0, L - t.numel()), value=1) for t in toks])
    emask = torch.stack([(torch.arange(L) < t.numel()).to(torch.int) for t in toks])
    with torch.no_grad():
        enc = oenc.encoder_forward(esd, ids, emask)
    st = odec.DecoderState(dsd, enc, emask, synth.synth_speakers(1, seed=33).repeat(2, 1))
    pre = torch.zeros(2, 4, 80)
    ends, idx, live, starts = [-1, -1], 0, [True, True], [1, 1]
    ref = [[], []]
    with torch.no_grad():
        for c in range(ncalls):
            frames = []
            for s in range(16):
                sp, pr = odec.step(dsd, st, masks[c][s])
                frames.append(sp)
                for i in range(2):
                    if ends[i] < 0 and (bool((pr[i] >= 0.5).any()) or 24 <= idx):
                        ends[i] = idx + 2
                idx += 1
            mel = otail.postnet_forward(psd, torch.cat(frames, 1))
            audio, pre = otail.tts_tail(vsd, csd, pre, mel)
            sl, fin, more = otail.unbatch_slices(audio.size(1), idx, starts, ends, live)
            for i in range(2):
                if sl[i] is not None:
                    ref[i].append(audio[i, sl[i][0]:sl[i][1]])
                if fin[i]:
                    live[i] = False
    assert ended == [1, 1] and ncalls == 2
    for i in range(2):
        a, r = torch.cat(got[i]), torch.cat(ref[i])
        print(f"sentence {i}: {a.numel()} samples, max |d audio| {float((a - r).abs().max()):.2e}")
        assert a.shape == r.shape and float((a - r).abs().max()) <= 1e-3


def test_bf16_encoder_into_the_bf16_decoder_against_the_oracle_encoder_states():
    """bf16 front half from token ids: the mel of GPU encoder -> GPU decoder is >= 40 dB against the same decoder fed the fp32 oracle's
    encoder states (same dropout masks, one batched call: the first three slots get the GPU states, the last three the oracle's)."""
    from infernos_b200.engine import TTSDecoder, TTSEncoder
    esd, dsd = synth.encoder_state_dict(), synth.decoder_state_dict()
    lengths = (40, 17, 64)
    ids, mask = synth.synth_token_ids(lengths, seed=24)
    ref_enc = _oracle(esd, ids, mask)
    spk = synth.synth_speakers(3, seed=25)
    g = torch.Generator().manual_seed(26)
    masks = (torch.rand(16, 2, 256, generator=g) < 0.5).float().cuda()
    enc = TTSEncoder("cuda:0", esd, mode="bf16", max_tokens=256, max_len=64)
    dec = TTSDecoder("cuda:0", dsd, mode="bf16", max_sessions=8, max_steps=32, max_enc_len=64)
    try:
        lens = mask.sum(1).to(torch.int32).cuda()
        gpu_states = enc(ids, mask)
        a, b = torch.arange(3, dtype=torch.int32).cuda(), torch.arange(3, 6, dtype=torch.int32).cuda()
        dec.start(a, gpu_states, lens, spk.cuda())
        dec.start(b, ref_enc.cuda(), lens, spk.cuda())
        mel, _ = dec.steps(torch.cat([a, b]), 16, masks=masks)
        enc.poll_errors(); dec.poll_errors()
        mel = mel.cpu()
    finally:
        enc.close(); dec.close()
    c = mel[3:].mean()
    snr = _snr(mel[3:] - c, mel[:3] - c)
    print(f"bf16 GPU encoder -> bf16 decoder vs oracle encoder states -> same decoder: mel SNR {snr:.2f} dB")
    assert snr >= 40.0


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def test_bf16_encoder_one_large_pass_is_bitwise_each_sentence_alone(sd):
    """About 4,000 rows in one pass of the default 16,384-row workspace: there qkv and ff1 run on 128 x 256 tiles, while each sentence alone
    (at most 200 rows) runs them on 128 x 128 tiles.  Every sentence's rows must still be bitwise what it gets alone on the same handle, padded
    rows zero, and six of them (the first, the last, the longest and three more) within the usual floors of the oracle."""
    from infernos_b200.engine import TTSEncoder
    g = torch.Generator().manual_seed(41)
    lengths = [int(x) for x in torch.randint(8, 201, (40,), generator=g)]
    ids, mask = synth.synth_token_ids(lengths, seed=42)
    rows = sum(lengths)
    assert -(-rows // 128) * (2304 // 128) > _sms(), f"{rows} rows do not put qkv (N = 2304) on 128 x 256 tiles"
    enc = TTSEncoder("cuda:0", sd, mode="bf16")
    try:
        cohort = enc(ids, mask).cpu()
        alone = [enc(ids[i:i + 1, :n], None).cpu()[0] for i, n in enumerate(lengths)]
        enc.poll_errors()
    finally:
        enc.close()
    m = mask.bool()
    assert float(cohort[~m].abs().max()) == 0.0, "padded rows must be zero"
    diff = [i for i, n in enumerate(lengths) if not torch.equal(cohort[i, :n], alone[i])]
    print(f"encoder bf16, {len(lengths)} sentences, {rows} rows in one pass: {len(lengths) - len(diff)} of {len(lengths)} bitwise equal to alone")
    assert not diff, f"sentences {diff}: a {rows}-row pass does not give the bits they get alone"
    longest = max(range(len(lengths)), key=lambda i: lengths[i])
    pick = sorted({0, len(lengths) - 1, longest, 10, 20, 30})
    Lp = max(lengths[i] for i in pick)
    sub_ids, sub_mask = ids[pick, :Lp], mask[pick, :Lp]
    _check("bf16", _oracle(sd, sub_ids, sub_mask)[sub_mask.bool()], cohort[pick, :Lp], sub_mask, f"sentences {pick} of a {rows}-row pass")


@pytest.mark.parametrize("max_tokens,lengths", [(64, (64, 30, 9, 57, 1)), (100, (100, 37, 63, 1, 88))])
def test_bf16_encoder_workspace_smaller_than_one_tile(sd, max_tokens, lengths):
    """max_tokens below the GEMM's 128-row box: the A maps span fewer rows than one tile, every pass is cut short of it.  Against the oracle,
    and bitwise against a handle with the default workspace."""
    from infernos_b200.engine import TTSEncoder
    ids, mask = synth.synth_token_ids(lengths, seed=44 + max_tokens)
    small = TTSEncoder("cuda:0", sd, mode="bf16", max_tokens=max_tokens, max_len=128)
    big = TTSEncoder("cuda:0", sd, mode="bf16", max_len=128)
    try:
        got = small(ids, mask).cpu()
        ref_big = big(ids, mask).cpu()
        small.poll_errors(); big.poll_errors()
    finally:
        small.close(); big.close()
    _check("bf16", _oracle(sd, ids, mask)[mask.bool()], got, mask, f"max_tokens {max_tokens}")
    assert torch.equal(got, ref_big)


def test_fp32_encoder_lengths_at_the_attention_tile_edges(sd):
    """k_enc_attend works on key tiles of 32 and query tiles of 64; lengths on either side of their edges, and the whole positional table
    (450).  The oracle runs per sentence at its own length."""
    from infernos_b200.engine import TTSEncoder
    lengths = (31, 32, 33, 63, 64, 65, 127, 128, 129, 320, 450)
    ids, mask = synth.synth_token_ids(lengths, seed=43)
    enc = TTSEncoder("cuda:0", sd, mode="fp32", max_tokens=2048, max_len=450)
    try:
        got = enc(ids, mask).cpu()
        enc.poll_errors()
    finally:
        enc.close()
    ref = torch.cat([_oracle(sd, ids[i:i + 1, :n], None)[0] for i, n in enumerate(lengths)])
    _check("fp32", ref, got, mask, "lengths at the attention kernel's tile edges")
