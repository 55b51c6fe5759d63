"""GPU parity of the autoregressive front half (b2_dec_*, SURVEY 8 f3) against oracle/decoder.py (pinned to the live transformers modules
by tests/test_oracle_decoder.py) and against the golden produced by the REAL modules (tests/golden/decoder_golden.npz): same synthetic
weights, same encoder states, same prenet dropout masks.  fp32 mode: max-abs <= 1e-3 on the mel frames; bf16 mode: >= 40 dB SNR."""
import os

import numpy as np
import pytest
import torch

from infernos_b200 import synth

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def sd():
    return synth.decoder_state_dict()


def _snr(ref, x):
    from oracle.tail import snr_db
    return snr_db(torch.as_tensor(ref), torch.as_tensor(x))


def _oracle(sd, enc, enc_mask, speaker, masks):
    from oracle import decoder as odec
    st = odec.DecoderState(sd, enc, enc_mask, speaker)
    specs, probs = [], []
    with torch.no_grad():
        for s in range(masks.size(0)):
            sp, pr = odec.step(sd, st, masks[s])
            specs.append(sp); probs.append(pr)
    return torch.cat(specs, 1), torch.stack(probs, 1)


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_decoder_replays_the_real_modules_golden(sd, mode):
    """16 steps (one reference infer() call) of 3 sentences with ragged encoder lengths, slots out of order."""
    from infernos_b200.engine import TTSDecoder
    d = np.load(os.path.join(G, "decoder_golden.npz"))
    enc, mask, spk, masks = (torch.from_numpy(d[k]) for k in ("enc", "enc_mask", "speaker", "masks"))
    dec = TTSDecoder("cuda:0", sd, mode=mode, max_sessions=8, max_steps=64, max_enc_len=16)
    try:
        slots = torch.tensor([5, 0, 3], dtype=torch.int32).cuda()
        dec.start(slots, enc.cuda(), mask.sum(1).to(torch.int32).cuda(), spk.cuda())
        mel, prob = dec.steps(slots, 16, masks=masks.cuda())
        dec.poll_errors()
        assert [dec.get_step(s) for s in (5, 0, 3)] == [16, 16, 16]
    finally:
        dec.close()
    mel, prob = mel.cpu().numpy(), prob.cpu().numpy()
    assert mel.shape == d["mel"].shape == (3, 32, 80) and prob.shape == d["prob"].shape
    err, snr = float(np.abs(mel - d["mel"]).max()), _snr(d["mel"] - d["mel"].mean(), mel - d["mel"].mean())
    print(f"decoder {mode}: max |d mel| {err:.2e}, SNR on the mean-removed mel {snr:.2f} dB, max |d prob| {np.abs(prob - d['prob']).max():.2e}")
    if mode == "fp32":
        assert err <= 1e-3 and np.abs(prob - d["prob"]).max() <= 1e-4
    else:
        assert snr >= 40.0


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_decoder_two_calls_continuous_batching_and_sub_passes(sd, mode):
    """Two consecutive 16-step calls (the KV cache carries over), a second cohort admitted between them, max_rows smaller than the batch
    (internal passes), against the oracle run per cohort."""
    from infernos_b200.engine import TTSDecoder
    g = torch.Generator().manual_seed(4)
    encA, encB = synth.synth_encoder_states(5, 9, seed=21), synth.synth_encoder_states(2, 14, seed=22)
    mA, mB = torch.ones(5, 9, dtype=torch.int), (torch.arange(14)[None] < torch.tensor([14, 6])[:, None]).to(torch.int)
    sA, sB = synth.synth_speakers(5, seed=23), synth.synth_speakers(2, seed=24)
    masks1 = (torch.rand(16, 2, 256, generator=g) < 0.5).float()
    masks2 = (torch.rand(16, 2, 256, generator=g) < 0.5).float()
    refA, _ = _oracle(sd, encA, mA, sA, torch.cat([masks1, masks2]))
    refB, _ = _oracle(sd, encB, mB, sB, masks2)
    dec = TTSDecoder("cuda:0", sd, mode=mode, max_sessions=16, max_rows=4, max_steps=40, max_enc_len=14)
    try:
        slA = torch.tensor([1, 2, 3, 4, 9], dtype=torch.int32).cuda()
        slB = torch.tensor([7, 0], dtype=torch.int32).cuda()
        dec.start(slA, encA.cuda(), None, sA.cuda())
        mel1, _ = dec.steps(slA, 16, masks=masks1.cuda())
        dec.start(slB, encB.cuda(), mB.sum(1).to(torch.int32).cuda(), sB.cuda())
        both = torch.cat([slB, slA])                                    # one batched call over both cohorts, newcomers first
        mel2, _ = dec.steps(both, 16, masks=masks2.cuda())
        dec.poll_errors()
        assert dec.get_step(9) == 32 and dec.get_step(7) == 16
        with pytest.raises(RuntimeError, match="max_steps"):            # 40 positions only: the third call runs the first cohort past them
            dec.steps(slA, 16, masks=masks1.cuda())
            dec.poll_errors()
    finally:
        dec.close()
    gotA = torch.cat([mel1.cpu(), mel2[2:].cpu()], dim=1)
    gotB = mel2[:2].cpu()
    if mode == "fp32":
        assert float((gotA - refA).abs().max()) <= 1e-3 and float((gotB - refB).abs().max()) <= 1e-3
    else:
        c = refA.mean()
        print(f"decoder bf16, 32 steps: SNR {_snr(refA - c, gotA - c):.2f} dB (cohort A), {_snr(refB - c, gotB - c):.2f} dB (cohort B)")
        assert _snr(refA - c, gotA - c) >= 40.0 and _snr(refB - c, gotB - c) >= 40.0


def test_decoder_feeds_the_tail_without_leaving_the_device(sd):
    """front half + tail: the decoder's feat_out frames go straight into b2_tts_tail2(B2_TAIL_APPLY_POSTNET)."""
    from infernos_b200.engine import TTSDecoder, TTSTail
    from oracle import codec as ocodec
    from oracle import tail as otail
    d = np.load(os.path.join(G, "decoder_golden.npz"))
    enc, mask, spk, masks = (torch.from_numpy(d[k]) for k in ("enc", "enc_mask", "speaker", "masks"))
    vsd, csd, psd = synth.hifigan_state_dict(), synth.chunker_state_dict(), synth.postnet_state_dict()
    dec = TTSDecoder("cuda:0", sd, mode="fp32", max_sessions=4, max_steps=32, max_enc_len=16)
    tail = TTSTail("cuda:0", vsd, csd, mode="fp32", max_sessions=4, max_windows=16, postnet_sd=psd)
    try:
        slots = torch.tensor([2, 0, 1], dtype=torch.int32).cuda()
        tail.reset_sessions([0, 1, 2])
        dec.start(slots, enc.cuda(), mask.sum(1).to(torch.int32).cuda(), spk.cuda())
        mel, _ = dec.steps(slots, 16, masks=masks.cuda())
        g, a = tail.tail(slots, mel, apply_postnet=True)
        tail.poll_errors()
        a, g = a.cpu(), g.cpu()
    finally:
        dec.close(); tail.close()
    with torch.no_grad():
        ref_mel = otail.postnet_forward(psd, torch.from_numpy(d["mel"]))
        ref, _ = otail.tts_tail(vsd, csd, torch.zeros(3, 4, 80), ref_mel)
    assert float((a - ref).abs().max()) <= 1e-3
    assert np.array_equal(g.numpy(), ocodec.encode_f32(a.numpy(), 0))


def test_engine_end_to_end_with_the_gpu_front_half(sd):
    """HelloSippyRTPipe with B200Frontend: text -> (scripted tokenizer / encoder, the per-sentence glue) -> GPU decoder -> GPU post-net + tail ->
    unbatch_and_dispatch, against the oracle chain decoder -> post-net -> tail -> unbatch arithmetic with the same dropout masks."""
    import uuid
    from infernos_b200.engine import TTSDecoder
    from infernos_b200.HelloSippyTTSRT.HelloSippyRTPipe import (B200Frontend, HelloSippyPipeState, HelloSippyPipeStateBatched, HelloSippyPlayRequest,
                                                                 HelloSippyRTPipe)
    from oracle import decoder as odec
    from oracle import tail as otail
    vsd, csd, psd = synth.hifigan_state_dict(), synth.chunker_state_dict(), synth.postnet_state_dict()
    texts = ["first sentence", "the second one is longer"]
    encs = {0: synth.synth_encoder_states(1, 9, seed=31)[0], 1: synth.synth_encoder_states(1, 13, seed=32)[0]}
    g = torch.Generator().manual_seed(8)
    masks = [(torch.rand(16, 2, 256, generator=g) < 0.5).float() for _ in range(4)]

    def tokenizer(text):
        i = texts.index(text)
        return torch.full((1, encs[i].size(0)), i + 4, dtype=torch.long)

    def encoder(ids, mask):
        L = ids.size(1)
        return torch.stack([torch.nn.functional.pad(encs[int(r[0]) - 4], (0, 0, 0, L - encs[int(r[0]) - 4].size(0))) for r in ids])

    dec = TTSDecoder("cuda:0", sd, mode="fp32", max_sessions=4, max_steps=64, max_enc_len=16)
    fe = B200Frontend(dec, tokenizer, encoder, mask_fn=lambda c: masks[c])
    pp = HelloSippyRTPipe("cuda:0", output_sr=8000, frontend=fe, vocoder_state_dict=vsd, chunker_state_dict=csd, postnet_state_dict=psd,
                          mode="fp32", max_sessions=4, speaker_embeddings=[synth.synth_speakers(1, seed=33)])
    pp.maxlenratio = 4.0                                    # maxlen = int(13 * 4 / 2) = 26 decoder steps for the batch: both sentences end in call 2
    got = [[], []]
    ended = [0, 0]

    def cb(i):
        def f(chunk):
            if chunk is None:
                ended[i] += 1
            else:
                got[i].append(chunk.clone())
        return f
    reqs = [HelloSippyPlayRequest(uuid.uuid4(), t, pp.get_voice(0), cb(i)) for i, t in enumerate(texts)]
    state = HelloSippyPipeStateBatched([HelloSippyPipeState(pp, r) for r in reqs], pp)
    assert (state.minlen, state.maxlen) == (0, 26)          # batch-wide, from the padded encoder length like the reference (:117-118)
    ncalls = 0
    while True:
        pp.infer(state)
        ncalls += 1
        if not pp.unbatch_and_dispatch(state):
            break
    dec.close()
    # oracle chain
    L = 13
    enc = torch.stack([torch.nn.functional.pad(encs[i], (0, 0, 0, L - encs[i].size(0))) for i in range(2)])
    emask = torch.stack([(torch.arange(L) < encs[i].size(0)).to(torch.int) for i in range(2)])
    spk = synth.synth_speakers(1, seed=33).repeat(2, 1)
    st = odec.DecoderState(sd, enc, emask, spk)
    pre = torch.zeros(2, 4, 80)
    ends, idx, live, starts = [-1, -1], 0, [True, True], [1, 1]
    ref = [[], []]
    with torch.no_grad():
        for c in range(ncalls):
            frames = []
            for s in range(16):
                sp, pr = odec.step(sd, st, masks[c][s])
                frames.append(sp)
                for i in range(2):
                    if ends[i] < 0 and (bool((pr[i] >= 0.5).any()) or 26 <= idx):
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
        assert a.shape == r.shape and float((a - r).abs().max()) <= 1e-3


def test_worker_with_gpu_front_half_reference_load_test_shape():
    """The reference's own load test (HelloSippyRTPipeTest.py:180-236) in miniature: requests queued at once on InfernTTSWorker(continuous=True)
    with the GPU front half and pre-encoded dispatch; every session ends, gets (ends_at - 1) * 256 samples (A.5) with as many payload bytes."""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    import session_bench
    r = session_bench.run(6, 24, "bf16")
    assert r["sessions"] == 6 and r["payload_bytes_equal_samples"] and r["all_faster_than_real_time"]
    # maxlen = 24 decoder steps -> ends_at = 26 -> (26 - 1) * 256 samples at 8 kHz
    assert abs(r["audio_s_per_session"] - 25 * 256 / 8000.0) < 1e-9
    assert r["time_to_first_frame_s"]["p99"] <= r["time_to_last_frame_s"]["p50"]


def test_bf16_decoder_800_sessions_against_the_oracle_and_a_small_handle(sd):
    """800 sessions in one pass with ragged encoder lengths up to 128: ff1 and (in start) xkv run on 128 x 256 tiles and k_attend on up to
    128 encoder positions.  Seven sessions (rows 0, 127, 128, 767, 768, 799 and the longest encoder sequence) are each >= 40 dB from the
    oracle run for that session alone, and bitwise what a handle of seven sessions (128 x 128 and 64-wide tiles throughout) gives them."""
    from infernos_b200.engine import TTSDecoder
    n, L = 800, 128
    g = torch.Generator().manual_seed(51)
    lens = torch.randint(1, L + 1, (n,), generator=g, dtype=torch.int32)
    lens[400], lens[401] = 1, L
    enc, spk = synth.synth_encoder_states(n, L, seed=52), synth.synth_speakers(n, seed=53)
    masks = (torch.rand(16, 2, 256, generator=g) < 0.5).float()
    pick = sorted({0, 127, 128, 767, 768, 799, int(lens.argmax())})
    big = TTSDecoder("cuda:0", sd, mode="bf16", max_sessions=n, max_steps=32, max_enc_len=L)
    try:
        slots = torch.arange(n, dtype=torch.int32).cuda()
        big.start(slots, enc.cuda(), lens.cuda(), spk.cuda())
        mel, _ = big.steps(slots, 16, masks=masks.cuda())
        big.poll_errors()
        mel = mel.cpu()
    finally:
        big.close()
    small = TTSDecoder("cuda:0", sd, mode="bf16", max_sessions=len(pick), max_steps=32, max_enc_len=L)
    try:
        ps = torch.arange(len(pick), dtype=torch.int32).cuda()
        small.start(ps, enc[pick].cuda(), lens[pick].cuda(), spk[pick].cuda())
        mel_small, _ = small.steps(ps, 16, masks=masks.cuda())
        small.poll_errors()
        mel_small = mel_small.cpu()
    finally:
        small.close()
    for j, i in enumerate(pick):
        n_i = int(lens[i])
        ref, _ = _oracle(sd, enc[i:i + 1, :n_i], torch.ones(1, n_i, dtype=torch.int), spk[i:i + 1], masks)
        c = ref.mean()
        snr = _snr(ref[0] - c, mel[i] - c)
        same = torch.equal(mel[i], mel_small[j])
        print(f"decoder bf16, 800 sessions: session {i} ({n_i} encoder positions) SNR {snr:.2f} dB, bitwise equal on a 7-session handle: {same}")
        assert snr >= 40.0, (i, snr)
        assert same, f"session {i}: an 800-session pass does not give the bits a 7-session handle gives"


def test_fp32_decoder_128_steps_over_long_encoder_sequences(sd):
    """Eight 16-step calls (128 self-attention positions, the KV cache carried across calls) over encoder sequences of 65, 128 and 200
    positions, against the oracle run over the same 128 steps."""
    from infernos_b200.engine import TTSDecoder
    lens, L = [65, 128, 200], 200
    g = torch.Generator().manual_seed(61)
    enc, spk = synth.synth_encoder_states(3, L, seed=62), synth.synth_speakers(3, seed=63)
    mask = (torch.arange(L)[None] < torch.tensor(lens)[:, None]).to(torch.int)
    masks = (torch.rand(128, 2, 256, generator=g) < 0.5).float()
    dec = TTSDecoder("cuda:0", sd, mode="fp32", max_sessions=4, max_steps=128, max_enc_len=L)
    try:
        slots = torch.tensor([2, 0, 3], dtype=torch.int32).cuda()
        dec.start(slots, enc.cuda(), torch.tensor(lens, dtype=torch.int32).cuda(), spk.cuda())
        got = torch.cat([dec.steps(slots, 16, masks=masks[16 * c:16 * c + 16].cuda())[0].cpu() for c in range(8)], 1)
        dec.poll_errors()
        assert [dec.get_step(s) for s in (2, 0, 3)] == [128] * 3
    finally:
        dec.close()
    ref, _ = _oracle(sd, enc, mask, spk, masks)
    ref64, _ = _oracle({k: v.double() for k, v in sd.items()}, enc.double(), mask, spk.double(), masks.double())
    per_call = [float((got[:, 32 * c:32 * c + 32] - ref[:, 32 * c:32 * c + 32]).abs().max()) for c in range(8)]
    drift = float((ref.double() - ref64).abs().max())
    print(f"decoder fp32, 128 steps, encoder lengths {lens}: max |d mel| per 16-step call {', '.join(f'{e:.1e}' for e in per_call)}; "
          f"against the float64 oracle {float((got.double() - ref64).abs().max()):.1e}; the oracle's own float32-vs-float64 drift {drift:.1e}")
    assert max(per_call) <= 1e-3
