"""GPU parity of the TTS tail (through the C-ABI) against the oracle and the golden vectors produced by the
real reference modules.  Tolerances are the ones north_star states: fp32 mode max-abs <= 1e-3 against the
torch fp32 SpeechT5HifiGan, bf16 (tensor-core) mode >= 40 dB SNR; G.711 bytes bit-exact from the same PCM."""
import os

import numpy as np
import pytest
import torch

from infernos_b200 import synth

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
FP32_TOL = 1e-3       # north_star: "within max-abs 1e-3 in fp32 mode"
BF16_SNR_DB = 40.0    # north_star: ">= 40 dB SNR in bf16 mode"


@pytest.fixture(scope="module")
def sds():
    return synth.hifigan_state_dict(), synth.chunker_state_dict()


@pytest.fixture(scope="module")
def tail32(sds):
    from infernos_b200.engine import TTSTail
    t = TTSTail("cuda:0", sds[0], sds[1], mode="fp32", max_sessions=64, max_windows=24)
    yield t
    t.close()


@pytest.fixture(scope="module")
def tail16(sds):
    from infernos_b200.engine import TTSTail
    t = TTSTail("cuda:0", sds[0], sds[1], mode="bf16", max_sessions=64, max_windows=24)
    yield t
    t.close()


def snr(ref, x):
    from oracle.tail import snr_db
    return snr_db(torch.as_tensor(ref), torch.as_tensor(x))


def test_vocoder_fp32_matches_real_hifigan_golden(tail32):
    d = np.load(os.path.join(G, "hifigan_golden.npz"))
    a = tail32.vocoder(torch.from_numpy(d["mel"]).cuda()).cpu().numpy()
    assert a.shape == d["audio"].shape
    assert np.abs(a - d["audio"]).max() <= FP32_TOL
    assert np.abs(a - d["audio"]).max() < 5e-5          # in practice fp32 summation-order noise only
    al = tail32.vocoder(torch.from_numpy(d["mel_long"]).cuda()).cpu().numpy()      # T = 20: general window length
    assert np.abs(al - d["audio_long"]).max() <= FP32_TOL
    un = tail32.vocoder(torch.from_numpy(d["mel_long"][0]).cuda()).cpu().numpy()   # un-batched form
    assert un.shape == (5120,) and np.array_equal(un, al[0])


def test_vocoder_fp32_matches_live_transformers_module(tail32, sds):
    """The real third-party module, run on this box's CPU (transformers is in the image; /root/reference is not needed)."""
    tr = pytest.importorskip("transformers")
    m = tr.SpeechT5HifiGan(tr.SpeechT5HifiGanConfig())
    m.load_state_dict(sds[0], strict=True)
    m.eval()
    mel = synth.synth_mel(5, 12, seed=123)
    with torch.no_grad():
        ref = m(mel)
    got = tail32.vocoder(mel.cuda()).cpu()
    assert (got - ref).abs().max() <= FP32_TOL


def test_chunker_matches_real_module_golden(tail32):
    d = np.load(os.path.join(G, "chunker_golden.npz"))
    c = tail32.chunker(torch.from_numpy(d["mel"]).cuda(), torch.from_numpy(d["audio"]).cuda()).cpu().numpy()
    assert np.abs(c - d["out"]).max() < 5e-5


def test_vocoder_bf16_snr(tail16):
    d = np.load(os.path.join(G, "hifigan_golden.npz"))
    a = tail16.vocoder(torch.from_numpy(d["mel"]).cuda()).cpu().numpy()
    print("bf16 vocoder SNR vs real fp32 SpeechT5HifiGan: %.2f dB" % snr(d["audio"], a))
    assert snr(d["audio"], a) >= BF16_SNR_DB
    al = tail16.vocoder(torch.from_numpy(d["mel_long"]).cuda()).cpu().numpy()
    assert snr(d["audio_long"], al) >= BF16_SNR_DB


def test_vocoder_bf16_tracks_its_cpu_emulation(tail16, sds):
    """The tcgen05 path against the same bf16 operand rounding restated on the CPU (oracle.tail.hifigan_forward_bf16emu).
    Both are ~45 dB roundings of the fp32 result whose bf16 rounding decisions flip with fp32 summation order, so they
    agree with each other to about the same SNR, and each clears the 40 dB bar against fp32 on its own."""
    from oracle import tail as otail
    mel = synth.synth_mel(3, 12, seed=21)
    with torch.no_grad():
        emu = otail.hifigan_forward_bf16emu(sds[0], mel)
    got = tail16.vocoder(mel.cuda()).cpu()
    assert snr(emu, got) >= 42.0


def test_vocoder_bf16_with_taps_matches_vocoder(tail16):
    """Recording the stage-boundary taps runs stage 3 differently: its upsampler is a launch of its own (the fused path never writes
    x to memory), and the k = 3 ResBlock then runs on the time-as-M kernel.  Only this path reaches them in bf16 mode.  The operands
    are rounded at the same points as in vocoder(); only the fp32 summation order differs."""
    mel = synth.synth_mel(8, 12, seed=314).cuda()
    ref = tail16.vocoder(mel).cpu()
    got, taps = tail16.vocoder_with_taps(mel, names=("up3",))
    assert taps["up3"].shape == (8, 32, 12 * 256)
    s = snr(ref, got.cpu())
    print("bf16 vocoder with taps vs without: %.1f dB" % s)
    assert s > 46.0


def _replay(tail, law=0):
    """Replays the scripted run of the REAL infer()/unbatch_and_dispatch() (tests/golden/infer_golden.npz)."""
    from oracle import tail as otail
    d = np.load(os.path.join(G, "infer_golden.npz"))
    plan = torch.from_numpy(d["plan"])
    B = plan.size(0)
    slots = torch.tensor([5, 0, 9], dtype=torch.int32)
    tail.reset_sessions(slots.tolist())
    audios, codes = [], []
    for c in range(int(d["ncalls_run"])):
        mel = plan[:, 32 * c:32 * (c + 1)].contiguous()
        g, a = tail.tail(slots.cuda(), mel.cuda(), law=law)
        audios.append(a.cpu())
        codes.append(g.cpu())
    return d, audios, codes, otail


def test_tail_fp32_matches_real_infer(tail32):
    from oracle import codec as ocodec
    d, audios, codes, otail = _replay(tail32)
    B = 3
    starts, live = [1] * B, [True] * B
    per_a = [[] for _ in range(B)]
    per_c = [[] for _ in range(B)]
    for c, (a, g) in enumerate(zip(audios, codes)):
        assert np.abs(a.numpy() - d["audio"][c]).max() <= FP32_TOL
        assert np.abs(a.numpy() - d["audio"][c]).max() < 1e-4
        # the bytes are exactly the G.711 codes of the 8 kHz floats this same call returned
        assert np.array_equal(g.numpy(), ocodec.encode_f32(a.numpy(), 0))
        sl, fin, more = otail.unbatch_slices(a.size(1), int(d["idx"][c]), starts, d["ends_at"][c].tolist(), live)
        for i in range(B):
            if sl[i] is not None:
                per_a[i].append(a[i, sl[i][0]:sl[i][1]])
                per_c[i].append(g[i, sl[i][0]:sl[i][1]])
            if fin[i]:
                live[i] = False
    for i in range(B):
        full = torch.cat(per_a[i]).numpy()
        ref = d[f"session{i}_audio"]
        assert full.shape == ref.shape
        pcm_mine = ocodec.f32_to_pcm16(full).astype(np.int32)
        pcm_ref = ocodec.f32_to_pcm16(ref).astype(np.int32)
        assert np.abs(pcm_mine - pcm_ref).max() <= 2          # |dPCM| of fp32 summation-order noise
        by = torch.cat(per_c[i]).numpy()
        ref_by = d[f"session{i}_ulaw"]
        assert by.shape == ref_by.shape
        assert (by != ref_by).mean() < 0.02                    # codes differ only where PCM sat on a step edge


def test_tail_bf16_snr_and_state(tail16):
    d, audios, codes, _ = _replay(tail16, law=1)
    ref = np.stack([d["audio"][c] for c in range(len(audios))])
    got = np.stack([a.numpy() for a in audios])
    print("bf16 tail SNR (after the chunker's tanh(gain * x) and the resampler) vs the real fp32 infer(): %.2f dB" % snr(ref, got))
    assert snr(ref, got) >= BF16_SNR_DB
    # pre_frames carried per session = last four mel frames of the last call
    last = d["plan"][:, 32 * len(audios) - 4:32 * len(audios)]
    for b, slot in enumerate([5, 0, 9]):
        assert np.array_equal(tail16.get_pre_frames(slot).numpy(), last[b])


def test_tail_sessions_are_independent_and_order_free(tail32):
    """Sharding property: a session's output does not depend on which other sessions share the batch."""
    mel = synth.synth_mel(6, 32, seed=77)
    tail32.reset_sessions(list(range(6)))
    g_all, a_all = tail32.tail(torch.arange(6, dtype=torch.int32).cuda(), mel.cuda())
    tail32.reset_sessions(list(range(6)))
    perm = torch.tensor([4, 2, 5], dtype=torch.int32)
    g_sub, a_sub = tail32.tail(perm.cuda(), mel[perm.long()].cuda())
    assert torch.equal(g_all[perm.long()].cpu(), g_sub.cpu())
    assert torch.equal(a_all[perm.long()].cpu(), a_sub.cpu())


def test_tail_more_windows_than_workspace(tail32):
    """B*nwin > max_windows exercises the internal sub-batching."""
    mel = synth.synth_mel(10, 32, seed=78)          # 40 windows > 24
    tail32.reset_sessions(list(range(10)))
    g1, _ = tail32.tail(torch.arange(10, dtype=torch.int32).cuda(), mel.cuda())
    tail32.reset_sessions(list(range(10)))
    g2a, _ = tail32.tail(torch.arange(5, dtype=torch.int32).cuda(), mel[:5].cuda())
    g2b, _ = tail32.tail(torch.arange(5, 10, dtype=torch.int32).cuda(), mel[5:].cuda())
    assert torch.equal(g1.cpu(), torch.cat([g2a, g2b]).cpu())


def test_tail_host_entry_matches_device_entry(tail32):
    mel = synth.synth_mel(4, 32, seed=79)
    slots = torch.arange(4, dtype=torch.int32)
    tail32.reset_sessions([0, 1, 2, 3])
    g_dev, a_dev = tail32.tail(slots.cuda(), mel.cuda())
    tail32.reset_sessions([0, 1, 2, 3])
    g = torch.empty(4, 4096, dtype=torch.uint8).pin_memory()
    a = torch.empty(4, 4096, dtype=torch.float32).pin_memory()
    tail32.tail_host(slots.pin_memory(), mel.pin_memory(), g, a)
    assert torch.equal(g, g_dev.cpu()) and torch.equal(a, a_dev.cpu())


def test_eight_frame_chunks(tail32, sds):
    """Config 2/4 shape: 8-frame chunks (one window per call) give the same 16 kHz audio as 32-frame calls;
    only the resampler's per-call edge transient differs (SURVEY App. A.3)."""
    from oracle import tail as otail
    mel = synth.synth_mel(2, 32, seed=80)
    tail32.reset_sessions([0, 1])
    outs = []
    for c in range(4):
        _, a = tail32.tail(torch.arange(2, dtype=torch.int32).cuda(), mel[:, 8 * c:8 * c + 8].contiguous().cuda())
        outs.append(a.cpu())
    pre = torch.zeros(2, 4, 80)
    with torch.no_grad():
        for c in range(4):
            ref, pre = otail.tts_tail(*sds, pre, mel[:, 8 * c:8 * c + 8])
            assert (outs[c] - ref).abs().max() < 1e-4


def test_bad_arguments_raise(tail32):
    with pytest.raises(RuntimeError):
        tail32.tail(torch.zeros(2, dtype=torch.int32).cuda(), torch.zeros(2, 12, 80).cuda())      # 12 % 8 != 0
    with pytest.raises(RuntimeError):
        tail32.vocoder(torch.zeros(1, 12, 80))                                                     # CPU tensor
