"""GPU parity: G.711 + resampler kernels (through the C-ABI) against the C oracle and the golden vectors.
Bit-exact for every integer/byte result."""
import hashlib
import json
import os

import numpy as np
import pytest
import torch

from infernos_b200 import synth

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def eng():
    from infernos_b200 import engine
    return engine


@pytest.fixture(scope="module")
def oc():
    from oracle import codec
    return codec


@pytest.fixture(scope="module")
def taps():
    return np.load(os.path.join(G, "resample_taps.npz"))


@pytest.mark.parametrize("law", [0, 1])
def test_encode_all_int16_bit_exact(eng, oc, law):
    t = np.load(os.path.join(G, "g711_tables.npz"))
    pcm = torch.arange(-32768, 32768, dtype=torch.int32).to(torch.int16).cuda()
    out = eng.g711_encode(pcm, law).cpu().numpy()
    assert np.array_equal(out, t["alaw_enc" if law else "ulaw_enc"])
    # unaligned / odd length path
    out2 = eng.g711_encode(pcm[3:3 + 1001], law).cpu().numpy()
    assert np.array_equal(out2, t["alaw_enc" if law else "ulaw_enc"][3:1004])


@pytest.mark.parametrize("law", [0, 1])
def test_decode_all_codes_bit_exact(eng, law):
    t = np.load(os.path.join(G, "g711_tables.npz"))
    codes = torch.arange(256, dtype=torch.int32).to(torch.uint8).cuda()
    pcm = eng.g711_decode(codes, law, torch.int16).cpu().numpy()
    assert np.array_equal(pcm, t["alaw_dec" if law else "ulaw_dec"])
    f = eng.g711_decode(codes.repeat(5)[1:], law).cpu().numpy()
    ref = (np.tile(t["alaw_dec" if law else "ulaw_dec"], 5)[1:].astype(np.float32) / np.float32(32767.0))
    assert np.array_equal(f, ref)


def test_reference_byte_streams(eng):
    with open(os.path.join(G, "g711_golden.json")) as f:
        gold = json.load(f)
    g1 = torch.linspace(-1.25, 1.25, 48001).cuda()
    assert sha(eng.g711_encode(g1).cpu().numpy()) == gold["G1_encode_linspace"]
    g2 = synth.synth_audio(64, 8192).cuda()
    assert sha(eng.g711_encode(g2).cpu().numpy()) == gold["G2_encode_rand"]
    codes = torch.arange(256, dtype=torch.int32).to(torch.uint8).cuda()
    assert sha(eng.g711_decode(codes).cpu().numpy()) == gold["G4_decode_all"]
    edge = torch.tensor(gold["edge_in"], dtype=torch.float32).cuda()
    assert eng.g711_encode(edge).cpu().tolist() == gold["edge_ulaw"]


def test_float_to_pcm_bit_exact(eng, oc):
    g = torch.Generator().manual_seed(5)
    x = torch.cat([(torch.rand(100000, generator=g) * 2.4 - 1.2), torch.tensor([0.0, -0.0, 1.0, -1.0, 0.5, -0.5, 3e-5, -3e-5]),
                   # far out of range, infinities and NaN: the clamp saturates, NaN becomes 0 (one saturating F2I.S16 in the kernel)
                   torch.tensor([1e9, -1e9, 3.4e38, -3.4e38, float("inf"), float("-inf"), float("nan"), 1.00001, -1.00004, 32768.0 / 32767.0])])
    assert np.array_equal(eng.f32_to_pcm16(x.cuda()).cpu().numpy(), oc.f32_to_pcm16(x.numpy()))


@pytest.mark.parametrize("law", [0, 1])
@pytest.mark.parametrize("rows,L", [(3, 8192), (5, 2048), (2, 512), (1, 16), (7, 320), (3, 1600), (2, 333), (1, 1), (4, 4096 + 16),
                                     # row ends on every lane of the flat kernel, one-chunk rows, and several grid-stride trips
                                     (70, 16), (40, 48), (33, 16 * 31), (300, 32), (9, 16 * 33), (3000, 1600), (40, 8192 * 2)])
def test_fused_resample_encode_bit_exact_vs_oracle(eng, oc, taps, law, rows, L):
    x = synth.synth_audio(rows, L, seed=L + rows)
    ref_u8 = oc.resample_2to1_encode(x.numpy(), taps["down"], law)
    ref_f = oc.resample_2to1(x.numpy(), taps["down"])
    got_u8 = eng.resample_g711_encode(x.cuda(), law).cpu().numpy()
    got_f = eng.resample_2to1(x.cuda()).cpu().numpy()
    assert got_u8.shape == ref_u8.shape == (rows, (L + 1) // 2)
    assert np.array_equal(got_f, ref_f)            # same fmaf chain -> identical floats
    assert np.array_equal(got_u8, ref_u8)


def test_resample_close_to_torchaudio_golden(eng, taps):
    y = eng.resample_2to1(torch.from_numpy(taps["x"]).cuda()).cpu().numpy()
    assert np.abs(y - taps["y_down"]).max() < 2e-6
    y = eng.resample_2to1(torch.from_numpy(taps["x_odd"]).cuda()).cpu().numpy()
    assert y.shape == taps["y_down_odd"].shape and np.abs(y - taps["y_down_odd"]).max() < 2e-6
    yu = eng.resample_1to2(torch.from_numpy(taps["x"][:, :200].copy()).cuda()).cpu().numpy()
    assert np.abs(yu - taps["y_up"]).max() < 2e-6


@pytest.mark.parametrize("law", [0, 1])
def test_decode_upsample_bit_exact_vs_oracle(eng, oc, taps, law):
    g = torch.Generator().manual_seed(9)
    codes = torch.randint(0, 256, (6, 160), generator=g).to(torch.uint8)
    x8 = oc.decode_f32(codes.numpy(), law)
    ref = oc.resample_1to2(x8, taps["up"])
    got = eng.g711_decode_upsample(codes.cuda(), law).cpu().numpy()
    assert np.array_equal(got, ref)
    d = np.load(os.path.join(G, "g711_decode16k.npz"))
    if law == 0:   # the reference codec's own 16 kHz decode (torch summation order): close, not bit-equal
        got = eng.g711_decode_upsample(torch.from_numpy(d["inp"]).cuda()[None], 0).cpu().numpy()[0]
        assert np.abs(got - d["out"]).max() < 2e-6


@pytest.mark.parametrize("law", [0, 1])
@pytest.mark.parametrize("rows,L", [(1, 4), (7, 8), (70, 12), (300, 40), (33, 4 * 255), (9, 4 * 257), (2000, 800), (5, 1024 * 3 + 4), (3, 333), (4, 162)])
def test_decode_upsample_shapes_bit_exact_vs_oracle(eng, oc, taps, law, rows, L):
    """Row ends on every thread of the flat 8k -> 16k kernel (one- and two-quad rows too), several grid-stride trips, and the
    scalar kernel's shapes (L % 4 != 0); also the fp32-input form of the same kernels."""
    g = torch.Generator().manual_seed(rows * 1000 + L)
    codes = torch.randint(0, 256, (rows, L), generator=g).to(torch.uint8)
    x8 = oc.decode_f32(codes.numpy(), law)
    ref = oc.resample_1to2(x8, taps["up"])
    got = eng.g711_decode_upsample(codes.cuda(), law).cpu().numpy()
    assert got.shape == (rows, 2 * L) and np.array_equal(got, ref)
    assert np.array_equal(eng.resample_1to2(torch.from_numpy(x8).cuda()).cpu().numpy(), ref)


@pytest.mark.parametrize("law", [0, 1])
def test_round_trip_properties_at_full_size(eng, law):
    """Size-independent properties at config-5 scale (100k streams x 160-byte packets)."""
    n = 100_000 * 160
    g = torch.Generator(device="cuda").manual_seed(1)
    x = (torch.rand(n, generator=g, device="cuda") * 2 - 1) * 0.95
    codes = eng.g711_encode(x, law)
    dec = eng.g711_decode(codes, law)
    # decode(encode(x)) re-encodes to the same code (idempotence of the quantiser)
    assert torch.equal(eng.g711_encode(dec, law), codes)
    # quantisation error bound of G.711 (largest step 1024 LSB at full scale for mu-law, 1024 for A-law)
    assert float((dec - x).abs().max()) <= 1056.0 / 32767.0
    # the quantiser is monotone: sorted input decodes to a non-decreasing sequence
    xs, _ = torch.sort(x[: 4_000_000])
    ds = eng.g711_decode(eng.g711_encode(xs, law), law)
    assert bool((ds[1:] >= ds[:-1]).all())
    # checksum of checksums: encoding the halves separately equals encoding the whole
    h = n // 2
    assert torch.equal(torch.cat([eng.g711_encode(x[:h], law), eng.g711_encode(x[h:], law)]), codes)


@pytest.mark.parametrize("law", [0, 1])
@pytest.mark.parametrize("up", [False, True])
def test_decode_many_ragged_and_uniform_bit_exact_vs_oracle(eng, oc, taps, law, up):
    """SURVEY 8 f4: the packets of many calls in one staging copy + one launch; every packet is decoded / resampled on its own
    (per-packet zero padding), exactly like one G711Codec.decode per packet."""
    from infernos_b200.Core.Codecs.G711 import G711ACodec, G711Codec
    rng = np.random.default_rng(17 + law)

    def ref_one(b):
        x8 = oc.decode_f32(np.frombuffer(b, dtype=np.uint8)[None], law)
        return (oc.resample_1to2(x8, taps["up"]) if up else x8)[0]
    for lens in ([160] * 257, [160, 80, 0, 1, 7, 333, 160, 1024, 3, 160, 800, 5]):       # uniform (flat kernel) / ragged, incl. empty
        pk = [rng.integers(0, 256, n, dtype=np.uint8).tobytes() for n in lens]
        l0 = eng.kernel_launch_count()
        got = eng.g711_decode_many(pk, law, upsample=up)
        assert eng.kernel_launch_count() - l0 == 1                                       # one launch for all packets
        assert len(got) == len(pk)
        for b, g in zip(pk, got):
            r = ref_one(b) if len(b) else np.empty(0, np.float32)
            assert g.shape == r.shape and np.array_equal(g.numpy(), r)
    codec = (G711ACodec if law else G711Codec)().to("cuda:0")
    pk = [rng.integers(0, 256, n, dtype=np.uint8).tobytes() for n in (160, 160, 320)]
    many = codec.decode_many(pk, sample_rate=16000 if up else 8000)
    for b, ch in zip(pk, many):
        one = codec.decode(b, sample_rate=16000 if up else 8000)
        assert ch.samplerate == one.samplerate and np.array_equal(ch.audio.numpy(), one.audio.cpu().numpy())
    assert codec.decode(b"").audio.numel() == 0 and eng.g711_decode_many([]) == []


def test_empty_inputs(eng):
    assert eng.g711_encode(torch.empty(0, device="cuda")).numel() == 0
    assert eng.resample_g711_encode(torch.empty(0, 64, device="cuda")).shape == (0, 32)
    assert eng.g711_decode(torch.empty(0, dtype=torch.uint8, device="cuda")).numel() == 0


def test_cpu_tensor_is_rejected(eng):
    with pytest.raises(RuntimeError):
        eng.g711_encode(torch.zeros(4))

