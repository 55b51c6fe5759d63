"""GPU parity of the fused ResBlock kernel (csrc/conv_resblock.cu) against a torch restatement of
transformers' HifiGanResidualBlock.forward (modeling_speecht5.py:2954-2962) with the kernel's operand rounding
(bf16 weights and bf16 leaky-ReLU'd activations, fp32/fp64 accumulation, fp32 residual stream)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _ref(x, ws, bs, k, dils, slope, acc, div, round_ops=True):
    """x (W,T,C) fp32; ws [6] (C,C,k); bs [6] (C,).  Returns (W,T,C) float64."""
    rb = (lambda t: t.bfloat16().double()) if round_ops else (lambda t: t.double())
    h = x.double().transpose(1, 2)
    for i, d in enumerate(dils):
        a = rb(F.leaky_relu(h, slope).float())
        y = F.conv1d(a, rb(ws[2 * i]), bs[2 * i].double(), dilation=d, padding=(k - 1) * d // 2)
        a2 = rb(F.leaky_relu(y, slope).float())
        h = h + F.conv1d(a2, rb(ws[2 * i + 1]), bs[2 * i + 1].double(), dilation=1, padding=(k - 1) // 2)
    h = h.transpose(1, 2)
    if acc is not None:
        h = acc.double() + h
    return h / div


def _run(x, ws, bs, k, dils, slope, acc, div, want32=True, wantb=True, outb_slope=0.1):
    from infernos_b200 import _lib
    lib = _lib.load()
    W, T, C = x.shape
    hw = torch.stack(ws).contiguous()
    hb = torch.stack(bs).contiguous()
    xd = x.cuda().contiguous()
    accd = acc.cuda().contiguous() if acc is not None else None
    out32 = torch.full((W, T, C), float("nan"), device="cuda", dtype=torch.float32) if want32 else None
    outb = torch.zeros(W, T, C, device="cuda", dtype=torch.bfloat16) if wantb else None
    rc = lib.b2_resblock_tc(xd.data_ptr(), hw.data_ptr(), hb.data_ptr(), W, T, C, k, dils[0], dils[1], dils[2],
                            accd.data_ptr() if accd is not None else None,
                            out32.data_ptr() if out32 is not None else None,
                            outb.data_ptr() if outb is not None else None,
                            slope, outb_slope, div, torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, "resblock_tc")
    torch.cuda.synchronize()
    return (out32.cpu() if want32 else None), (outb.float().cpu() if wantb else None)


def _make(W, T, C, k, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(W, T, C, generator=g)
    ws = [torch.randn(C, C, k, generator=g) / (C * k) ** 0.5 for _ in range(6)]
    bs = [torch.randn(C, generator=g) * 0.1 for _ in range(6)]
    acc = torch.randn(W, T, C, generator=g)
    return x, ws, bs, acc


SHAPES = [
    # (W, T, C, k)
    (3, 3072, 32, 11), (2, 3072, 32, 7), (2, 3072, 32, 3),
    (2, 768, 64, 11), (3, 768, 64, 7), (2, 768, 64, 3),
    (3, 100, 32, 7), (2, 700, 64, 11), (1, 393, 32, 11), (5, 1, 32, 3), (2, 513, 64, 3),
    (2, 900, 32, 5), (2, 700, 32, 9), (1, 3072, 32, 9),       # tap counts that take the stacked-output kernel's table-driven MMA loop
    (3, 192, 128, 3), (2, 192, 128, 7), (3, 192, 128, 11), (2, 600, 128, 7), (1, 257, 128, 3), (2, 40, 128, 11),
]


@pytest.fixture(autouse=True, scope="module")
def _stacked_kernel_for_every_tap_count():
    """C = 32 shapes go to the stacked-output kernel (conv_resblock_t.cu) from five taps up by default; in this module also the three-tap
    shapes do, so that both of its MMA issue paths (unrolled k = 3 / 7 / 11, table-driven otherwise) are checked against torch.  The
    time-as-M kernel's C = 32 path is covered by test_time_as_m_kernel_c32 below and, inside the bf16 tail, by the stage-boundary taps
    test of tests/test_gpu_tail.py."""
    from infernos_b200 import _lib
    lib = _lib.load()
    lib.b2_debug_set_stacked_min_taps(3)
    yield
    lib.b2_debug_set_stacked_min_taps(0)


@pytest.mark.parametrize("shape", SHAPES)
def test_fused_resblock_matches_torch(shape):
    W, T, C, k = shape
    x, ws, bs, acc = _make(W, T, C, k, seed=sum(shape))
    dils = (1, 3, 5)
    out, outb = _run(x, ws, bs, k, dils, 0.1, acc, 3.0)
    ref = _ref(x, ws, bs, k, dils, 0.1, acc, 3.0)
    assert torch.isfinite(out).all()
    err = (out.double() - ref).abs()
    snr = 10 * torch.log10((ref ** 2).sum() / (err ** 2).sum().clamp_min(1e-30)).item()
    # same operand rounding as the kernel: what is left is fp32 accumulation order plus the odd bf16 rounding flip of an
    # intermediate activation
    assert snr > 60.0, f"snr {snr:.1f} dB, max err {err.max().item():.3e}"
    assert err.max().item() < 2e-2
    assert (outb.double() - F.leaky_relu(ref, 0.1)).abs().max().item() < 5e-2
    # against the un-rounded fp64 ResBlock: bf16 operands only
    ref_exact = _ref(x, ws, bs, k, dils, 0.1, acc, 3.0, round_ops=False)
    snr_exact = 10 * torch.log10((ref_exact ** 2).sum() / ((out.double() - ref_exact) ** 2).sum()).item()
    assert snr_exact > 40.0, snr_exact


@pytest.mark.parametrize("shape", [(2, 3072, 32, 3), (2, 1000, 32, 7), (1, 3072, 32, 11)])
def test_time_as_m_kernel_c32(shape):
    """the same check with every C = 32 block on the time-as-M kernel (conv_resblock.cu), which the product keeps for three-tap blocks"""
    from infernos_b200 import _lib
    lib = _lib.load()
    lib.b2_debug_set_stacked_min_taps(99)
    try:
        W, T, C, k = shape
        x, ws, bs, acc = _make(W, T, C, k, seed=sum(shape))
        out, _ = _run(x, ws, bs, k, (1, 3, 5), 0.1, acc, 3.0)
        ref = _ref(x, ws, bs, k, (1, 3, 5), 0.1, acc, 3.0)
        err = (out.double() - ref).abs()
        snr = 10 * torch.log10((ref ** 2).sum() / (err ** 2).sum().clamp_min(1e-30)).item()
        assert snr > 60.0 and err.max().item() < 2e-2, (snr, err.max().item())
    finally:
        lib.b2_debug_set_stacked_min_taps(3)


def test_fused_resblock_output_options():
    W, T, C, k = 2, 900, 32, 7
    x, ws, bs, acc = _make(W, T, C, k, seed=99)
    dils = (1, 3, 5)
    ref = _ref(x, ws, bs, k, dils, 0.1, None, 1.0)
    out, _ = _run(x, ws, bs, k, dils, 0.1, None, 1.0, want32=True, wantb=False)
    assert (out.double() - ref).abs().max().item() < 2e-2
    _, outb = _run(x, ws, bs, k, dils, 0.1, None, 1.0, want32=False, wantb=True, outb_slope=0.01)
    assert (outb.double() - F.leaky_relu(ref, 0.01)).abs().max().item() < 5e-2


def test_fused_resblock_rejects_unsupported_width():
    from infernos_b200 import _lib
    lib = _lib.load()
    x = torch.zeros(1, 8, 256, device="cuda")
    w = torch.zeros(6, 256, 256, 3)
    b = torch.zeros(6, 256)
    o = torch.zeros(1, 8, 256, device="cuda")
    rc = lib.b2_resblock_tc(x.data_ptr(), w.data_ptr(), b.data_ptr(), 1, 8, 256, 3, 1, 3, 5, None, o.data_ptr(), None, 0.1, 0.1, 1.0, None)
    assert rc != 0
    assert b"unsupported" in lib.b2_last_error(None)
