"""One Linear at a time (b2_linear: the packing and launch the encoder and decoder use, tile choice included) against a float64 reference.

bf16 mode runs the tcgen05 GEMM k_gemm_tc; its reference rounds A and W to bf16 first (round-to-nearest-even, like __float2bfloat16_rn) and
then computes act(A W^T + b) * colscale in float64.  fp32 mode runs the CUDA-core kernel against the unrounded operands.  Every output
element must lie within  c * S + 1e-6  of the reference, S = sum_k |a_k w_k| (times |colscale|): a per-element bound, so that an error in
a few elements of a large tensor cannot hide under a max-abs tolerance set by its largest values.  Shapes are every Linear of the two models
at their packed sizes, at row counts that reach every instantiation of the launcher, with rows of A past M poisoned with NaN and the
outputs past M fenced with a sentinel.

Run as a script (python tests/test_gpu_linear.py out.npz CASE...), it computes the named bf16 cases and saves what the GPU returned: the
runtime switches B2_GEMM_NT256 / B2_GEMM_DEEP are read once per process, so their variants run in subprocesses."""
import ctypes
import os
import subprocess
import sys
import warnings

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# c of the bound per mode: at most 8x the worst |got - ref| / S measured over the cases below on an NVIDIA B200 (1,000 W power limit):
# 4.55e-7 in bf16 mode (ff2, K = 3,072), 3.54e-7 in fp32 mode (ff1); DESIGN.md section 2
C_BF16 = 3e-6
C_FP32 = 2.5e-6
SENTINEL = 2.0 ** 20        # exact in bf16 too

# id: (K, N, M, act, colscale, outputs, spare rows of A past M).  Layers at the sizes finalize_dec / finalize_enc pack them.
BF16_CASES = {
    "prenet0_m16": (128, 256, 16, 1, True, "both", 112),      # the decoder's A map spans its workspace: 128 rows here
    "prenet1_m129": (256, 256, 129, 1, True, "both", 40),
    "fin_m300": (256, 768, 300, 0, False, "32", 20),
    "spkl_m127": (1280, 768, 127, 0, False, "32", 0),         # a_rows == M: the map's own edge inside the last 128-row box
    "qkv_m1": (768, 2304, 1, 0, False, "32", 0),
    "qkv_m128": (768, 2304, 128, 0, False, "32", 64),
    "qkv_m1025": (768, 2304, 1025, 0, False, "32", 100),      # 9 x 18 tiles of 128 x 128 > 148 SMs: 128 x 256 tiles
    "self_m4096": (768, 768, 4096, 0, False, "32", 7),        # so / xq / xo / o
    "ff1_m300": (768, 3072, 300, 2, False, "both", 33),      # both outputs: the GELU epilogue at fp32 precision
    "ff1_m769": (768, 3072, 769, 2, False, "b", 1),           # 7 x 24 > 148: 128 x 256 tiles
    "ff1_m16384": (768, 3072, 16384, 2, False, "b", 0),       # the encoder's default workspace
    "ff2_m129": (3072, 768, 129, 0, False, "32", 64),
    "xkv_m128": (768, 9216, 128, 0, False, "32", 0),
    "xkv_m257": (768, 9216, 257, 0, False, "32", 31),         # 3 x 72 > 148: 128 x 256 tiles
    "outl_m769": (768, 192, 769, 0, False, "32", 5),
    "k64_m300": (64, 256, 300, 0, False, "both", 12),         # one K block: fewer than the ring's stages
    "n2048_m1025": (256, 2048, 1025, 0, False, "both", 3),    # the only shape on 128 x 128 tiles with a 4-stage ring
    "n2176_m4096": (768, 2176, 4096, 0, False, "32", 9),      # N >= 2048 but no 256 map (N % 256 != 0): stays on 128 x 128
}
FP32_CASES = {
    "prenet0_m16": (128, 256, 16, 1, True, "32", 5),
    "qkv_m129": (768, 2304, 129, 0, False, "32", 3),
    "ff1_m769": (768, 3072, 769, 2, False, "32", 0),
    "ff2_m300": (3072, 768, 300, 0, False, "32", 17),
    "k64_m1": (64, 256, 1, 0, False, "32", 0),
    "outl_m127": (768, 192, 127, 0, False, "32", 1),
}
# the cases whose launch each switch changes
VARIANTS = {
    "B2_GEMM_NT256": ["qkv_m1025", "ff1_m769", "xkv_m257", "ff1_m16384"],
    "B2_GEMM_DEEP": ["spkl_m127", "qkv_m128", "self_m4096", "ff2_m129", "xkv_m128", "outl_m769", "n2176_m4096"],
}


def _inputs(case, seed):
    K, N, M, act, cs, outs, spare = case
    g = torch.Generator().manual_seed(seed)
    a = torch.randn(M, K, generator=g)
    w = torch.randn(N, K, generator=g) / K ** 0.5
    b = torch.randn(N, generator=g) * 0.1
    colscale = (torch.rand(N, generator=g) < 0.5).float() * 2.0 if cs else None      # the prenet's dropout keep-mask x 1 / (1 - p)
    return a, w, b, colscale


def _seed(name, bf16):
    return sum(map(ord, name)) * 2 + (1 if bf16 else 0)


def _bf16_round_np(x):
    """float64 -> float32 -> bf16 (round to nearest even) -> float64, in numpy"""
    u = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32).astype(np.uint64)
    u = ((u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000).astype(np.uint32)
    return u.view(np.float32).astype(np.float64)


def reference(a, w, b, act, colscale, bf16):
    """-> (act(A W^T + b) * colscale, S = (|A| |W|^T) * |colscale|), float64, on the operands the kernel sees"""
    A = (a.bfloat16() if bf16 else a).double()
    W = (w.bfloat16() if bf16 else w).double()
    y = A @ W.T + b.double()
    if act == 1:
        y = y.clamp_min(0.0)
    elif act == 2:
        y = 0.5 * y * (1.0 + torch.erf(y / 2 ** 0.5))
    S = A.abs() @ W.abs().T
    if colscale is not None:
        y = y * colscale.double()
        S = S * colscale.double().abs()
    return y, S


def outside(got, ref, S, c, rounded=False):
    """bool mask of the elements outside the bound (NaN counts as outside).  rounded: `got` was rounded to bf16 after the fp32 result."""
    tol = c * S + 1e-6
    if rounded:
        tol = tol * (1 + 2.0 ** -8) + 2.0 ** -8 * ref.abs()
    return ~((got.double() - ref).abs() <= tol)


def run_linear(case, bf16, seed):
    """-> (out32 or None, outb or None, (tile N, stages)): the outputs with their spare rows past M"""
    from infernos_b200 import _lib
    lib = _lib.load()
    K, N, M, act, cs, outs, spare = case
    a, w, b, colscale = _inputs(case, seed)
    dt = torch.bfloat16 if bf16 else torch.float32
    ain = torch.full((M + spare, K), float("nan"), dtype=dt)
    ain[:M] = a.to(dt)
    ain = ain.cuda()
    out32 = torch.full((M + 3, N), SENTINEL, device="cuda") if outs in ("32", "both") else None
    outb = torch.full((M + 3, N), SENTINEL, device="cuda", dtype=torch.bfloat16) if outs in ("b", "both") else None
    cs_d = colscale.cuda() if colscale is not None else None
    launched = (ctypes.c_int * 2)(-1, -1)
    rc = lib.b2_linear(torch.cuda.current_device(), _lib.MODE_BF16 if bf16 else _lib.MODE_FP32, ain.data_ptr(), M, M + spare,
                       w.contiguous().data_ptr(), b.contiguous().data_ptr(), N, K, act, cs_d.data_ptr() if cs_d is not None else None,
                       out32.data_ptr() if out32 is not None else None, outb.data_ptr() if outb is not None else None, launched,
                       torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, "b2_linear")
    return (out32.cpu() if out32 is not None else None, outb.cpu() if outb is not None else None, (launched[0], launched[1]))


def expected_launch(case, sms, nt256=True, deep=True):
    """(tile N, ring stages) the launcher is meant to pick (layers.cuh gemm_tile_n, decoder.cu gemm_tc_stages)"""
    K, N, M = case[:3]
    nt = 128 if N % 128 == 0 and N >= 2048 else 64
    if nt256 and nt == 128 and N % 256 == 0 and -(-M // 128) * (N // 128) > sms:
        nt = 256
    return nt, (6 if nt == 128 else 8) if deep and K >= 512 and nt != 256 else 4


_REF = {}            # (case, bf16) -> float64 (ref, S): about 1 GB with ff1_m16384, dropped when this module's tests are done


@pytest.fixture(scope="module", autouse=True)
def _drop_references():
    yield
    _REF.clear()


def _ref(name, bf16):
    key = (name, bf16)
    if key not in _REF:
        case = (BF16_CASES if bf16 else FP32_CASES)[name]
        a, w, b, colscale = _inputs(case, _seed(name, bf16))
        _REF[key] = reference(a, w, b, case[3], colscale, bf16)
    return _REF[key]


def check_case(name, bf16, out32, outb, what=""):
    """bound on rows < M, sentinel untouched on rows >= M, bf16 output == bf16(fp32 output); -> worst |got - ref| / S"""
    K, N, M = (BF16_CASES if bf16 else FP32_CASES)[name][:3]
    c = C_BF16 if bf16 else C_FP32
    ref, S = _ref(name, bf16)
    worst = 0.0
    for got, rounded in ((out32, False), (outb, True)):
        if got is None:
            continue
        assert bool((got[M:].float() == SENTINEL).all()), f"{name}{what}: rows at or past M = {M} were written"
        g = got[:M].double()
        assert bool(torch.isfinite(g).all()), f"{name}{what}: non-finite outputs below row M (NaN rows of A past M leaked in?)"
        bad = outside(g, ref, S, c, rounded)
        if not rounded:
            pos = S > 0
            worst = float(((g - ref).abs()[pos] / S[pos]).max()) if bool(pos.any()) else 0.0
        assert not bool(bad.any()), (f"{name}{what}: {int(bad.sum())} of {bad.numel()} elements outside {c:g} * S + 1e-6 "
                                     f"(first at {tuple(bad.nonzero()[0].tolist())})")
    if out32 is not None and outb is not None:
        assert torch.equal(outb[:M], out32[:M].bfloat16()), f"{name}{what}: the bf16 output is not bf16(fp32 output)"
    return worst


def _sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


# ------------------------------------------------------------------------------------------------ the bound itself (CPU)
@pytest.mark.parametrize("c", [C_BF16, C_FP32])
def test_the_bound_rejects_a_dropped_k_step_a_shifted_row_and_bf16_rounding(c):
    """The bound must be tight enough to matter: on a qkv-sized Linear it accepts the float64 result rounded to fp32 and rejects three
    faults of the kind a GEMM makes -- one 16-wide K step (one MMA) left out, one output row taken from its neighbour, the fp32 result
    rounded to bf16."""
    rng = np.random.default_rng(5)
    M, K, N = 300, 768, 768
    A = _bf16_round_np(rng.standard_normal((M, K)))
    W = _bf16_round_np(rng.standard_normal((N, K)) / K ** 0.5)
    b = rng.standard_normal(N) * 0.1
    ref = A @ W.T + b
    S = np.abs(A) @ np.abs(W).T

    def rejects(got):
        return bool(outside(torch.from_numpy(got), torch.from_numpy(ref), torch.from_numpy(S), c).any())

    assert not rejects(ref.astype(np.float32).astype(np.float64))
    k0 = 16 * 17
    assert rejects(ref - A[:, k0:k0 + 16] @ W[:, k0:k0 + 16].T)
    shifted = ref.copy()
    shifted[129] = ref[130]
    assert rejects(shifted)
    assert rejects(_bf16_round_np(ref))


def test_bad_arguments_fail_with_a_message_and_m0_is_a_no_op():
    """Checked before any device is touched: these run without a GPU."""
    from infernos_b200 import _lib
    from infernos_b200 import build
    build.build()
    lib = _lib.load()
    w, b = torch.zeros(256, 128), torch.zeros(256)
    launched = (ctypes.c_int * 2)(-1, -1)

    def call(mode=1, M=4, a_rows=4, N=256, K=128, act=0, out32=16, outb=None):
        return lib.b2_linear(0, mode, 16, M, a_rows, w.data_ptr(), b.data_ptr(), N, K, act, None, out32, outb, launched, None)

    for kw, msg in (({"mode": 2}, b"mode"), ({"K": 96}, b"K 96"), ({"K": 0}, b"K 0"), ({"N": 200}, b"N 200"), ({"a_rows": 3}, b"a_rows 3"),
                    ({"act": 3}, b"act 3"), ({"mode": 0, "outb": 16}, b"fp32 mode"), ({"mode": 0, "out32": None}, b"fp32 mode")):
        assert call(**kw) != 0, kw
        assert msg in lib.b2_last_error(None), (kw, lib.b2_last_error(None))
    assert call(M=0, a_rows=0) == 0
    assert tuple(launched) == (0, 0)


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
def test_tcgen05_linear_against_float64_every_layer_and_instantiation():
    sms = _sms()
    reached, worst = {}, {}
    for name, case in BF16_CASES.items():
        out32, outb, launched = run_linear(case, True, _seed(name, True))
        assert launched == expected_launch(case, sms), (name, launched, expected_launch(case, sms))
        worst[name] = check_case(name, True, out32, outb)
        reached.setdefault(launched, []).append(name)
        print(f"bf16 {name:14s} K {case[0]:5d} N {case[1]:5d} M {case[2]:6d}: k_gemm_tc<{launched[0]}, {launched[1]}>, "
              + (f"worst |d| / S {worst[name]:.2e}" if case[5] != "b" else "bf16 output only: within the bound + bf16 rounding"))
    print(f"bf16: worst |d| / S over all cases {max(worst.values()):.2e}, c = {C_BF16:g}; instantiations reached: "
          + ", ".join(f"<{t}, {s}> x{len(v)}" for (t, s), v in sorted(reached.items())))
    assert set(reached) == {expected_launch(case, sms) for case in BF16_CASES.values()}
    missing = {(64, 4), (64, 8), (128, 4), (128, 6), (256, 4)} - set(reached)
    wide = {"ff1_m769", "qkv_m1025", "xkv_m257"} - set(reached.get((256, 4), []))
    if missing or wide:     # the row counts are chosen for 148 SMs; elsewhere the tile choice moves and coverage shrinks
        warnings.warn(f"{sms} SMs: k_gemm_tc instantiations not reached {sorted(missing)}, 128 x 256 cases on 128 x 128 tiles {sorted(wide)}")
    if sms == 148:
        assert not missing and not wide


@pytest.mark.gpu
def test_cuda_core_linear_against_float64():
    worst = {}
    for name, case in FP32_CASES.items():
        out32, _, launched = run_linear(case, False, _seed(name, False))
        assert launched == (0, 0)
        worst[name] = check_case(name, False, out32, None)
        print(f"fp32 {name:14s} K {case[0]:5d} N {case[1]:5d} M {case[2]:6d}: worst |d| / S {worst[name]:.2e}")
    print(f"fp32: worst |d| / S over all cases {max(worst.values()):.2e}, c = {C_FP32:g}")
    assert C_FP32 <= 1e-4


def _run_variant(tmp_path, env, names):
    out = str(tmp_path / "variant.npz")
    e = dict(os.environ)
    e.update(env)
    subprocess.run([sys.executable, os.path.abspath(__file__), out, *names], check=True, env=e, timeout=600)
    return np.load(out)


@pytest.mark.gpu
@pytest.mark.parametrize("switch", sorted(VARIANTS))
def test_runtime_switch_variant_meets_the_same_bound(tmp_path, switch):
    """B2_GEMM_NT256=0 keeps the wide layers on 128 x 128 tiles, B2_GEMM_DEEP=0 gives every GEMM a 4-stage ring.  Each variant meets the
    same float64 bound and gives the default launch's bits (measured: it does).  The encoder's and decoder's promise that a sentence's
    output does not depend on its companions rests on the 128 x 256 and 128 x 128 tiles agreeing bit for bit, because a large pass runs
    the wide layers on the former and the same sentence alone on the latter."""
    names = VARIANTS[switch]
    got = _run_variant(tmp_path, {switch: "0"}, names)
    sms = _sms()
    for name in names:
        case = BF16_CASES[name]
        launched = tuple(int(x) for x in got[name + ".launched"])
        want = expected_launch(case, sms, nt256=switch != "B2_GEMM_NT256", deep=switch != "B2_GEMM_DEEP")
        assert launched == want != expected_launch(case, sms), (name, launched, want)
        out32 = torch.from_numpy(got[name + ".out32"]) if name + ".out32" in got else None
        outb = torch.from_numpy(got[name + ".outb"]).view(torch.bfloat16) if name + ".outb" in got else None
        worst = check_case(name, True, out32, outb, f" ({switch}=0)")
        d32, db, _ = run_linear(case, True, _seed(name, True))
        same = (out32 is None or torch.equal(out32, d32)) and (outb is None or torch.equal(outb, db))
        print(f"{switch}=0 {name:14s}: k_gemm_tc<{launched[0]}, {launched[1]}> instead of <{expected_launch(case, sms)[0]}, "
              f"{expected_launch(case, sms)[1]}>, worst |d| / S {worst:.2e}, bitwise equal to the default launch: {same}")
        assert same, f"{name}: k_gemm_tc<{launched[0]}, {launched[1]}> does not give the default launch's bits"


if __name__ == "__main__":
    res = {}
    for name in sys.argv[2:]:
        o32, ob, la = run_linear(BF16_CASES[name], True, _seed(name, True))
        res[name + ".launched"] = np.array(la)
        if o32 is not None:
            res[name + ".out32"] = o32.numpy()
        if ob is not None:
            res[name + ".outb"] = ob.view(torch.int16).numpy()
    np.savez(sys.argv[1], **res)
