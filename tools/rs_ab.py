#!/usr/bin/env python
"""Timing of the fused resample+encode kernel at several row lengths."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from infernos_b200 import engine
def timed(fn, iters=20):
    for _ in range(3): fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters
for rows, L in ((100_000, 320), (100_000, 1600), (20_000, 8192), (4096, 8192), (1024, 8192)):
    x = (torch.rand(rows, L, device="cuda") * 2 - 1) * 0.9
    ms = timed(lambda: engine.resample_g711_encode(x))
    nb = 9.0 * rows * (L // 2)
    print(rows, L, round(ms, 4), "ms", round(nb / ms / 1e6), "GB/s", round(nb / ms / 1e6 / 6446.6, 3))

# 8k -> 16k side (G711Codec.decode + AudioChunk.resample): 0.5 B in + 4 B out per 16 kHz output sample
for rows, L in ((100_000, 160), (100_000, 800), (20_000, 4096)):
    codes = torch.randint(0, 256, (rows, L), device="cuda").to(torch.uint8)
    ms = timed(lambda: engine.g711_decode_upsample(codes))
    nb = 9.0 * rows * L
    print("decode+upsample", rows, L, round(ms, 4), "ms", round(nb / ms / 1e6), "GB/s", round(nb / ms / 1e6 / 6446.6, 3))
# what a read-dominated stream can reach on this GPU: torch's reduction over 4 GB, and a copy (the MEASURED_PEAKS method)
big = torch.empty(1 << 30, dtype=torch.float32, device="cuda").normal_()
ms = timed(lambda: big.sum(), iters=5)
print("read-only probe (torch.sum over 4 GiB):", round(4 * (1 << 30) / ms / 1e6), "GB/s")
dst = torch.empty_like(big)
ms = timed(lambda: dst.copy_(big), iters=5)
print("copy probe (read+write, 8 GiB moved):", round(8 * (1 << 30) / ms / 1e6), "GB/s")
