#!/usr/bin/env python
"""Text-encoder throughput: the library's ragged encoder (engine.TTSEncoder, b2_enc_*) against the transformers module in torch bf16, padded
the way B200Frontend.start pads a cohort (every sentence to the longest), on the same synthetic weights and token ids, alternating in one
process.  Two cohorts of 1,024 sentences: all 64 tokens, and lengths drawn uniformly from [8, 200].  Also the admission cost of a cohort:
encoder + b2_dec_start (cross-attention keys / values of the six decoder layers).

Rates are over USEFUL work, computed from shapes: 169.9 MFLOP per valid token for the Linears (12 layers x (768 x 2304 + 768 x 768 +
2 x 768 x 3072) x 2) plus 6 x len x 768 per token and layer for the attention of a sentence of `len` tokens (q.k, q.pe_k, p.v).  The padded
torch arm does more work than that; it is charged the same useful FLOPs.  The weights (170 MB in bf16) and a pass's activations exceed the
126 MB L2, so nothing is timed out of cache.  Prints one JSON line with the card's name and power limit read in the same run.

    python tools/encoder_bench.py [--iters 10] [--warmup 3] [--mode bf16] [--out encoder_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

LINEAR_FLOP_PER_TOKEN = 12 * (768 * 2304 + 768 * 768 + 2 * 768 * 3072) * 2


def useful_flop(lengths):
    return sum(n * LINEAR_FLOP_PER_TOKEN + 12 * 6 * n * n * 768 for n in lengths)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
    name, power, clk = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clk}


def torch_module(sd, device):
    import torch
    import transformers as tr
    from infernos_b200.engine import decoder_position_table
    cfg = tr.SpeechT5Config()
    with torch.device("meta"):
        enc = tr.models.speecht5.modeling_speecht5.SpeechT5EncoderWithTextPrenet(cfg)
    enc = enc.to_empty(device="cpu")
    enc.load_state_dict({k[len("speecht5.encoder."):]: v for k, v in sd.items() if k.startswith("speecht5.encoder.")}, strict=False)
    enc.prenet.encode_positions.pe = decoder_position_table(cfg.max_text_positions)[None]
    return enc.to(device=device, dtype=torch.bfloat16).eval()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--mode", default="bf16")
    ap.add_argument("--sessions", type=int, default=1024)
    ap.add_argument("--max-tokens", type=int, default=16384)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from infernos_b200 import synth
    from infernos_b200.engine import TTSDecoder, TTSEncoder
    if not torch.cuda.is_available():
        raise SystemExit("encoder_bench needs a GPU")
    dev = torch.device("cuda:0")
    info = card()
    esd = synth.encoder_state_dict()
    g = torch.Generator().manual_seed(3)
    cohorts = {
        "fixed64": [64] * a.sessions,
        "ragged8_200": torch.randint(8, 201, (a.sessions,), generator=g).tolist(),
    }
    enc = TTSEncoder(dev, esd, mode=a.mode, max_tokens=a.max_tokens, max_len=200)
    ref = torch_module(esd, dev)
    dec = TTSDecoder(dev, synth.decoder_state_dict(), mode=a.mode, max_sessions=a.sessions, max_rows=min(a.sessions, 1024), max_steps=32, max_enc_len=200)
    spk = synth.synth_speakers(a.sessions, seed=5).to(dev)
    slots = torch.arange(a.sessions, dtype=torch.int32, device=dev)
    res = {}

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    for name, lengths in cohorts.items():
        ids, mask = synth.synth_token_ids(lengths, seed=7)
        ids_d, mask_d = ids.to(dev), mask.to(dev)
        lens_d = mask_d.sum(1).to(torch.int32)
        tokens = int(sum(lengths))
        flop = useful_flop(lengths)
        with torch.no_grad():
            runs = {
                "gpu_encoder": lambda: enc(ids_d, mask_d),
                "torch_bf16_padded": lambda: ref(input_values=ids_d, attention_mask=mask_d, return_dict=True).last_hidden_state,
                "admission": lambda: dec.start(slots, enc(ids_d, mask_d), lens_d, spk),
            }
            for _ in range(a.warmup):
                for fn in runs.values():
                    fn()
            torch.cuda.synchronize()
            ms = {k: [] for k in runs}
            for _ in range(a.iters):                     # alternating, same process
                for k, fn in runs.items():
                    ms[k].append(timed(fn))
            got = enc(ids_d, mask_d).float()
            want = ref(input_values=ids_d, attention_mask=mask_d, return_dict=True).last_hidden_state.float()
        enc.poll_errors(); dec.poll_errors()
        m = mask_d.bool()
        diff = (got[m] - want[m])
        snr = float(10 * torch.log10((want[m] ** 2).sum() / (diff ** 2).sum()))
        r = {"sessions": len(lengths), "tokens": tokens, "padded_tokens": len(lengths) * max(lengths), "useful_gflop": round(flop / 1e9, 1),
             "gpu_vs_torch_bf16_snr_db": round(snr, 1)}
        for k, v in ms.items():
            v = sorted(v)
            med = v[len(v) // 2]
            r[k] = {"ms_median": round(med, 3), "ms_min": round(v[0], 3), "ms_max": round(v[-1], 3),
                    "tokens_per_s": round(tokens / (med / 1e3)), "useful_tflops": round(flop / (med / 1e3) / 1e12, 1)}
        r["speedup_vs_torch"] = round(r["torch_bf16_padded"]["ms_median"] / r["gpu_encoder"]["ms_median"], 2)
        r["dec_start_ms_by_difference"] = round(r["admission"]["ms_median"] - r["gpu_encoder"]["ms_median"], 3)
        res[name] = r
    enc.close(); dec.close()
    line = json.dumps({"tool": "encoder_bench", **info, "mode": a.mode, "max_tokens": a.max_tokens, "iters": a.iters, "cohorts": res})
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
