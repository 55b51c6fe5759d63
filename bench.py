#!/usr/bin/env python
"""Benchmark of the B200 TTS tail (mel chunks -> HiFiGAN -> chunker -> 16k->8k -> G.711).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

Metric (BASELINE.json): concurrent real-time 8 kHz G.711 TTS streams per job at RTF <= 1
= seconds of audio produced per second of device time.  A step is one reference `infer()` tail
(HelloSippyRTPipe.py:231-240) over every session of the batch: 32 new mel frames -> 4 windows of 12 frames
-> 8,192 samples @16 kHz -> 4,096 G.711 bytes (0.512 s of audio) per session.

Prints ONE JSON line on rank 0.  `value` is timed with inputs resident in HBM; `e2e` goes through the
host-buffer C-ABI entry (pinned H2D of the mel, D2H of the G.711 bytes, inside the timed region).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

AUDIO_S_PER_FRAME = 256 / 16000.0
# algorithmic work per 12-frame window (BASELINE.md section 3, SURVEY.md 8d)
FLOP_PER_WINDOW_TC = 12 * 2 * (4 * 33.030144e6 + 4 * 1.048576e6 + 0.28672e6) + 2 * 10.22e6   # tcgen05 kernels: upsamplers, ResBlocks,
                                                                                            # conv_pre, chunker upsamplers + ResBlock
FLOP_PER_WINDOW_ALL = 12 * 273.318e6 + 25.68e6 + 0.057e6 * 4
# the three stages the fused ResBlock kernel covers (C = 128, 64, 32): 33.03 MMAC per frame per stage, algorithmic (no halo rows)
FLOP_PER_WINDOW_RESBLOCK_STAGE = 12 * 2 * 33.030144e6
CODEC_BYTES_PER_OUT = 9.0                                            # 2 fp32 in + 1 byte out per 8 kHz sample
DUMP_BYTES = 60 << 20                                                # --dump-outputs: all files of one run together, under 64 MB with headers


def dump_outputs(out_dir: str, arrays: dict, rank: int = 0, world: int = 1) -> None:
    """Writes what the timed path returned in its last step as out_dir/<name>.npy (float32), so that two builds can be compared
    output for output.  Each rank gets an equal share of DUMP_BYTES; an array larger than its share keeps a fixed, seeded sample
    of its rows (sessions), in row order, so the same arguments select the same rows in every run."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // (len(arrays) * world)
    for name, t in arrays.items():
        a = t.cpu().numpy().astype(np.float32)
        keep = max(1, share // max(a[0].nbytes, 1))
        if a.shape[0] > keep:
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
        np.save(os.path.join(out_dir, f"{name}_rank{rank}.npy" if world > 1 else f"{name}.npy"), a)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm_gbs=d["hbm_gbs"], tf_sustained=d["bf16_tflops_sustained"], tf_burst=d["bf16_tflops"], source="measured")
    return dict(hbm_gbs=6650.0, tf_sustained=1400.0, tf_burst=1590.0, source="fallback")


def load_traffic():
    """DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture (profiles/): measured under the
    profiler at a smaller session count, scaled per window; {} when the summary is absent."""
    for name in ("r3_resblock_traffic.json", "r2z_resblock_traffic.json", "r2_resblock_traffic.json", "r1_resblock_traffic.json"):          # the newest capture that is committed
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                d = json.load(f)
            d["file"] = "profiles/" + name
            return d
        except Exception:
            continue
    return {}


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.rows, self.proc, self.all_rows, self.t0 = index, [], None, [], 0.0

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.all_rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def mark_begin(self):
        """nvidia-smi takes a few hundred ms to start streaming, so it is launched before the warm-up; only samples that
        arrive between mark_begin() (start of the timed region) and stop() are reported."""
        self.t0 = time.time()

    def samples_under_load(self) -> int:
        return sum(1 for t, _ in self.all_rows if t >= self.t0)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.rows = [r for t, r in self.all_rows if t >= self.t0]
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower() == "active" for r in self.rows)]
        pw = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "power_w_max": max(pw) if pw else None}


# ----------------------------------------------------------------------------------------------- CPU arm
def cpu_tail_fn(dtype=None):
    """The reference's own CPU arithmetic for the path: transformers SpeechT5HifiGan (the third-party module the
    reference calls) when importable, the oracle's restatements for AmendmentNetwork1 / Resample / G711Codec.encode
    (their sources live in /root/reference, which does not exist on the GPU box)."""
    import torch
    from infernos_b200 import synth
    from oracle import codec as ocodec
    from oracle import tail as otail
    vsd, csd = synth.hifigan_state_dict(), synth.chunker_state_dict()
    dtype = dtype or torch.float32
    if dtype != torch.float32:          # the reference's product precision: maybe_half() on every module (HelloSippyRTPipe.py:57,171-186)
        vsd = {k: v.to(dtype) for k, v in vsd.items()}
        csd = {k: v.to(dtype) for k, v in csd.items()}
    kind = "port"
    try:
        from transformers import SpeechT5HifiGan, SpeechT5HifiGanConfig
        voc = SpeechT5HifiGan(SpeechT5HifiGanConfig())
        voc.load_state_dict({k: v.float() for k, v in vsd.items()}, strict=True)
        voc = voc.to(dtype)
        voc.eval()
        vocoder = lambda win: voc(win)
        desc = "transformers.SpeechT5HifiGan + oracle AmendmentNetwork1/Resample/G.711 restatements"
    except Exception:
        vocoder = lambda win: otail.hifigan_forward(vsd, win)
        desc = "oracle torch restatement of HiFiGAN/AmendmentNetwork1/Resample/G.711"

    def step(pre, mel):
        with torch.no_grad():
            B = mel.size(0)
            win, new_pre = otail.build_windows(pre, mel)
            audio = vocoder(win)
            audio = otail.chunker_forward(csd, win, audio)
            audio = torch.cat(audio.split(B, dim=0), dim=1).float()
            audio = otail.resample(audio, 16000, 8000)
            by = ocodec.encode_f32(audio.numpy(), 0)
        return new_pre, by

    return step, kind, desc


def run_cpu(sessions: int, steps: int, warmup: int, frames: int = 32, dtype=None):
    import torch
    from infernos_b200 import synth
    torch.set_num_threads(os.cpu_count() or 1)
    dtype = dtype or torch.float32
    step, kind, desc = cpu_tail_fn(dtype)
    mel = synth.synth_mel(sessions, frames, seed=7).to(dtype)
    pre = torch.zeros(sessions, 4, 80, dtype=dtype)
    for _ in range(warmup):
        pre, _ = step(pre, mel)
    t0 = time.perf_counter()
    for _ in range(steps):
        pre, _ = step(pre, mel)
    dt = time.perf_counter() - t0
    streams = sessions * frames * AUDIO_S_PER_FRAME * steps / dt
    return dict(value=streams, ms_per_step=dt / steps * 1e3, kind=kind, cores=torch.get_num_threads(),
                sample=f"{sessions} sessions x {frames} mel frames per step, {steps} steps, {'fp32' if dtype == torch.float32 else 'bf16'}, {desc}")


def main_cpu_sweep(args):
    """SURVEY section 8(d) CPU baseline table: the reference tail on this box's host cores, fp32 and bf16, B in {1, 8, 64},
    one warm-up + three timed steps each (bf16 B=64 is skipped when bf16 B=8 already takes > 20 s per step)."""
    import torch
    rows = []
    for dtype, name in ((torch.float32, "fp32"), (torch.bfloat16, "bf16")):
        slow = False
        for B in (1, 8, 64):
            if slow:
                rows.append({"dtype": name, "sessions": B, "skipped": "previous batch size took > 20 s per step"})
                continue
            r = run_cpu(B, 3, 1, dtype=dtype)
            rows.append({"dtype": name, "sessions": B, "ms_per_step": round(r["ms_per_step"], 1), "streams_rtf1": round(r["value"], 2),
                         "vocoder_msamples_per_s": round(B * 32 * 256 / r["ms_per_step"] / 1e3, 3), "cores": r["cores"], "kind": r["kind"]})
            print(rows[-1], file=sys.stderr, flush=True)
            slow = r["ms_per_step"] > 20000
    print(json.dumps({"impl": "reference", "cpu_sweep": rows, "os_cpu_count": os.cpu_count(), "torch_threads": torch.get_num_threads()}), flush=True)


def main_reference(args, rank, world):
    if rank != 0:
        return
    if args.cpu_sweep:
        return main_cpu_sweep(args)
    import torch
    sessions = args.ref_sessions
    rdt = torch.bfloat16 if args.ref_dtype == "bf16" else torch.float32
    r = run_cpu(sessions, args.steps, min(args.warmup, 5), dtype=rdt)      # warm-ups matter: the first bf16 calls build oneDNN primitives
    out = {
        "impl": "reference", "metric": "real-time G.711 TTS streams (RTF<=1)", "value": round(r["value"], 3), "unit": "streams",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": min(args.warmup, 5), "ms_per_step": round(r["ms_per_step"], 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16" if args.ref_dtype == "bf16" else "f32", "data": "synthetic",
        "config": {"workload": f"TTS tail (HiFiGAN+chunker+16k->8k+G.711), {sessions} sessions x 32-frame calls on host CPU cores, {args.ref_dtype} "
                               "(the reference casts every module to bf16, HelloSippyRTPipe.py:57,164-186, and batches 8 requests, Cluster/InfernTTSWorker.py:57)",
                   "sessions_per_step": sessions, "frames_per_call": 32},
        "cpu_baseline": {"value": round(r["value"], 3), "unit": "streams", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
        "e2e": {"value": round(r["value"], 3), "unit": "streams", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


# ----------------------------------------------------------------------------------------------- serving-loop legs
def _poll_all(sched, want, out_rows, stop_evt=None, timeout_s=120.0):
    """Consumer: drains completions into out_rows (numpy structured arrays) until `want` chunks have arrived."""
    import numpy as np
    from infernos_b200.engine import _Completion
    dt = np.dtype([("tag", "u8"), ("t_enq", "i8"), ("t_launch", "i8"), ("t_done", "i8"), ("off", "i8"), ("slot", "i4"), ("nbytes", "i4"),
                   ("bs", "i4"), ("pad", "i4")])
    assert dt.itemsize == __import__("ctypes").sizeof(_Completion)
    n, t0 = 0, time.time()
    while n < want and time.time() - t0 < timeout_s and not (stop_evt is not None and stop_evt.is_set() and n >= want):
        recs, _ = sched.poll(timeout_ms=20, want_bytes=True)
        if len(recs):
            out_rows.append(np.frombuffer(sched._recs, dtype=dt, count=len(recs)).copy())
            n += len(recs)
    return n


def run_e2e_pipelined(tail, slots_h, mel_h, steps, warmup):
    """e2e through the serving loop with HOST buffers: every step's mel is copied H2D from pinned staging and its G.711 bytes D2H into
    pinned memory inside the timed region; step n+1's copy-in overlaps step n's compute (two sub-batches in flight)."""
    import numpy as np
    from infernos_b200.engine import TailScheduler
    S, F = mel_h.size(0), mel_h.size(1)
    sched = TailScheduler(tail, nframes=F, depth=2, use_graphs=True, max_batch=S, poll_capacity=max(4096, S))
    rows = []
    try:
        for phase, k in (("warm", max(5, warmup)), ("timed", steps)):      # >= one step per staging buffer: each has its own graph
            rows.clear()
            th = threading.Thread(target=_poll_all, args=(sched, k * S, rows))
            th.start()
            t0 = time.monotonic_ns()
            for _ in range(k):
                sched.submit(slots_h, mel_h)
            th.join()
            r = np.concatenate(rows)
            assert r.shape[0] == k * S, "the serving loop lost chunks"
            ms = (int(r["t_done"].max()) - t0) / 1e6
        st = sched.stats()
    finally:
        sched.close()
    return ms, st


def run_latency(dev, sessions, seconds, chunk_frames=8, mode="bf16", max_windows=2048, tick_ms=0.5, depth=1, max_batch=0, policy=(0, 0)):
    """north_star's joint target: `sessions` concurrent real-time streams, each delivering one chunk_frames-frame mel chunk every
    chunk period (8 frames = 128 ms), arrivals staggered uniformly over the period; latency of a chunk = its nominal arrival time ->
    its G.711 bytes in pinned host memory.  Served by the native sub-batch scheduler (b2_sched_*).  depth = sub-batches in flight: 1 closes the
    next sub-batch the moment the previous one completes (lowest latency: a chunk waits for at most one sub-batch ahead of its own; measured
    p99 at 20,000 sessions 11.9 ms against 16.9 ms with depth 2, profiles/r2c_latency_sweep.json); 2 overlaps the copies with compute."""
    import numpy as np
    import torch
    from infernos_b200 import synth
    from infernos_b200.engine import TailScheduler, TTSTail
    period_ns = int(chunk_frames * AUDIO_S_PER_FRAME * 1e9)
    tail = TTSTail(dev, synth.hifigan_state_dict(), synth.chunker_state_dict(), mode=mode, max_sessions=sessions, max_windows=max_windows)
    sched = TailScheduler(tail, nframes=chunk_frames, depth=depth, use_graphs=True, poll_capacity=8192, max_batch=max_batch)
    if policy != (0, 0):
        sched.set_policy(*policy)
    sched.prebuild(0)                  # every bucket's CUDA graph exists before the first chunk: none is built on the serving path (a backlog
    graphs_pre = sched.stats()["graphs_built"]         # after a host hiccup would otherwise meet sub-batch sizes never seen in the warm-up)
    mel = synth.synth_mel(sessions, chunk_frames, seed=11).pin_memory()
    slots = torch.arange(sessions, dtype=torch.int32)
    phase = (np.arange(sessions, dtype=np.int64) * period_ns) // sessions          # staggered: session i arrives at phase_i + k * period
    rows, stop = [], threading.Event()
    nper = max(2, int(round(seconds * 1e9 / period_ns)))
    warm_periods = 3                                                              # graph buckets get captured here; not reported
    total = (nper + warm_periods) * sessions
    th = threading.Thread(target=_poll_all, args=(sched, total, rows, None, seconds + 60))
    th.start()
    t0 = time.monotonic_ns() + 2_000_000
    sent = 0                                                                      # chunks submitted so far, in arrival order
    late_ticks = 0
    try:
        while sent < total:
            now = time.monotonic_ns()
            due = min(total, int((now - t0) // period_ns) * sessions + int(np.searchsorted(phase, (now - t0) % period_ns, side="right"))) if now >= t0 else 0
            while sent < due:
                k, i = divmod(sent, sessions)
                j = min(sessions, i + (due - sent))
                te = torch.from_numpy(t0 + k * period_ns + phase[i:j])
                sched.submit(slots[i:j], mel[i:j], t_enqueue_ns=te)
                sent += j - i
            spent = (time.monotonic_ns() - now) / 1e6
            if spent > 2 * tick_ms:
                late_ticks += 1
            time.sleep(max(0.0, (tick_ms - spent) / 1e3))
        th.join()
        st = sched.stats()
    finally:
        sched.close()
        tail.close()
    r = np.concatenate(rows) if rows else np.zeros(0)
    r = r[r["t_enq"] >= t0 + warm_periods * period_ns]
    lat = (r["t_done"] - r["t_enq"]) / 1e6
    qd = (r["t_launch"] - r["t_enq"]) / 1e6
    wall_s = (int(r["t_done"].max()) - int(r["t_enq"].min())) / 1e9
    return {"sessions": sessions, "chunk_frames": chunk_frames, "chunk_period_ms": period_ns / 1e6, "chunks": int(lat.size),
            "steps": int(st["sub_batches"]), "p50_ms": round(float(np.percentile(lat, 50)), 3), "p99_ms": round(float(np.percentile(lat, 99)), 3),
            "p999_ms": round(float(np.percentile(lat, 99.9)), 3), "max_ms": round(float(lat.max()), 3), "mean_ms": round(float(lat.mean()), 3),
            "queue_p99_ms": round(float(np.percentile(qd, 99)), 3),
            "mean_sub_batch": round(st["sessions"] / max(1, st["sub_batches"]), 1), "max_sub_batch": int(st["max_sub_batch"]),
            "padded_frac": round(st["padded_sessions"] / max(1, st["sessions"]), 4), "graphs_built": int(st["graphs_built"]),
            "graphs_built_while_serving": int(st["graphs_built"]) - int(graphs_pre),
            "streams_sustained": round(lat.size * chunk_frames * AUDIO_S_PER_FRAME / wall_s, 1), "rtf_ok": bool(lat.max() < period_ns / 1e6),
            "loadgen_late_ticks": late_ticks, "depth": depth, "max_batch": max_batch or max_windows * 8 // chunk_frames, "target_p99_ms": 20.0, "met": bool(np.percentile(lat, 99) < 20.0),
            "definition": "latency = nominal arrival of a session's mel chunk (staggered uniformly over the chunk period) -> its G.711 bytes in "
                          "pinned host memory; H2D and D2H inside; sub-batches formed adaptively, one CUDA graph launch each"}


def run_front_half(dev, tail, slots_d, sessions, calls=8, enc_len=64, mode="bf16"):
    """SURVEY 8 f3: the autoregressive decoder (b2_dec_*) in front of the tail, both on the GPU, frames never leaving the device.
    `calls` consecutive reference infer() calls (16 decoder steps + post-net + tail each) for `sessions` sentences of `enc_len` encoder
    positions; the decoder's attention cost grows with the step count, so per-call times are reported from the first to the last call."""
    import torch
    from infernos_b200 import synth
    from infernos_b200.engine import TTSDecoder
    dec = TTSDecoder(dev, synth.decoder_state_dict(), mode=mode, max_sessions=sessions, max_rows=min(sessions, 1024), max_steps=16 * (calls + 2) + 1,
                     max_enc_len=enc_len)
    try:
        enc = synth.synth_encoder_states(min(sessions, 64), enc_len, seed=5).to(dev).repeat((sessions + 63) // 64, 1, 1)[:sessions].contiguous()
        spk = synth.synth_speakers(sessions, seed=6).to(dev)
        tail.reset_sessions(list(range(sessions)))
        # two warm-up calls: the first runs every kernel eagerly, the second captures the decoder's graph
        dec.start(slots_d, enc, None, spk)
        for _ in range(2):
            mel, _ = dec.steps(slots_d, 16)
            tail.tail(slots_d, mel, want_audio=False, apply_postnet=tail.has_postnet)
        dec.start(slots_d, enc, None, spk)
        torch.cuda.synchronize(dev)
        rows = []
        for c in range(calls):
            e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            e[0].record()
            mel, prob = dec.steps(slots_d, 16)
            e[1].record()
            tail.tail(slots_d, mel, want_audio=False, apply_postnet=tail.has_postnet)
            e[2].record()
            torch.cuda.synchronize(dev)
            rows.append((e[0].elapsed_time(e[1]), e[1].elapsed_time(e[2])))
        dec.poll_errors()
        dms, tms = [r[0] for r in rows], [r[1] for r in rows]
        tot = sum(dms) + sum(tms)
        return {"sessions": sessions, "calls": calls, "encoder_positions": enc_len, "decoder_ms_per_call_first_last": [round(dms[0], 3), round(dms[-1], 3)],
                "decoder_ms_per_call_mean": round(sum(dms) / calls, 3), "tail_ms_per_call_mean": round(sum(tms) / calls, 3),
                "streams_front_plus_tail": round(sessions * 32 * AUDIO_S_PER_FRAME * calls / (tot / 1e3), 1),
                "decoder_hbm_bytes": dec.device_bytes,
                "note": "decoder: prenet + 6 layers + feat_out/prob_out, 16 steps per call as one CUDA graph launch, bf16 tcgen05 GEMMs fed by TMA, "
                        "bf16 KV cache; tail: post-net + vocoder + chunker + resample + G.711 on the decoder's frames in HBM; the text encoder (once "
                        "per sentence) is outside"}
    finally:
        dec.close()


# ----------------------------------------------------------------------------------------------- GPU arm
def main_b200(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    from infernos_b200 import sharding, synth
    from infernos_b200.engine import TTSTail, kernel_launch_count

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # stdout carries exactly ONE JSON line: until it is printed, file descriptor 1 points at stderr, so that anything a native library
    # writes there (NCCL prints its version banner to stdout whatever NCCL_DEBUG_FILE says) cannot land next to it
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    F = args.frames
    first, S = sharding.shard_range(args.sessions * world, world, rank)      # weak scaling: a fixed block of sessions per GPU
    nwin = F // 8
    max_windows = min(S * nwin, args.max_windows)
    tail = TTSTail(dev, synth.hifigan_state_dict(), synth.chunker_state_dict(), mode=args.mode, max_sessions=S, max_windows=max_windows)
    ctx_bytes = tail.device_bytes
    mel_h = synth.synth_mel(S, F, seed=7 + rank).pin_memory()
    slots_h = torch.arange(S, dtype=torch.int32).pin_memory()
    g_h = torch.empty(S, F * 128, dtype=torch.uint8).pin_memory()
    mel_d, slots_d = mel_h.to(dev), slots_h.to(dev)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(ms: float) -> float:
        return sharding.max_over_ranks(ms, device=dev)

    # ---- device-resident timing -------------------------------------------------------------------
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        tail.tail(slots_d, mel_d, want_audio=False)
    barrier()
    sampler.mark_begin()
    l0 = kernel_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        g711, _ = tail.tail(slots_d, mel_d, want_audio=False)
    e1.record()
    barrier()
    launches = kernel_launch_count() - l0
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    audio_s = S * world * F * AUDIO_S_PER_FRAME * args.steps
    value = audio_s / (ms_total / 1e3)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"g711": g711}, rank, world)

    # ---- end-to-end timing with HOST buffers -----------------------------------------------------------
    # (a) the blocking C-ABI call (b2_tts_tail_host: H2D -> tail -> D2H -> sync, nothing overlapped): what a caller pays per call
    for _ in range(min(args.warmup, 3)):
        tail.tail_host(slots_h, mel_h, g_h)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        tail.tail_host(slots_h, mel_h, g_h)
    torch.cuda.synchronize(dev)
    sync_ms = max_over_ranks((time.perf_counter() - t0) * 1e3)
    barrier()
    # (b) the serving loop (b2_sched_*): the same steps from the same pinned host buffers, step n+1's H2D and step n-1's D2H under step n
    e2e_ms, e2e_st = run_e2e_pipelined(tail, slots_h, mel_h, args.steps, min(args.warmup, 3))
    e2e_ms = max_over_ranks(e2e_ms)
    barrier()
    e2e_value = audio_s / (e2e_ms / 1e3)
    # clocks: sampled every 100 ms across both timed regions; a short run (10 steps = 0.23 s) is extended with untimed steps of
    # the same load until three samples are in (bounded), so the line never goes out without clocks
    if rank == 0:
        t_lim = time.time() + 3.0
        while sampler.proc is not None and sampler.samples_under_load() < 3 and time.time() < t_lim:
            tail.tail(slots_d, mel_d, want_audio=False)
            torch.cuda.synchronize(dev)
    clocks = sampler.stop() if rank == 0 else None
    barrier()

    # ---- per-kernel-class timing for the roofline (separate pass, events around every launch) --------
    tail.profile_begin()
    psteps = max(1, min(args.steps, 3))
    for _ in range(psteps):
        tail.tail(slots_d, mel_d, want_audio=False)
    ms_cls, n_cls = tail.profile_end()
    peaks = load_peaks()
    W_step = S * nwin
    bf = args.mode == "bf16"
    tc_ms = (ms_cls["conv_tc"] + ms_cls["resblock_tc"]) if bf else ms_cls["conv_f32"]
    tc_n = (n_cls["conv_tc"] + n_cls["resblock_tc"]) if bf else n_cls["conv_f32"]
    step_ms = max(sum(ms_cls.values()), 1e-9)
    roofline = codec_roof = family_roof = None
    traffic = load_traffic()
    if bf and ms_cls["resblock_tc"] > 0:
        # the dominant kernel: one fused launch per ResBlock for the C = 128 / 64 / 32 stages (9 launches per sub-batch)
        rb_ms, rb_n = ms_cls["resblock_tc"], n_cls["resblock_tc"]
        tf = 3 * FLOP_PER_WINDOW_RESBLOCK_STAGE * W_step * psteps / (rb_ms / 1e3) / 1e12
        roofline = {"bound": "tensor", "kernel": "k_resblock<C> / k_resblock_t (fused tcgen05 ResBlock: six convolutions per launch, residual stream in TMEM; "
                                                 "stages C=128/64/32, 9 launches per sub-batch; the three stage-3 launches stack four output "
                                                 "time steps into the MMA's N dimension and compute the stage's upsampler themselves -- its FLOPs, "
                                                 "done three times, are not counted here)",
                    "achieved": round(tf, 2), "peak": peaks["tf_sustained"], "unit": "TFLOP/s", "frac": round(tf / peaks["tf_sustained"], 4),
                    "peak_source": f"{peaks['source']} bf16 sustained (kernel timed inside a long step)",
                    "traffic": traffic.get("k_resblock_bytes_per_launch"), "traffic_note": traffic.get("note"), "traffic_file": traffic.get("file"),
                    "flop_per_launch": round(3 * FLOP_PER_WINDOW_RESBLOCK_STAGE * W_step * psteps / rb_n),
                    "launches": rb_n, "avg_launch_ms": round(rb_ms / max(rb_n, 1), 4), "share_of_step": round(rb_ms / step_ms, 4),
                    "note": "M128xN32/N64 MMAs cap at 40 % / 67 % of the tensor peak (operand fetch from shared memory: 32 + N/4 cycles "
                            "per K=16 step, tools/mma_rate.cu) -- the time-as-M kernel's bound at C=32/64; the stacked-output kernel (C=32) "
                            "issues N=128 MMAs at the full rate but spends (k+3)/k of the useful cycles; halo rows and structural-zero columns "
                            "are not counted as work"}
    if tc_ms > 0:
        tf = FLOP_PER_WINDOW_TC * W_step * psteps / (tc_ms / 1e3) / 1e12
        fam = {"bound": "tensor", "kernel": "all tcgen05 kernels (k_resblock / k_resblock_t + per-layer k_conv_umma / k_conv_umma_p: conv_pre, upsamplers 0-2, "
                                            "stage-0 ResBlock convs as CTA pairs on tcgen05.mma.cta_group::2, chunker convs)" if bf else "k_conv_simt",
               "achieved": round(tf, 2), "peak": peaks["tf_sustained"], "unit": "TFLOP/s", "frac": round(tf / peaks["tf_sustained"], 4),
               "peak_source": f"{peaks['source']} bf16 sustained (kernel timed inside a long step)", "traffic": None,
               "launches": tc_n, "avg_launch_ms": round(tc_ms / max(tc_n, 1), 4), "share_of_step": round(tc_ms / step_ms, 4)}
        if roofline is None:
            roofline = fam
        else:
            family_roof = fam
    if ms_cls["resample_g711"] > 0:
        # the fused resample + G.711 kernel handles only 4 MB inside a TTS step (launch-latency bound), so its HBM roofline is
        # measured on its own at BASELINE config 5's size: 100k streams x one 100 ms mux quantum (640 MB in, 80 MB out > L2)
        from infernos_b200 import engine as _eng
        cs, cl = 100_000, 1600
        xc = (torch.rand(cs, cl, device=dev) * 2 - 1) * 0.9
        for _ in range(3):
            _eng.resample_g711_encode(xc)
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev)
        c0.record()
        for _ in range(20):
            _eng.resample_g711_encode(xc)
        c1.record()
        torch.cuda.synchronize(dev)
        c_ms = c0.elapsed_time(c1) / 20
        del xc
        gbs = CODEC_BYTES_PER_OUT * cs * (cl // 2) / (c_ms / 1e3) / 1e9
        in_step_ms = ms_cls["resample_g711"] / max(n_cls["resample_g711"], 1)
        codec_roof = {"bound": "hbm", "kernel": "k_resample_2to1_flat (fused 16k->8k + G.711: flat chunk mapping, warp-shuffle halo, FFMA2 tap pairs)",
                      "achieved": round(gbs, 1), "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": round(gbs / peaks["hbm_gbs"], 4),
                      "peak_source": peaks["source"], "traffic": 682162432,
                      "traffic_note": "dram read+write of one launch, ncu --set full (profiles/r1c_ncu_full_resample_g711_100k_streams.csv); algorithmic 720 MB "
                                      "(the 80 MB of output bytes were still in L2 when the capture ended)",
                      "workload": "100,000 streams x 1,600 samples (100 ms at 16 kHz) -> 800 G.711 bytes each; 9 algorithmic bytes per output byte; "
                                  "20 back-to-back launches timed with CUDA events, input (640 MB) larger than L2",
                      "avg_launch_ms": round(c_ms, 4), "in_step_launch_ms": round(in_step_ms, 4),
                      "in_step_note": f"inside the TTS step the same kernel handles {S * F * 128 * 9 / 1e6:.1f} MB per launch: launch-latency bound"}

    # ---- control-plane stats gather (the only collective; NCCL) -----------------------------------
    allstats = sharding.gather_stats({"sessions": S, "steps": args.steps, "g711_bytes": S * F * 128 * args.steps,
                                      "kernel_launches": launches, "device_ms": e0.elapsed_time(e1)}, device=dev)

    # ---- BASELINE config 3 as written: 1,024 calls in TOTAL, block-partitioned over the GPUs (strong scaling) ---------------------
    strong = None
    if not args.no_strong:
        shapes = [args.strong_total // world] if world > 1 else [args.strong_total // g for g in (2, 4, 8)]
        rows_s = []
        for Ss in shapes:
            Ss = max(1, min(Ss, S))
            sl, ml = slots_d[:Ss].contiguous(), mel_d[:Ss].contiguous()
            for _ in range(3):
                tail.tail(sl, ml, want_audio=False)
            barrier()
            evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
            for a, b in evs:
                a.record()
                tail.tail(sl, ml, want_audio=False)
                b.record()
            barrier()
            per = sorted(a.elapsed_time(b) for a, b in evs)
            tot = max_over_ranks(evs[0][0].elapsed_time(evs[-1][1]))
            worst = max_over_ranks(per[-1])
            rows_s.append({"sessions_per_gpu": Ss, "sessions_total": Ss * world, "value": round(Ss * world * F * AUDIO_S_PER_FRAME * args.steps / (tot / 1e3), 1),
                           "ms_per_step": round(tot / args.steps, 3), "call_ms_median": round(per[len(per) // 2], 3), "call_ms_max": round(worst, 3),
                           "per_gpu_efficiency_vs_1024": round((Ss * F * AUDIO_S_PER_FRAME * args.steps / (tot / 1e3)) / (value / world), 4)})
        strong = {"config": "BASELINE configs[2]: 1,024 concurrent calls in total, sharded by session across the GPUs (bf16)",
                  "n_gpus": world, "rows": rows_s,
                  "note": ("this run: one row, the shape each GPU gets at this GPU count" if world > 1 else
                           "single GPU: the per-GPU shapes of 2 / 4 / 8 GPUs (512 / 256 / 128 sessions) timed on one GPU; there is no data-plane "
                           "collective, so the N-GPU strong-scaling value is N x these") +
                          "; efficiency is against this run's own 1,024-sessions-per-GPU rate; what it loses is wave quantisation of the small "
                          "grids (stage 0/1 at 512 windows) and the fixed ~41 launches per call"}

    # ---- SURVEY 8 f3: AR decoder + tail, both on the GPU ------------------------------------------------------------------------------
    front = None
    if rank == 0 and world == 1 and not args.no_front and args.mode == "bf16":
        try:
            front = run_front_half(dev, tail, slots_d, S)
        except Exception as e:
            front = {"error": repr(e)[:300]}

    # ---- the reference's own load-test shape (HelloSippyRTPipeTest.py:180-236) through the plugin API: per-session TTFF / TTLF / rtr -------------
    session_test = None
    if rank == 0 and world == 1 and not args.no_sessions and args.mode == "bf16":
        tail.close()
        tail = None
        torch.cuda.empty_cache()
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import session_bench
            session_test = [session_bench.run(n, 96, args.mode, device=f"cuda:{local_rank}") for n in args.session_counts]
            for r in session_test:
                r.pop("what", None)
        except Exception as e:
            session_test = {"error": repr(e)[:300]}

    # ---- north_star's joint target: p99 chunk latency at >= 5,000 concurrent real-time streams ---------------------------------------
    latency = None
    if rank == 0 and world == 1 and not args.no_latency:
        if tail is not None:
            tail.close()
            tail = None
        torch.cuda.empty_cache()
        latency = []
        for nsess in args.latency_sessions:
            try:
                latency.append(run_latency(dev, nsess, args.latency_seconds, mode=args.mode))
            except Exception as e:                                      # keep the line: report what failed
                latency.append({"sessions": nsess, "error": repr(e)[:300]})

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        r = run_cpu(args.ref_sessions, 5, 2, dtype=torch.bfloat16 if args.ref_dtype == "bf16" else torch.float32)
        cpu = {"value": round(r["value"], 3), "unit": "streams", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]}

    if rank == 0:
        out = {
            "metric": "real-time G.711 TTS streams (RTF<=1)", "value": round(value, 1), "unit": "streams", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_total / args.steps, 3), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16" if args.mode == "bf16" else "f32", "data": "synthetic",
            "config": {"workload": f"batched vocoder+chunker+resample+G.711, {S} concurrent sessions per GPU, {F}-frame calls "
                                   f"({nwin} windows of 12 frames, 8 emitted each), {args.mode} conv path",
                       "sessions_per_gpu": S, "frames_per_call": F, "mode": args.mode, "sharding": "sessions block-partitioned, no data-plane collective",
                       "l2": "per-step working set (GBs of activations) exceeds the 126 MB L2; no explicit flush",
                       "vocoder_msamples_per_s": round(S * world * F * 256 * args.steps / (ms_total / 1e3) / 1e6, 1)},
            "clocks": clocks,
            "e2e": {"value": round(e2e_value, 1), "unit": "streams", "h2d_bytes_per_step": int(mel_h.numel() * 4 + slots_h.numel() * 4) * world,
                    "d2h_bytes_per_step": int(g_h.numel()) * world, "ms_per_step": round(e2e_ms / args.steps, 3),
                    "path": "b2_sched_submit / b2_sched_poll (native serving loop): pinned H2D + one CUDA-graph launch + D2H per step, two steps in flight",
                    "blocking_call_ms_per_step": round(sync_ms / args.steps, 3),
                    "blocking_call_value": round(audio_s / (sync_ms / 1e3), 1)},
            "gpu_launches": int(sum(s["kernel_launches"] for s in allstats)),
            "roofline": roofline, "roofline_conv_family": family_roof, "roofline_codec": codec_roof,
            "kernel_ms_per_step": {k: round(v / psteps, 3) for k, v in ms_cls.items()},
            "cpu_baseline": cpu,
            "latency": latency, "strong": strong, "front_half": front, "session_test": session_test,
            "per_gpu_stats": [{"sessions": int(s["sessions"]), "steps": int(s["steps"]), "g711_bytes": int(s["g711_bytes"]),
                               "device_ms": round(s["device_ms"], 3)} for s in allstats],
            "hbm_bytes_ctx": ctx_bytes,
        }
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(out), flush=True)
        os.dup2(2, 1)
    if tail is not None:
        tail.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps (at least 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--sessions", type=int, default=1024, help="concurrent sessions per GPU")
    ap.add_argument("--frames", type=int, default=32, help="mel frames per session per call (reference: 32)")
    ap.add_argument("--mode", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--max-windows", type=int, default=4096, help="workspace capacity in 12-frame windows (sub-batch size)")
    ap.add_argument("--ref-sessions", type=int, default=8, help="sessions per step of the CPU arm's bounded sample (reference: max_batch_size = 8)")
    ap.add_argument("--ref-dtype", default="bf16", choices=["bf16", "fp32"], help="precision of the CPU arm (the reference runs bf16: maybe_half)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-latency", action="store_true", help="skip the p99 chunk-latency legs (5,000 / 20,000 staggered real-time sessions)")
    ap.add_argument("--latency-sessions", type=int, nargs="*", default=[5000, 20000])
    ap.add_argument("--latency-seconds", type=float, default=3.0)
    ap.add_argument("--no-sessions", action="store_true", help="skip the reference-style session test (TTFF / TTLF / rtr through InfernTTSWorker + GPU front half)")
    ap.add_argument("--session-counts", type=int, nargs="*", default=[50, 1000])
    ap.add_argument("--no-front", action="store_true", help="skip the AR-decoder + tail leg (SURVEY 8 f3)")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling block (BASELINE config 3 as written)")
    ap.add_argument("--strong-total", type=int, default=1024)
    ap.add_argument("--cpu-sweep", action="store_true", help="with --impl reference: fp32/bf16 x B in {1,8,64} CPU table (SURVEY 8d)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="GPU arm: after the timed steps, write the G.711 codes of the last timed step (sessions x samples) as DIR/g711.npy "
                         "(float32, at most 64 MB; larger outputs keep a fixed, seeded sample of sessions)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the GPU arm's outputs (--impl b200)")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        main_reference(args, rank, world)
        return
    if world == 1 and args.gpus > 1:
        # launched without torchrun: re-exec under it so that there is one process per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
               "--master-port", str(29500 + os.getpid() % 1000), os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    main_b200(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
