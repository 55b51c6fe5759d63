#!/usr/bin/env python
"""Latency of whole sentences through the sentence server (engine.TTSServer, b2_tts_server_*): token ids in, G.711 chunks out.

Synthetic weights (synth.*_state_dict), sentences of 8-200 tokens arriving as a Poisson process whose rate keeps `level` sentences
playing at once if each lasted its audio length (rate = level / audio seconds per sentence).  2 x level sentences per level.  The random
decoder's stop probability stays low, so every sentence runs to maxlen = max_steps - 20 decoder steps (8 engine calls, 3.6 s of audio).
Per level:
  TTFF          submit -> the call holding the sentence's first bytes was in pinned host memory (t_done_ns), p50 / p99 / max
  underruns     chunks that arrived after the playout of the bytes before them, counted from the arrival of the first bytes
  rt_streams    audio seconds produced per wall second while sentences were arriving (the real-time streams the run sustained)
  live/call     mean sentences live on the device per engine call;  ms/call: wall time between consecutive call completions
With --compare N (default 1000) the same arrivals also go through InfernTTSWorker(continuous=True) -> HelloSippyRTPipe -> B200Frontend with
the library's encoder and decoder (the path of tools/session_bench.py), timed at its dispatch callbacks.
With --barge-in FRAC every level and depth runs twice on the same arrivals: without cancels, then with a fraction FRAC of the sentences
cancelled by the polling thread (where a caller's barge-in arrives) right after it polls the k-th record of the sentence, k uniform in 1..7
(between the first bytes and the natural end).  Per cancelled sentence:
  cancel_ms     cancel() call -> t_done_ns of the cancelled record, p50 / p99 / max
  cancel_calls  engine calls from the latest call polled at cancel() to the cancelled record
  bytes_after_cancel   bytes of the sentence polled after cancel() returned (calls already built)
  ended_before_cancel  cancels that a call already in flight beat: the sentence ended on its own

    python tools/tts_serve_bench.py [--levels 1000 5000 10000] [--depth 1 2] [--mode bf16] [--barge-in 0.3] [--out profiles/r6_tts_serve_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CHUNK_S = 4096 / 8000.0
MAX_STEPS = 132                  # maxlen = 112 steps: the sentence ends in call 8
CALLS_PER_SENTENCE = 8


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as e:           # the card name is reported, not required
        return f"unknown ({e!r})"


def workload(level, seed):
    import torch
    from infernos_b200 import synth
    g = torch.Generator().manual_seed(seed)
    n = 2 * level
    lens = torch.randint(8, 201, (n,), generator=g).tolist()
    ids = [torch.randint(4, 81, (k,), generator=g).tolist() for k in lens]
    spk = synth.synth_speakers(16, seed=seed + 1)
    audio_s = 8 * CHUNK_S - 3 * 256 / 8000.0          # 112 + 2 steps after the first: 114 * 256 - 256 bytes
    rate = level / audio_s
    gaps = torch.empty(n).exponential_(generator=g) / rate
    t = gaps.cumsum(0).tolist()
    return ids, [spk[i % 16] for i in range(n)], t


def pct(xs, q):
    import numpy as np
    return float(np.percentile(np.asarray(xs), q)) if xs else None


def summarize(first_ns, chunks, t_sub, arrival_end_ns, t0_ns):
    """chunks: tag -> [(t_ns, nbytes)] in order; first_ns: tag -> t of first bytes"""
    ttff = [(first_ns[k] - t_sub[k]) / 1e6 for k in first_ns]
    under, under_sent, audio = 0, 0, 0.0
    for k, cs in chunks.items():
        t_first, played, bad = cs[0][0], 0, 0
        for t, nb in cs:
            if t > t_first + played / 8000.0 * 1e9 + 1e6:       # 1 ms of slack for the clock reads
                bad += 1
            played += nb
        under += bad
        under_sent += bad > 0
        audio += sum(nb for t, nb in cs if t <= arrival_end_ns) / 8000.0
    window = (arrival_end_ns - t0_ns) / 1e9
    return dict(sentences=len(first_ns), ttff_ms_p50=pct(ttff, 50), ttff_ms_p99=pct(ttff, 99), ttff_ms_max=max(ttff) if ttff else None,
                underrun_chunks=under, sentences_with_underrun=under_sent, chunks=sum(len(c) for c in chunks.values()),
                rt_streams=audio / window if window > 0 else None)


def serve_level(level, depth, mode, seed, barge_ins):
    """One set of handles; the same arrivals once per barge-in fraction, each on a fresh server"""
    from infernos_b200 import synth
    from infernos_b200.engine import TTSDecoder, TTSEncoder, TTSTail
    pool = int(level * 1.25) + 64
    tail = TTSTail("cuda:0", synth.hifigan_state_dict(), synth.chunker_state_dict(), mode=mode, max_sessions=pool, max_windows=4 * pool,
                   postnet_sd=synth.postnet_state_dict())
    enc = TTSEncoder("cuda:0", synth.encoder_state_dict(), mode=mode, max_tokens=16384, max_len=200)
    dec = TTSDecoder("cuda:0", synth.decoder_state_dict(), mode=mode, max_sessions=pool, max_steps=MAX_STEPS, max_enc_len=200)
    try:
        return [serve_once(tail, enc, dec, level, depth, mode, seed, b) for b in barge_ins]
    finally:
        tail.close(); enc.close(); dec.close()


def serve_once(tail, enc, dec, level, depth, mode, seed, barge_in):
    import random
    from infernos_b200.engine import TTSServer
    ids, spk, arr = workload(level, seed)
    # barge-in: a fraction of the sentences is cancelled right after the poller sees its k-th record, k uniform over the records between
    # the first bytes and the natural end (CALLS_PER_SENTENCE records, the last one ending the sentence)
    rng = random.Random(seed * 1000003 + level)
    plan = {i: rng.randint(1, CALLS_PER_SENTENCE - 1) for i in range(len(ids)) if rng.random() < barge_in}
    srv = TTSServer(tail, enc, dec, depth=depth, seed=seed, poll_capacity=65536)
    try:
        # warm-up: a burst at the level's size builds the decoder's and the tail's graph buckets and the encoder's workspaces
        for lo in (1, 8, 32, 128, 512, level):
            srv.submit_many(ids[:lo], spk[:lo], list(range(10 ** 9, 10 ** 9 + lo)))
            srv.flush()
            while srv.poll(0):
                pass
        s0 = srv.stats()
        n = len(ids)
        t_sub, first, chunks, ended = {}, {}, {}, [0]
        seen, last_call = {}, [-1]
        cancels = {}                                  # tag -> dict(t_ns, call, after): cancel() time, latest call polled, bytes since
        done = threading.Event()

        def poller():
            while ended[0] < n:
                for rec, b in srv.poll(timeout_ms=50):
                    k = rec["tag"]
                    last_call[0] = max(last_call[0], rec["call"])
                    if k in cancels:
                        c = cancels[k]
                        c["after"] += rec["nbytes"]
                        if rec["ended"]:
                            c.update(cancelled=rec["cancelled"], lat_ms=(rec["t_done_ns"] - c["t_ns"]) / 1e6, calls=rec["call"] - c["call"])
                    if rec["nbytes"]:
                        first.setdefault(k, rec["t_done_ns"])
                        chunks.setdefault(k, []).append((rec["t_done_ns"], rec["nbytes"]))
                    t_sub[k] = rec["t_submit_ns"]
                    ended[0] += rec["ended"]
                    seen[k] = seen.get(k, 0) + 1
                    if k in plan and seen[k] == plan[k] and not rec["ended"]:
                        t_ns = time.monotonic_ns()
                        if srv.cancel(k):
                            cancels[k] = dict(t_ns=t_ns, call=last_call[0], after=0)
            done.set()
        th = threading.Thread(target=poller, daemon=True)
        th.start()
        t0 = time.monotonic_ns()
        for i in range(n):
            wait = t0 + int(arr[i] * 1e9) - time.monotonic_ns()
            if wait > 0:
                time.sleep(wait / 1e9)
            srv.submit(ids[i], spk[i], i)
        t_end = time.monotonic_ns()
        assert done.wait(1800), "sentences did not finish"
        s1 = srv.stats()
        calls = s1["calls"] - s0["calls"]
        out = summarize(first, chunks, t_sub, t_end, t0)
        dones = sorted({c[0] for cs in chunks.values() for c in cs})
        gaps = [(b - a) / 1e6 for a, b in zip(dones, dones[1:])]
        out.update(level=level, depth=depth, mode=mode, barge_in=barge_in, calls=calls, live_per_call=(s1["live_rows"] - s0["live_rows"]) / max(1, calls),
                   rows_per_call=(s1["rows"] - s0["rows"]) / max(1, calls), ms_per_call_mean=sum(gaps) / len(gaps) if gaps else None,
                   ms_per_call_p50=pct(gaps, 50), admission_rounds=s1["admission_rounds"] - s0["admission_rounds"], arrival_s=(t_end - t0) / 1e9)
        if plan:
            hit = [c for c in cancels.values() if c.get("cancelled")]
            lat, ncalls, after = [c["lat_ms"] for c in hit], [c["calls"] for c in hit], [c["after"] for c in cancels.values()]
            out.update(cancels=len(cancels), cancelled=len(hit), ended_before_cancel=len(cancels) - len(hit),
                       cancel_ms_p50=pct(lat, 50), cancel_ms_p99=pct(lat, 99), cancel_ms_max=max(lat) if lat else None,
                       cancel_calls_p50=pct(ncalls, 50), cancel_calls_max=max(ncalls) if ncalls else None,
                       bytes_after_cancel_total=sum(after), bytes_after_cancel_mean=sum(after) / len(after) if after else None,
                       bytes_after_cancel_max=max(after) if after else None)
        return out
    finally:
        srv.close()


def worker_level(level, mode, seed):
    """The same arrivals through InfernTTSWorker(continuous=True) with B200Frontend.from_state_dict (library encoder and decoder)."""
    import torch
    import uuid
    from infernos_b200 import synth
    from infernos_b200.Cluster.InfernTTSWorker import InfernTTSWorker
    from infernos_b200.HelloSippyTTSRT.HelloSippyRTPipe import B200Frontend, HelloSippyPlayRequest
    ids, spk, arr = workload(level, seed)
    pool = int(level * 1.25) + 64
    by_text = {f"#{i}": torch.tensor([x]) for i, x in enumerate(ids)}
    fe = B200Frontend.from_state_dict({**synth.encoder_state_dict(), **synth.decoder_state_dict()}, lambda t: by_text[t], "cuda:0", mode=mode,
                                      max_sessions=pool, max_steps=MAX_STEPS, max_enc_len=200, seed=seed)
    w = InfernTTSWorker("en", 8000, device="cuda:0", continuous=True, frontend=fe, vocoder_state_dict=synth.hifigan_state_dict(),
                        chunker_state_dict=synth.chunker_state_dict(), postnet_state_dict=synth.postnet_state_dict(), mode=mode, max_sessions=pool,
                        max_windows=4 * pool)
    n = len(ids)
    t_sub, first, chunks, left = {}, {}, {}, [n]
    done = threading.Event()
    lock = threading.Lock()

    def cb(i):
        def f(chunk):
            t = time.monotonic_ns()
            with lock:
                if chunk is None:
                    left[0] -= 1
                    if left[0] == 0:
                        done.set()
                    return
                first.setdefault(i, t)
                chunks.setdefault(i, []).append((t, len(chunk.payload)))
        return f
    w.start()
    try:
        warm = threading.Event()
        w.infer(HelloSippyPlayRequest(uuid.uuid4(), "#0", spk[0][None], lambda c: warm.set() if c is None else None, pre_encoded=True))
        assert warm.wait(600)
        t0 = time.monotonic_ns()
        for i in range(n):
            wait = t0 + int(arr[i] * 1e9) - time.monotonic_ns()
            if wait > 0:
                time.sleep(wait / 1e9)
            t_sub[i] = time.monotonic_ns()
            w.infer(HelloSippyPlayRequest(uuid.uuid4(), f"#{i}", spk[i][None], cb(i), pre_encoded=True))
        t_end = time.monotonic_ns()
        ok = done.wait(3600)
    finally:
        w.stop()
        fe.close()
    out = summarize(first, chunks, {k: t_sub[k] for k in first}, t_end, t0)
    out.update(level=level, path="InfernTTSWorker(continuous=True) + B200Frontend", finished=bool(ok), arrival_s=(t_end - t0) / 1e9)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--levels", type=int, nargs="+", default=[1000, 5000, 10000])
    ap.add_argument("--depth", type=int, nargs="+", default=[1, 2])
    ap.add_argument("--mode", default="bf16")
    ap.add_argument("--compare", type=int, default=1000, help="level at which the worker path runs the same arrivals (0: none)")
    ap.add_argument("--barge-in", type=float, default=0.0,
                    help="fraction of sentences cancelled between their first bytes and their natural end; the same arrivals also run without")
    ap.add_argument("--seed", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not 0.0 <= a.barge_in <= 1.0:
        raise SystemExit("--barge-in must be in [0, 1]")
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("tts_serve_bench needs a CUDA device")
    res = dict(card=card(), mode=a.mode, max_steps=MAX_STEPS, barge_in=a.barge_in, server=[], worker=None)
    print("card (name, power limit, max SM clock):", res["card"], flush=True)
    for lv in a.levels:
        for d in a.depth:
            for r in serve_level(lv, d, a.mode, a.seed, [0.0, a.barge_in] if a.barge_in > 0 else [0.0]):
                res["server"].append(r)
                print(json.dumps(r), flush=True)
    if a.compare:
        res["worker"] = worker_level(a.compare, a.mode, a.seed)
        print(json.dumps(res["worker"]), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
