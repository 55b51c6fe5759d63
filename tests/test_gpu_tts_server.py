"""GPU: the sentence server (b2_tts_server_*, engine.TTSServer) against the host code it replaces.

Every server run is replayed with the public per-call APIs -- TTSEncoder, a fresh TTSDecoder making the same sequence of steps() calls,
TTSTail.tail(apply_postnet=True) -- and the stop rule and slicing of HelloSippyRTPipe._front_half / unbatch_prepare on the host, on the
admission schedule the server's records report.  Bytes per record, end calls and the absence of records after a sentence's last one are
compared exactly.  One cohort is also compared with what InfernTTSWorker.process_batch emits for the same requests."""
import os
import threading
import time
import uuid

import pytest
import torch

from infernos_b200 import synth

pytestmark = pytest.mark.gpu

SEED = 12345


@pytest.fixture(scope="module")
def sds():
    return dict(esd=synth.encoder_state_dict(), dsd=synth.decoder_state_dict(), vsd=synth.hifigan_state_dict(), csd=synth.chunker_state_dict(),
                psd=synth.postnet_state_dict())


def _handles(sds, mode, pool, max_steps, max_enc_len):
    from infernos_b200.engine import TTSDecoder, TTSEncoder, TTSTail
    tail = TTSTail("cuda:0", sds["vsd"], sds["csd"], mode=mode, max_sessions=pool, max_windows=4 * pool, postnet_sd=sds["psd"])
    enc = TTSEncoder("cuda:0", sds["esd"], mode=mode, max_tokens=4096, max_len=max_enc_len)
    dec = TTSDecoder("cuda:0", sds["dsd"], mode=mode, max_sessions=pool, max_steps=max_steps, max_enc_len=max_enc_len)
    return tail, enc, dec


def _sentences(lengths, seed):
    g = torch.Generator().manual_seed(seed)
    spk = synth.synth_speakers(len(lengths), seed=seed + 1)
    return {1000 + i: (torch.randint(4, 81, (n,), generator=g).tolist(), spk[i]) for i, n in enumerate(lengths)}


def _collect(srv, n, timeout=300.0):
    """tag -> [(call, bytes, ended)], plus the records themselves"""
    got, raw, ended, t0 = {}, [], 0, time.time()
    while ended < n:
        assert time.time() - t0 < timeout, f"only {ended} of {n} sentences ended in {timeout} s"
        for rec, b in srv.poll(timeout_ms=100):
            got.setdefault(rec["tag"], []).append((rec["call"], b, rec["ended"]))
            raw.append(rec)
            ended += rec["ended"]
    return got, raw


def _replay(sds, mode, pool, max_steps, max_enc_len, sents, raw, ncalls, threshold=0.5, minlenratio=0.0, maxlenratio=20.0, law=0):
    """The server's schedule (admit_call of every sentence) through the public per-call APIs and the host stop rule / slicing."""
    tail, enc, dec = _handles(sds, mode, pool, max_steps, max_enc_len)
    admit = {}
    for r in raw:
        admit.setdefault(r["admit_call"], set()).add(r["tag"])
    cap = max(1, max_steps - 16 - 4)
    free, st, live, out = list(range(pool)), {}, [], {}
    try:
        for c in range(ncalls):
            new = sorted(admit.get(c, ()))
            if new:
                L = max(len(sents[t][0]) for t in new)
                ids = torch.zeros(len(new), L, dtype=torch.long)
                mask = torch.zeros(len(new), L, dtype=torch.int)
                for i, t in enumerate(new):
                    ids[i, :len(sents[t][0])] = torch.tensor(sents[t][0])
                    mask[i, :len(sents[t][0])] = 1
                slots = [free.pop(0) for _ in new]
                e = enc(ids, mask)
                dec.start(torch.tensor(slots, dtype=torch.int32).cuda(), e, mask.sum(1).to(torch.int32).cuda(),
                          torch.stack([sents[t][1] for t in new]).cuda())
                tail.reset_sessions(slots)
                minlen, maxlen = int(L * minlenratio / 2), min(int(L * maxlenratio / 2), cap)
                for t, s in zip(new, slots):
                    st[t] = dict(slot=s, idx=0, ends=-1, minlen=minlen, maxlen=maxlen)
                live += new
            rows = [st[t]["slot"] for t in live] or [-1]
            mel, prob = dec.steps(torch.tensor(rows, dtype=torch.int32).cuda(), 16, seed=SEED)
            if not live:
                continue
            g, _ = tail.tail(torch.tensor(rows, dtype=torch.int32).cuda(), mel, law=law, want_audio=False, apply_postnet=True)
            g, prob = g.cpu(), prob.cpu()
            gone = []
            for i, t in enumerate(live):
                s = st[t]
                for k in range(16):                       # HelloSippyRTPipe._front_half, :417-421
                    stop = bool((prob[i, k] >= threshold).sum() > 0)
                    if s["ends"] < 0 and s["minlen"] <= s["idx"] and (stop or s["maxlen"] <= s["idx"]):
                        s["ends"] = s["idx"] + 2
                    s["idx"] += 1
                idx, ends = s["idx"], s["ends"]            # unbatch_prepare, :503-527
                startoff = max(0, 4096 - (idx - 1) * 256)
                endoff = min(4096, 4096 - ((idx - ends) * 256 if ends >= 0 else 0))
                ended = 0 <= ends <= idx - 1
                if startoff != endoff or ended:
                    out.setdefault(t, []).append((c, g[i, startoff:endoff].numpy().tobytes(), ended))
                if ended:
                    gone.append(t)
                    free.append(s["slot"])
            live = [t for t in live if t not in gone]
        dec.poll_errors(); enc.poll_errors(); tail.poll_errors()
    finally:
        tail.close(); enc.close(); dec.close()
    return out, st


def _check_against_replay(got, ref, sents):
    assert set(got) == set(sents) == set(ref)
    for t in sents:
        g, r = got[t], ref[t]
        assert [x[2] for x in g].count(True) == 1 and g[-1][2], f"sentence {t}: the ended record must be its last and only one"
        assert [(c, e) for c, _, e in g] == [(c, e) for c, _, e in r], f"sentence {t}: calls / end differ: {[(c, e) for c, _, e in g]} vs " \
                                                                          f"{[(c, e) for c, _, e in r]}"
        assert all(a[1] == b[1] for a, b in zip(g, r)), f"sentence {t}: bytes differ from the replay"


def _serve(sds, mode, pool, max_steps, max_enc_len, submit, n, **kw):
    from infernos_b200.engine import TTSServer
    tail, enc, dec = _handles(sds, mode, pool, max_steps, max_enc_len)
    srv = TTSServer(tail, enc, dec, seed=SEED, **kw)
    try:
        th = threading.Thread(target=submit, args=(srv,), daemon=True)
        th.start()
        got, raw = _collect(srv, n)
        th.join(60)
        srv.flush(60000)
        stats = srv.stats()
        srv.close()
        dec.poll_errors()                                  # nothing ran past max_steps, no bad slot
        enc.poll_errors()
    finally:
        srv.close(); tail.close(); enc.close(); dec.close()
    return got, raw, stats


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_one_cohort_equals_the_worker_drop_in(sds, mode):
    """The same requests through InfernTTSWorker.process_batch (HelloSippyRTPipe + B200Frontend.from_state_dict, same seed, law and post-net):
    every sentence's concatenated bytes and its end call are bitwise those of the server."""
    from infernos_b200.Cluster.InfernBatchedWorker import InfernBatchedWorker
    from infernos_b200.Cluster.InfernTTSWorker import InfernTTSWorker
    from infernos_b200.HelloSippyTTSRT.HelloSippyRTPipe import B200Frontend, HelloSippyPlayRequest, HelloSippyRTPipe
    lengths = (3, 17, 9, 20, 1, 12)
    sents = _sentences(lengths, seed=5)
    by_text = {f"s{t}": torch.tensor([ids]) for t, (ids, _) in sents.items()}
    fe = B200Frontend.from_state_dict({**sds["esd"], **sds["dsd"]}, lambda text: by_text[text], "cuda:0", mode=mode, max_sessions=8, max_steps=64,
                                      max_enc_len=32, max_tokens=4096, seed=SEED)
    pp = HelloSippyRTPipe("cuda:0", output_sr=8000, frontend=fe, vocoder_state_dict=sds["vsd"], chunker_state_dict=sds["csd"],
                          postnet_state_dict=sds["psd"], mode=mode, max_sessions=8)
    w = InfernTTSWorker.__new__(InfernTTSWorker)
    InfernBatchedWorker.__init__(w)
    w.continuous, w.output_sr, w.tts_engine = False, 8000, pp
    calls = [0]
    infer = pp.infer

    def counted(state):
        infer(state)
        calls[0] += 1
    pp.infer = counted
    ref_bytes, ref_end = {t: b"" for t in sents}, {}

    def cbs(t):
        def d(chunk):
            if chunk is None:
                ref_end[t] = calls[0] - 1
        def g(b):
            ref_bytes[t] += b
        return d, g
    reqs = []
    for t, (ids, spk) in sents.items():
        d, g = cbs(t)
        reqs.append(HelloSippyPlayRequest(uuid.uuid4(), f"s{t}", spk[None], d, dispatch_g711=g))
    try:
        w.process_batch(reqs)
    finally:
        fe.close(); pp.tail.close()
    tags = list(sents)
    got, raw, stats = _serve(sds, mode, 8, 64, 32, lambda srv: srv.submit_many([sents[t][0] for t in tags], [sents[t][1] for t in tags], tags),
                             len(tags))
    assert stats["admission_rounds"] == 1
    for t in tags:
        assert b"".join(b for _, b, _ in got[t]) == ref_bytes[t], f"sentence {t}: bytes differ from process_batch"
        assert got[t][-1][0] == ref_end[t], f"sentence {t}: ends at call {got[t][-1][0]}, process_batch at {ref_end[t]}"
    print(f"{mode}: {len(tags)} sentences, {stats['calls']} calls, bytes and end calls equal process_batch")


@pytest.mark.parametrize("depth", [1, 2])
def test_staggered_admission_equals_the_replay(sds, depth):
    """Sentences arrive from another thread at random times, more than the pool holds (back-pressure, slot reuse); a sentence shares
    decoder passes with whatever is live, whichever call admitted it."""
    g = torch.Generator().manual_seed(60 + depth)
    n = 80
    lengths = torch.randint(1, 31, (n,), generator=g).tolist()
    sents = _sentences(lengths, seed=61)
    gaps = (torch.rand(n, generator=g) * 0.02).tolist()

    def submit(srv):
        for (t, (ids, spk)), dt in zip(sents.items(), gaps):
            time.sleep(dt)
            srv.submit(ids, spk, t)
    kw = dict(depth=depth, maxlenratio=2.0)
    got, raw, stats = _serve(sds, "bf16", 24, 64, 32, submit, n, **kw)
    ref, _ = _replay(sds, "bf16", 24, 64, 32, sents, raw, stats["calls"], maxlenratio=2.0)
    _check_against_replay(got, ref, sents)
    assert stats["admission_rounds"] > 1 and stats["ended"] == n
    print(f"depth {depth}: {n} sentences, {stats['calls']} calls, {stats['admission_rounds']} admission rounds, "
          f"{stats['live_rows'] / stats['calls']:.1f} live sentences per call")


@pytest.mark.parametrize("depth", [1, 2])
def test_stop_rule_edges(sds, depth):
    """One cohort, L = 10 tokens: maxlen = int(10 * 3.0 / 2) = 15 fires in the last step of call 0 (the sentence ends in call 1), minlen = 5,
    one-token sentences, and a threshold at the median of the sentences' largest stop probability over steps 5..14, so that about half
    of them stop on probability.  max_steps = 36: a sentence left stepping after its end (no retirement) would run past it in call 2."""
    from infernos_b200.engine import TTSDecoder, TTSEncoder
    lengths = (1, 1, 10, 4, 7, 10, 2, 9, 6, 3, 8, 5)
    sents = _sentences(lengths, seed=70)
    tags = list(sents)
    # the stop probabilities of the cohort do not depend on the threshold: read them once to place it
    enc = TTSEncoder("cuda:0", sds["esd"], mode="bf16", max_tokens=4096, max_len=32)
    dec = TTSDecoder("cuda:0", sds["dsd"], mode="bf16", max_sessions=16, max_steps=36, max_enc_len=32)
    try:
        ids = torch.zeros(len(tags), 10, dtype=torch.long)
        mask = torch.zeros(len(tags), 10, dtype=torch.int)
        for i, t in enumerate(tags):
            ids[i, :len(sents[t][0])] = torch.tensor(sents[t][0]); mask[i, :len(sents[t][0])] = 1
        sl = torch.arange(len(tags), dtype=torch.int32).cuda()
        dec.start(sl, enc(ids, mask), mask.sum(1).to(torch.int32).cuda(), torch.stack([sents[t][1] for t in tags]).cuda())
        _, prob = dec.steps(sl, 16, seed=SEED)
        peak = prob.cpu()[:, 5:15].amax(dim=(1, 2))
    finally:
        enc.close(); dec.close()
    thr = float(peak.median())
    kw = dict(depth=depth, threshold=thr, minlenratio=1.0, maxlenratio=3.0)
    got, raw, stats = _serve(sds, "bf16", 16, 36, 32,
                             lambda srv: srv.submit_many([sents[t][0] for t in tags], [sents[t][1] for t in tags], tags), len(tags), **kw)
    ref, st = _replay(sds, "bf16", 16, 36, 32, sents, raw, stats["calls"], threshold=thr, minlenratio=1.0, maxlenratio=3.0)
    _check_against_replay(got, ref, sents)
    on_prob = [t for t in tags if st[t]["ends"] - 2 < 15]
    at_max = [t for t in tags if st[t]["ends"] - 2 == 15]
    print(f"depth {depth}: threshold {thr:.4f}: {len(on_prob)} sentences stopped on probability, {len(at_max)} at maxlen (step 15, the last of call 0)")
    assert on_prob and at_max
    assert all(st[t]["ends"] - 2 >= 5 for t in tags), "minlen = 5"
    assert all(got[t][-1][0] == 1 for t in at_max)


@pytest.mark.parametrize("use_graphs", [True, False])
def test_graph_buckets_and_pool_reuse(sds, use_graphs):
    """130 sentences at once, then 60 more one by one into a pool of 160: live counts cross the bucket edges, slots are reused, and bytes
    are the replay's (the plain tail call) with and without the graph buckets."""
    g = torch.Generator().manual_seed(80)
    first = torch.randint(1, 25, (130,), generator=g).tolist()
    more = torch.randint(1, 25, (60,), generator=g).tolist()
    sents = _sentences(first + more, seed=81)
    tags = list(sents)

    def submit(srv):
        srv.submit_many([sents[t][0] for t in tags[:130]], [sents[t][1] for t in tags[:130]], tags[:130])
        for t in tags[130:]:
            time.sleep(0.01)
            srv.submit(sents[t][0], sents[t][1], t)
    kw = dict(depth=2, maxlenratio=2.0, use_graphs=use_graphs)
    got, raw, stats = _serve(sds, "bf16", 160, 64, 32, submit, len(tags), **kw)
    ref, _ = _replay(sds, "bf16", 160, 64, 32, sents, raw, stats["calls"], maxlenratio=2.0)
    _check_against_replay(got, ref, sents)
    per_call = {}
    for r in raw:
        per_call[r["call"]] = per_call.get(r["call"], 0) + 1
    counts = sorted(per_call.values())
    print(f"graphs {use_graphs}: {stats['calls']} calls, live sentences per call {counts[0]}..{counts[-1]}, graphs built {stats['graphs_built']}, "
          f"padded rows {stats['padded_rows']}")
    assert counts[-1] > 128 and counts[0] <= 32 and stats["admitted"] == len(tags)
    assert (stats["graph_launches"] == stats["calls"]) if use_graphs else (stats["graph_launches"] == 0)


def _server_threads():
    names = []
    for t in os.listdir("/proc/self/task"):
        try:
            with open(f"/proc/self/task/{t}/comm") as f:
                names.append(f.read().strip())
        except OSError:
            pass
    return [n for n in names if n.startswith("b2-tts-")]


def test_errors_and_destroy_with_work_in_flight(sds):
    import ctypes
    from infernos_b200.engine import TTSServer
    tail, enc, dec = _handles(sds, "bf16", 8, 64, 32)
    spk = synth.synth_speakers(1, seed=3)[0]
    try:
        srv = TTSServer(tail, enc, dec, seed=SEED)
        with pytest.raises(RuntimeError, match="more than"):
            srv.submit([5] * 33, spk, 1)                   # max_enc_len = 32
        with pytest.raises(RuntimeError, match="at least one token"):
            srv.submit([], spk, 2)
        with pytest.raises(RuntimeError, match="outside"):
            srv.submit([5, 81, 6], spk, 3)
        with pytest.raises(RuntimeError, match="outside"):
            srv.submit_many([[5, 6], [7, -1]], [spk, spk], [4, 5])
        lib = srv.lib
        ids = (ctypes.c_int32 * 3)(5, 6, 7)
        lens = (ctypes.c_int32 * 1)(3)
        sp = (ctypes.c_float * 512)()
        tg = (ctypes.c_uint64 * 1)(9)
        assert lib.b2_tts_server_submit(srv.h, None, lens, 1, sp, tg) != 0
        assert lib.b2_tts_server_submit(srv.h, ids, None, 1, sp, tg) != 0
        assert lib.b2_tts_server_submit(srv.h, ids, lens, 1, None, tg) != 0
        assert lib.b2_tts_server_submit(srv.h, ids, lens, 1, sp, None) != 0
        assert lib.b2_tts_server_submit(None, ids, lens, 1, sp, tg) != 0
        zero = (ctypes.c_int32 * 1)(0)
        assert lib.b2_tts_server_submit(srv.h, ids, zero, 1, sp, tg) != 0
        assert srv.stats()["submitted"] == 0 and srv.poll(timeout_ms=50) == []
        assert sorted(_server_threads()) == ["b2-tts-complete", "b2-tts-driver"]
        for i in range(8):
            srv.submit([4 + i] * (5 + i), spk, 100 + i)
        time.sleep(0.005)
        t0 = time.time()
        srv.close()                                        # calls in flight: returns, threads joined
        assert time.time() - t0 < 30
        assert _server_threads() == []
    finally:
        tail.close(); enc.close(); dec.close()
