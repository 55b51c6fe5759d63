"""GPU: cancelling sentences in the sentence server (b2_tts_server_cancel, engine.TTSServer.cancel).

Every run is replayed as in test_gpu_tts_server.py: the public per-call APIs on the admission schedule the server's records report, with the
host stop rule and slicing, and with each cancelled sentence dropped from the rows at the call its cancelled record names.  Bytes are compared
exactly.  A cancelled sentence must have the replay's records of the calls before that one, then one record with no bytes, then nothing;
every other sentence, including those admitted later into slots a cancel freed, must be the replay's."""
import ctypes
import random
import threading
import time

import pytest
import torch

from infernos_b200 import synth
from test_gpu_tts_server import SEED, _handles, _sentences, _server_threads

pytestmark = pytest.mark.gpu

NATURAL, CANCELLED = 1, 2                 # the kind of a sentence's last record; 0 for the others


@pytest.fixture(scope="module")
def sds():
    return dict(esd=synth.encoder_state_dict(), dsd=synth.decoder_state_dict(), vsd=synth.hifigan_state_dict(), csd=synth.chunker_state_dict(),
                psd=synth.postnet_state_dict())


def _collect(srv, n, on_record=None, timeout=300.0):
    """Polls until n sentences have their last record: tag -> [(call, bytes, kind)] and the records.  on_record(rec) runs on this thread,
    the one that polls, which is where a barge-in would be noticed."""
    got, raw, ended, t0 = {}, [], 0, time.time()
    while ended < n:
        assert time.time() - t0 < timeout, f"only {ended} of {n} sentences ended in {timeout} s"
        for rec, b in srv.poll(timeout_ms=20):
            got.setdefault(rec["tag"], []).append((rec["call"], b, CANCELLED if rec["cancelled"] else int(rec["ended"])))
            raw.append(rec)
            ended += rec["ended"]
            if on_record is not None:
                on_record(rec)
    return got, raw


def _replay(mk, pool, sents, raw, ncalls, cancel_at, threshold=0.5, minlenratio=0.0, maxlenratio=20.0, max_steps=64):
    """test_gpu_tts_server._replay with cancels: the sentences of cancel_at = {tag: call} leave the rows at that call, where their record
    is (call, b"", CANCELLED).  mk() -> fresh (tail, encoder, decoder)."""
    tail, enc, dec = mk()
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
            for t in live:
                if cancel_at.get(t) == c:
                    out.setdefault(t, []).append((c, b"", CANCELLED))
                    free.append(st[t]["slot"])
            live = [t for t in live if cancel_at.get(t) != c]
            rows = [st[t]["slot"] for t in live] or [-1]
            mel, prob = dec.steps(torch.tensor(rows, dtype=torch.int32).cuda(), 16, seed=SEED)
            if not live:
                continue
            g, _ = tail.tail(torch.tensor(rows, dtype=torch.int32).cuda(), mel, law=0, want_audio=False, apply_postnet=True)
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
                    out.setdefault(t, []).append((c, g[i, startoff:endoff].numpy().tobytes(), NATURAL if ended else 0))
                if ended:
                    gone.append(t)
                    free.append(s["slot"])
            live = [t for t in live if t not in gone]
        dec.poll_errors(); enc.poll_errors(); tail.poll_errors()
    finally:
        tail.close(); enc.close(); dec.close()
    return out, st


def _cancel_calls(got):
    """tag -> call of its cancelled record, for the sentences a cancel ended after their admission"""
    return {t: g[-1][0] for t, g in got.items() if g[-1][2] == CANCELLED and g[-1][0] >= 0}


def _check_against_replay(got, ref, tags):
    for t in tags:
        g, r = got[t], ref.get(t, [])
        kinds = [k for _, _, k in g]
        assert sum(k != 0 for k in kinds) == 1 and kinds[-1] != 0, f"sentence {t}: one last record, and nothing after it: {kinds}"
        assert [(c, k) for c, _, k in g] == [(c, k) for c, _, k in r], f"sentence {t}: calls / kinds differ: {[(c, k) for c, _, k in g]} vs " \
                                                                          f"{[(c, k) for c, _, k in r]}"
        assert all(a[1] == b[1] for a, b in zip(g, r)), f"sentence {t}: bytes differ from the replay"
        if kinds[-1] == CANCELLED:
            assert g[-1][1] == b""


def _serve(mk, submit, n, on_record, **kw):
    """(tail, enc, dec) = mk(); a server on them, submit(srv) on another thread, the records collected with on_record(srv, rec) on this one"""
    from infernos_b200.engine import TTSServer
    tail, enc, dec = mk()
    srv = TTSServer(tail, enc, dec, seed=SEED, **kw)
    try:
        th = threading.Thread(target=submit, args=(srv,), daemon=True)
        th.start()
        got, raw = _collect(srv, n, lambda rec: on_record(srv, rec))
        th.join(60)
        srv.flush(60000)
        stats = srv.stats()
        srv.close()
        dec.poll_errors()                                  # no row stepped past max_steps, no bad slot
        enc.poll_errors()
    finally:
        srv.close(); tail.close(); enc.close(); dec.close()
    return got, raw, stats


@pytest.mark.parametrize("depth,use_graphs", [(1, True), (2, True), (1, False), (2, False)])
def test_mid_sentence_cancels_equal_the_replay(sds, depth, use_graphs):
    """60 sentences arrive from another thread into a pool of 24; the polling thread cancels about a third of them a random number of
    records after their first.  max_steps = 100 (maxlen 80 steps, 6 calls): a row left stepping after its end would run past it."""
    g = torch.Generator().manual_seed(90 + depth)
    n = 60
    lengths = torch.randint(1, 31, (n,), generator=g).tolist()
    sents = _sentences(lengths, seed=91)
    gaps = (torch.rand(n, generator=g) * 0.02).tolist()
    rng = random.Random(92 + depth)
    plan = {t: rng.randint(1, 4) for t in sents if rng.random() < 1 / 3}
    seen, asked = {}, {}

    def submit(srv):
        for (t, (ids, spk)), dt in zip(sents.items(), gaps):
            time.sleep(dt)
            srv.submit(ids, spk, t)

    def on_record(srv, rec):
        t = rec["tag"]
        seen[t] = seen.get(t, 0) + 1
        if t in plan and seen[t] == plan[t] and not rec["ended"]:
            found = srv.cancel(t)                           # 0 when a later call, not polled yet, has already ended it
            assert found in (0, 1)
            if found:
                asked[t] = rec["call"]
    mk = lambda: _handles(sds, "bf16", 24, 100, 32)
    kw = dict(depth=depth, maxlenratio=20.0, use_graphs=use_graphs)
    got, raw, stats = _serve(mk, submit, n, on_record, **kw)
    cancel_at = _cancel_calls(got)
    assert set(cancel_at) <= set(asked), "only the sentences asked for were cancelled"
    assert all(cancel_at[t] > asked[t] for t in cancel_at)
    assert cancel_at and stats["ended"] == n
    assert any(r["admit_call"] > min(cancel_at.values()) for r in raw), "sentences were admitted after the first cancel freed a slot"
    ref, _ = _replay(mk, 24, sents, raw, stats["calls"], cancel_at, maxlenratio=20.0, max_steps=100)
    _check_against_replay(got, ref, sents)
    lag = sorted(cancel_at[t] - asked[t] for t in cancel_at)
    print(f"depth {depth} graphs {use_graphs}: {stats['calls']} calls, {len(asked)} cancels asked, {len(cancel_at)} cancelled, "
          f"{len(asked) - len(cancel_at)} ended on their own first; calls from the polled record to the cancelled one {lag[0]}..{lag[-1]}")


def _handles_9_slots_8_rows(sds):
    """9 slots but tail room for 8 rows per call: a 9th sentence waits in the queue while 8 are live, and a 10th submit blocks"""
    from infernos_b200.engine import TTSDecoder, TTSEncoder, TTSTail
    tail = TTSTail("cuda:0", sds["vsd"], sds["csd"], mode="bf16", max_sessions=9, max_windows=32, postnet_sd=sds["psd"])
    enc = TTSEncoder("cuda:0", sds["esd"], mode="bf16", max_tokens=4096, max_len=32)
    dec = TTSDecoder("cuda:0", sds["dsd"], mode="bf16", max_sessions=9, max_steps=2000, max_enc_len=32)
    return tail, enc, dec


@pytest.mark.parametrize("depth", [1, 2])
def test_pending_cancel_and_back_pressure(sds, depth):
    """8 long sentences fill the rows (maxlen 1,980 steps, 124 calls; the stop probability never fires), a 9th is pending, a 10th submit
    blocks.  Cancelling the pending one makes its record at once and unblocks the 10th; cancelling a live one lets the 10th in within a
    few calls, and its bytes are the replay's."""
    from infernos_b200.engine import TTSServer
    sents = _sentences([30] * 9 + [1], seed=95)
    tags = list(sents)
    longs, pend, late = tags[:8], tags[8], tags[9]
    kw = dict(depth=depth, threshold=2.0, maxlenratio=132.0)
    tail, enc, dec = _handles_9_slots_8_rows(sds)
    srv = TTSServer(tail, enc, dec, seed=SEED, **kw)
    recs = []

    def drain(until, timeout=60.0):
        t0 = time.time()
        while not until():
            assert time.time() - t0 < timeout
            recs.extend(srv.poll(timeout_ms=5))
    try:
        srv.submit_many([sents[t][0] for t in longs], [sents[t][1] for t in longs], longs)
        srv.submit(*sents[pend], pend)
        done = threading.Event()
        th = threading.Thread(target=lambda: (srv.submit(*sents[late], late), done.set()), daemon=True)
        th.start()
        assert not done.wait(0.05), "the 10th submit blocks while 9 sentences are unfinished in 9 slots"
        st = srv.stats()
        assert st["submitted"] == 9 and st["admitted"] == 8
        assert srv.cancel(pend) == 1
        recs.extend(srv.poll(timeout_ms=0))
        mine = [(r, b) for r, b in recs if r["tag"] == pend]
        assert len(mine) == 1, "the pending sentence's record is there at once"
        r, b = mine[0]
        assert (r["call"], r["admit_call"], r["nbytes"], r["ended"], r["cancelled"], b) == (-1, -1, 0, True, True, b"")
        assert r["t_done_ns"] >= r["t_submit_ns"]
        assert srv.cancel(pend) == 0
        assert done.wait(10), "cancelling the pending sentence freed its place for the blocked submit"
        th.join(10)
        assert srv.stats()["admitted"] == 8, "the 10th waits for a row"
        assert srv.cancel(longs[0]) == 1
        c1 = srv.stats()["calls"]
        drain(lambda: any(r["tag"] == late for r, _ in recs))
        first_late = next(r for r, _ in recs if r["tag"] == late)
        drain(lambda: any(r["tag"] == late and r["ended"] for r, _ in recs))
        gone = next(r for r, _ in recs if r["tag"] == longs[0] and r["ended"])
        assert gone["cancelled"] and gone["call"] <= c1 + depth
        assert first_late["admit_call"] <= c1 + 2 * depth, f"admitted at call {first_late['admit_call']}, cancel after call {c1}"
        assert not any(r["ended"] for r, _ in recs if r["tag"] in longs[1:]), "the long sentences were still running (timing premise)"
        assert srv.cancel(longs[1:]) == 7
        srv.flush(60000)
        recs.extend(srv.poll(timeout_ms=0))
        st = srv.stats()
        assert st["ended"] == st["submitted"] == 10 and st["admitted"] == 9
        srv.close()
        dec.poll_errors()
    finally:
        srv.close(); tail.close(); enc.close(); dec.close()
    got, raw = {}, []
    for r, b in recs:
        got.setdefault(r["tag"], []).append((r["call"], b, CANCELLED if r["cancelled"] else int(r["ended"])))
        raw.append(r)
    assert got[pend] == [(-1, b"", CANCELLED)]
    ref, _ = _replay(lambda: _handles_9_slots_8_rows(sds), 9, sents, raw, st["calls"], _cancel_calls(got), threshold=2.0, maxlenratio=132.0,
                     max_steps=2000)
    _check_against_replay(got, ref, longs + [late])
    assert got[late][-1][2] == NATURAL
    print(f"depth {depth}: cancel of a live sentence after call {c1}: its cancelled record at call {gone['call']}, the waiting sentence admitted "
          f"at call {first_late['admit_call']}; {st['calls']} calls")


@pytest.mark.parametrize("depth", [1, 2, 4])
def test_cancel_racing_a_natural_end(sds, depth):
    """12 sentences of L = 10 tokens, maxlen = 10 * 8 / 2 = 40 steps and no stop on probability: all end in call E = 2 (step 42 falls in
    steps 32..47).  All are cancelled as soon as the first record of call E - 1 is polled.  Each ends either on its own at E with the
    replay's bytes, or by the cancel at E after the replay's records of the calls before; never later.  At depth >= 2 call E has normally
    been built before the cancel arrives; at depth 1 the cancel races the driver's build of call E."""
    E = 2
    lengths = (10, 3, 7, 10, 1, 5, 9, 10, 2, 8, 6, 4)
    sents = _sentences(lengths, seed=97)
    tags = list(sents)
    fired = []

    def on_record(srv, rec):
        if not fired and rec["call"] == E - 1:
            fired.append(srv.cancel(tags))
    mk = lambda: _handles(sds, "bf16", 16, 64, 32)
    kw = dict(depth=depth, threshold=2.0, maxlenratio=8.0)
    got, raw, stats = _serve(mk, lambda srv: srv.submit_many([sents[t][0] for t in tags], [sents[t][1] for t in tags], tags), len(tags),
                             on_record, **kw)
    assert fired and 0 <= fired[0] <= len(tags)
    cancel_at = _cancel_calls(got)
    ref, _ = _replay(mk, 16, sents, raw, stats["calls"], cancel_at, threshold=2.0, maxlenratio=8.0, max_steps=64)
    _check_against_replay(got, ref, tags)
    assert all(got[t][-1][0] == E for t in tags), f"every last record is at call {E}: {[got[t][-1][0] for t in tags]}"
    print(f"depth {depth}: cancel returned {fired[0]}; {len(tags) - len(cancel_at)} ended on their own at call {E}, {len(cancel_at)} by the cancel")


def test_cancel_semantics(sds):
    from infernos_b200.engine import TTSServer
    tail, enc, dec = _handles(sds, "bf16", 8, 200, 32)
    sents = _sentences([1, 20, 20, 20], seed=99)
    (ids4, spk4), (ids1, spk1), (ids7a, spk7a), (ids7b, spk7b) = sents.values()
    try:
        srv = TTSServer(tail, enc, dec, seed=SEED, threshold=2.0, maxlenratio=20.0)
        lib = srv.lib
        tg = (ctypes.c_uint64 * 1)(1)
        assert lib.b2_tts_server_cancel(srv.h, None, 1) < 0
        assert lib.b2_tts_server_cancel(srv.h, tg, -1) < 0
        assert lib.b2_tts_server_cancel(srv.h, None, 0) == 0
        srv.submit(ids4, spk4, 4)                          # one token: maxlen 10, ends in call 0
        srv.flush(60000)
        assert srv.cancel(4) == 0, "an ended sentence"
        srv.submit_many([ids1, ids7a, ids7b], [spk1, spk7a, spk7b], [1, 7, 7])          # maxlen 180 steps: 12 calls
        assert srv.cancel(7) == 2, "both sentences of a shared tag"
        assert srv.cancel([7]) == 0, "a second cancel"
        assert srv.cancel(1) == 1
        assert srv.cancel((1, 1)) == 0
        assert srv.cancel(12345) == 0 and srv.cancel([]) == 0
        srv.flush(60000)
        recs = srv.poll(timeout_ms=0)
        assert srv.cancel([1, 4, 7]) == 0
        assert srv.poll(timeout_ms=100) == [], "no record after a sentence's last one"
        last = [(r["tag"], r["cancelled"]) for r, _ in recs if r["ended"]]
        assert sorted(last) == [(1, True), (4, False), (7, True), (7, True)]
        assert all(r["nbytes"] == 0 for r, _ in recs if r["cancelled"])
        st = srv.stats()
        assert st["ended"] == st["submitted"] == 4
        srv.close()
        with pytest.raises(RuntimeError, match="closed"):
            srv.cancel(1)
        dec.poll_errors()
        # a cancel with calls in flight, then close
        srv = TTSServer(tail, enc, dec, seed=SEED, depth=2)
        for i in range(8):
            srv.submit([4 + i] * (5 + i), spk1, 100 + i)
        time.sleep(0.005)
        assert srv.cancel(range(100, 104)) in range(0, 5)
        t0 = time.time()
        srv.close()
        assert time.time() - t0 < 30
        assert _server_threads() == []
    finally:
        tail.close(); enc.close(); dec.close()
