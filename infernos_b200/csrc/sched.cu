// Latency-bounded serving loop around the fused tail (SURVEY.md section 7 step 6; north_star: ">= 5,000 concurrent real-time streams
// per B200 with p99 per-chunk latency < 20 ms").
//
// What it replaces in the reference: the strictly serial worker loop  infer() -> unbatch_and_dispatch()  of
// Cluster/InfernTTSWorker.py:83-92 and the three overlapping executors of HelloSippyTTSRT/HelloSippyRTPipeTest.py:126-161
// (generate / dispatch / collect).  Here:
//
//   submit() (any thread)   copies a session's mel chunk straight into the pinned staging buffer of the OPEN sub-batch
//   launcher thread         closes the open sub-batch as soon as the pipeline has room (adaptive batching: small sub-batches when
//                           the GPU is idle, larger ones under load), then enqueues   H2D (stream in) -> tail (stream compute,
//                           ONE cudaGraphLaunch per sub-batch, graphs cached per (bucket, staging buffer)) -> D2H (stream out)
//   completer thread        waits for the D2H event of the oldest sub-batch, stamps the completion time of its chunks and hands them to
//                           poll(); the staging buffer goes back to the pool
//
// With `depth` sub-batches in flight the H2D of sub-batch n+1 and the D2H of n-1 overlap the compute of n; the compute of successive
// sub-batches is serialised on one stream (they share the context's workspaces).  Sessions per sub-batch are padded up to a bucket
// size with a scratch session (slot id max_sessions) so that a few dozen graphs cover every batch size.
#include "serve.cuh"
#include "../../include/infernos_b200.h"

#include <string.h>
#include <condition_variable>
#include <deque>
#include <map>
#include <mutex>
#include <thread>
#include <vector>

using namespace b2;

namespace {

struct Batch {
    int id = 0;
    // pinned host staging
    int32_t *h_slots = nullptr;
    float *h_mel = nullptr;
    uint8_t *h_out = nullptr;
    // device staging
    int32_t *d_slots = nullptr;
    float *d_mel = nullptr;
    uint8_t *d_out = nullptr;
    std::vector<uint64_t> tags;
    std::vector<int64_t> t_enq;
    int reserved = 0;                    // sessions handed out to submitters (under the scheduler mutex)
    std::atomic<int> filled{0};          // sessions whose mel has been copied in
    int n = 0, nb = 0;                   // sessions, padded sessions of the launch
    int64_t t_first = 0;                 // arrival of the first chunk (max_wait policy)
    int64_t t_launch = 0, t_done = 0;
    cudaEvent_t ev_in = nullptr, ev_c = nullptr, ev_out = nullptr;
    int polled = 0;                      // completions already handed to poll()
    std::map<int, std::pair<cudaGraphExec_t, int>> graphs;   // bucket -> (instantiated graph over THIS buffer's pointers, kernels in it)
};

}  // namespace

struct b2_sched {
    b2_ctx *ctx = nullptr;
    int nframes = 0, law = 0, flags = 0, cap = 0, depth = 2, use_graphs = 1, max_wait_us = 0, min_batch = 0;
    size_t mel_per = 0, out_per = 0;
    cudaStream_t s_in = nullptr, s_c = nullptr, s_out = nullptr;
    std::vector<Batch *> pool;
    std::mutex mu;
    std::condition_variable cv_submit, cv_launch, cv_complete, cv_poll;
    Batch *open = nullptr;
    std::deque<Batch *> free_q, inflight, done_q;
    bool stop = false;
    std::string async_error;
    std::thread th_launch, th_complete;
    // stats
    uint64_t n_batches = 0, n_sessions = 0, n_padded = 0, n_graph_launches = 0, n_graphs = 0, max_batch_seen = 0;
    std::vector<uint8_t> seen;           // host-side duplicate check of a sub-batch
    std::vector<int> seen_list;
};

namespace {

int sched_fail(b2_sched *s, const char *what) {
    std::lock_guard<std::mutex> lk(s->mu);
    if (s->async_error.empty()) s->async_error = std::string(what) + ": " + g_last_error;
    s->stop = true;
    s->cv_submit.notify_all(); s->cv_launch.notify_all(); s->cv_complete.notify_all(); s->cv_poll.notify_all();
    return 1;
}

// captures the tail over `b`'s device staging buffers at a padded sub-batch size `nb` and instantiates it (nothing is launched)
int build_graph(b2_sched *s, Batch *b, int nb) {
    cudaGraphExec_t ge = nullptr;
    int nk = 0;
    if (capture_tail_graph(s->ctx, b->d_slots, b->d_mel, nb, s->nframes, s->law, (s->flags & B2_TAIL_APPLY_POSTNET) != 0, b->d_out, s->s_c, &ge, &nk))
        return 1;
    b->graphs.emplace(nb, std::make_pair(ge, nk));
    s->n_graphs++;
    return 0;
}

int enqueue_batch(b2_sched *s, Batch *b) {
    b2_ctx *c = s->ctx;
    const int n = b->n;
    const int nb = s->use_graphs ? bucket_of(n, s->cap) : n;
    for (int i = n; i < nb; i++) b->h_slots[i] = c->max_sessions;          // the scratch session: its audio is computed and dropped
    b->nb = nb;
    B2_CUDA_OK(cudaMemcpyAsync(b->d_slots, b->h_slots, (size_t)nb * sizeof(int32_t), cudaMemcpyHostToDevice, s->s_in));
    B2_CUDA_OK(cudaMemcpyAsync(b->d_mel, b->h_mel, (size_t)n * s->mel_per * sizeof(float), cudaMemcpyHostToDevice, s->s_in));
    B2_CUDA_OK(cudaEventRecord(b->ev_in, s->s_in));
    B2_CUDA_OK(cudaStreamWaitEvent(s->s_c, b->ev_in, 0));
    const bool pn = (s->flags & B2_TAIL_APPLY_POSTNET) != 0;
    if (s->use_graphs && !c->prof.on) {
        auto it = b->graphs.find(nb);
        if (it == b->graphs.end()) {
            if (build_graph(s, b, nb)) return 1;
            it = b->graphs.find(nb);
        }
        B2_CUDA_OK(cudaGraphLaunch(it->second.first, s->s_c));
        count_launch(it->second.second);
        s->n_graph_launches++;
    } else {
        if (tail_device(c, b->d_slots, b->d_mel, nb, s->nframes, s->law, pn, b->d_out, nullptr, s->s_c, false, true)) return 1;
    }
    B2_CUDA_OK(cudaEventRecord(b->ev_c, s->s_c));
    B2_CUDA_OK(cudaStreamWaitEvent(s->s_out, b->ev_c, 0));
    B2_CUDA_OK(cudaMemcpyAsync(b->h_out, b->d_out, (size_t)n * s->out_per, cudaMemcpyDeviceToHost, s->s_out));
    B2_CUDA_OK(cudaEventRecord(b->ev_out, s->s_out));
    return 0;
}

void launcher_main(b2_sched *s) {
    cudaSetDevice(s->ctx->device);
    std::unique_lock<std::mutex> lk(s->mu);
    while (true) {
        // something to launch, and room in the pipeline
        s->cv_launch.wait(lk, [&] { return s->stop || (s->open && s->open->reserved > 0 && (int)s->inflight.size() < s->depth); });
        if (s->stop) break;
        Batch *b = s->open;
        if (s->max_wait_us > 0 && b->reserved < s->min_batch) {
            // small sub-batch: give it until max_wait_us after its first chunk to grow (off by default)
            const int64_t deadline = b->t_first + (int64_t)s->max_wait_us * 1000;
            const int64_t t = now_ns();
            if (t < deadline) {
                s->cv_launch.wait_for(lk, std::chrono::nanoseconds(deadline - t));
                continue;
            }
        }
        // close it; submitters move on to the next free buffer (or wait for one)
        s->open = nullptr;
        if (!s->free_q.empty()) { s->open = s->free_q.front(); s->free_q.pop_front(); }
        b->n = b->reserved;
        s->cv_submit.notify_all();
        lk.unlock();
        while (b->filled.load(std::memory_order_acquire) < b->n) { /* a submitter is still copying its chunk in: microseconds */ }
        b->t_launch = now_ns();
        const int rc = enqueue_batch(s, b);
        lk.lock();
        if (rc) {
            lk.unlock();
            sched_fail(s, "sub-batch launch");
            lk.lock();
            break;
        }
        s->n_batches++; s->n_sessions += (uint64_t)b->n; s->n_padded += (uint64_t)(b->nb - b->n);
        s->max_batch_seen = std::max<uint64_t>(s->max_batch_seen, (uint64_t)b->n);
        s->inflight.push_back(b);
        s->cv_complete.notify_all();
    }
}

void completer_main(b2_sched *s) {
    cudaSetDevice(s->ctx->device);
    std::unique_lock<std::mutex> lk(s->mu);
    while (true) {
        s->cv_complete.wait(lk, [&] { return !s->inflight.empty() || s->stop; });
        if (s->inflight.empty()) { if (s->stop) break; continue; }
        Batch *b = s->inflight.front();
        lk.unlock();
        const cudaError_t e = cudaEventSynchronize(b->ev_out);      // spins: the completion time is what is being measured
        b->t_done = now_ns();
        if (e != cudaSuccess) {
            set_error("cudaEventSynchronize: %s", cudaGetErrorString(e));
            sched_fail(s, "sub-batch completion");
            lk.lock();
            break;
        }
        lk.lock();
        s->inflight.pop_front();
        b->polled = 0;
        s->done_q.push_back(b);
        s->cv_launch.notify_all();
        s->cv_poll.notify_all();
    }
}

void recycle(b2_sched *s, Batch *b) {      // under the mutex
    b->reserved = 0; b->n = 0; b->nb = 0; b->polled = 0; b->t_first = 0;
    b->filled.store(0, std::memory_order_relaxed);
    if (!s->open) s->open = b; else s->free_q.push_back(b);
    s->cv_submit.notify_all();
    s->cv_launch.notify_all();
}

}  // namespace

namespace b2 {

int capture_tail_graph(b2_ctx *c, const int32_t *d_slots, const float *d_mel, int nb, int nframes, int law, bool apply_postnet, uint8_t *d_g711,
                       cudaStream_t st, cudaGraphExec_t *exec, int *nk) {
    cudaGraph_t g = nullptr;
    cudaGraphExec_t ge = nullptr;
    const uint64_t l0 = g_launches.load();
    B2_CUDA_OK(cudaStreamBeginCapture(st, cudaStreamCaptureModeRelaxed)      /* relaxed: a kernel's first launch may set its function attributes */);
    const int rc = tail_device(c, d_slots, d_mel, nb, nframes, law, apply_postnet, d_g711, nullptr, st, false, true);
    cudaError_t e = cudaStreamEndCapture(st, &g);
    if (rc) { if (g) cudaGraphDestroy(g); return 1; }
    if (e != cudaSuccess) return set_error("cudaStreamEndCapture: %s", cudaGetErrorString(e));
    e = cudaGraphInstantiate(&ge, g, 0);
    cudaGraphDestroy(g);
    if (e != cudaSuccess) return set_error("cudaGraphInstantiate: %s", cudaGetErrorString(e));
    *nk = (int)(g_launches.load() - l0);                   // kernel nodes: counted by the launch wrappers while capturing
    g_launches.fetch_sub((uint64_t)*nk);                   // ... and only charged when the graph actually runs
    *exec = ge;
    return 0;
}

int warm_tail(b2_ctx *c, int32_t *d_slots, const float *d_mel, int nb, int nframes, int law, bool apply_postnet, uint8_t *d_g711, cudaStream_t st) {
    std::vector<int32_t> pad((size_t)nb, c->max_sessions);
    B2_CUDA_OK(cudaMemcpyAsync(d_slots, pad.data(), (size_t)nb * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    if (tail_device(c, d_slots, d_mel, nb, nframes, law, apply_postnet, d_g711, nullptr, st, false, true)) return 1;
    B2_CUDA_OK(cudaStreamSynchronize(st));
    return 0;
}

}  // namespace b2

extern "C" {

b2_sched *b2_sched_create(b2_ctx *c, int nframes, int law, int flags, int max_batch, int depth, int use_graphs) {
    if (!c || !c->finalized) { set_error("b2_sched_create: the context has no finalized weights"); return nullptr; }
    if (nframes < 8 || nframes % 8) { set_error("b2_sched_create: nframes must be a positive multiple of 8"); return nullptr; }
    if (law != B2_LAW_ULAW && law != B2_LAW_ALAW) { set_error("b2_sched_create: bad law %d", law); return nullptr; }
    if (flags & ~B2_TAIL_APPLY_POSTNET) { set_error("b2_sched_create: unknown flags"); return nullptr; }
    if ((flags & B2_TAIL_APPLY_POSTNET) && !c->has_postnet) { set_error("b2_sched_create: B2_TAIL_APPLY_POSTNET without post-net weights"); return nullptr; }
    const int nwin = nframes / 8;
    const int fit = c->max_windows / nwin;                       // one pass of the tail per sub-batch
    if (fit < 1) { set_error("b2_sched_create: nframes=%d needs more windows than the context's workspace", nframes); return nullptr; }
    if (max_batch <= 0 || max_batch > fit) max_batch = fit;
    if (depth < 1) depth = 2;
    if (depth > 6) depth = 6;
    if (cudaSetDevice(c->device) != cudaSuccess) { set_error("cudaSetDevice failed"); return nullptr; }
    b2_sched *s = new b2_sched();
    s->ctx = c; s->nframes = nframes; s->law = law; s->flags = flags; s->cap = max_batch; s->depth = depth; s->use_graphs = use_graphs ? 1 : 0;
    s->mel_per = (size_t)nframes * 80; s->out_per = (size_t)nframes * 128;
    s->seen.assign((size_t)c->max_sessions, 0);
    bool ok = cudaStreamCreateWithFlags(&s->s_in, cudaStreamNonBlocking) == cudaSuccess &&
              cudaStreamCreateWithFlags(&s->s_c, cudaStreamNonBlocking) == cudaSuccess &&
              cudaStreamCreateWithFlags(&s->s_out, cudaStreamNonBlocking) == cudaSuccess;
    const int nbuf = depth + 2;                                   // `depth` in flight + one open + one being drained by poll()
    for (int i = 0; ok && i < nbuf; i++) {
        Batch *b = new Batch();
        b->id = i;
        s->pool.push_back(b);
        b->tags.resize((size_t)max_batch); b->t_enq.resize((size_t)max_batch);
        ok = cudaHostAlloc((void **)&b->h_slots, (size_t)max_batch * sizeof(int32_t), cudaHostAllocDefault) == cudaSuccess &&
             cudaHostAlloc((void **)&b->h_mel, (size_t)max_batch * s->mel_per * sizeof(float), cudaHostAllocDefault) == cudaSuccess &&
             cudaHostAlloc((void **)&b->h_out, (size_t)max_batch * s->out_per, cudaHostAllocDefault) == cudaSuccess &&
             cudaMalloc((void **)&b->d_slots, (size_t)max_batch * sizeof(int32_t)) == cudaSuccess &&
             cudaMalloc((void **)&b->d_mel, (size_t)max_batch * s->mel_per * sizeof(float)) == cudaSuccess &&
             cudaMalloc((void **)&b->d_out, (size_t)max_batch * s->out_per) == cudaSuccess &&
             cudaEventCreateWithFlags(&b->ev_in, cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&b->ev_c, cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&b->ev_out, cudaEventDisableTiming) == cudaSuccess;
        if (ok) {
            memset(b->h_mel, 0, (size_t)max_batch * s->mel_per * sizeof(float));
            ok = cudaMemset(b->d_mel, 0, (size_t)max_batch * s->mel_per * sizeof(float)) == cudaSuccess;
        }
    }
    if (!ok) {
        set_error("b2_sched_create: allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
        b2_sched_destroy(s);
        return nullptr;
    }
    if (warm_tail(c, s->pool[0]->d_slots, s->pool[0]->d_mel, std::min(8, max_batch), nframes, law, (flags & B2_TAIL_APPLY_POSTNET) != 0, s->pool[0]->d_out, s->s_c)) {
        b2_sched_destroy(s);
        return nullptr;
    }
    s->open = s->pool[0];
    for (int i = 1; i < nbuf; i++) s->free_q.push_back(s->pool[i]);
    s->th_launch = std::thread(launcher_main, s);
    s->th_complete = std::thread(completer_main, s);
    return s;
}

void b2_sched_destroy(b2_sched *s) {
    if (!s) return;
    {
        std::lock_guard<std::mutex> lk(s->mu);
        s->stop = true;
    }
    s->cv_submit.notify_all(); s->cv_launch.notify_all(); s->cv_complete.notify_all(); s->cv_poll.notify_all();
    if (s->th_launch.joinable()) s->th_launch.join();
    if (s->th_complete.joinable()) s->th_complete.join();
    cudaSetDevice(s->ctx->device);
    if (s->s_c) cudaStreamSynchronize(s->s_c);
    if (s->s_in) cudaStreamSynchronize(s->s_in);
    if (s->s_out) cudaStreamSynchronize(s->s_out);
    for (Batch *b : s->pool) {
        for (auto &kv : b->graphs) cudaGraphExecDestroy(kv.second.first);
        if (b->h_slots) cudaFreeHost(b->h_slots);
        if (b->h_mel) cudaFreeHost(b->h_mel);
        if (b->h_out) cudaFreeHost(b->h_out);
        if (b->d_slots) cudaFree(b->d_slots);
        if (b->d_mel) cudaFree(b->d_mel);
        if (b->d_out) cudaFree(b->d_out);
        if (b->ev_in) cudaEventDestroy(b->ev_in);
        if (b->ev_c) cudaEventDestroy(b->ev_c);
        if (b->ev_out) cudaEventDestroy(b->ev_out);
        delete b;
    }
    if (s->s_in) cudaStreamDestroy(s->s_in);
    if (s->s_c) cudaStreamDestroy(s->s_c);
    if (s->s_out) cudaStreamDestroy(s->s_out);
    delete s;
}

int b2_sched_set_policy(b2_sched *s, int min_batch, int max_wait_us) {
    if (!s) return set_error("null scheduler");
    std::lock_guard<std::mutex> lk(s->mu);
    s->min_batch = std::max(0, min_batch);
    s->max_wait_us = std::max(0, max_wait_us);
    return 0;
}

int b2_sched_submit(b2_sched *s, const int32_t *h_slots, const float *h_mel, int n, const int64_t *t_enqueue_ns, const uint64_t *tags) {
    if (!s) return set_error("null scheduler");
    if (n < 0 || (n > 0 && (!h_slots || !h_mel))) return set_error("b2_sched_submit: bad arguments");
    const int64_t t_now = now_ns();
    for (int i = 0; i < n; i++)
        if (h_slots[i] < 0 || h_slots[i] >= s->ctx->max_sessions) return set_error("b2_sched_submit: slot %d is outside the pool of %d", h_slots[i], s->ctx->max_sessions);
    int done = 0;
    while (done < n) {
        Batch *b = nullptr;
        int at = 0, k = 0;
        {
            std::unique_lock<std::mutex> lk(s->mu);
            // back-pressure: every staging buffer is busy.  Buffers come back through b2_sched_poll, so a caller that submits and polls on ONE
            // thread can starve itself: rather than hang, give up after a while and say so
            if (!s->cv_submit.wait_for(lk, std::chrono::seconds(20), [&] { return s->stop || (s->open && s->open->reserved < s->cap); }))
                return set_error("b2_sched_submit: no staging buffer became free in 20 s (%d of %d chunks of this call were accepted); finished sub-batches "
                                 "are recycled by b2_sched_poll -- poll from another thread, or between smaller submits", done, n);
            if (s->stop) return set_error("b2_sched_submit: the scheduler has stopped%s%s", s->async_error.empty() ? "" : ": ", s->async_error.c_str());
            b = s->open;
            at = b->reserved;
            // a session may appear once per sub-batch (its pre_frames are read and written by that launch); a second chunk of the same
            // session closes this sub-batch for it and goes into the next one
            k = 0;
            if (at == 0) { for (int q : s->seen_list) s->seen[(size_t)q] = 0; s->seen_list.clear(); }
            while (k < std::min(s->cap - at, n - done)) {
                const int sl = h_slots[done + k];
                if (s->seen[(size_t)sl]) break;
                s->seen[(size_t)sl] = 1; s->seen_list.push_back(sl);
                k++;
            }
            if (k == 0) {
                // the next chunk's session is already in the open sub-batch: wait until that one has been closed
                s->cv_launch.notify_all();
                if (!s->cv_submit.wait_for(lk, std::chrono::seconds(20), [&] { return s->stop || s->open != b || b->reserved == 0; }))
                    return set_error("b2_sched_submit: the open sub-batch was not launched within 20 s (pipeline full and nobody polling?)");
                continue;
            }
            if (at == 0) b->t_first = t_now;
            b->reserved = at + k;
        }
        memcpy(b->h_slots + at, h_slots + done, (size_t)k * sizeof(int32_t));
        memcpy(b->h_mel + (size_t)at * s->mel_per, h_mel + (size_t)done * s->mel_per, (size_t)k * s->mel_per * sizeof(float));
        for (int i = 0; i < k; i++) {
            b->tags[(size_t)(at + i)] = tags ? tags[done + i] : (uint64_t)h_slots[done + i];
            b->t_enq[(size_t)(at + i)] = (t_enqueue_ns && t_enqueue_ns[done + i] > 0) ? t_enqueue_ns[done + i] : t_now;
        }
        b->filled.fetch_add(k, std::memory_order_release);
        done += k;
        s->cv_launch.notify_all();
    }
    return 0;
}

int b2_sched_poll(b2_sched *s, b2_completion *out, int max_out, uint8_t *h_g711, size_t g711_capacity, int timeout_ms) {
    if (!s) return -set_error("null scheduler");
    if (!out || max_out < 1) return -set_error("b2_sched_poll: bad arguments");
    std::unique_lock<std::mutex> lk(s->mu);
    if (s->done_q.empty() && timeout_ms != 0) {
        auto pred = [&] { return !s->done_q.empty() || s->stop; };
        if (timeout_ms < 0) s->cv_poll.wait(lk, pred);
        else s->cv_poll.wait_for(lk, std::chrono::milliseconds(timeout_ms), pred);
    }
    if (s->done_q.empty()) {
        if (!s->async_error.empty()) return -set_error("b2_sched_poll: %s", s->async_error.c_str());
        return 0;
    }
    int cnt = 0;
    size_t off = 0;
    while (cnt < max_out && !s->done_q.empty()) {
        Batch *b = s->done_q.front();
        while (cnt < max_out && b->polled < b->n) {
            if (h_g711 && off + s->out_per > g711_capacity) goto full;
            b2_completion &r = out[cnt];
            const int i = b->polled;
            r.tag = b->tags[(size_t)i]; r.slot = b->h_slots[i]; r.nbytes = (int32_t)s->out_per;
            r.t_enqueue_ns = b->t_enq[(size_t)i]; r.t_launch_ns = b->t_launch; r.t_done_ns = b->t_done;
            r.batch_sessions = b->n; r.g711_offset = h_g711 ? (int64_t)off : -1;
            if (h_g711) { memcpy(h_g711 + off, b->h_out + (size_t)i * s->out_per, s->out_per); off += s->out_per; }
            b->polled++; cnt++;
        }
        if (b->polled < b->n) break;
        s->done_q.pop_front();
        recycle(s, b);
    }
full:
    return cnt;
}

int b2_sched_flush(b2_sched *s, int timeout_ms) {
    if (!s) return set_error("null scheduler");
    std::unique_lock<std::mutex> lk(s->mu);
    auto idle = [&] { return s->stop || ((!s->open || s->open->reserved == 0) && s->inflight.empty()); };
    s->cv_launch.notify_all();
    // completions wake cv_poll; use it as the progress signal
    const auto deadline = std::chrono::steady_clock::now() + std::chrono::milliseconds(timeout_ms < 0 ? 3600000 : timeout_ms);
    while (!idle()) {
        if (s->cv_poll.wait_until(lk, deadline) == std::cv_status::timeout && !idle()) return set_error("b2_sched_flush: timed out");
    }
    if (!s->async_error.empty()) return set_error("b2_sched_flush: %s", s->async_error.c_str());
    return 0;
}

int b2_sched_prebuild(b2_sched *s, int max_sessions) {
    if (!s) return set_error("null scheduler");
    if (!s->use_graphs || s->ctx->prof.on) return 0;
    std::unique_lock<std::mutex> lk(s->mu);
    if (!((!s->open || s->open->reserved == 0) && s->inflight.empty())) return set_error("b2_sched_prebuild: the scheduler is not idle");
    if (cudaSetDevice(s->ctx->device) != cudaSuccess) return set_error("b2_sched_prebuild: cudaSetDevice failed");
    const int top = bucket_of(std::max(1, std::min(max_sessions <= 0 ? s->cap : max_sessions, s->cap)), s->cap);
    // every staging buffer has its own graphs (they bake the buffer's device pointers in)
    for (Batch *b : s->pool)
        for (int n = 1; n <= top;) {
            const int nb = bucket_of(n, s->cap);
            if (!b->graphs.count(nb) && build_graph(s, b, nb)) return 1;
            n = nb + 1;
        }
    if (cudaStreamSynchronize(s->s_c) != cudaSuccess) return set_error("b2_sched_prebuild: %s", cudaGetErrorString(cudaGetLastError()));
    return 0;
}

int b2_sched_get_stats(b2_sched *s, b2_sched_stats *st) {
    if (!s || !st) return set_error("b2_sched_get_stats: null pointer");
    std::lock_guard<std::mutex> lk(s->mu);
    st->sub_batches = s->n_batches; st->sessions = s->n_sessions; st->padded_sessions = s->n_padded;
    st->graph_launches = s->n_graph_launches; st->graphs_built = s->n_graphs; st->max_sub_batch = s->max_batch_seen;
    st->capacity = (uint64_t)s->cap; st->depth = (uint64_t)s->depth;
    return 0;
}

}  // extern "C"
