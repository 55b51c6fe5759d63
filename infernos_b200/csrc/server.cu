// Sentence server: token ids in, G.711 chunks out, with the stop rule on the device (include/infernos_b200.h, b2_tts_server_*).
//
// What it replaces in the reference: the worker loop  infer() -> unbatch_and_dispatch()  of Cluster/InfernTTSWorker.py:83-92 around
// HelloSippyTTSRT/HelloSippyRTPipe.py:195-259 (the decoder loop, the stop rule, the tail, the slicing).  Here:
//
//   submit() (any thread)   validates one sentence on the host and queues it (blocks while every slot holds a sentence that has not ended)
//   driver thread           one engine call after another, `depth` of them in flight, all on one compute stream:
//                             admission round (pending sentences -> free slots: H2D of the packed ids, b2_enc_forward, b2_dec_start,
//                             k_tts_admit) -> k_tts_rows -> b2_dec_steps(16) over every live slot -> k_tts_stop -> fused tail with the
//                             post-net (one graph launch) -> D2H of the bytes and of the (startoff, endoff, ended) triples on a copy stream
//   completer thread        waits for a call's D2H, turns its triples into records (bytes copied out of the call's pinned buffer, so the
//                             buffer is free again at once) and returns the slots of ended sentences to the pool
//
// The host only learns that a sentence ended when its call completes.  With depth > 1 the next call has already been built with that
// sentence in its row list, so k_tts_stop retires an ending row on the device (live[slot] = 0) and k_tts_rows of every later call turns the
// row into the decoder's padding id -1 (the scratch slot: no step counted, nothing flagged) and the tail's scratch session.
//
// Cancellation (b2_tts_server_cancel) uses the same retirement.  A pending sentence is dropped from the queue on the host.  An admitted one
// is queued as (slot, admission sequence number); the next build_call puts it into that call's cancel list if the slot still holds the same
// admission, and k_tts_cancel clears live[slot] and marks the row, so k_tts_rows pads it and k_tts_stop reports {0, 0, 2}.  Whether the
// sentence ended on its own in a call already in flight is known only on the device: there live[slot] is already 0 and the cancel does
// nothing.  live goes from 1 to 0 once per admission, so every sentence gets exactly one last record.
#include "serve.cuh"
#include "../../include/infernos_b200.h"

#include <pthread.h>
#include <string.h>
#include <condition_variable>
#include <deque>
#include <functional>
#include <map>
#include <mutex>
#include <thread>
#include <vector>

using namespace b2;

namespace {

constexpr int NSTEPS = 16;                      // decoder steps per engine call (B200Frontend.steps_per_call)
constexpr int NFRAMES = 2 * NSTEPS;             // mel frames per call: reduction factor 2
constexpr int NBYTES = NFRAMES * 128;           // G.711 bytes per sentence and call (8 kHz)
constexpr int STEP_BYTES = 256;                 // bytes per decoder step at 8 kHz (unbatch_and_dispatch's stepsize, :505)
constexpr int STARTS_AT = 1;                    // post_nframes // reduction_factor (:98)
constexpr int END_DELAY = 2;                    // (pre_nframes + post_nframes) // reduction_factor (:420)
constexpr int SPK = 512, NMEL = 80;

// ---------------------------------------------------------------------------------------------------- kernels
// a new sentence in `slot`: its stop-rule state, and zero pre_frames in the tail's pool (HelloSippyPipeState, :77, :98-99)
__global__ void k_tts_admit(const int32_t *__restrict__ adm, int n, int32_t *__restrict__ idx, int32_t *__restrict__ ends, int32_t *__restrict__ minlen,
                            int32_t *__restrict__ maxlen, int32_t *__restrict__ live, float *__restrict__ pre_pool) {
    const int i = blockIdx.x;
    if (i >= n) return;
    const int sl = adm[i];                      // adm = [slots | minlen | maxlen], n each
    for (int c = threadIdx.x; c < 4 * NMEL; c += blockDim.x) pre_pool[(size_t)sl * 4 * NMEL + c] = 0.0f;
    if (threadIdx.x == 0) {
        idx[sl] = 0; ends[sl] = -1; minlen[sl] = adm[n + i]; maxlen[sl] = adm[2 * n + i]; live[sl] = 1;
    }
}

// rows of this call: the host's list of slots it believes live -> decoder slots (-1 once retired on the device) and tail slots (the
// scratch session for retired rows and for the padding up to the graph bucket nb)
__global__ void k_tts_rows(const int32_t *__restrict__ rows, int n, int nb, const int32_t *__restrict__ live, int scratch, int32_t *__restrict__ dslots,
                           int32_t *__restrict__ tslots) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nb) return;
    if (i < n) {
        const int sl = rows[i];
        const bool on = live[sl] != 0;
        dslots[i] = on ? sl : -1;
        tslots[i] = on ? sl : scratch;
    } else {
        tslots[i] = scratch;
    }
}

// cancels of this call: can[2i] = row, can[2i + 1] = slot.  A sentence still live on the device is retired and its row marked; one that a
// call in flight already retired (a natural end) is left alone.  One thread per cancel.
__global__ void k_tts_cancel(const int32_t *__restrict__ can, int n, int32_t *__restrict__ live, int32_t *__restrict__ mark) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int sl = can[2 * i + 1];
    if (live[sl]) { live[sl] = 0; mark[can[2 * i]] = 1; }
}

// The stop rule of HelloSippyRTPipe._front_half (:417-421), step by step over this call's stop probabilities, then unbatch_prepare's slice
// (:503-527): tri[i] = {startoff, endoff, ended} in bytes of this call's 4,096.  An ended sentence is retired (live = 0).  One thread per row.
// mark (NULL when the call has no cancel): rows k_tts_cancel retired get {0, 0, 2}; the marks are cleared for the next call.
__global__ void k_tts_stop(const int32_t *__restrict__ dslots, const float *__restrict__ prob, int n, float threshold, int32_t *__restrict__ idx,
                           int32_t *__restrict__ ends, const int32_t *__restrict__ minlen, const int32_t *__restrict__ maxlen, int32_t *__restrict__ live,
                           int32_t *__restrict__ mark, int32_t *__restrict__ tri) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int sl = dslots[i];
    if (sl < 0) {
        int cancelled = 0;
        if (mark) { cancelled = mark[i] ? 2 : 0; mark[i] = 0; }
        tri[3 * i] = 0; tri[3 * i + 1] = 0; tri[3 * i + 2] = cancelled;
        return;
    }
    int t = idx[sl], e = ends[sl];
    const int lo = minlen[sl], hi = maxlen[sl];
    for (int s = 0; s < NSTEPS; s++) {
        const float *p = prob + ((size_t)i * NSTEPS + s) * 2;
        const bool stop = p[0] >= threshold || p[1] >= threshold;
        if (e < 0 && lo <= t && (stop || hi <= t)) e = t + END_DELAY;
        t++;
    }
    idx[sl] = t; ends[sl] = e;
    const int startoff = max(0, NBYTES - (t - STARTS_AT) * STEP_BYTES);
    const int endoff = min(NBYTES, NBYTES - (e >= 0 ? (t - e) * STEP_BYTES : 0));
    const int ended = (e >= 0 && e <= t - 1) ? 1 : 0;
    tri[3 * i] = startoff; tri[3 * i + 1] = endoff; tri[3 * i + 2] = ended;
    if (ended) live[sl] = 0;
}

struct Pending {
    std::vector<int32_t> ids;
    std::vector<float> spk;
    uint64_t tag = 0;
    int64_t t_submit = 0;
};

struct SlotInfo {
    uint64_t tag = 0;
    uint64_t seq = 0;                          // admission sequence number: tells this sentence from a later one in the same slot
    int64_t t_submit = 0, admit_call = 0;
    bool live = false;
    bool cancelled = false;                    // a cancel of this admission has been accepted
};

struct Done {                                  // the records of one completed call, waiting for poll()
    std::vector<b2_tts_chunk> recs;
    std::vector<uint8_t> bytes;                // record r's bytes at recs[r].g711_offset (rewritten for the caller by poll)
    size_t polled = 0;
};

// one engine call's pinned staging and device outputs; graphs bake this buffer's d_out in
struct Call {
    int32_t *h_ids = nullptr, *h_len = nullptr, *h_adm = nullptr, *h_rows = nullptr, *h_tri = nullptr;
    int32_t *h_can = nullptr;                  // cancel list: n_can (row, slot) pairs
    float *h_spk = nullptr;
    uint8_t *h_out = nullptr, *d_out = nullptr;
    int32_t *d_tri = nullptr;
    cudaEvent_t ev_c = nullptr, ev_out = nullptr;
    std::map<int, std::pair<cudaGraphExec_t, int>> graphs;    // bucket -> (instantiated tail graph, kernels in it)
    int64_t call = 0;
    int n = 0, nb = 0, n_adm = 0, L = 0, n_can = 0;
    std::vector<int32_t> row_slot;
    std::vector<SlotInfo> row_info;            // the sentence each row belonged to when the call was built
};

}  // namespace

struct b2_tts_server {
    b2_ctx *ctx = nullptr;
    b2_enc *enc = nullptr;
    b2_dec *dec = nullptr;
    int law = 0, depth = 2, use_graphs = 1;
    float threshold = 0.5f, minlenratio = 0.0f, maxlenratio = 20.0f;
    uint64_t seed = 0;
    int nslots = 0, cap = 0, adm_cap = 0, max_len = 0, max_tokens = 0, vocab = 0, max_steps = 0;
    cudaStream_t s_c = nullptr, s_out = nullptr;
    // device state, indexed by slot
    int32_t *d_idx = nullptr, *d_ends = nullptr, *d_minlen = nullptr, *d_maxlen = nullptr, *d_live = nullptr;
    // device workspaces shared by the calls (stream-ordered on s_c); d_mark (by row) is all zero between calls
    int32_t *d_ids = nullptr, *d_len = nullptr, *d_adm = nullptr, *d_rows = nullptr, *d_dslots = nullptr, *d_tslots = nullptr;
    int32_t *d_can = nullptr, *d_mark = nullptr;
    float *d_spk = nullptr, *d_enc = nullptr, *d_mel = nullptr, *d_prob = nullptr;
    std::vector<Call *> calls_pool;
    std::mutex mu;
    std::condition_variable cv_submit, cv_drive, cv_complete, cv_poll;
    std::deque<Pending> pending;
    std::vector<SlotInfo> slots;
    std::vector<int> free_slots;               // a stack: the lowest ids are handed out first
    std::vector<int> live_list;                // slots of admitted sentences not known to have ended, in admission order
    std::vector<std::pair<int, uint64_t>> cancels;    // (slot, admission seq) accepted by cancel, for the next call built
    std::vector<int> row_of;                   // by slot: row in the call being built (scratch of build_call)
    std::deque<Call *> free_q, inflight;
    std::deque<Done *> done_q;
    int64_t next_call = 0;
    uint64_t next_seq = 0;
    int unfinished = 0;                        // submitted sentences whose ended record has not been made yet
    bool stop = false;
    std::string async_error;
    std::thread th_drive, th_complete;
    b2_tts_server_stats st = {};
};

namespace {

int server_fail(b2_tts_server *s, const char *what) {
    std::lock_guard<std::mutex> lk(s->mu);
    if (s->async_error.empty()) s->async_error = std::string(what) + ": " + g_last_error;
    s->stop = true;
    s->cv_submit.notify_all(); s->cv_drive.notify_all(); s->cv_complete.notify_all(); s->cv_poll.notify_all();
    return 1;
}

// everything of one engine call, enqueued without a host synchronisation
int enqueue_call(b2_tts_server *s, Call *b) {
    b2_ctx *c = s->ctx;
    cudaStream_t st = s->s_c;
    const int n = b->n, na = b->n_adm;
    if (na > 0) {
        const int L = b->L;
        B2_CUDA_OK(cudaMemcpyAsync(s->d_ids, b->h_ids, (size_t)na * L * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        B2_CUDA_OK(cudaMemcpyAsync(s->d_len, b->h_len, (size_t)na * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        B2_CUDA_OK(cudaMemcpyAsync(s->d_adm, b->h_adm, (size_t)3 * na * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        B2_CUDA_OK(cudaMemcpyAsync(s->d_spk, b->h_spk, (size_t)na * SPK * sizeof(float), cudaMemcpyHostToDevice, st));
        if (b2_enc_forward(s->enc, s->d_ids, b->h_len, na, L, s->d_enc, st)) return 1;
        if (b2_dec_start(s->dec, s->d_adm, s->d_enc, s->d_len, s->d_spk, na, L, st)) return 1;
        k_tts_admit<<<na, 128, 0, st>>>(s->d_adm, na, s->d_idx, s->d_ends, s->d_minlen, s->d_maxlen, s->d_live, c->pre_pool);
        B2_LAUNCH_OK("k_tts_admit");
    }
    const int nc = b->n_can;
    if (nc > 0) {
        B2_CUDA_OK(cudaMemcpyAsync(s->d_can, b->h_can, (size_t)2 * nc * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        k_tts_cancel<<<cdiv(nc, 128), 128, 0, st>>>(s->d_can, nc, s->d_live, s->d_mark);
        B2_LAUNCH_OK("k_tts_cancel");
    }
    const int nb = b->nb;
    B2_CUDA_OK(cudaMemcpyAsync(s->d_rows, b->h_rows, (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    k_tts_rows<<<cdiv(nb, 128), 128, 0, st>>>(s->d_rows, n, nb, s->d_live, c->max_sessions, s->d_dslots, s->d_tslots);
    B2_LAUNCH_OK("k_tts_rows");
    if (b2_dec_steps(s->dec, s->d_dslots, n, NSTEPS, nullptr, s->seed, s->d_mel, s->d_prob, st)) return 1;
    k_tts_stop<<<cdiv(n, 128), 128, 0, st>>>(s->d_dslots, s->d_prob, n, s->threshold, s->d_idx, s->d_ends, s->d_minlen, s->d_maxlen, s->d_live,
                                             nc > 0 ? s->d_mark : nullptr, b->d_tri);
    B2_LAUNCH_OK("k_tts_stop");
    if (s->use_graphs && !c->prof.on) {
        auto it = b->graphs.find(nb);
        if (it == b->graphs.end()) {
            cudaGraphExec_t ge = nullptr;
            int nk = 0;
            if (capture_tail_graph(c, s->d_tslots, s->d_mel, nb, NFRAMES, s->law, true, b->d_out, st, &ge, &nk)) return 1;
            it = b->graphs.emplace(nb, std::make_pair(ge, nk)).first;
            std::lock_guard<std::mutex> lk(s->mu);
            s->st.graphs_built++;
        }
        B2_CUDA_OK(cudaGraphLaunch(it->second.first, st));
        count_launch(it->second.second);
        std::lock_guard<std::mutex> lk(s->mu);
        s->st.graph_launches++;
    } else {
        if (tail_device(c, s->d_tslots, s->d_mel, nb, NFRAMES, s->law, true, b->d_out, nullptr, st, false, true)) return 1;
    }
    B2_CUDA_OK(cudaEventRecord(b->ev_c, st));
    B2_CUDA_OK(cudaStreamWaitEvent(s->s_out, b->ev_c, 0));
    B2_CUDA_OK(cudaMemcpyAsync(b->h_out, b->d_out, (size_t)n * NBYTES, cudaMemcpyDeviceToHost, s->s_out));
    B2_CUDA_OK(cudaMemcpyAsync(b->h_tri, b->d_tri, (size_t)3 * n * sizeof(int32_t), cudaMemcpyDeviceToHost, s->s_out));
    B2_CUDA_OK(cudaEventRecord(b->ev_out, s->s_out));
    return 0;
}

// under the mutex: the next call's admission round and row list.  -> false when there is nothing to run.
bool build_call(b2_tts_server *s, Call *b) {
    // sentences the completer has seen end leave the row list
    size_t w = 0;
    for (int sl : s->live_list) if (s->slots[(size_t)sl].live) s->live_list[w++] = sl;
    s->live_list.resize(w);
    const int64_t call = s->next_call;
    int na = 0, L = 0;
    while (na < (int)s->pending.size() && na < s->adm_cap && na < (int)s->free_slots.size() && (int)s->live_list.size() + na < s->cap) {
        L = std::max(L, (int)s->pending[(size_t)na].ids.size());
        na++;
    }
    if (na == 0 && s->live_list.empty()) return false;
    // maxlen / minlen of B200Frontend.length_bounds: from the padded token length L of this round; maxlen capped so that the KV cache
    // (max_steps positions) holds the sentence up to its end 2 steps later, rounded up to a whole call
    const int cap_steps = std::max(1, s->max_steps - NSTEPS - 4);
    const int minlen = (int)((double)L * (double)s->minlenratio / 2.0);
    const int maxlen = std::min((int)((double)L * (double)s->maxlenratio / 2.0), cap_steps);
    for (int i = 0; i < na; i++) {
        Pending &p = s->pending.front();
        const int sl = s->free_slots.back();
        s->free_slots.pop_back();
        const int len = (int)p.ids.size();
        memcpy(b->h_ids + (size_t)i * L, p.ids.data(), (size_t)len * sizeof(int32_t));
        memset(b->h_ids + (size_t)i * L + len, 0, (size_t)(L - len) * sizeof(int32_t));
        memcpy(b->h_spk + (size_t)i * SPK, p.spk.data(), SPK * sizeof(float));
        b->h_len[i] = len;
        b->h_adm[i] = sl; b->h_adm[na + i] = minlen; b->h_adm[2 * na + i] = maxlen;
        SlotInfo &si = s->slots[(size_t)sl];
        si.tag = p.tag; si.t_submit = p.t_submit; si.admit_call = call; si.live = true;
        si.seq = s->next_seq++; si.cancelled = false;
        s->live_list.push_back(sl);
        s->pending.pop_front();
    }
    const int n = (int)s->live_list.size();
    b->call = call; b->n = n; b->n_adm = na; b->L = L;
    b->nb = s->use_graphs ? bucket_of(n, s->cap) : n;
    b->row_slot.assign(s->live_list.begin(), s->live_list.end());
    b->row_info.resize((size_t)n);
    for (int i = 0; i < n; i++) {
        b->h_rows[i] = s->live_list[(size_t)i];
        b->row_info[(size_t)i] = s->slots[(size_t)s->live_list[(size_t)i]];
    }
    // every accepted cancel enters this call, if its slot still holds the admission it was accepted for: the completer may have freed the
    // slot on a natural end since, and this round may have given it to a newcomer
    int nc = 0;
    if (!s->cancels.empty()) {
        for (int i = 0; i < n; i++) s->row_of[(size_t)s->live_list[(size_t)i]] = i;
        for (const auto &q : s->cancels) {
            const SlotInfo &si = s->slots[(size_t)q.first];
            if (!si.live || si.seq != q.second) continue;
            b->h_can[2 * nc] = s->row_of[(size_t)q.first]; b->h_can[2 * nc + 1] = q.first;
            nc++;
        }
        s->cancels.clear();
    }
    b->n_can = nc;
    s->next_call++;
    if (na) { s->st.admission_rounds++; s->st.admitted += (uint64_t)na; }
    s->st.rows += (uint64_t)n; s->st.padded_rows += (uint64_t)(b->nb - n);
    s->st.max_rows = std::max<uint64_t>(s->st.max_rows, (uint64_t)n);
    return true;
}

void driver_main(b2_tts_server *s) {
    pthread_setname_np(pthread_self(), "b2-tts-driver");
    cudaSetDevice(s->ctx->device);
    std::unique_lock<std::mutex> lk(s->mu);
    while (true) {
        s->cv_drive.wait(lk, [&] {
            if (s->stop) return true;
            if (s->free_q.empty()) return false;
            for (int sl : s->live_list) if (s->slots[(size_t)sl].live) return true;
            return !s->pending.empty() && !s->free_slots.empty();
        });
        if (s->stop) break;
        Call *b = s->free_q.front();
        if (!build_call(s, b)) continue;
        s->free_q.pop_front();
        s->cv_submit.notify_all();
        lk.unlock();
        const int rc = enqueue_call(s, b);
        lk.lock();
        if (rc) {
            lk.unlock();
            server_fail(s, "engine call");
            lk.lock();
            break;
        }
        s->inflight.push_back(b);
        s->cv_complete.notify_all();
    }
}

void completer_main(b2_tts_server *s) {
    pthread_setname_np(pthread_self(), "b2-tts-complete");
    cudaSetDevice(s->ctx->device);
    std::unique_lock<std::mutex> lk(s->mu);
    while (true) {
        s->cv_complete.wait(lk, [&] { return !s->inflight.empty() || s->stop; });
        if (s->stop) break;
        Call *b = s->inflight.front();
        lk.unlock();
        const cudaError_t e = cudaEventSynchronize(b->ev_out);
        const int64_t t_done = now_ns();
        if (e != cudaSuccess) {
            set_error("cudaEventSynchronize: %s", cudaGetErrorString(e));
            server_fail(s, "engine call completion");
            return;
        }
        Done *d = new Done();
        size_t total = 0;
        int nlive = 0;
        for (int i = 0; i < b->n; i++) {
            const int32_t *t = b->h_tri + 3 * i;
            if (t[1] > t[0] || t[2]) {
                const SlotInfo &si = b->row_info[(size_t)i];
                b2_tts_chunk r = {};
                r.tag = si.tag; r.call = b->call; r.admit_call = si.admit_call; r.t_submit_ns = si.t_submit; r.t_done_ns = t_done;
                r.nbytes = t[1] - t[0]; r.ended = t[2]; r.g711_offset = (int64_t)total;
                total += (size_t)r.nbytes;
                d->recs.push_back(r);
            }
            nlive += (t[1] > t[0] || t[2] == 1) ? 1 : 0;          // a cancelled row (ended 2) took no step
        }
        d->bytes.resize(total);
        size_t k = 0;
        for (int i = 0; i < b->n; i++) {
            const int32_t *t = b->h_tri + 3 * i;
            if (!(t[1] > t[0] || t[2])) continue;
            memcpy(d->bytes.data() + d->recs[k].g711_offset, b->h_out + (size_t)i * NBYTES + t[0], (size_t)(t[1] - t[0]));
            k++;
        }
        lk.lock();
        int nended = 0;
        for (int i = 0, j = 0; i < b->n; i++) {
            const int32_t *t = b->h_tri + 3 * i;
            if (!(t[1] > t[0] || t[2])) continue;
            if (d->recs[(size_t)j++].ended) {
                const int sl = b->row_slot[(size_t)i];
                s->slots[(size_t)sl].live = false;
                s->free_slots.push_back(sl);
                nended++;
            }
        }
        std::sort(s->free_slots.begin(), s->free_slots.end(), std::greater<int>());
        s->unfinished -= nended;
        s->st.ended += (uint64_t)nended; s->st.calls++; s->st.live_rows += (uint64_t)nlive;
        s->inflight.pop_front();
        s->free_q.push_back(b);
        s->done_q.push_back(d);
        s->cv_drive.notify_all(); s->cv_submit.notify_all(); s->cv_poll.notify_all();
    }
}

}  // namespace

extern "C" {

b2_tts_server *b2_tts_server_create(b2_ctx *c, b2_enc *enc, b2_dec *dec, int law, int depth, int use_graphs, float threshold, float minlenratio,
                                    float maxlenratio, uint64_t seed) {
    if (!c || !c->finalized) { set_error("b2_tts_server_create: the context has no finalized weights"); return nullptr; }
    if (!c->has_postnet) { set_error("b2_tts_server_create: the context has no post-net weights"); return nullptr; }
    if (!enc || !dec) { set_error("b2_tts_server_create: null encoder or decoder handle"); return nullptr; }
    if (law != B2_LAW_ULAW && law != B2_LAW_ALAW) { set_error("b2_tts_server_create: bad law %d", law); return nullptr; }
    if (depth < 1 || depth > 4) { set_error("b2_tts_server_create: depth must be 1..4"); return nullptr; }
    if (!(threshold == threshold) || !(minlenratio >= 0.0f) || !(maxlenratio >= 0.0f)) { set_error("b2_tts_server_create: bad stop-rule parameters"); return nullptr; }
    int dec_sessions = 0, max_steps = 0, max_enc = 0, max_tokens = 0, enc_len = 0, vocab = 0;
    dec_limits(dec, &dec_sessions, &max_steps, &max_enc);
    enc_limits(enc, &max_tokens, &enc_len, &vocab);
    if (max_steps < NSTEPS + 8) { set_error("b2_tts_server_create: the decoder's max_steps=%d is too small for %d steps per call", max_steps, NSTEPS); return nullptr; }
    if (cudaSetDevice(c->device) != cudaSuccess) { set_error("cudaSetDevice failed"); return nullptr; }
    b2_tts_server *s = new b2_tts_server();
    s->ctx = c; s->enc = enc; s->dec = dec; s->law = law; s->depth = depth; s->use_graphs = use_graphs ? 1 : 0;
    s->threshold = threshold; s->minlenratio = minlenratio; s->maxlenratio = maxlenratio; s->seed = seed;
    s->nslots = std::min(c->max_sessions, dec_sessions);
    s->cap = std::min(s->nslots, c->max_windows / (NFRAMES / 8));           // one tail pass per call
    s->adm_cap = std::min(s->cap, 512);
    s->max_len = std::min(enc_len, max_enc); s->max_tokens = max_tokens; s->vocab = vocab; s->max_steps = max_steps;
    s->st.capacity = (uint64_t)s->cap; s->st.depth = (uint64_t)depth;
    if (s->cap < 1) { set_error("b2_tts_server_create: the context's workspace holds no session of %d frames", NFRAMES); delete s; return nullptr; }
    s->slots.resize((size_t)s->nslots);
    s->row_of.resize((size_t)s->nslots);
    for (int i = s->nslots - 1; i >= 0; i--) s->free_slots.push_back(i);
    const size_t S = (size_t)s->nslots, R = (size_t)s->cap, A = (size_t)s->adm_cap, Lm = (size_t)s->max_len;
    auto dal = [](auto **p, size_t n) { return cudaMalloc((void **)p, n * sizeof(**p)) == cudaSuccess; };
    auto hal = [](auto **p, size_t n) { return cudaHostAlloc((void **)p, n * sizeof(**p), cudaHostAllocDefault) == cudaSuccess; };
    bool ok = cudaStreamCreateWithFlags(&s->s_c, cudaStreamNonBlocking) == cudaSuccess &&
              cudaStreamCreateWithFlags(&s->s_out, cudaStreamNonBlocking) == cudaSuccess &&
              dal(&s->d_idx, S) && dal(&s->d_ends, S) && dal(&s->d_minlen, S) && dal(&s->d_maxlen, S) && dal(&s->d_live, S) &&
              dal(&s->d_ids, A * Lm) && dal(&s->d_len, A) && dal(&s->d_adm, 3 * A) && dal(&s->d_rows, R) && dal(&s->d_dslots, R) &&
              dal(&s->d_tslots, R) && dal(&s->d_spk, A * SPK) && dal(&s->d_enc, A * Lm * 768) && dal(&s->d_mel, R * NFRAMES * NMEL) &&
              dal(&s->d_prob, R * NSTEPS * 2) && dal(&s->d_can, 2 * R) && dal(&s->d_mark, R) &&
              cudaMemset(s->d_live, 0, S * sizeof(int32_t)) == cudaSuccess && cudaMemset(s->d_mark, 0, R * sizeof(int32_t)) == cudaSuccess &&
              cudaMemset(s->d_mel, 0, R * NFRAMES * NMEL * sizeof(float)) == cudaSuccess;
    for (int i = 0; ok && i < depth; i++) {
        Call *b = new Call();
        s->calls_pool.push_back(b);
        ok = hal(&b->h_ids, A * Lm) && hal(&b->h_len, A) && hal(&b->h_adm, 3 * A) && hal(&b->h_rows, R) && hal(&b->h_tri, 3 * R) && hal(&b->h_can, 2 * R) &&
             hal(&b->h_spk, A * SPK) && hal(&b->h_out, R * NBYTES) && dal(&b->d_out, R * NBYTES) && dal(&b->d_tri, 3 * R) &&
             cudaEventCreateWithFlags(&b->ev_c, cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&b->ev_out, cudaEventDisableTiming) == cudaSuccess;
    }
    if (!ok) {
        set_error("b2_tts_server_create: allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
        b2_tts_server_destroy(s);
        return nullptr;
    }
    if (warm_tail(c, s->d_tslots, s->d_mel, std::min(8, s->cap), NFRAMES, law, true, s->calls_pool[0]->d_out, s->s_c)) {
        b2_tts_server_destroy(s);
        return nullptr;
    }
    for (Call *b : s->calls_pool) s->free_q.push_back(b);
    s->th_drive = std::thread(driver_main, s);
    s->th_complete = std::thread(completer_main, s);
    return s;
}

void b2_tts_server_destroy(b2_tts_server *s) {
    if (!s) return;
    {
        std::lock_guard<std::mutex> lk(s->mu);
        s->stop = true;
    }
    s->cv_submit.notify_all(); s->cv_drive.notify_all(); s->cv_complete.notify_all(); s->cv_poll.notify_all();
    if (s->th_drive.joinable()) s->th_drive.join();
    if (s->th_complete.joinable()) s->th_complete.join();
    cudaSetDevice(s->ctx->device);
    if (s->s_c) cudaStreamSynchronize(s->s_c);
    if (s->s_out) cudaStreamSynchronize(s->s_out);
    for (Call *b : s->calls_pool) {
        for (auto &kv : b->graphs) cudaGraphExecDestroy(kv.second.first);
        for (void *p : {(void *)b->h_ids, (void *)b->h_len, (void *)b->h_adm, (void *)b->h_rows, (void *)b->h_tri, (void *)b->h_can, (void *)b->h_spk,
                        (void *)b->h_out})
            if (p) cudaFreeHost(p);
        if (b->d_out) cudaFree(b->d_out);
        if (b->d_tri) cudaFree(b->d_tri);
        if (b->ev_c) cudaEventDestroy(b->ev_c);
        if (b->ev_out) cudaEventDestroy(b->ev_out);
        delete b;
    }
    for (void *p : {(void *)s->d_idx, (void *)s->d_ends, (void *)s->d_minlen, (void *)s->d_maxlen, (void *)s->d_live, (void *)s->d_ids, (void *)s->d_len,
                    (void *)s->d_adm, (void *)s->d_rows, (void *)s->d_dslots, (void *)s->d_tslots, (void *)s->d_spk, (void *)s->d_enc, (void *)s->d_mel,
                    (void *)s->d_prob, (void *)s->d_can, (void *)s->d_mark})
        if (p) cudaFree(p);
    for (Done *d : s->done_q) delete d;
    if (s->s_c) cudaStreamDestroy(s->s_c);
    if (s->s_out) cudaStreamDestroy(s->s_out);
    delete s;
}

int b2_tts_server_submit(b2_tts_server *s, const int32_t *h_ids, const int32_t *h_lens, int n, const float *h_speakers, const uint64_t *tags) {
    if (!s) return set_error("null server");
    const int64_t t_now = now_ns();
    if (n < 0 || (n > 0 && (!h_ids || !h_lens || !h_speakers || !tags))) return set_error("b2_tts_server_submit: null pointer or n < 0");
    const int lim = std::min(s->max_len, s->max_tokens);
    std::vector<Pending> ps((size_t)n);
    size_t off = 0;
    for (int j = 0; j < n; j++) {
        const int len = h_lens[j];
        if (len < 1) return set_error("b2_tts_server_submit: sentence %d has %d tokens (at least one is needed)", j, len);
        if (len > lim)
            return set_error("b2_tts_server_submit: sentence %d has %d tokens, more than the encoder's max_len / max_tokens or the decoder's max_enc_len allow "
                             "(%d)", j, len, lim);
        for (int i = 0; i < len; i++)
            if (h_ids[off + i] < 0 || h_ids[off + i] >= s->vocab)
                return set_error("b2_tts_server_submit: sentence %d: token id %d at position %d is outside [0, %d)", j, h_ids[off + i], i, s->vocab);
        Pending &p = ps[(size_t)j];
        p.ids.assign(h_ids + off, h_ids + off + len);
        p.spk.assign(h_speakers + (size_t)j * SPK, h_speakers + (size_t)(j + 1) * SPK);
        p.tag = tags[j]; p.t_submit = t_now;
        off += (size_t)len;
    }
    int done = 0;
    while (done < n) {
        std::unique_lock<std::mutex> lk(s->mu);
        // back-pressure: every slot holds a sentence that has not ended (slots come back when the completer sees a sentence end, whether or
        // not anybody polls).  Sentences that fit are enqueued together, so that they can share one admission round.
        if (!s->cv_submit.wait_for(lk, std::chrono::seconds(20), [&] { return s->stop || s->unfinished < s->nslots; }))
            return set_error("b2_tts_server_submit: no slot became free in 20 s (%d of %d sentences of this call were accepted)", done, n);
        if (s->stop) return set_error("b2_tts_server_submit: the server has stopped%s%s", s->async_error.empty() ? "" : ": ", s->async_error.c_str());
        const int k = std::min(n - done, s->nslots - s->unfinished);
        for (int j = 0; j < k; j++) s->pending.push_back(std::move(ps[(size_t)(done + j)]));
        s->unfinished += k;
        s->st.submitted += (uint64_t)k;
        done += k;
        s->cv_drive.notify_all();
    }
    return 0;
}

int b2_tts_server_cancel(b2_tts_server *s, const uint64_t *tags, int n) {
    if (!s) return -set_error("null server");
    if (n < 0 || (n > 0 && !tags)) return -set_error("b2_tts_server_cancel: null tags or n < 0");
    const int64_t t_now = now_ns();
    std::vector<uint64_t> want(tags, tags + n);
    std::sort(want.begin(), want.end());
    auto wanted = [&](uint64_t t) { return std::binary_search(want.begin(), want.end(), t); };
    std::lock_guard<std::mutex> lk(s->mu);
    if (s->stop) return -set_error("b2_tts_server_cancel: the server has stopped%s%s", s->async_error.empty() ? "" : ": ", s->async_error.c_str());
    // pending sentences were never admitted: they leave the queue and get their last record now
    Done *d = nullptr;
    size_t w = 0;
    for (size_t i = 0; i < s->pending.size(); i++) {
        Pending &p = s->pending[i];
        if (!wanted(p.tag)) {
            if (w != i) s->pending[w] = std::move(p);
            w++;
            continue;
        }
        if (!d) d = new Done();
        b2_tts_chunk r = {};
        r.tag = p.tag; r.call = -1; r.admit_call = -1; r.t_submit_ns = p.t_submit; r.t_done_ns = t_now; r.ended = 2;
        d->recs.push_back(r);
    }
    s->pending.resize(w);
    const int npend = d ? (int)d->recs.size() : 0;
    if (d) {
        s->done_q.push_back(d);
        s->unfinished -= npend;
        s->st.ended += (uint64_t)npend;
    }
    // admitted sentences: the device decides in the next call (build_call), since a call in flight may end them first
    int nlive = 0;
    for (int sl : s->live_list) {
        SlotInfo &si = s->slots[(size_t)sl];
        if (!si.live || si.cancelled || !wanted(si.tag)) continue;
        si.cancelled = true;
        s->cancels.emplace_back(sl, si.seq);
        nlive++;
    }
    if (npend) { s->cv_submit.notify_all(); s->cv_poll.notify_all(); }
    if (nlive) s->cv_drive.notify_all();
    return npend + nlive;
}

int b2_tts_server_poll(b2_tts_server *s, b2_tts_chunk *out, int max_out, uint8_t *h_g711, size_t g711_capacity, int timeout_ms) {
    if (!s) return -set_error("null server");
    if (!out || max_out < 1) return -set_error("b2_tts_server_poll: bad arguments");
    std::unique_lock<std::mutex> lk(s->mu);
    if (s->done_q.empty() && timeout_ms != 0) {
        auto pred = [&] { return !s->done_q.empty() || s->stop; };
        if (timeout_ms < 0) s->cv_poll.wait(lk, pred);
        else s->cv_poll.wait_for(lk, std::chrono::milliseconds(timeout_ms), pred);
    }
    if (s->done_q.empty() && !s->async_error.empty()) return -set_error("b2_tts_server_poll: %s", s->async_error.c_str());
    int cnt = 0;
    size_t off = 0;
    while (cnt < max_out && !s->done_q.empty()) {
        Done *d = s->done_q.front();
        while (cnt < max_out && d->polled < d->recs.size()) {
            const b2_tts_chunk &r = d->recs[d->polled];
            if (h_g711 && off + (size_t)r.nbytes > g711_capacity) return cnt;
            out[cnt] = r;
            out[cnt].g711_offset = h_g711 ? (int64_t)off : -1;
            if (h_g711) { memcpy(h_g711 + off, d->bytes.data() + r.g711_offset, (size_t)r.nbytes); off += (size_t)r.nbytes; }
            d->polled++; cnt++;
        }
        if (d->polled < d->recs.size()) break;
        s->done_q.pop_front();
        delete d;
    }
    return cnt;
}

int b2_tts_server_flush(b2_tts_server *s, int timeout_ms) {
    if (!s) return set_error("null server");
    std::unique_lock<std::mutex> lk(s->mu);
    auto idle = [&] { return s->stop || (s->unfinished == 0 && s->inflight.empty()); };
    const auto deadline = std::chrono::steady_clock::now() + std::chrono::milliseconds(timeout_ms < 0 ? 3600000 : timeout_ms);
    while (!idle()) {
        if (s->cv_poll.wait_until(lk, deadline) == std::cv_status::timeout && !idle()) return set_error("b2_tts_server_flush: timed out");
    }
    if (!s->async_error.empty()) return set_error("b2_tts_server_flush: %s", s->async_error.c_str());
    return 0;
}

int b2_tts_server_get_stats(b2_tts_server *s, b2_tts_server_stats *out) {
    if (!s || !out) return set_error("b2_tts_server_get_stats: null pointer");
    std::lock_guard<std::mutex> lk(s->mu);
    *out = s->st;
    return 0;
}

}  // extern "C"
