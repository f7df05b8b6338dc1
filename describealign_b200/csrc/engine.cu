// Batch engine: many pairs in flight on one GPU, driven by ONE scheduler thread inside the library.
//
// The reference's batch mode is a sequential loop over file pairs (describealign.py:1077).  Here a pair
// occupies a slot (a dab_pair: device buffers + its own CUDA stream) and walks through
//     upload + features + stage A  ->  copy of what the host fit needs  ->  [host fit, caller's code]
//     ->  stage B  ->  copy of the final path  ->  [caller reads the result]  ->  slot released
// Every device stage is enqueued in one go (no host round trip inside a stage: the counts that size
// later kernels stay on the device, common.cuh DC_*), and the scheduler only looks at events: it never
// blocks on a stream, so one thread keeps any number of slots moving and the caller needs no thread
// per pair.  The caller's side is a queue: dab_engine_next hands out pairs whose stage A or stage B
// results have landed in the slot's page-locked host buffers.
#include <string.h>
#include <time.h>

#include <chrono>
#include <condition_variable>
#include <deque>
#include <thread>

#include "common.cuh"

namespace {

enum SlotState { S_FREE = 0, S_A_RUN, S_A_COPY, S_A_HOST, S_B_PENDING, S_B_RUN, S_B_COPY, S_B_HOST };

struct PinBuf {
  void *p = nullptr;
  size_t cap = 0;
  int ensure(size_t bytes) {
    if (bytes <= cap && p) return 0;
    if (p) dab_free_pinned(p);
    cap = bytes + bytes / 4 + 4096;
    p = dab_alloc_pinned(cap);
    if (!p) { cap = 0; return 1; }
    return 0;
  }
  void release() { if (p) dab_free_pinned(p); p = nullptr; cap = 0; }
};

struct Slot {
  dab_pair *pair = nullptr;
  SlotState state = S_FREE;
  dab_job job = {};
  cudaEvent_t ev = nullptr;          // recorded after the last command of the phase in flight
  int status = DAB_OK;
  std::string err;
  int attempts = 0;
  PinBuf path_x, path_y, feat[2][3], rows, cor;   // cor: the line clusters of the stage-B input
  dab_stage_b_in b_in = {};
  int64_t host_us = 0;               // scheduler time spent enqueueing this pair's work
  int64_t t_submit_us = 0, t_a_done_us = 0, t_b_submit_us = 0;
};

int64_t now_us() {
  return std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

}  // namespace

struct dab_engine {
  dab_ctx *ctx = nullptr;
  std::vector<Slot> slots;
  std::thread thread;
  std::mutex mu;
  std::condition_variable cv_out;      // results for the caller
  std::condition_variable cv_in;       // work for the scheduler
  std::deque<dab_job> pending;         // submitted, waiting for a free slot
  std::deque<int> b_requests;          // slots whose stage-B input has arrived
  std::deque<int> releases;
  std::deque<dab_event> out;           // finished stage A / stage B results
  bool stop = false;
  int in_flight = 0;                   // slots not free + pending jobs
  int64_t loops = 0, idle_sleeps = 0;
};

namespace {

void fail_slot(dab_engine *e, Slot &s, int slot, int rc, int kind) {
  s.status = rc;
  s.err = dab_last_error(e->ctx);
  dab_event evt;
  memset(&evt, 0, sizeof evt);
  evt.kind = kind; evt.tag = s.job.tag; evt.slot = slot; evt.status = rc;
  s.state = kind == DAB_EVENT_STAGE_A ? S_A_HOST : S_B_HOST;
  std::lock_guard<std::mutex> g(e->mu);
  e->out.push_back(evt);
  e->cv_out.notify_all();
}

#define ENG_TRY(expr, kind)                                   \
  do {                                                        \
    int rc__ = (expr);                                        \
    if (rc__ != DAB_OK) { fail_slot(e, s, slot, rc__, kind); return; } \
  } while (0)

#define ENG_CUDA(call, kind)                                  \
  do {                                                        \
    cudaError_t ce__ = (call);                                \
    if (ce__ != cudaSuccess) {                                \
      dab_set_err(e->ctx, std::string(#call) + " failed: " + cudaGetErrorString(ce__)); \
      fail_slot(e, s, slot, DAB_E_CUDA, kind);                \
      return;                                                 \
    }                                                         \
  } while (0)

void enqueue_a(dab_engine *e, int slot, bool upload) {
  Slot &s = e->slots[slot];
  dab_pair *pr = s.pair;
  StreamScope scope__(pr->stream);
  const int64_t t0 = now_us();
  if (upload) {
    for (int t = 0; t < 2; ++t)
      ENG_TRY(dab_pair_set_pcm(pr, t, s.job.pcm[t], s.job.samples[t], s.job.channels[t], s.job.format, s.job.on_device),
              DAB_EVENT_STAGE_A);
  }
  ENG_TRY(dab_check_stage_a_inputs(pr, "stage_a"), DAB_EVENT_STAGE_A);
  ENG_TRY(dab_enqueue_stage_a(pr, nullptr, 0, INT64_MAX, true), DAB_EVENT_STAGE_A);
  ENG_CUDA(cudaEventRecord(s.ev, pr->stream), DAB_EVENT_STAGE_A);
  s.state = S_A_RUN;
  s.host_us += now_us() - t0;
}

// stage A has run: counts are on the host.  Grow-and-retry on overflow, else bring back the pass-1 path and
// the three feature vectors per track the host fit reads (describealign.py:735).
void after_a(dab_engine *e, int slot) {
  Slot &s = e->slots[slot];
  dab_pair *pr = s.pair;
  StreamScope scope__(pr->stream);
  const int64_t t0 = now_us();
  const int rc = dab_collect_stage_a(pr, nullptr, true);
  if (rc == DAB_E_CAPACITY && ++s.attempts < DAB_STAGE_A_ATTEMPTS) { enqueue_a(e, slot, false); return; }
  ENG_TRY(rc, DAB_EVENT_STAGE_A);
  cudaStream_t st = pr->stream;
  const size_t pb = sizeof(int32_t) * (size_t)pr->n_path1;
  if (s.path_x.ensure(pb + 4) || s.path_y.ensure(pb + 4)) { dab_set_err(e->ctx, "out of page-locked memory"); fail_slot(e, s, slot, DAB_E_CUDA, DAB_EVENT_STAGE_A); return; }
  if (pb) {
    ENG_CUDA(cudaMemcpyAsync(s.path_x.p, pr->path1_x.p, pb, cudaMemcpyDeviceToHost, st), DAB_EVENT_STAGE_A);
    ENG_CUDA(cudaMemcpyAsync(s.path_y.p, pr->path1_y.p, pb, cudaMemcpyDeviceToHost, st), DAB_EVENT_STAGE_A);
  }
  for (int t = 0; t < 2; ++t) {
    Track &tk = pr->trk[t];
    const void *src[3] = {tk.energy.p, tk.zc.p, tk.b0.p};
    const int64_t len[3] = {tk.Le, tk.L, tk.L};
    for (int f = 0; f < 3; ++f) {
      const size_t fb = sizeof(float) * (size_t)len[f];
      if (s.feat[t][f].ensure(fb + 4)) { dab_set_err(e->ctx, "out of page-locked memory"); fail_slot(e, s, slot, DAB_E_CUDA, DAB_EVENT_STAGE_A); return; }
      if (fb) ENG_CUDA(cudaMemcpyAsync(s.feat[t][f].p, src[f], fb, cudaMemcpyDeviceToHost, st), DAB_EVENT_STAGE_A);
    }
  }
  ENG_CUDA(cudaEventRecord(s.ev, st), DAB_EVENT_STAGE_A);
  s.state = S_A_COPY;
  s.host_us += now_us() - t0;
}

void publish_a(dab_engine *e, int slot) {
  Slot &s = e->slots[slot];
  dab_pair *pr = s.pair;
  dab_event evt;
  memset(&evt, 0, sizeof evt);
  evt.kind = DAB_EVENT_STAGE_A; evt.tag = s.job.tag; evt.slot = slot; evt.status = DAB_OK;
  evt.n_path1 = pr->n_path1;
  evt.path_x = reinterpret_cast<const int32_t *>(s.path_x.p);
  evt.path_y = reinterpret_cast<const int32_t *>(s.path_y.p);
  for (int t = 0; t < 2; ++t) {
    Track &tk = pr->trk[t];
    const int64_t len[3] = {tk.Le, tk.L, tk.L};
    for (int f = 0; f < 3; ++f) {
      evt.features[t][f] = reinterpret_cast<const float *>(s.feat[t][f].p);
      evt.feature_len[t][f] = len[f];
    }
  }
  evt.stats = pr->stats;
  s.state = S_A_HOST;
  s.t_a_done_us = now_us();
  std::lock_guard<std::mutex> g(e->mu);
  e->out.push_back(evt);
  e->cv_out.notify_all();
}

void enqueue_b(dab_engine *e, int slot) {
  Slot &s = e->slots[slot];
  dab_pair *pr = s.pair;
  StreamScope scope__(pr->stream);
  const int64_t t0 = now_us();
  const dab_stage_b_in &b = s.b_in;
  ENG_TRY(dab_enqueue_stage_b_clusters(pr, b.gain, b.audio_std, b.n_audio, b.n_video, reinterpret_cast<const dab_cluster *>(s.cor.p),
                                       b.n_clusters, 0, INT64_MAX, true, "dab_pair_stage_b_clusters"), DAB_EVENT_STAGE_B);
  ENG_CUDA(cudaEventRecord(s.ev, pr->stream), DAB_EVENT_STAGE_B);
  s.state = S_B_RUN;
  s.host_us += now_us() - t0;
}

void after_b(dab_engine *e, int slot) {
  Slot &s = e->slots[slot];
  dab_pair *pr = s.pair;
  const int64_t t0 = now_us();
  ENG_TRY(dab_collect_stage_b(pr, true), DAB_EVENT_STAGE_B);
  const size_t rb = sizeof(double) * 5 * (size_t)pr->n_path2;
  if (s.rows.ensure(rb + 8)) { dab_set_err(e->ctx, "out of page-locked memory"); fail_slot(e, s, slot, DAB_E_CUDA, DAB_EVENT_STAGE_B); return; }
  if (rb) ENG_CUDA(cudaMemcpyAsync(s.rows.p, pr->path2.p, rb, cudaMemcpyDeviceToHost, pr->stream), DAB_EVENT_STAGE_B);
  ENG_CUDA(cudaEventRecord(s.ev, pr->stream), DAB_EVENT_STAGE_B);
  s.state = S_B_COPY;
  s.host_us += now_us() - t0;
}

void publish_b(dab_engine *e, int slot) {
  Slot &s = e->slots[slot];
  dab_pair *pr = s.pair;
  dab_event evt;
  memset(&evt, 0, sizeof evt);
  evt.kind = DAB_EVENT_STAGE_B; evt.tag = s.job.tag; evt.slot = slot; evt.status = DAB_OK;
  evt.n_path1 = pr->n_path1;
  evt.n_path2 = pr->n_path2;
  evt.rows = reinterpret_cast<const double *>(s.rows.p);
  evt.stats = pr->stats;
  dab_pair_get_timings(pr, evt.timings_ms);      // the stream is idle: no waiting
  evt.timings_ms[10] = (float)(s.host_us / 1e3);  // scheduler time spent on this pair (all enqueues)
  evt.timings_ms[11] = (float)((s.t_a_done_us - s.t_submit_us) / 1e3);   // submit -> stage A results on the host
  evt.timings_ms[12] = (float)((now_us() - s.t_b_submit_us) / 1e3);      // stage B input -> final path on the host
  evt.timings_ms[13] = 0.f;
  s.state = S_B_HOST;
  std::lock_guard<std::mutex> g(e->mu);
  e->out.push_back(evt);
  e->cv_out.notify_all();
}

void scheduler(dab_engine *e) {
  cudaSetDevice(e->ctx->device);
  const int n = (int)e->slots.size();
  for (;;) {
    bool progressed = false;
    // ---- take requests ----
    {
      std::unique_lock<std::mutex> lk(e->mu);
      if (e->stop) return;
      while (!e->releases.empty()) {
        const int slot = e->releases.front();
        e->releases.pop_front();
        Slot &s = e->slots[slot];
        if (s.state == S_A_HOST || s.state == S_B_HOST) { s.state = S_FREE; --e->in_flight; progressed = true; }
      }
      while (!e->b_requests.empty()) {
        const int slot = e->b_requests.front();
        e->b_requests.pop_front();
        if (e->slots[slot].state == S_A_HOST) { e->slots[slot].state = S_B_PENDING; progressed = true; }
      }
      for (int k = 0; k < n && !e->pending.empty(); ++k) {
        Slot &s = e->slots[k];
        if (s.state != S_FREE) continue;
        s.job = e->pending.front();
        e->pending.pop_front();
        s.status = DAB_OK; s.attempts = 0; s.host_us = 0; s.err.clear();
        s.t_submit_us = now_us();
        s.state = S_A_RUN;     // claimed; the work is enqueued below, outside the lock
        s.attempts = -1;       // marker: not enqueued yet
        progressed = true;
      }
      if (e->in_flight == 0 && e->pending.empty()) {
        e->cv_in.wait_for(lk, std::chrono::milliseconds(50));
        continue;
      }
    }
    // ---- move every slot as far as it can go ----
    for (int k = 0; k < n; ++k) {
      Slot &s = e->slots[k];
      switch (s.state) {
        case S_A_RUN:
          if (s.attempts < 0) { s.attempts = 0; enqueue_a(e, k, true); progressed = true; break; }
          if (cudaEventQuery(s.ev) == cudaSuccess) { after_a(e, k); progressed = true; }
          break;
        case S_A_COPY:
          if (cudaEventQuery(s.ev) == cudaSuccess) { publish_a(e, k); progressed = true; }
          break;
        case S_B_PENDING:
          enqueue_b(e, k);
          progressed = true;
          break;
        case S_B_RUN:
          if (cudaEventQuery(s.ev) == cudaSuccess) { after_b(e, k); progressed = true; }
          break;
        case S_B_COPY:
          if (cudaEventQuery(s.ev) == cudaSuccess) { publish_b(e, k); progressed = true; }
          break;
        default:
          break;
      }
    }
    cudaGetLastError();    // cudaErrorNotReady from the queries is not sticky, but keep the slate clean
    ++e->loops;
    if (!progressed) {
      ++e->idle_sleeps;
      struct timespec ts = {0, 20000};
      nanosleep(&ts, nullptr);
    }
  }
}

}  // namespace

extern "C" {

int dab_engine_create(dab_ctx *ctx, int32_t slots, dab_engine **out) {
  if (!ctx || !out || slots < 1 || slots > 1024) return DAB_E_ARG;
  *out = nullptr;
  DAB_CUDA(cudaSetDevice(ctx->device));
  dab_engine *e = new (std::nothrow) dab_engine();
  if (!e) return DAB_E_CUDA;
  e->ctx = ctx;
  e->slots.resize((size_t)slots);
  for (auto &s : e->slots) {
    int rc = dab_pair_create(ctx, &s.pair);
    if (rc == DAB_OK && cudaEventCreateWithFlags(&s.ev, cudaEventDisableTiming) != cudaSuccess) rc = DAB_E_CUDA;
    if (rc != DAB_OK) {
      for (auto &t : e->slots) { if (t.pair) dab_pair_destroy(t.pair); if (t.ev) cudaEventDestroy(t.ev); }
      delete e;
      return rc;
    }
  }
  e->thread = std::thread(scheduler, e);
  *out = e;
  return DAB_OK;
}

void dab_engine_destroy(dab_engine *e) {
  if (!e) return;
  {
    std::lock_guard<std::mutex> g(e->mu);
    e->stop = true;
  }
  e->cv_in.notify_all();
  if (e->thread.joinable()) e->thread.join();
  cudaSetDevice(e->ctx->device);
  for (auto &s : e->slots) {
    if (s.pair) dab_pair_destroy(s.pair);      // waits for the slot's stream
    if (s.ev) cudaEventDestroy(s.ev);
    s.path_x.release(); s.path_y.release(); s.rows.release(); s.cor.release();
    for (int t = 0; t < 2; ++t)
      for (int f = 0; f < 3; ++f) s.feat[t][f].release();
  }
  delete e;
}

int dab_engine_submit(dab_engine *e, const dab_job *job) {
  if (!e || !job || !job->pcm[0] || !job->pcm[1]) return DAB_E_ARG;
  for (int t = 0; t < 2; ++t)
    if (job->samples[t] < 0 || (job->channels[t] != 1 && job->channels[t] != 2)) return DAB_E_ARG;
  if (job->format != DAB_PCM_S16 && job->format != DAB_PCM_F16) return DAB_E_ARG;
  {
    std::lock_guard<std::mutex> g(e->mu);
    e->pending.push_back(*job);
    ++e->in_flight;
  }
  e->cv_in.notify_all();
  return DAB_OK;
}

int dab_engine_next(dab_engine *e, dab_event *out, int32_t timeout_ms) {
  if (!e || !out) return DAB_E_ARG;
  std::unique_lock<std::mutex> lk(e->mu);
  if (e->out.empty()) {
    if (timeout_ms == 0) return DAB_E_TIMEOUT;
    if (timeout_ms < 0) e->cv_out.wait(lk, [&] { return !e->out.empty(); });
    else if (!e->cv_out.wait_for(lk, std::chrono::milliseconds(timeout_ms), [&] { return !e->out.empty(); })) return DAB_E_TIMEOUT;
  }
  *out = e->out.front();
  e->out.pop_front();
  return DAB_OK;
}

int dab_engine_submit_b(dab_engine *e, int32_t slot, const dab_stage_b_in *in) {
  if (!e || !in || slot < 0 || slot >= (int)e->slots.size() || in->n_clusters < 0 || (in->n_clusters > 0 && !in->clusters))
    return DAB_E_ARG;
  Slot &s = e->slots[(size_t)slot];
  // the slot is in S_A_HOST: it belongs to the caller until this request is queued
  if (s.cor.ensure(sizeof(dab_cluster) * (size_t)(in->n_clusters + 1))) return DAB_E_CUDA;
  if (in->n_clusters) memcpy(s.cor.p, in->clusters, sizeof(dab_cluster) * (size_t)in->n_clusters);
  s.b_in = *in;
  s.b_in.clusters = nullptr;
  s.t_b_submit_us = now_us();
  {
    std::lock_guard<std::mutex> g(e->mu);
    e->b_requests.push_back(slot);
  }
  e->cv_in.notify_all();
  return DAB_OK;
}

int dab_engine_release(dab_engine *e, int32_t slot) {
  if (!e || slot < 0 || slot >= (int)e->slots.size()) return DAB_E_ARG;
  {
    std::lock_guard<std::mutex> g(e->mu);
    e->releases.push_back(slot);
  }
  e->cv_in.notify_all();
  return DAB_OK;
}

const char *dab_engine_slot_error(dab_engine *e, int32_t slot) {
  if (!e || slot < 0 || slot >= (int)e->slots.size()) return "";
  return e->slots[(size_t)slot].err.c_str();
}

void *dab_engine_slot_pair(dab_engine *e, int32_t slot) {
  if (!e || slot < 0 || slot >= (int)e->slots.size()) return nullptr;
  return e->slots[(size_t)slot].pair;
}

void dab_engine_counters(dab_engine *e, int64_t out[4]) {
  if (!e || !out) return;
  out[0] = e->loops; out[1] = e->idle_sleeps; out[2] = 0; out[3] = 0;
}

}  // extern "C"
