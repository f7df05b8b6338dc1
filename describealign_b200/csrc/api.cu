// C ABI of describealign_b200 (include/describealign_b200.h).
#include <string.h>

#include <new>

#include <time.h>

#include "common.cuh"

static std::string g_create_err;

int dab_g_wait_mode = 0;

cudaError_t dab_wait_stream(cudaStream_t st) {
  if (dab_g_wait_mode != 2) return cudaStreamSynchronize(st);
  // poll and sleep: 20 us at first, backing off to 400 us (a DP kernel runs for tens of milliseconds)
  long ns = 20000;
  for (;;) {
    const cudaError_t e = cudaStreamQuery(st);
    if (e != cudaErrorNotReady) return e;
    struct timespec ts = {0, ns};
    nanosleep(&ts, nullptr);
    if (ns < 400000) ns += ns / 2;
  }
}

// ---- pinned host memory pool ----------------------------------------------------------------
// Results (features, paths) are copied device -> host asynchronously; with pageable destinations
// the runtime stages every copy through its own bounce buffer and serialises the pairs in flight.
// Buffers are handed out in power-of-two size classes and go back to a free list, so a batch in
// steady state performs no cudaHostAlloc / cudaFreeHost (both synchronise the device).
#include <map>
#include <mutex>
namespace {
std::mutex g_pin_mu;
std::multimap<size_t, void *> g_pin_free;        // size class -> buffer
std::map<void *, size_t> g_pin_live;             // buffer -> size class
size_t pin_class(size_t bytes) {
  size_t c = 4096;
  while (c < bytes) c <<= 1;
  return c;
}
}  // namespace

#include <atomic>
#include <chrono>
static std::atomic<int64_t> g_alloc_calls{0}, g_alloc_us{0}, g_pin_calls{0}, g_pin_us{0};
static inline int64_t now_us() {
  return std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// Device buffers only ever grow, and are freed with cudaFreeAsync on the pair's stream: a plain
// cudaFree would wait for every other pair's kernels (the frontier DPs run for ~0.1 s).
thread_local cudaStream_t dab_t_stream = nullptr;
int64_t ApiTimer::now() { return now_us(); }

int dab_ensure(dab_ctx *ctx, DevBuf &b, size_t bytes) {
  if (bytes <= b.cap && b.p) return DAB_OK;
  const int64_t t0 = now_us();
  cudaStream_t st = dab_t_stream;
  if (b.p) {
    if (b.pooled && st) DAB_CUDA(cudaFreeAsync(b.p, st));
    else DAB_CUDA(cudaFree(b.p));
    b.p = nullptr;
    b.cap = 0;
  }
  size_t want = bytes + bytes / 4 + 256;   // head-room so that similar pairs reuse the buffer
  if (st) {
    DAB_CUDA(cudaMallocAsync(&b.p, want, st));
    b.pooled = true;
  } else {
    DAB_CUDA(cudaMalloc(&b.p, want));
    b.pooled = false;
  }
  b.cap = want;
  g_alloc_calls += 1;
  g_alloc_us += now_us() - t0;
  return DAB_OK;
}

static void free_buf(DevBuf &b) {
  if (b.p) cudaFree(b.p);     // also valid for stream-ordered allocations (synchronises)
  b.p = nullptr;
  b.cap = 0;
}

static void free_prep(Prep &p) {
  for (DevBuf *b : {&p.ms, &p.nrm, &p.pack, &p.code, &p.nq_flag, &p.nq_list}) free_buf(*b);
}

static void free_video_side(VideoSide &vs) {
  free_prep(vs.prep);
  for (DevBuf *b : {&vs.tbl_start, &vs.tbl_items, &vs.v_rec}) free_buf(*b);
}

extern "C" {

int dab_abi_version(void) { return DAB_ABI_VERSION; }

void *dab_alloc_pinned(size_t bytes) {
  const size_t c = pin_class(bytes ? bytes : 1);
  {
    std::lock_guard<std::mutex> g(g_pin_mu);
    auto it = g_pin_free.find(c);
    if (it != g_pin_free.end()) {
      void *p = it->second;
      g_pin_free.erase(it);
      g_pin_live[p] = c;
      return p;
    }
  }
  void *p = nullptr;
  const int64_t t0 = now_us();
  if (cudaHostAlloc(&p, c, cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  g_pin_calls += 1;
  g_pin_us += now_us() - t0;
  std::lock_guard<std::mutex> g(g_pin_mu);
  g_pin_live[p] = c;
  return p;
}

void dab_free_pinned(void *p) {
  if (!p) return;
  std::lock_guard<std::mutex> g(g_pin_mu);
  auto it = g_pin_live.find(p);
  if (it == g_pin_live.end()) return;
  g_pin_free.emplace(it->second, p);
  g_pin_live.erase(it);
}

void dab_host_copy(void *dst, const void *src, size_t bytes) {
  if (dst && src && bytes) memcpy(dst, src, bytes);
}

void dab_alloc_stats(int64_t out[4]) {
  if (!out) return;
  out[0] = g_alloc_calls; out[1] = g_alloc_us; out[2] = g_pin_calls; out[3] = g_pin_us;
}

void dab_trim_pinned(void) {
  std::multimap<size_t, void *> drop;
  {
    std::lock_guard<std::mutex> g(g_pin_mu);
    drop.swap(g_pin_free);
  }
  for (auto &kv : drop) cudaFreeHost(kv.second);
}

int dab_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

const char *dab_last_error(const dab_ctx *ctx) {
  static thread_local std::string copy;
  if (!ctx) return g_create_err.c_str();
  dab_ctx *c = const_cast<dab_ctx *>(ctx);
  std::lock_guard<std::mutex> g(c->err_mu);
  copy = c->err;
  return copy.c_str();
}

int dab_set_host_wait(int device, int mode) {
  if (mode < 0 || mode > 2) return -DAB_E_ARG;
  if (device >= 0 && cudaSetDevice(device) != cudaSuccess) { cudaGetLastError(); return -DAB_E_CUDA; }
  unsigned flags = 0;
  if (cudaGetDeviceFlags(&flags) != cudaSuccess) { cudaGetLastError(); return -DAB_E_CUDA; }
  flags = (flags & ~(unsigned)cudaDeviceScheduleMask) |
          (mode == 1 ? (unsigned)cudaDeviceScheduleBlockingSync : (unsigned)cudaDeviceScheduleAuto);
  if (cudaSetDeviceFlags(flags) != cudaSuccess) { cudaGetLastError(); return -DAB_E_CUDA; }
  if (cudaGetDeviceFlags(&flags) != cudaSuccess) { cudaGetLastError(); return -DAB_E_CUDA; }
  dab_g_wait_mode = mode;
  return (int)(flags & (unsigned)cudaDeviceScheduleMask);
}

int dab_create(int device, dab_ctx **out) {
  if (!out) return DAB_E_ARG;
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    g_create_err = std::string("no CUDA device available (describealign_b200 has no CPU fallback): ") +
                   (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    return DAB_E_CUDA;
  }
  if (device < 0) {
    if (cudaGetDevice(&device) != cudaSuccess) device = 0;
  }
  if (device >= n) { g_create_err = "device index out of range"; return DAB_E_ARG; }
  e = cudaSetDevice(device);
  if (e != cudaSuccess) { g_create_err = cudaGetErrorString(e); return DAB_E_CUDA; }
  dab_ctx *ctx = new (std::nothrow) dab_ctx();
  if (!ctx) return DAB_E_CUDA;
  ctx->device = device;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) ctx->sm_count = prop.multiProcessorCount;
  cudaMemPool_t pool = nullptr;
  if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess && pool) {
    uint64_t keep = UINT64_MAX;   // freed buffers stay in the pool instead of going back to the OS
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
  }
  cudaGetLastError();
  *out = ctx;
  return DAB_OK;
}

void dab_destroy(dab_ctx *ctx) { delete ctx; }

int dab_set_option(dab_ctx *ctx, const char *name, int64_t value) {
  if (!ctx || !name) return DAB_E_ARG;
  if (strcmp(name, "dp2_impl") == 0 && (value == 0 || value == 2)) { ctx->opt_dp2_impl = (int)value; return DAB_OK; }
  dab_set_err(ctx, std::string("dab_set_option: unknown option ") + name);
  return DAB_E_ARG;
}

int64_t dab_launch_count(const dab_ctx *ctx) { return ctx ? ctx->launches.load() : 0; }

}  // extern "C"

// A few words from device memory into the pair's mapped host block, written by a one-warp kernel.
// A cudaMemcpyAsync of 4 bytes would do the same, but copies share the copy engines' queues with
// the bulk PCM uploads of the other pairs in flight, and a 4-byte read-back was seen to wait
// 100-200 ms behind them (profiles/r1_v10_timeline_e2e.txt); a store over PCIe does not queue.
__global__ void readback_kernel(uint32_t *dst, const uint32_t *src, int n_words) {
  if ((int)threadIdx.x < n_words) dst[threadIdx.x] = src[threadIdx.x];
  __threadfence_system();
}

cudaError_t dab_readback(dab_pair *pr, void *host_dst, const void *dev_src, size_t bytes) {
  const ptrdiff_t off = reinterpret_cast<const char *>(host_dst) - reinterpret_cast<const char *>(pr->h_counters);
  if (off < 0 || off + (ptrdiff_t)bytes > (ptrdiff_t)(sizeof(int64_t) * 32) || bytes % 4 != 0 || bytes > 128)
    return cudaErrorInvalidValue;
  pr->ctx->launches++;
  readback_kernel<<<1, 32, 0, pr->stream>>>(reinterpret_cast<uint32_t *>(reinterpret_cast<char *>(pr->d_counters_map) + off),
                                            reinterpret_cast<const uint32_t *>(dev_src), (int)(bytes / 4));
  return cudaGetLastError();
}

// a stage-A step enqueued on the pair's stream, waited for and collected; run again while the collect reports an
// overflow (it has grown the buffer)
template <typename Enqueue, typename Collect>
static int grow_and_retry(dab_pair *pr, Enqueue enqueue, Collect collect) {
  dab_ctx *ctx = pr->ctx;
  int rc = DAB_E_CAPACITY;
  for (int attempt = 0; attempt < DAB_STAGE_A_ATTEMPTS && rc == DAB_E_CAPACITY; ++attempt) {
    DAB_TRY(enqueue());
    DAB_CUDA(dab_wait_stream(pr->stream));
    rc = collect();
  }
  return rc;
}

// stage A against a shared index, or against the pair's own video side (ix null)
static int stage_a_sync(dab_pair *pr, const dab_index *ix, int64_t row_lo, int64_t row_hi, bool with_dp) {
  return grow_and_retry(pr, [&] { return dab_enqueue_stage_a(pr, ix, row_lo, row_hi, with_dp); },
                        [&] { return dab_collect_stage_a(pr, ix, with_dp); });
}

extern "C" {

void dab_pair_destroy(dab_pair *pr);

int dab_pair_create(dab_ctx *ctx, dab_pair **out) {
  if (!ctx || !out) return DAB_E_ARG;
  *out = nullptr;
  DAB_CUDA(cudaSetDevice(ctx->device));
  dab_pair *pr = new (std::nothrow) dab_pair();
  if (!pr) return DAB_E_CUDA;
  pr->ctx = ctx;
  // on a failure half-way the pair built so far is torn down again (dab_pair_destroy copes with missing parts)
  cudaError_t e = cudaStreamCreateWithFlags(&pr->stream, cudaStreamNonBlocking);
  for (int k = 0; k < 32 && e == cudaSuccess; ++k) e = cudaEventCreate(&pr->ev[k]);
  // mapped: kernels write the counts the host waits for straight into this block (dab_readback)
  if (e == cudaSuccess)
    e = cudaHostAlloc(reinterpret_cast<void **>(&pr->h_counters), sizeof(int64_t) * 32, cudaHostAllocMapped | cudaHostAllocPortable);
  if (e == cudaSuccess) {
    memset(pr->h_counters, 0, sizeof(int64_t) * 32);
    e = cudaHostGetDevicePointer(reinterpret_cast<void **>(&pr->d_counters_map), pr->h_counters, 0);
  }
  if (e != cudaSuccess) {
    dab_set_err(ctx, std::string("dab_pair_create: ") + cudaGetErrorString(e));
    dab_pair_destroy(pr);
    return DAB_E_CUDA;
  }
  *out = pr;
  return DAB_OK;
}

void dab_pair_destroy(dab_pair *pr) {
  if (!pr) return;
  cudaSetDevice(pr->ctx->device);
  if (pr->stream) dab_wait_stream(pr->stream);
  for (int t = 0; t < 2; ++t) {
    Track &k = pr->trk[t];
    DevBuf *bs[] = {&k.pcm, &k.feat_ticket, &k.feat_mid, &k.energy, &k.zc, &k.b0, &k.b1, &k.b2, &k.gate};
    for (DevBuf *b : bs) free_buf(*b);
  }
  free_prep(pr->prep_a);
  free_video_side(pr->video);
  DevBuf *bs[] = {&pr->scan_tmp, &pr->tbl_sb, &pr->tbl_ent, &pr->clusters, &pr->refine_partial, &pr->maxes, &pr->row_count, &pr->row_off, &pr->row_stash, &pr->gate_rec, &pr->gate_best, &pr->gate_big,
                  &pr->cand_tmp, &pr->cand_s, &pr->cand_i, &pr->cand_q, &pr->keep_flag, &pr->keep_off, &pr->pt_i,
                  &pr->pt_s, &pr->pt_q, &pr->counters, &pr->tree1, &pr->back1, &pr->dpres,
                  &pr->path1_x, &pr->path1_y, &pr->a_scaled, &pr->v_scaled, &pr->corridors,
                  &pr->row2_count, &pr->row2_off, &pr->p2_i, &pr->p2_c, &pr->p2_rank, &pr->p2_j, &pr->p2_q,
                  &pr->tree2, &pr->cache2, &pr->cluster_best2, &pr->back2, &pr->path2,
                  &pr->p2_k, &pr->pm2, &pr->tb_up, &pr->tb_mark};
  for (DevBuf *b : bs) free_buf(*b);
  for (int k = 0; k < 32; ++k)
    if (pr->ev[k]) cudaEventDestroy(pr->ev[k]);
  if (pr->h_counters) cudaFreeHost(pr->h_counters);
  if (pr->stream) cudaStreamDestroy(pr->stream);
  delete pr;
}

int dab_pair_sync(dab_pair *pr) {
  if (!pr) return DAB_E_ARG;
  dab_ctx *ctx = pr->ctx;
  DAB_CUDA(dab_wait_stream(pr->stream));
  return DAB_OK;
}

void *dab_pair_stream(dab_pair *pr) { return pr ? reinterpret_cast<void *>(pr->stream) : nullptr; }

int dab_pair_set_pcm(dab_pair *pr, int track, const void *pcm, int64_t samples, int channels, int format,
                     int on_device) {
  if (!pr) return DAB_E_ARG;
  dab_ctx *ctx = pr->ctx;
  StreamScope scope__(pr->stream);
  if (track == DAB_TRACK_VIDEO) pr->api_us[0] = 0;     // a new pair starts with its video track
  ApiTimer timer__(&pr->api_us[0]);
  if (track < 0 || track > 1 || !pcm || samples < 0 || (channels != 1 && channels != 2) ||
      (format != DAB_PCM_S16 && format != DAB_PCM_F16)) {
    dab_set_err(ctx, "dab_pair_set_pcm: invalid argument");
    return DAB_E_ARG;
  }
  DAB_CUDA(cudaSetDevice(ctx->device));
  Track &tk = pr->trk[track];
  tk.S = samples;
  tk.ch = channels;
  tk.have_features = false;
  tk.have_gate = false;
  if (pr->points_side == &pr->video) pr->points_side = nullptr;
  if (track == DAB_TRACK_VIDEO) { pr->api_us[1] = pr->api_us[2] = pr->api_us[3] = 0; }
  const void *d_pcm = pcm;
  cudaEvent_t e0 = pr->ev[2 * track], e1 = pr->ev[2 * track + 1];
  if (!on_device) {
    const size_t bytes = sizeof(int16_t) * (size_t)samples * (size_t)channels;
    DAB_TRY(dab_ensure(ctx, tk.pcm, bytes + 16));
    DAB_CUDA(cudaMemcpyAsync(tk.pcm.p, pcm, bytes, cudaMemcpyHostToDevice, pr->stream));
    d_pcm = tk.pcm.p;
  }
  DAB_CUDA(cudaEventRecord(e0, pr->stream));
  DAB_TRY(dab_run_features(pr, track, d_pcm, format));
  DAB_CUDA(cudaEventRecord(e1, pr->stream));
  pr->ev_used[track] = true;
  return DAB_OK;
}

int dab_pair_set_features(dab_pair *pr, int track, const float *energy, int64_t n_energy, const float *zc,
                          const float *band0, const float *band1, const double *band2, int64_t n) {
  if (!pr) return DAB_E_ARG;
  dab_ctx *ctx = pr->ctx;
  StreamScope scope__(pr->stream);
  ApiTimer timer__(&pr->api_us[0]);
  if (track < 0 || track > 1 || !energy || !zc || !band0 || !band1 || !band2 || n < 0 ||
      (n_energy != n && n_energy != n + 1)) {
    dab_set_err(ctx, "dab_pair_set_features: invalid argument (len(energy) must be n or n + 1)");
    return DAB_E_ARG;
  }
  DAB_CUDA(cudaSetDevice(ctx->device));
  Track &tk = pr->trk[track];
  tk.L = n;
  tk.Le = n_energy;
  tk.S = n * 210;
  tk.have_gate = false;
  if (pr->points_side == &pr->video) pr->points_side = nullptr;
  DAB_TRY(dab_ensure(ctx, tk.energy, sizeof(float) * (size_t)(n_energy + 1)));
  DAB_TRY(dab_ensure(ctx, tk.zc, sizeof(float) * (size_t)(n + 1)));
  DAB_TRY(dab_ensure(ctx, tk.b0, sizeof(float) * (size_t)(n + 1)));
  DAB_TRY(dab_ensure(ctx, tk.b1, sizeof(float) * (size_t)(n + 1)));
  DAB_TRY(dab_ensure(ctx, tk.b2, sizeof(double) * (size_t)(n + 1)));
  cudaStream_t st = pr->stream;
  DAB_CUDA(cudaMemcpyAsync(tk.energy.p, energy, sizeof(float) * (size_t)n_energy, cudaMemcpyHostToDevice, st));
  DAB_CUDA(cudaMemcpyAsync(tk.zc.p, zc, sizeof(float) * (size_t)n, cudaMemcpyHostToDevice, st));
  DAB_CUDA(cudaMemcpyAsync(tk.b0.p, band0, sizeof(float) * (size_t)n, cudaMemcpyHostToDevice, st));
  DAB_CUDA(cudaMemcpyAsync(tk.b1.p, band1, sizeof(float) * (size_t)n, cudaMemcpyHostToDevice, st));
  DAB_CUDA(cudaMemcpyAsync(tk.b2.p, band2, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, st));
  DAB_CUDA(dab_wait_stream(st));   // the caller may free its arrays right after (describealign.py:1107)
  tk.have_features = true;
  return DAB_OK;
}

int dab_pair_set_gate_energy(dab_pair *pr, int track, const float *energy, int64_t n_energy) {
  if (!pr) return DAB_E_ARG;
  dab_ctx *ctx = pr->ctx;
  StreamScope scope__(pr->stream);
  if (track < 0 || track > 1 || !energy) { dab_set_err(ctx, "dab_pair_set_gate_energy: invalid argument"); return DAB_E_ARG; }
  Track &tk = pr->trk[track];
  if (!tk.have_features) { dab_set_err(ctx, "dab_pair_set_gate_energy: set the track's features first"); return DAB_E_STATE; }
  if (n_energy != tk.Le) { dab_set_err(ctx, "dab_pair_set_gate_energy: the energy argument must have the length of features[0]"); return DAB_E_ARG; }
  DAB_CUDA(cudaSetDevice(ctx->device));
  DAB_TRY(dab_ensure(ctx, tk.gate, sizeof(float) * (size_t)(n_energy + 1)));
  DAB_CUDA(cudaMemcpyAsync(tk.gate.p, energy, sizeof(float) * (size_t)n_energy, cudaMemcpyHostToDevice, pr->stream));
  DAB_CUDA(dab_wait_stream(pr->stream));
  tk.have_gate = true;
  if (pr->points_side == &pr->video) pr->points_side = nullptr;
  return DAB_OK;
}

int dab_pair_feature_lens(dab_pair *pr, int track, int64_t lens[5]) {
  if (!pr || track < 0 || track > 1 || !lens) return DAB_E_ARG;
  Track &tk = pr->trk[track];
  if (!tk.have_features) { dab_set_err(pr->ctx, "no features computed for this track"); return DAB_E_STATE; }
  lens[0] = tk.Le;
  lens[1] = lens[2] = lens[3] = lens[4] = tk.L;
  return DAB_OK;
}

int dab_pair_get_features(dab_pair *pr, int track, float *energy, float *zc, float *band0, float *band1,
                          double *band2) {
  if (!pr || track < 0 || track > 1) return DAB_E_ARG;
  dab_ctx *ctx = pr->ctx;
  ApiTimer timer__(&pr->api_us[3]);
  Track &tk = pr->trk[track];
  if (!tk.have_features) { dab_set_err(ctx, "no features computed for this track"); return DAB_E_STATE; }
  DAB_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = pr->stream;
  if (energy && tk.Le > 0) DAB_CUDA(cudaMemcpyAsync(energy, tk.energy.p, sizeof(float) * (size_t)tk.Le, cudaMemcpyDeviceToHost, st));
  if (tk.L > 0) {
    if (zc) DAB_CUDA(cudaMemcpyAsync(zc, tk.zc.p, sizeof(float) * (size_t)tk.L, cudaMemcpyDeviceToHost, st));
    if (band0) DAB_CUDA(cudaMemcpyAsync(band0, tk.b0.p, sizeof(float) * (size_t)tk.L, cudaMemcpyDeviceToHost, st));
    if (band1) DAB_CUDA(cudaMemcpyAsync(band1, tk.b1.p, sizeof(float) * (size_t)tk.L, cudaMemcpyDeviceToHost, st));
    if (band2) DAB_CUDA(cudaMemcpyAsync(band2, tk.b2.p, sizeof(double) * (size_t)tk.L, cudaMemcpyDeviceToHost, st));
  }
  DAB_CUDA(dab_wait_stream(st));
  return DAB_OK;
}

int dab_pair_stage_a(dab_pair *pr, int64_t *n_points, int64_t *n_path) {
  if (!pr) return DAB_E_ARG;
  dab_ctx *ctx = pr->ctx;
  StreamScope scope__(pr->stream);
  ApiTimer timer__(&pr->api_us[1]);
  DAB_TRY(dab_check_stage_a_inputs(pr, "stage_a"));
  DAB_CUDA(cudaSetDevice(ctx->device));
  DAB_TRY(stage_a_sync(pr, nullptr, 0, INT64_MAX, true));
  if (n_points) *n_points = pr->n_points1;
  if (n_path) *n_path = pr->n_path1;
  return DAB_OK;
}

int dab_pair_get_path1(dab_pair *pr, int32_t *x_audio, int32_t *y_video) {
  if (!pr) return DAB_E_ARG;
  dab_ctx *ctx = pr->ctx;
  ApiTimer timer__(&pr->api_us[3]);
  DAB_CUDA(cudaSetDevice(ctx->device));
  const size_t bytes = sizeof(int32_t) * (size_t)pr->n_path1;
  if (bytes) {
    if (x_audio) DAB_CUDA(cudaMemcpyAsync(x_audio, pr->path1_x.p, bytes, cudaMemcpyDeviceToHost, pr->stream));
    if (y_video) DAB_CUDA(cudaMemcpyAsync(y_video, pr->path1_y.p, bytes, cudaMemcpyDeviceToHost, pr->stream));
  }
  DAB_CUDA(dab_wait_stream(pr->stream));
  return DAB_OK;
}

}  // extern "C"

namespace {
__global__ void ranks_to_frames_kernel(const int32_t *pt_s, const int32_t *v_sel, int64_t n, int32_t *out) {
  int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k < n) out[k] = v_sel[pt_s[k]];
}
}  // namespace

extern "C" {

static int export_points1(dab_pair *pr, int32_t *i_audio, int32_t *v_video, double *qual, int dst_on_device) {
  dab_ctx *ctx = pr->ctx;
  if (pr->points_side && pr->points_side != &pr->video) {
    dab_set_err(ctx, "export_points1: the points of stage_a_against are ranks into the index's hashed frames, not this pair's");
    return DAB_E_STATE;
  }
  StreamScope scope__(pr->stream);
  ApiTimer timer__(&pr->api_us[3]);
  DAB_CUDA(cudaSetDevice(ctx->device));
  const cudaMemcpyKind kind = dst_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
  const int64_t n = pr->n_points1;
  if (n > 0) {
    cudaStream_t st = pr->stream;
    if (i_audio) DAB_CUDA(cudaMemcpyAsync(i_audio, pr->pt_i.p, sizeof(int32_t) * (size_t)n, kind, st));
    if (qual) DAB_CUDA(cudaMemcpyAsync(qual, pr->pt_q.p, sizeof(double) * (size_t)n, kind, st));
    if (v_video) {
      DAB_TRY(dab_ensure(ctx, pr->cand_tmp, sizeof(int32_t) * (size_t)(n + 1)));
      ranks_to_frames_kernel<<<(unsigned)cdiv(n, 256), 256, 0, st>>>(pr->pt_s.as<int32_t>(),
                                                                      pr->video.prep.nq_list.as<int32_t>(), n,
                                                                      pr->cand_tmp.as<int32_t>());
      ctx->launches += 1;
      DAB_CUDA(cudaMemcpyAsync(v_video, pr->cand_tmp.p, sizeof(int32_t) * (size_t)n, kind, st));
    }
  }
  DAB_CUDA(dab_wait_stream(pr->stream));
  return DAB_OK;
}

int dab_pair_get_points1(dab_pair *pr, int32_t *i_audio, int32_t *v_video, double *qual) {
  if (!pr) return DAB_E_ARG;
  return export_points1(pr, i_audio, v_video, qual, 0);
}

int dab_pair_export_points1(dab_pair *pr, int32_t *i_audio, int32_t *v_video, double *qual, int dst_on_device) {
  if (!pr) return DAB_E_ARG;
  return export_points1(pr, i_audio, v_video, qual, dst_on_device);
}

static void index_destroy(dab_index *ix) {
  free_video_side(ix->side);
  free_buf(ix->counters);
  if (ix->ready) cudaEventDestroy(ix->ready);
  delete ix;
}

int dab_index_build(dab_pair *src, dab_index **out) {
  if (!src || !out) return DAB_E_ARG;
  *out = nullptr;
  dab_ctx *ctx = src->ctx;
  StreamScope scope__(src->stream);
  const Track &S = src->trk[DAB_TRACK_VIDEO];
  if (!S.have_features) { dab_set_err(ctx, "index_build: the pair's video track has no features"); return DAB_E_STATE; }
  if ((S.Le < S.L ? S.Le : S.L) < 2 * DAB_WIN) { dab_set_err(ctx, "index_build: track shorter than 82 frames"); return DAB_E_TOO_SHORT; }
  DAB_CUDA(cudaSetDevice(ctx->device));
  dab_index *ix = new (std::nothrow) dab_index();
  if (!ix) return DAB_E_CUDA;
  ix->ctx = ctx;
  int rc = DAB_OK;
  const cudaError_t e = cudaEventCreateWithFlags(&ix->ready, cudaEventDisableTiming);
  if (e != cudaSuccess) { dab_set_err(ctx, std::string("index_build: ") + cudaGetErrorString(e)); rc = DAB_E_CUDA; }
  if (rc == DAB_OK) {
    rc = grow_and_retry(src, [&] { return dab_enqueue_index(src, ix); }, [&] { return dab_collect_index(src, ix); });
    if (rc == DAB_E_CAPACITY) dab_set_err(ctx, "dab_index_build: the hash tables overflowed on every attempt");
  }
  if (rc != DAB_OK) {
    dab_wait_stream(src->stream);
    index_destroy(ix);
    return rc;
  }
  *out = ix;
  return DAB_OK;
}

int dab_index_free(dab_index *ix) {
  if (!ix) return DAB_OK;
  int idle = 0;
  if (!ix->users.compare_exchange_strong(idle, -1)) {
    dab_set_err(ix->ctx, "index_free: " + std::to_string(idle) + " stage_a_against call(s) still running against this index");
    return DAB_E_STATE;
  }
  cudaSetDevice(ix->ctx->device);
  index_destroy(ix);
  return DAB_OK;
}

int dab_index_info(const dab_index *ix, int64_t out[4]) {
  if (!ix || !out) return DAB_E_ARG;
  out[0] = ix->side.prep.L; out[1] = ix->side.n_vsel; out[2] = ix->side.n_entries; out[3] = ix->users.load();
  return DAB_OK;
}

int dab_pair_stage_a_against(dab_pair *pr, const dab_index *ix, int64_t *n_points, int64_t *n_path) {
  if (!pr || !ix) return DAB_E_ARG;
  dab_ctx *ctx = pr->ctx;
  StreamScope scope__(pr->stream);
  ApiTimer timer__(&pr->api_us[1]);
  if (ix->ctx->device != ctx->device) { dab_set_err(ctx, "stage_a_against: the index lives on another device"); return DAB_E_ARG; }
  const Track &A = pr->trk[DAB_TRACK_AUDIO];
  if (!A.have_features) { dab_set_err(ctx, "stage_a_against: features of the description track are required first"); return DAB_E_STATE; }
  if ((A.Le < A.L ? A.Le : A.L) < 2 * DAB_WIN) { dab_set_err(ctx, "stage_a_against: track shorter than 82 frames"); return DAB_E_TOO_SHORT; }
  int u = ix->users.load();
  do {
    if (u < 0) { dab_set_err(ctx, "stage_a_against: the index is being freed"); return DAB_E_STATE; }
  } while (!ix->users.compare_exchange_weak(u, u + 1));
  struct Release {
    const dab_index *ix;
    ~Release() { ix->users.fetch_sub(1); }
  } release__{ix};
  DAB_CUDA(cudaSetDevice(ctx->device));
  DAB_TRY(stage_a_sync(pr, ix, 0, INT64_MAX, true));
  if (n_points) *n_points = pr->n_points1;
  if (n_path) *n_path = pr->n_path1;
  return DAB_OK;
}

int dab_pair_stage_a_match(dab_pair *pr, int64_t row_lo, int64_t row_hi, int64_t *n_points) {
  if (!pr) return DAB_E_ARG;
  dab_ctx *ctx = pr->ctx;
  StreamScope scope__(pr->stream);
  ApiTimer timer__(&pr->api_us[1]);
  if (row_lo < 0 || row_hi < row_lo) { dab_set_err(ctx, "dab_pair_stage_a_match: invalid row range"); return DAB_E_ARG; }
  DAB_TRY(dab_check_stage_a_inputs(pr, "stage_a_match"));
  DAB_CUDA(cudaSetDevice(ctx->device));
  DAB_TRY(stage_a_sync(pr, nullptr, row_lo, row_hi, false));
  if (n_points) *n_points = pr->n_points1;
  return DAB_OK;
}

int dab_pair_import_points1(dab_pair *pr, const int32_t *i_audio, const int32_t *v_video, const double *qual,
                            int64_t n, int src_on_device) {
  if (!pr) return DAB_E_ARG;
  dab_ctx *ctx = pr->ctx;
  StreamScope scope__(pr->stream);
  if (n < 0 || (n > 0 && (!i_audio || !v_video || !qual))) { dab_set_err(ctx, "dab_pair_import_points1: invalid argument"); return DAB_E_ARG; }
  if (pr->points_side != &pr->video) { dab_set_err(ctx, "import_points1: run stage_a_match on this pair first (it builds the hashed-frame list)"); return DAB_E_STATE; }
  DAB_CUDA(cudaSetDevice(ctx->device));
  return dab_run_import_points1(pr, i_audio, v_video, qual, n, src_on_device);
}

int dab_pair_dp1(dab_pair *pr, int64_t *n_path) {
  if (!pr) return DAB_E_ARG;
  dab_ctx *ctx = pr->ctx;
  StreamScope scope__(pr->stream);
  ApiTimer timer__(&pr->api_us[1]);
  if (pr->points_side != &pr->video) { dab_set_err(ctx, "dp1: no match points (run stage_a_match / import_points1 first)"); return DAB_E_STATE; }
  DAB_CUDA(cudaSetDevice(ctx->device));
  DAB_TRY(dab_enqueue_stage_a_dp(pr));
  DAB_TRY(dab_enqueue_counts(pr));
  DAB_CUDA(dab_wait_stream(pr->stream));
  dab_collect_stage_a_dp(pr);
  if (n_path) *n_path = pr->n_path1;
  return DAB_OK;
}

// the end of every synchronous stage-B entry: wait for the enqueued stage and its counts, collect
static int finish_stage_b(dab_pair *pr, bool with_dp, int64_t *n_points, int64_t *n_path) {
  dab_ctx *ctx = pr->ctx;
  DAB_CUDA(dab_wait_stream(pr->stream));
  DAB_TRY(dab_collect_stage_b(pr, with_dp));
  if (n_points) *n_points = pr->n_points2;
  if (n_path) *n_path = pr->n_path2;
  return DAB_OK;
}

int dab_pair_stage_b(dab_pair *pr, const float *audio_scaled, int64_t n_audio, const float *video_scaled,
                     int64_t n_video, const dab_corridor *corridors, int32_t n_corridors, int32_t n_clusters,
                     int64_t *n_points, int64_t *n_path) {
  if (!pr) return DAB_E_ARG;
  dab_ctx *ctx = pr->ctx;
  StreamScope scope__(pr->stream);
  ApiTimer timer__(&pr->api_us[2]);
  if (!audio_scaled || !video_scaled || n_audio <= 0 || n_video <= 8 || n_corridors < 0 || n_clusters < 0 ||
      (n_corridors > 0 && !corridors)) {
    dab_set_err(ctx, "dab_pair_stage_b: invalid argument");
    return DAB_E_ARG;
  }
  for (int k = 0; k < n_corridors; ++k) {
    const dab_corridor &c = corridors[k];
    if (c.cluster < 0 || c.cluster >= n_clusters || c.lo < 0 || c.hi > n_audio ||
        (k > 0 && c.cluster <= corridors[k - 1].cluster)) {
      dab_set_err(ctx, "dab_pair_stage_b: corridors must be in ascending cluster order with rows inside the audio track");
      return DAB_E_ARG;
    }
    if (c.hi > c.lo) {
      // the line must stay inside the video feature array for every scored row (:898-899)
      const double j0 = c.slope * (double)c.lo + c.offset, j1 = c.slope * (double)(c.hi - 1) + c.offset;
      const double jmin = j0 < j1 ? j0 : j1, jmax = j0 < j1 ? j1 : j0;
      if (!(jmin >= 0.0) || !(jmax < (double)(n_video - 1))) {
        dab_set_err(ctx, "dab_pair_stage_b: corridor line leaves the video track");
        return DAB_E_ARG;
      }
    }
  }
  DAB_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = pr->stream;
  DAB_TRY(dab_ensure(ctx, pr->a_scaled, sizeof(float) * 3 * (size_t)n_audio));
  DAB_TRY(dab_ensure(ctx, pr->v_scaled, sizeof(float) * 3 * (size_t)n_video));
  DAB_CUDA(cudaMemcpyAsync(pr->a_scaled.p, audio_scaled, sizeof(float) * 3 * (size_t)n_audio, cudaMemcpyHostToDevice, st));
  DAB_CUDA(cudaMemcpyAsync(pr->v_scaled.p, video_scaled, sizeof(float) * 3 * (size_t)n_video, cudaMemcpyHostToDevice, st));
  DAB_TRY(dab_enqueue_column_maxes(pr, n_audio, n_video));
  DAB_TRY(dab_ensure(ctx, pr->corridors, sizeof(dab_corridor) * (size_t)(n_corridors + 1)));
  if (n_corridors > 0)
    DAB_CUDA(cudaMemcpyAsync(pr->corridors.p, corridors, sizeof(dab_corridor) * (size_t)n_corridors, cudaMemcpyHostToDevice, st));
  dab_set_stage_b_plan(pr, n_audio, n_video, std::vector<dab_corridor>(corridors, corridors + n_corridors), n_clusters, false);
  DAB_TRY(dab_enqueue_stage_b(pr, 0, INT64_MAX, true));
  return finish_stage_b(pr, true, n_points, n_path);   // (the caller's arrays have been consumed once it returns)
}

int dab_pair_stage_b_clusters(dab_pair *pr, const float gain[3], const float audio_std[3], int64_t n_audio,
                              int64_t n_video, const dab_cluster *clusters, int32_t n_clusters,
                              int64_t *n_points, int64_t *n_path) {
  if (!pr) return DAB_E_ARG;
  StreamScope scope__(pr->stream);
  ApiTimer timer__(&pr->api_us[2]);
  DAB_TRY(dab_enqueue_stage_b_clusters(pr, gain, audio_std, n_audio, n_video, clusters, n_clusters, 0, INT64_MAX, true,
                                       "dab_pair_stage_b_clusters"));
  return finish_stage_b(pr, true, n_points, n_path);
}

// ---- stage B in steps, for one very long pair split over several GPUs (SURVEY.md 8e) ----
int dab_pair_stage_b_score(dab_pair *pr, const float gain[3], const float audio_std[3], int64_t n_audio, int64_t n_video,
                           const dab_cluster *clusters, int32_t n_clusters, int64_t row_lo, int64_t row_hi,
                           int64_t *n_points, int64_t *first_point, int64_t *n_mine) {
  if (!pr) return DAB_E_ARG;
  StreamScope scope__(pr->stream);
  ApiTimer timer__(&pr->api_us[2]);
  DAB_TRY(dab_enqueue_stage_b_clusters(pr, gain, audio_std, n_audio, n_video, clusters, n_clusters, row_lo, row_hi, false,
                                       "dab_pair_stage_b_score"));
  DAB_TRY(finish_stage_b(pr, false, nullptr, nullptr));
  int64_t first = 0, count = 0;
  DAB_TRY(dab_row_range_points2(pr, row_lo, row_hi, &first, &count));
  if (n_points) *n_points = pr->n_points2;
  if (first_point) *first_point = first;
  if (n_mine) *n_mine = count;
  return DAB_OK;
}

int dab_pair_export_quals2(dab_pair *pr, double *q, int64_t first, int64_t count, int dst_on_device) {
  if (!pr) return DAB_E_ARG;
  dab_ctx *ctx = pr->ctx;
  if (first < 0 || count < 0 || first + count > pr->n_points2 || (count > 0 && !q)) {
    dab_set_err(ctx, "dab_pair_export_quals2: range outside the pair's points");
    return DAB_E_ARG;
  }
  DAB_CUDA(cudaSetDevice(ctx->device));
  if (count > 0)
    DAB_CUDA(cudaMemcpyAsync(q, pr->p2_q.as<double>() + first, sizeof(double) * (size_t)count,
                             dst_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, pr->stream));
  DAB_CUDA(dab_wait_stream(pr->stream));
  return DAB_OK;
}

int dab_pair_import_quals2(dab_pair *pr, const double *q_all, int64_t n, int src_on_device) {
  if (!pr) return DAB_E_ARG;
  dab_ctx *ctx = pr->ctx;
  StreamScope scope__(pr->stream);
  if (n != pr->n_points2 || (n > 0 && !q_all)) {
    dab_set_err(ctx, "dab_pair_import_quals2: one qual per pass-2 point of the pair is required");
    return DAB_E_ARG;
  }
  DAB_CUDA(cudaSetDevice(ctx->device));
  if (n == 0) return DAB_OK;
  const double *src = q_all;
  if (!src_on_device) {
    DAB_TRY(dab_ensure(ctx, pr->cand_q, sizeof(double) * (size_t)(n + 1)));
    DAB_CUDA(cudaMemcpyAsync(pr->cand_q.p, q_all, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, pr->stream));
    src = pr->cand_q.as<double>();
  }
  DAB_TRY(dab_enqueue_set_quals2(pr, src));
  DAB_CUDA(dab_wait_stream(pr->stream));
  return DAB_OK;
}

int dab_pair_dp2(dab_pair *pr, int64_t *n_path) {
  if (!pr) return DAB_E_ARG;
  dab_ctx *ctx = pr->ctx;
  StreamScope scope__(pr->stream);
  ApiTimer timer__(&pr->api_us[2]);
  DAB_CUDA(cudaSetDevice(ctx->device));
  DAB_TRY(dab_enqueue_stage_b_dp(pr));
  DAB_TRY(dab_enqueue_counts(pr));
  return finish_stage_b(pr, true, nullptr, n_path);
}

int dab_pair_get_corridors(dab_pair *pr, dab_corridor *out, int32_t cap, int32_t *n_corridors) {
  if (!pr || !n_corridors) return DAB_E_ARG;
  dab_ctx *ctx = pr->ctx;
  const int32_t n = (int32_t)pr->plan_b.cor.size();
  *n_corridors = n;
  if (!out || cap <= 0 || n == 0) return DAB_OK;
  const int32_t m = n < cap ? n : cap;
  DAB_CUDA(cudaSetDevice(ctx->device));
  DAB_CUDA(cudaMemcpyAsync(out, pr->corridors.p, sizeof(dab_corridor) * (size_t)m, cudaMemcpyDeviceToHost, pr->stream));
  DAB_CUDA(dab_wait_stream(pr->stream));
  return DAB_OK;
}

int dab_pair_get_path2(dab_pair *pr, double *rows) {
  if (!pr) return DAB_E_ARG;
  dab_ctx *ctx = pr->ctx;
  ApiTimer timer__(&pr->api_us[3]);
  DAB_CUDA(cudaSetDevice(ctx->device));
  if (rows && pr->n_path2 > 0)
    DAB_CUDA(cudaMemcpyAsync(rows, pr->path2.p, sizeof(double) * 5 * (size_t)pr->n_path2, cudaMemcpyDeviceToHost, pr->stream));
  DAB_CUDA(dab_wait_stream(pr->stream));
  return DAB_OK;
}

int dab_pair_get_points2(dab_pair *pr, int32_t *i_audio, double *j_video, int32_t *cluster, double *qual) {
  if (!pr) return DAB_E_ARG;
  dab_ctx *ctx = pr->ctx;
  ApiTimer timer__(&pr->api_us[3]);
  DAB_CUDA(cudaSetDevice(ctx->device));
  const size_t n = (size_t)pr->n_points2;
  cudaStream_t st = pr->stream;
  if (n > 0) {
    if (i_audio) DAB_CUDA(cudaMemcpyAsync(i_audio, pr->p2_i.p, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, st));
    if (j_video) DAB_CUDA(cudaMemcpyAsync(j_video, pr->p2_j.p, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
    if (cluster) DAB_CUDA(cudaMemcpyAsync(cluster, pr->p2_c.p, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, st));
    if (qual) DAB_CUDA(cudaMemcpyAsync(qual, pr->p2_q.p, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
  }
  DAB_CUDA(dab_wait_stream(st));
  return DAB_OK;
}

int dab_pair_get_stats(dab_pair *pr, dab_stats *out) {
  if (!pr || !out) return DAB_E_ARG;
  *out = pr->stats;
  return DAB_OK;
}

int dab_pair_get_timings(dab_pair *pr, float ms[16]) {
  if (!pr || !ms) return DAB_E_ARG;
  dab_ctx *ctx = pr->ctx;
  DAB_CUDA(cudaSetDevice(ctx->device));
  DAB_CUDA(dab_wait_stream(pr->stream));
  for (int s = 0; s < 16; ++s) {
    ms[s] = 0.0f;
    if (s < 9 && pr->ev_used[s]) {
      float t = 0.0f;
      if (cudaEventElapsedTime(&t, pr->ev[2 * s], pr->ev[2 * s + 1]) == cudaSuccess) ms[s] = t;
    }
    if (s >= 10 && s <= 13) ms[s] = (float)(pr->api_us[s - 10] / 1e3);
    if (s == 9 && pr->ev_used[8]) {
      float t = 0.0f;
      if (cudaEventElapsedTime(&t, pr->ev[16], pr->ev[18]) == cudaSuccess) ms[s] = t;
    }
  }
  return DAB_OK;
}

int dab_pair_get_timeline(dab_pair *pr, void *ref_event, float start_ms[9], float end_ms[9]) {
  if (!pr || !ref_event || !start_ms || !end_ms) return DAB_E_ARG;
  dab_ctx *ctx = pr->ctx;
  DAB_CUDA(cudaSetDevice(ctx->device));
  DAB_CUDA(dab_wait_stream(pr->stream));
  cudaEvent_t ref = reinterpret_cast<cudaEvent_t>(ref_event);
  for (int s = 0; s < 9; ++s) {
    start_ms[s] = end_ms[s] = -1.0f;
    if (!pr->ev_used[s]) continue;
    float t0 = 0.0f, t1 = 0.0f;
    if (cudaEventElapsedTime(&t0, ref, pr->ev[2 * s]) == cudaSuccess &&
        cudaEventElapsedTime(&t1, ref, pr->ev[2 * s + 1]) == cudaSuccess) { start_ms[s] = t0; end_ms[s] = t1; }
    cudaGetLastError();
  }
  return DAB_OK;
}

}  // extern "C"
