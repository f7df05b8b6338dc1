// describealign_b200 - shared declarations of the CUDA implementation (sm_100a).
// All arithmetic files are compiled with -fmad=false: the reference's numpy code never
// contracts a*b+c, and where OpenBLAS does (its ddot kernels), fma() is written explicitly.
#pragma once

#include <cuda_runtime.h>
#include <atomic>
#include <mutex>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>

#include "../../include/describealign_b200.h"

#define DAB_NCODE 823543  // 7^7 digit codes per hash table (reference describealign.py:610-628)
#define DAB_WIN 41        // frames in the correlation / norm window (:597)

struct DevBuf {
  void *p = nullptr;
  size_t cap = 0;
  bool pooled = false;   // allocated with cudaMallocAsync
  template <typename T> T *as() const { return reinterpret_cast<T *>(p); }
};

struct dab_ctx {
  int device = 0;
  std::string err;                    // last error; written under err_mu (pairs of one context run on several host threads)
  std::mutex err_mu;
  std::atomic<int64_t> launches{0};   // kernels launched through this context (many host threads)
  int sm_count = 148;
  int opt_dp2_impl = 0;      // 0 scan kernel (dp2_scan.cuh), 2 generic tree DP (both exact; the tests compare them)
};

// Features of one track, device resident.
struct Track {
  int64_t S = 0;       // samples per channel
  int ch = 1;
  int64_t L = 0;       // frames = S / 210 (length of zc / bands)
  int64_t Le = 0;      // length of the energy feature (L or L + 1)
  bool have_features = false;
  DevBuf pcm;          // staging for host PCM
  DevBuf energy, zc, b0, b1, b2;   // f32 x4, f64
  DevBuf feat_ticket;  // u32: tile ticket of the persistent feature kernel
  DevBuf feat_mid;     // per-frame intermediates between the two feature kernels (features.cu: FeatMid), 212 B per frame
  DevBuf gate;         // the separate *_energy argument of align() when it is not features[0] (:629, :657)
  bool have_gate = false;
};

// Stage-A prep of one track's features (features 0..2 keep ms / nrm for scoring; 3, 4 only feed the codes)
struct Prep {
  int64_t L = 0, Le = 0;   // the feature lengths it was made from
  DevBuf ms;           // f64 [3][Lp]   Lp = min feature length
  DevBuf nrm;          // f64 [3][Lp-40]
  DevBuf pack;         // u32 [5][Lp-40] one digit per nibble (bits 0-2), bit 3 of the nibble = flag (video)
  DevBuf code;         // i32 [5][Lp-40] base-7 code (audio: lookup key)
  DevBuf nq_flag;      // i32 [n] not-quiet flags, then their exclusive scan
  DevBuf nq_list;      // i32 selected frame list (video: every 4th not-quiet; audio: all not-quiet)
};

// The video side of the match stage, as the gate, scoring and DP 1 read it: the video track's prep, the hash tables
// over its hashed frames and the records of those frames.  A pair builds its own in every stage-A run; a shared
// index (dab_index) builds one once, and any number of pairs then only read it.
struct VideoSide {
  Prep prep;
  DevBuf tbl_start;   // i32 [5*NCODE + 1]
  DevBuf tbl_items;   // i32 sel-ranks
  DevBuf v_rec;       // uint4[2] per hashed video frame: its five digit packs (gate)
  int64_t n_vsel = 0, n_entries = 0;   // hashed frames, table entries
  int64_t cap_entries = 0;             // capacity of the tables (grown on overflow)
};

// What one stage-B call decided, read by every later step of that call (points, DP 2, the exchange of
// quals of a row-sharded pair).  Set once per call by dab_set_stage_b_plan.
struct StageBPlan {
  int64_t n_audio = 0, n_video = 0;
  std::vector<dab_corridor> cor;   // host row bounds; device-planned: ranges that contain the planned ones
  int32_t n_clusters = 0;          // cluster indices are below this
  bool device_planned = false;     // corridors planned on the device from clusters, not uploaded
  int64_t pm_off[32] = {};         // first PM row of each corridor (scan DP)
  int64_t rows = 0;                // total corridor rows: bounds the pass-2 points
  bool scan_dp = false;            // the corridor-state DP runs, not the generic tree DP
};

struct dab_pair {
  dab_ctx *ctx = nullptr;
  cudaStream_t stream = nullptr;
  Track trk[2];
  // scan scratch
  DevBuf scan_tmp;            // single-pass scan: ticket counter + tile status words
  unsigned int scan_epoch = 0;
  // stage A
  Prep prep_a;                // of the audio track
  VideoSide video;            // of the video track
  // the video side whose hashed frames the pass-1 points refer to: &video, a shared index's (export refused), or
  // null (a run in flight, or the own side out of date after new features).  Only compared, never read through.
  const VideoSide *points_side = nullptr;
  // table build scratch
  DevBuf tbl_sb;      // i32: per super-bucket of 4096 slots its entry count, offset (+ total) and scatter cursor
  DevBuf tbl_ent;     // u32 x2 [entries]: (slot within its super-bucket, rank), grouped by super-bucket
  // gate / scoring
  DevBuf row_count, row_off;   // i32 [n_queries + 1]
  DevBuf row_stash;            // i32 [n_queries][4]: first candidates of each row (gate count pass)
  DevBuf gate_big;             // i32: rows with more than 4 candidates (work list of the fill pass)
  DevBuf gate_rec;             // per query: digit words + its two buckets (32 B)
  DevBuf gate_best;            // per query: i64 exclusive scan of the bucket entries to visit, then those i32 counts
  DevBuf cand_tmp, cand_s, cand_i;  // i32 [n_cand]
  DevBuf cand_q;               // f64 [n_cand]
  DevBuf keep_flag, keep_off;  // i32 [n_cand + 1]
  DevBuf pt_i, pt_s, pt_q;     // match points of pass 1
  DevBuf counters;             // i64 [16] device counters
  // dp1
  DevBuf tree1;                // Node16 levels
  DevBuf back1;                // BackRec [n_points]
  DevBuf dpres;                // i32/i64 results (end id, path len)
  DevBuf path1_x, path1_y;     // i32
  int64_t n_points1 = 0, n_path1 = 0;
  int64_t cap_cand = 0, cap_points1 = 0;   // capacities of device-sized buffers (grown on overflow)
  // stage B
  DevBuf a_scaled, v_scaled;   // f32 (n,3)
  DevBuf corridors;            // dab_corridor[]
  DevBuf row2_count, row2_off; // i32 [n_audio + 1]
  DevBuf p2_i, p2_c, p2_rank, p2_k;  // i32
  DevBuf pm2;                  // corridor-state DP: per-corridor running maxima
  DevBuf tb_up, tb_mark;       // traceback scratch of both DPs (they run one after the other on the stream)
  StageBPlan plan_b;
  DevBuf p2_j, p2_q;           // f64
  DevBuf tree2;                // frontier tree of pass 2
  DevBuf cache2;               // prev_cache rows
  DevBuf cluster_best2;        // tree DP: per cluster, cum - 50 of its best point (f64) and its id (i32)
  DevBuf back2;                // BackRec [n_points]
  DevBuf path2;                // f64 (n,5)
  int64_t n_points2 = 0, n_path2 = 0;
  DevBuf clusters, refine_partial, maxes;
  dab_stats stats = {};
  cudaEvent_t ev[32] = {};
  bool ev_used[16] = {};
  // pinned host mirror of small results
  int64_t *h_counters = nullptr;       // pinned + mapped host block
  int64_t *d_counters_map = nullptr;   // its device-side address
  // host time spent inside the library's calls for this pair since the last set_pcm (microseconds):
  // [0] set_pcm / set_features, [1] stage A, [2] stage B, [3] get_* copies
  int64_t api_us[4] = {0, 0, 0, 0};
};

// A video side built once per video and then only read: any number of pairs, each on its own stream, run their
// description track against it (dab_pair_stage_a_against).
struct dab_index {
  dab_ctx *ctx = nullptr;           // the context of the pair it was built from (device, error messages)
  VideoSide side;
  DevBuf counters;                  // the build's device counts
  cudaEvent_t ready = nullptr;      // recorded after the last command of the build; every user's stream waits on it
  mutable std::atomic<int> users{0};   // stage-A calls running against the index; -1 once it is being freed
};

inline void dab_set_err(dab_ctx *ctx, const std::string &msg) {
  std::lock_guard<std::mutex> g(ctx->err_mu);
  ctx->err = msg;
}

struct ApiTimer {
  int64_t *slot;
  int64_t t0;
  static int64_t now();
  explicit ApiTimer(int64_t *s) : slot(s), t0(now()) {}
  ~ApiTimer() { *slot += now() - t0; }
};

#define DAB_CUDA(call)                                                                     \
  do {                                                                                     \
    cudaError_t e__ = (call);                                                              \
    if (e__ != cudaSuccess) {                                                              \
      char b__[512];                                                                       \
      snprintf(b__, sizeof b__, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__),   \
               __FILE__, __LINE__);                                                        \
      dab_set_err(ctx, b__);                                                                    \
      return DAB_E_CUDA;                                                                   \
    }                                                                                      \
  } while (0)

#define DAB_TRY(expr)              \
  do {                             \
    int rc__ = (expr);             \
    if (rc__ != DAB_OK) return rc__; \
  } while (0)

// Device buffers are allocated stream-ordered (cudaMallocAsync / cudaFreeAsync on the stream of the
// pair whose API call is running): cudaMalloc / cudaFree would wait for every other pair's kernels.
extern thread_local cudaStream_t dab_t_stream;
struct StreamScope {
  cudaStream_t prev;
  explicit StreamScope(cudaStream_t s) : prev(dab_t_stream) { dab_t_stream = s; }
  ~StreamScope() { dab_t_stream = prev; }
};
int dab_ensure(dab_ctx *ctx, DevBuf &b, size_t bytes);
// Host thread waits for everything queued in `st`.  Mode 0/1: cudaStreamSynchronize (spinning or
// blocking, as the device's schedule flags say); mode 2: cudaStreamQuery + short sleeps with back-off
// (see dab_set_host_wait).
extern int dab_g_wait_mode;
cudaError_t dab_wait_stream(cudaStream_t st);
cudaError_t dab_readback(dab_pair *pr, void *host_dst, const void *dev_src, size_t bytes);
static inline int64_t cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }

// exclusive scan of n non-negative int32 values; out[n] receives the total (out has n + 1 entries).  n_dev
// (optional): device-side count of valid elements (<= n; launches are sized for n); total_out (optional): device
// word that also receives the total.  int32 sums saturate at INT32_MAX; the int64 scan writes its total to
// total_out[0] (low word) and total_out[1] (high word).
int dab_exclusive_scan(dab_pair *pr, const int32_t *in, int32_t *out, int64_t n, const int32_t *n_dev = nullptr,
                       int32_t *total_out = nullptr);
int dab_exclusive_scan(dab_pair *pr, const int32_t *in, int64_t *out, int64_t n, const int32_t *n_dev = nullptr,
                       int32_t *total_out = nullptr);

// Counts that only the device knows while a stage is in flight (int32 words of dab_pair::counters).  Every
// kernel of a stage reads the counts it needs from here, so a whole stage is enqueued without a host
// round trip; the block is copied to the pair's mapped host page when the stage ends.
enum {
  DC_N_VNQ = 0,        // not-quiet video frames
  DC_N_AQ_ALL = 1,     // not-quiet audio frames
  DC_N_ENTRIES = 2,    // expanded table entries
  DC_N_VSEL = 3,       // hashed video frames (every 4th not-quiet)
  DC_ENUM_LO = 4, DC_ENUM_HI = 5,   // u64: bucket entries visited by the gate (low, high word; written by its scan)
  DC_N_CAND = 6,
  DC_N_PTS1 = 7,
  DC_DP1_END = 8,      // end id (-1: no path), written by dp1_kernel
  DC_N_PATH1 = 9,      // path length, written by the traceback
  DC_Q_LO = 10, DC_Q_HI = 11, DC_N_Q = 12,    // query range of this shard in the not-quiet audio list
  DC_OVERFLOW = 13,    // bit 0 table entries, bit 1 candidates, bit 2 > 32 corridors on a row, bit 3 pass-2 points
  DC_BAD_IMPORT = 14,
  DC_N_BIGROWS = 15,   // gate rows with more than GATE_STASH candidates
  DC_N_PTS2 = 16,
  DC_OVERFLOW_B = 17,  // stage B: bit 2 more than 32 corridors on one audio row
  DC_DP2_END = 18,     // end id, then the frontier value (double at words 20-21)
  DC_N_PATH2 = 19,     // path length, written by the traceback
  DC_NEED_ENTRIES = 22, DC_NEED_CAND = 23,    // unclamped table-entry and candidate totals (sizes the next run;
                                              // the candidate total saturates at INT32_MAX)
  DC_DP2_CNT = 24,     // 4 x u64 DP-2 work counters
  DC_WORDS = 32
};
enum { DAB_OVF_ENTRIES = 1, DAB_OVF_CAND = 2, DAB_OVF_ROWCOR = 4, DAB_OVF_PTS2 = 8 };

// stage entry points implemented in the .cu files
int dab_run_features(dab_pair *pr, int track, const void *d_pcm, int format);
// A device stage is enqueued on the pair's stream without waiting (counts stay on the device) and ends with
// dab_enqueue_counts, which copies the counts block to the mapped host page; once the stream has passed that
// point, dab_collect_* interprets it.
int dab_enqueue_counts(dab_pair *pr);
// Stage A.  On a capacity overflow dab_collect_stage_a grows the buffer to at least the total the run needed and
// returns DAB_E_CAPACITY: the caller enqueues the stage again, up to DAB_STAGE_A_ATTEMPTS runs in all.  An
// entries overflow leaves the tables empty, so the candidate total is only known one run later: three runs at most.
// A run that needs more candidates than the int32-indexed candidate arrays hold (DAB_MAX_CANDIDATES) is not run
// again: the collect returns DAB_E_CAPACITY with the count, and the next enqueue refuses at once.
constexpr int DAB_STAGE_A_ATTEMPTS = 8;
constexpr int64_t DAB_MAX_CANDIDATES = 0x7ffffffeLL;   // INT32_MAX - 1: a candidate total of INT32_MAX is saturated
int dab_check_stage_a_inputs(dab_pair *pr, const char *who);
// match points of audio rows [row_lo, row_hi) against a shared index (ix), or against the pair's own video side,
// built in the same run; then DP 1 + traceback if with_dp, then the counts
int dab_enqueue_stage_a(dab_pair *pr, const dab_index *ix, int64_t row_lo, int64_t row_hi, bool with_dp);
int dab_collect_stage_a(dab_pair *pr, const dab_index *ix, bool with_dp);
int dab_enqueue_stage_a_dp(dab_pair *pr);      // DP 1 + traceback over the pair's points (its own video side)
void dab_collect_stage_a_dp(dab_pair *pr);
// the video side of src's video track into ix, then the counts (to src's mapped page); the collect records
// ix->ready, or grows the tables after an overflow and returns DAB_E_CAPACITY
int dab_enqueue_index(dab_pair *src, dab_index *ix);
int dab_collect_index(dab_pair *src, dab_index *ix);
int dab_run_import_points1(dab_pair *pr, const int32_t *i_audio, const int32_t *v_video, const double *qual,
                           int64_t n, int src_on_device);
// Stage B.  Its sizes come from pr->plan_b, set by device planning from clusters or by the explicit upload of
// dab_pair_stage_b.
void dab_set_stage_b_plan(dab_pair *pr, int64_t n_audio, int64_t n_video, std::vector<dab_corridor> cor, int32_t n_clusters,
                          bool device_planned);
int dab_enqueue_column_maxes(dab_pair *pr, int64_t n_audio, int64_t n_video);
// checks, scaling, corridor planning, then dab_enqueue_stage_b (`who` names the caller in argument errors)
int dab_enqueue_stage_b_clusters(dab_pair *pr, const float gain[3], const float audio_std[3], int64_t n_audio, int64_t n_video,
                                 const dab_cluster *clusters, int32_t n_clusters, int64_t row_lo, int64_t row_hi, bool with_dp,
                                 const char *who);
// points with quals for audio rows [row_lo, row_hi), then DP 2 + traceback if with_dp, then the counts
int dab_enqueue_stage_b(dab_pair *pr, int64_t row_lo, int64_t row_hi, bool with_dp);
int dab_enqueue_stage_b_dp(dab_pair *pr);
int dab_enqueue_set_quals2(dab_pair *pr, const double *d_q_all);
int dab_row_range_points2(dab_pair *pr, int64_t lo, int64_t hi, int64_t *first, int64_t *count);
int dab_collect_stage_b(dab_pair *pr, bool with_dp);

// What both frontier DPs keep per point for the traceback: the value the point started from and its
// predecessor's id (-1: the seed).  A predecessor always has a smaller id than its point.
struct __align__(16) BackRec {
  double best;
  int32_t pred;
  int32_t pad;
};

// What the traceback writes for every path point, in path order.
struct Path1Out {              // pass 1: audio frame x, video frame y
  const int32_t *pt_i, *pt_s, *v_sel;
  int32_t *x, *y;
};
struct Path2Out {              // pass 2: rows (j, i, cluster, qual, cum)
  const int32_t *p_i, *p_c;
  const double *p_j, *p_q;
  double *rows;
};
// Traceback (traceback.cu) from the end id result[0] (-1: empty path) through the back records of the *n_dev <= cap
// points; the path length goes to *n_path.  Pass 2 also reads the end point's frontier value, a double at result + 2.
int dab_enqueue_traceback(dab_pair *pr, const BackRec *back, const int32_t *n_dev, const int32_t *result, int64_t cap,
                          int32_t *n_path, const Path1Out &out);
int dab_enqueue_traceback(dab_pair *pr, const BackRec *back, const int32_t *n_dev, const int32_t *result, int64_t cap,
                          int32_t *n_path, const Path2Out &out);

#define DAB_LAUNCHED(pr) ((pr)->ctx->launches++)

// ------------------------------------------------------------------------------------------
// OpenBLAS 0.3.30 SkylakeX ddot summation order (what np.dot / np.convolve do on f64 in the
// reference, SURVEY.md B.2 iv): blocks of 32 through 4 x 8 FMA lanes folded to 4 x 4, blocks
// of 16 through 4 x 4 FMA lanes, tail as one FMA chain.  X(i), Y(i) are accessor macros.
// ------------------------------------------------------------------------------------------
template <typename FX, typename FY>
__device__ __forceinline__ double ddot_skx(FX X, FY Y, int n) {
  double a[4][4];
#pragma unroll
  for (int k = 0; k < 4; ++k)
#pragma unroll
    for (int l = 0; l < 4; ++l) a[k][l] = 0.0;
  int n1 = n & ~15;
  int n32 = n1 & ~31;
  int i = 0;
  if (n32) {
    double z[4][8];
#pragma unroll
    for (int k = 0; k < 4; ++k)
#pragma unroll
      for (int l = 0; l < 8; ++l) z[k][l] = 0.0;
    for (; i < n32; i += 32) {
#pragma unroll
      for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int l = 0; l < 8; ++l) z[k][l] = fma(X(i + 8 * k + l), Y(i + 8 * k + l), z[k][l]);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k)
#pragma unroll
      for (int l = 0; l < 4; ++l) a[k][l] = z[k][l] + z[k][l + 4];
  }
  for (; i < n1; i += 16) {
#pragma unroll
    for (int k = 0; k < 4; ++k)
#pragma unroll
      for (int l = 0; l < 4; ++l) a[k][l] = fma(X(i + 4 * k + l), Y(i + 4 * k + l), a[k][l]);
  }
  double s0 = ((a[0][0] + a[1][0]) + a[2][0]) + a[3][0];
  double s1 = ((a[0][1] + a[1][1]) + a[2][1]) + a[3][1];
  double s2 = ((a[0][2] + a[1][2]) + a[2][2]) + a[3][2];
  double s3 = ((a[0][3] + a[1][3]) + a[2][3]) + a[3][3];
  double dot = (s0 + s2) + (s1 + s3);
  for (; i < n; ++i) dot = fma(Y(i), X(i), dot);
  return dot;
}

// Fixed n = 41 specialisation: one 32-block, no 16-block, 9-element tail.
template <typename FX, typename FY>
__device__ __forceinline__ double ddot41_skx(FX X, FY Y) {
  double z[4][8];
#pragma unroll
  for (int k = 0; k < 4; ++k)
#pragma unroll
    for (int l = 0; l < 8; ++l) z[k][l] = fma(X(8 * k + l), Y(8 * k + l), 0.0);
  double s[4];
#pragma unroll
  for (int l = 0; l < 4; ++l) {
    double a0 = z[0][l] + z[0][l + 4];
    double a1 = z[1][l] + z[1][l + 4];
    double a2 = z[2][l] + z[2][l + 4];
    double a3 = z[3][l] + z[3][l + 4];
    s[l] = ((a0 + a1) + a2) + a3;
  }
  double dot = (s[0] + s[2]) + (s[1] + s[3]);
#pragma unroll
  for (int i = 32; i < 41; ++i) dot = fma(Y(i), X(i), dot);
  return dot;
}
