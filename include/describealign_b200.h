/*
 * describealign_b200 - C ABI of the B200 alignment hot path.
 *
 * Drop-in boundary for the part of julbean/describealign between "PCM decoded" and the
 * returned alignment (reference describealign.py:545-1027).  The reference has no FFI for
 * this path - it is plain Python calling numpy - so the entry points below are what a
 * binding for the reference's four hot-path functions needs (INTEGRATION.md shows the
 * ctypes stub):
 *
 *   reference function (describealign.py)            replaced by
 *   ------------------------------------------------------------------------------------
 *   parse_audio_from_file tail  :156  (int16->f16)   dab_pair_set_pcm (conversion on device)
 *   get_energy                  :545-555             dab_pair_set_pcm + dab_pair_get_features
 *   get_zero_crossings          :557-566             "
 *   get_freq_bands              :575-593             "
 *   align, device stage A       :596-700             dab_pair_stage_a + dab_pair_get_path1
 *   align, host stage           :702-893             stays in Python (describealign_b200/host_fit.py)
 *   align, device stage B       :895-993             dab_pair_stage_b_clusters + dab_pair_get_path2
 *
 * Conventions: plain pointers and sizes only; every function returns 0 on success or a
 * DAB_E_* code, with a message available from dab_last_error(); the caller owns every
 * buffer it passes; "host" pointers may be pageable or pinned; nothing here is
 * thread-safe per context (the reference calls the path from one thread, :1098-1122) but
 * any number of pairs may be in flight on one context - calls that enqueue work are
 * asynchronous on the pair's own CUDA stream and dab_pair_get_* / dab_pair_sync wait for it.
 * There is no CPU fallback: without a CUDA device dab_create fails.
 */
#ifndef DESCRIBEALIGN_B200_H
#define DESCRIBEALIGN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DAB_ABI_VERSION 2

enum {
  DAB_OK = 0,
  DAB_E_CUDA = 1,       /* a CUDA runtime call failed */
  DAB_E_ARG = 2,        /* invalid argument */
  DAB_E_STATE = 3,      /* call sequence violated (e.g. stage_a before features) */
  DAB_E_CAPACITY = 4,   /* an internal buffer overflowed even after growing */
  DAB_E_TOO_SHORT = 5,  /* track shorter than the 41-frame window */
  DAB_E_TIMEOUT = 6     /* dab_engine_next: nothing finished within the timeout */
};

/* sample formats accepted by dab_pair_set_pcm */
enum {
  DAB_PCM_S16 = 0,      /* interleaved int16, as ffmpeg's s16le stream (describealign.py:152) */
  DAB_PCM_F16 = 1       /* interleaved IEEE half, i.e. the memory behind the reference's
                           float16 (ch, S) array, which is an F-ordered view (describealign.py:156) */
};

enum { DAB_TRACK_VIDEO = 0, DAB_TRACK_AUDIO = 1 };

typedef struct dab_ctx dab_ctx;    /* one per process and GPU */
typedef struct dab_pair dab_pair;  /* one (video, description) pair: device-resident state */

/* One scored corridor of stage B: audio rows [lo, hi) on the line j = slope * i + offset,
 * belonging to line cluster `cluster` (describealign.py:931-941). */
typedef struct {
  int32_t cluster;
  int32_t lo;
  int32_t hi;
  int32_t reserved;
  double slope;
  double offset;
} dab_corridor;

/* One line cluster of the host fit (describealign.py:861-893): first and last audio coordinate of its
 * points and the fitted line j = slope * i + offset.  Stage B plans the scored corridor from it on the
 * device (:895-932): row limits, sub-frame offset refinement, +-30 s extension. */
typedef struct {
  int32_t cluster;
  int32_t reserved;
  double x_first, x_last;
  double offset, slope;
} dab_cluster;

/* Work counters of the last stage_a / stage_b run (for measurement, SURVEY.md appendix D). */
typedef struct {
  int64_t n_video_frames, n_audio_frames;
  int64_t n_video_selected;   /* hashed video frames (every 4th not-quiet) */
  int64_t n_audio_queries;    /* not-quiet audio frames */
  int64_t n_table_entries;    /* expanded entries per table, summed over the 5 tables */
  int64_t n_enumerated;       /* bucket entries visited by the gate */
  int64_t n_candidates;       /* candidates scored */
  int64_t n_points1;          /* match points of pass 1 */
  int64_t n_path1;
  int64_t n_points2;
  int64_t n_path2;
  int64_t n_dp2_queries;      /* pass-2 points that needed a real frontier query */
  int64_t n_dp2_refills;      /* 16-row refills of the per-corridor running-max windows */
  int64_t n_dp2_neighbour;    /* pass-2 points with another corridor within 2 cells / 2 rows */
  int64_t n_dp2_run_points;   /* pass-2 points committed by block evaluation (dp2_block_kernel) */
} dab_stats;

int dab_abi_version(void);
int dab_device_count(void);

/* Page-locked host buffers from a process-wide pool (power-of-two size classes, recycled on free).
 * Passing such buffers as the host pointers of dab_pair_set_pcm / dab_pair_get_* / dab_pair_stage_b
 * makes those copies asynchronous DMA instead of staged pageable copies; any host pointer works.
 * dab_alloc_pinned returns NULL when no CUDA device is available.  dab_trim_pinned releases the
 * free list back to the driver. */
void *dab_alloc_pinned(size_t bytes);
void dab_free_pinned(void *p);
void dab_trim_pinned(void);
/* Plain host memcpy.  Exists so that a Python host can move results between its pinned staging
 * buffers and ordinary arrays without holding the interpreter lock (ctypes releases it). */
void dab_host_copy(void *dst, const void *src, size_t bytes);
/* Allocator activity since load: out[0] device (re)allocations, out[1] microseconds spent in them,
 * out[2] page-locked allocations that missed the pool, out[3] microseconds spent in them.  A batch in
 * steady state should show no growth: both kinds of call synchronise the whole device. */
void dab_alloc_stats(int64_t out[4]);

/* How host threads wait for the device inside the stage calls.  mode 0: cudaStreamSynchronize with the
 * CUDA default, which spins when the process has fewer contexts than the host has cores; 1: the same call
 * with cudaDeviceScheduleBlockingSync (the thread sleeps until the driver wakes it); 2: cudaStreamQuery
 * polling with 20-400 us sleeps in between.  A batch driver that keeps more pairs in flight (one host
 * thread each) than there are host cores must not use 0: the spinning waiters starve the threads that
 * have kernels to launch.  Measured with 64 pairs in flight on 16 cores (profiles/r1_v9_pairs_in_flight.txt):
 * mode 1 wakes a thread only milliseconds after its stream drained, mode 2 within the sleep it was in.
 * Returns the device's schedule flags after the call (>= 0) or a negative DAB_E_* code.  device < 0:
 * current device. */
int dab_set_host_wait(int device, int mode);

/* device < 0: current device. */
int dab_create(int device, dab_ctx **out);
void dab_destroy(dab_ctx *ctx);
/* Testing switch.  "dp2_impl" = 2 forces the generic tree-based pass-2 DP (the fallback for more than 32
 * corridors or non-positive slopes) instead of the scan DP ("dp2_impl" = 0, the default); both are exact and
 * the tests compare them.  Unknown names or values return DAB_E_ARG. */
int dab_set_option(dab_ctx *ctx, const char *name, int64_t value);
const char *dab_last_error(const dab_ctx *ctx);   /* ctx may be NULL for dab_create failures */

/* "Native numpy" parity (reference :554, :590 call np.log10 on float32): numpy's bundled SIMD log10 differs
 * from glibc's log10f - which the feature kernel restates - by up to 2 ulp when the host has AVX-512.
 * nibbles: one 4-bit entry per float32 from 1.0f upwards (two per byte, low nibble first) holding
 * (bits of the host's log10f(x)) - (bits of dab_eval_log10f without a correction) + 8; count entries.
 * count = 0 removes the table (glibc behaviour, the default).  Applies to the context's device.
 * dab_eval_log10f evaluates the feature kernel's log10f for n host values >= 1 (with the current table). */
int dab_set_log10f_correction(dab_ctx *ctx, const unsigned char *nibbles, uint64_t count);
int dab_eval_log10f(dab_ctx *ctx, const float *x, float *y, int64_t n);

int dab_pair_create(dab_ctx *ctx, dab_pair **out);
void dab_pair_destroy(dab_pair *pair);
int dab_pair_sync(dab_pair *pair);
/* the CUDA stream (cudaStream_t) the pair's work is enqueued on, for event timing */
void *dab_pair_stream(dab_pair *pair);

/* ---- features (reference :545-593) ------------------------------------------------------
 * Computes the five 210 Hz feature vectors of one track from interleaved PCM of
 * `samples` samples per channel, `channels` in {1, 2}.  `pcm` is a host pointer, or a
 * device pointer when on_device != 0.  Results stay on the device inside the pair. */
int dab_pair_set_pcm(dab_pair *pair, int track, const void *pcm, int64_t samples, int channels,
                     int format, int on_device);

/* Alternatively upload features computed elsewhere (the reference-level align() boundary,
 * :595): energy[n_energy], zc[n], band0[n], band1[n] float32 and band2[n] float64 (host). */
int dab_pair_set_features(dab_pair *pair, int track, const float *energy, int64_t n_energy,
                          const float *zc, const float *band0, const float *band1, const double *band2,
                          int64_t n);

/* align()'s separate video_energy / audio_desc_energy arguments (:595) decide which frames are "not
 * quiet" (:629, :657).  The reference's only caller passes features[0] for them (:1121), which is what
 * the pair uses by default; a caller that passes something else uploads it here after the features
 * (n_energy must equal len(features[0])). */
int dab_pair_set_gate_energy(dab_pair *pair, int track, const float *energy, int64_t n_energy);

/* lens[0] = len(energy) (n or n + 1, :555), lens[1..4] = n. */
int dab_pair_feature_lens(dab_pair *pair, int track, int64_t lens[5]);
/* Copies features to host buffers of at least lens[] elements; any pointer may be NULL. */
int dab_pair_get_features(dab_pair *pair, int track, float *energy, float *zc, float *band0,
                          float *band1, double *band2);

/* ---- stage A (reference :596-700) -------------------------------------------------------
 * prep + codes + tables + gate + scoring + frontier DP #1 + traceback, all on the device.
 * Blocks until the path length is known.  n_points / n_path may be NULL. */
int dab_pair_stage_a(dab_pair *pair, int64_t *n_points, int64_t *n_path);
/* pass-1 path, ascending: audio frame x[k], video frame y[k] (int32, n_path entries each). */
int dab_pair_get_path1(dab_pair *pair, int32_t *x_audio, int32_t *y_video);
/* pass-1 match points sorted by (audio frame, video frame); any pointer may be NULL. */
int dab_pair_get_points1(dab_pair *pair, int32_t *i_audio, int32_t *v_video, double *qual);

/* ---- stage A of many combinations: one video index shared by many descriptions ----------------
 * Which description belongs to which video is decided by stage A itself (its pass-1 path length against
 * the reference's minimum, :698-699); the video side of stage A (prep, codes, hashed-frame list, hash
 * tables) depends on the video track only, so it is built once per video.
 * dab_index_build: the video side of `src`'s video track (features required) into a new index, on src's
 *   stream; blocks until the index's table capacity is settled, then src may be reused.  The index is
 *   read-only from then on; an event on it marks it ready and every user's stream waits on it.
 * dab_pair_stage_a_against: prep of `pair`'s description track (features of the audio track required),
 *   then gate, scoring, DP 1 and traceback against the index, enqueued without a host round trip; grows and
 *   reruns on a candidate overflow like dab_pair_stage_a.  Blocks until the counts are back; nothing else
 *   leaves the device (dab_pair_get_path1 copies the path on request; dab_pair_get_stats has the candidate
 *   count).  The points are ranks into the index's hashed frames: dab_pair_get_points1 / export_points1
 *   refuse them, and dab_pair_dp1 / import_points1 need the pair's own stage_a_match again.  Any number of
 *   pairs, each on its own stream and host thread, may run against one index at once.
 * dab_index_free: DAB_E_STATE (nothing freed) while a dab_pair_stage_a_against call on the index is running.
 * dab_index_info: out[0] video frames, [1] hashed frames, [2] table entries, [3] calls running against it. */
typedef struct dab_index dab_index;
int dab_index_build(dab_pair *src, dab_index **out);
int dab_index_free(dab_index *index);
int dab_index_info(const dab_index *index, int64_t out[4]);
int dab_pair_stage_a_against(dab_pair *pair, const dab_index *index, int64_t *n_points, int64_t *n_path);

/* ---- stage A in two steps, for one very long pair split over several GPUs (SURVEY.md 8e) ----
 * dab_pair_stage_a_match: prep + codes + tables for the whole pair, then gate + scoring only for the
 * audio frames row_lo <= i < row_hi (pass 0, INT64_MAX for all rows); the match points stay on the
 * device.  Ranks exchange them with dab_pair_export_points1 / dab_pair_import_points1 (pointers may be
 * device pointers, e.g. NCCL buffers, when *_on_device != 0); imported points must be sorted by
 * (audio frame, video frame) without duplicates, have quals > 0 and lie on hashed video frames of this pair
 * - concatenating the shards in row order gives exactly that; anything else is rejected with DAB_E_ARG.
 * dab_pair_dp1 then runs frontier DP #1 + traceback (reference :674-700) on the pair's points. */
int dab_pair_stage_a_match(dab_pair *pair, int64_t row_lo, int64_t row_hi, int64_t *n_points);
int dab_pair_export_points1(dab_pair *pair, int32_t *i_audio, int32_t *v_video, double *qual, int dst_on_device);
int dab_pair_import_points1(dab_pair *pair, const int32_t *i_audio, const int32_t *v_video, const double *qual,
                            int64_t n, int src_on_device);
int dab_pair_dp1(dab_pair *pair, int64_t *n_path);

/* ---- stage B (reference :895-993) -------------------------------------------------------
 * The explicit-input entry, used by tests to feed inputs no line cluster can produce.
 * audio_scaled / video_scaled: float32 row-major (n, 3) arrays (:740-741), host pointers.
 * corridors: the scored clusters in cluster order with their final (refined) lines.
 * n_clusters: number of line clusters (>= max cluster index + 1).  np.max of the energy
 * columns (:908-909) is taken on the device. */
int dab_pair_stage_b(dab_pair *pair, const float *audio_scaled, int64_t n_audio,
                     const float *video_scaled, int64_t n_video, const dab_corridor *corridors,
                     int32_t n_corridors, int32_t n_clusters, int64_t *n_points, int64_t *n_path);
/* The whole of stage B on the device for a pair that still holds its feature vectors there (after
 * dab_pair_set_pcm or dab_pair_set_features), from the host fit's line clusters (in cluster order,
 * ascending cluster index).  The scaled arrays of describealign.py:737-741 are produced on the device
 * from the least-squares gains and the audio standard deviations of the first three features (numpy
 * float32 roundings: audio / std ; video * gain / std), so only 6 floats travel instead of
 * 12 (n_audio + n_video) bytes.  n_audio / n_video: lengths of the scaled arrays (the shortest of the
 * three vectors of each track).  Then corridor planning incl. the offset refinement (:895-932), np.max
 * of the scaled energy columns (:908-909), scoring, DP #2, traceback.  The refinement's least-squares
 * coefficient is the quotient of float64 sums (the reference: np.linalg.lstsq), so refined offsets
 * agree with the reference's to ~1e-15 relative rather than bit for bit. */
int dab_pair_stage_b_clusters(dab_pair *pair, const float gain[3], const float audio_std[3], int64_t n_audio,
                              int64_t n_video, const dab_cluster *clusters, int32_t n_clusters,
                              int64_t *n_points, int64_t *n_path);
/* ---- stage B in steps, for one very long pair split over several GPUs (SURVEY.md 8e) ----
 * dab_pair_stage_b_score: scaling, corridor planning and the sorted pass-2 point list for the whole pair
 * (identical on every rank: it only depends on the corridors), but the quals - the part that reads the
 * features - only for the audio rows row_lo <= i < row_hi; those are the points [*first_point,
 * *first_point + *n_mine).  Ranks exchange their qual slices (dab_pair_export_quals2, e.g. into NCCL
 * buffers), one rank imports the concatenation (dab_pair_import_quals2, n = *n_points) and runs
 * dab_pair_dp2: DP #2 + traceback (reference :946-993), which do not shard. */
int dab_pair_stage_b_score(dab_pair *pair, const float gain[3], const float audio_std[3], int64_t n_audio,
                           int64_t n_video, const dab_cluster *clusters, int32_t n_clusters, int64_t row_lo,
                           int64_t row_hi, int64_t *n_points, int64_t *first_point, int64_t *n_mine);
int dab_pair_export_quals2(dab_pair *pair, double *qual, int64_t first_point, int64_t count, int dst_on_device);
int dab_pair_import_quals2(dab_pair *pair, const double *qual_all, int64_t n, int src_on_device);
int dab_pair_dp2(dab_pair *pair, int64_t *n_path);

/* the corridors of the last stage_b call as scored (for _clusters: as planned on the device); cap entries */
int dab_pair_get_corridors(dab_pair *pair, dab_corridor *out, int32_t cap, int32_t *n_corridors);
/* final path rows (video j, audio i, cluster, qual, cum), float64 row-major (n_path, 5),
 * in frames (the /210 scaling of :1026 is the caller's). */
int dab_pair_get_path2(dab_pair *pair, double *rows);
/* pass-2 points sorted by (i, j, cluster); any pointer may be NULL. */
int dab_pair_get_points2(dab_pair *pair, int32_t *i_audio, double *j_video, int32_t *cluster, double *qual);

int dab_pair_get_stats(dab_pair *pair, dab_stats *out);

/* Device-side time of the kernels of the last stage_a / stage_b / set_pcm call on this pair,
 * in milliseconds, measured with CUDA events on the pair's stream; slots:
 * 0 features(video) 1 features(audio) 2 prep+codes 3 tables 4 gate 5 score 6 dp1+traceback
 * 7 corridor scoring 8 dp2+traceback 9 dp2 alone; and HOST wall time spent inside the library for
 * this pair since its last video set_pcm: 10 set_pcm/set_features 11 stage A 12 stage B 13 get_*
 * copies.  Slots not run since creation are 0. */
int dab_pair_get_timings(dab_pair *pair, float ms[16]);
/* Where on the device's clock the stages 0-8 above started and ended, in milliseconds after
 * `ref_event` (a cudaEvent_t recorded with timing by the caller, e.g. at the start of a batch);
 * -1 for stages not run.  With many pairs in flight this is the timeline of the batch. */
int dab_pair_get_timeline(dab_pair *pair, void *ref_event, float start_ms[9], float end_ms[9]);
/* number of kernel launches issued by this context since creation */
int64_t dab_launch_count(const dab_ctx *ctx);

/* ---- batch engine (reference describealign.py:1077, the per-pair loop of batch mode) -----------------
 * Many pairs in flight on one GPU without a host thread per pair: the caller submits jobs and then
 * serves a queue of events.  A pair occupies one of the engine's slots (device buffers + a CUDA stream)
 * and goes   submit -> [upload, features, stage A on the device] -> DAB_EVENT_STAGE_A
 *            -> caller runs the host fit (:702-893) and answers with dab_engine_submit_b
 *            -> [stage B on the device] -> DAB_EVENT_STAGE_B -> caller reads the path, dab_engine_release.
 * One scheduler thread inside the library enqueues every device stage in one go and polls CUDA events;
 * it never blocks on a stream.  All result pointers of an event are page-locked host memory owned by the
 * slot, valid until the slot's next dab_engine_submit_b (stage A results) or dab_engine_release.
 * The PCM buffers of a job must stay valid until the job's DAB_EVENT_STAGE_A (page-locked memory makes
 * the uploads asynchronous DMA).  Any thread may call these functions; events are handed out once. */
typedef struct dab_engine dab_engine;

typedef struct {
  uint64_t tag;             /* caller's id of the pair, returned with its events */
  const void *pcm[2];       /* [DAB_TRACK_VIDEO], [DAB_TRACK_AUDIO]: interleaved samples, host or device memory */
  int64_t samples[2];       /* per channel */
  int32_t channels[2];      /* 1 or 2 */
  int32_t format;           /* DAB_PCM_* */
  int32_t on_device;        /* != 0: pcm[] are device pointers (no upload) */
} dab_job;

enum { DAB_EVENT_STAGE_A = 1, DAB_EVENT_STAGE_B = 2 };

typedef struct {
  int32_t kind;             /* DAB_EVENT_* */
  int32_t slot;             /* handle for dab_engine_submit_b / dab_engine_release */
  uint64_t tag;
  int32_t status;           /* DAB_OK, or the DAB_E_* code the pair failed with (dab_engine_slot_error) */
  int32_t reserved;
  /* stage A: pass-1 path (audio frame x, video frame y) and the first three feature vectors of each track
   * (what the host fit reads, :706-741) */
  int64_t n_path1;
  const int32_t *path_x, *path_y;
  const float *features[2][3];
  int64_t feature_len[2][3];
  /* stage B: final path rows (video j, audio i, cluster, qual, cum), row-major (n_path2, 5), in frames */
  int64_t n_path2;
  const double *rows;
  dab_stats stats;
  /* as dab_pair_get_timings, except slots 10-13: [10] scheduler time spent enqueueing this pair's work,
   * [11] submit -> stage A results on the host, [12] stage-B input -> final path on the host (ms) */
  float timings_ms[16];
} dab_event;

/* input of stage B, as dab_pair_stage_b_clusters */
typedef struct {
  float gain[3], audio_std[3];
  int64_t n_audio, n_video;
  int32_t n_clusters;
  const dab_cluster *clusters;     /* n_clusters line clusters (copied by dab_engine_submit_b) */
} dab_stage_b_in;

int dab_engine_create(dab_ctx *ctx, int32_t slots, dab_engine **out);
void dab_engine_destroy(dab_engine *engine);
int dab_engine_submit(dab_engine *engine, const dab_job *job);     /* queued; starts when a slot is free */
/* timeout_ms < 0: wait for ever; 0: poll.  Returns DAB_OK, DAB_E_TIMEOUT or DAB_E_ARG. */
int dab_engine_next(dab_engine *engine, dab_event *out, int32_t timeout_ms);
int dab_engine_submit_b(dab_engine *engine, int32_t slot, const dab_stage_b_in *in);
int dab_engine_release(dab_engine *engine, int32_t slot);
const char *dab_engine_slot_error(dab_engine *engine, int32_t slot);
/* the dab_pair behind a slot, for introspection between DAB_EVENT_STAGE_B and dab_engine_release */
void *dab_engine_slot_pair(dab_engine *engine, int32_t slot);
/* out[0] scheduler loop iterations, out[1] iterations that found nothing to do and slept 20 us */
void dab_engine_counters(dab_engine *engine, int64_t out[4]);

/* ---------------------------------------------------------------------------------------------------------
 * Host stage in native code (SURVEY.md 8f N1): the parts of the "rate-change fit" of align() that are plain
 * array arithmetic - reference describealign.py:706-724 (continuity error), :743-767 (70 -> 1 compression of
 * the pass-1 path) and :769-836 (assembly of the L1 programme).  scipy.optimize.linprog itself stays with the
 * caller.  Every sum is formed in numpy's / OpenBLAS' order (csrc/host_stage.cpp); no device is needed.
 * --------------------------------------------------------------------------------------------------------- */
/* err[n - (deriv != 0)]; n >= 51.  x, y: the pass-1 path (audio frame, video frame). */
int dab_host_continuity_error(const int64_t *x, const int64_t *y, int64_t n, int deriv, double *err);
/* the same on float64 input (either the float or the integer pair of pointers is given, the other is NULL) */
int dab_host_continuity_error_f64(const double *x, const double *y, const int64_t *xi, const int64_t *yi, int64_t n,
                                  int deriv, double *err);
/* out_x, out_y: room for n entries; *n_out = number of fit points.  DAB_E_ARG when the path is too short
 * (n <= 90: the reference raises "Alignment failed, are the input files mismatched?"). */
int dab_host_compress_path(const int64_t *x, const int64_t *y, int64_t n, double *out_x, double *out_y, int64_t *n_out);
/* cost[12n-9]; A_eq (3n-4 rows x 12n-9 columns) in CSC with sorted row indices: indptr[12n-8], indices / data
 * with room for 24n entries (23n - 21 are written), *nnz = entries written; b_eq[3n-4].  n >= 51. */
/* Grouping of the fitted path into co-linear clusters (describealign.py:861-884).  x, y: the n fit points with the fit
 * error removed from y; slopes[n + 1].  out_x / out_y: room for 2n points (a point can vote twice); cluster_start: room
 * for 2n + 1 entries; cluster c is out_*[cluster_start[c] .. cluster_start[c + 1]).  The line fit per cluster
 * (np.linalg.lstsq, describealign.py:886-891) stays with the caller. */
int dab_host_line_clusters(const double *x, const double *y, const double *slopes, int64_t n, double *out_x, double *out_y,
                           int64_t *cluster_start, int64_t *n_clusters);
int dab_host_lp_assemble(const double *x, const double *y, int64_t n, double *cost, int32_t *indptr, int32_t *indices,
                         double *data, double *b_eq, int64_t *nnz);

/* ---------------------------------------------------------------------------------------------------------
 * Decode hand-off (SURVEY.md 8f N2): replaces the tail of parse_audio_from_file, reference
 * describealign.py:149-157 (ffmpeg's s16le pipe -> bytes -> int16 -> float16 on the host).  A reader thread inside
 * the library read()s the decoder's pipe into two page-locked chunks in turn and copies each chunk to the device
 * while the decoder is still running; the int16 -> float16 conversion happens in the feature kernel.
 * --------------------------------------------------------------------------------------------------------- */
typedef struct dab_pcm_reader dab_pcm_reader;
/* fd: read end of the decoder's pipe (or any file descriptor); expected_bytes: size hint (duration x rate x
 * channels x 2) or 0 - the device buffer then grows geometrically.  Returns at once; reading goes on in a thread. */
int dab_pcm_reader_open(dab_ctx *ctx, int fd, int64_t expected_bytes, dab_pcm_reader **out);
int64_t dab_pcm_reader_progress(dab_pcm_reader *reader);       /* bytes handed to the copy engine so far */
/* Blocks until EOF and until every chunk is on the device.  *device_pcm (int16, interleaved) stays valid until
 * dab_pcm_reader_close: pass it to dab_pair_set_pcm(pair, track, ptr, bytes / (2 * channels), channels,
 * DAB_PCM_S16, 1) and close the reader after that pair's features have been computed. */
int dab_pcm_reader_wait(dab_pcm_reader *reader, void **device_pcm, int64_t *bytes);
/* the samples back on the host (int16, interleaved), for --stretch_audio (describealign.py:1142-1150) */
int dab_pcm_reader_copy_to_host(dab_pcm_reader *reader, void *dst, int64_t bytes);
void dab_pcm_reader_close(dab_pcm_reader *reader);

/* ---------------------------------------------------------------------------------------------------------
 * --stretch_audio resynthesis (SURVEY.md 8f N3): the jump search of the reference's pitch-preserving time stretch,
 * describealign.py:252-304 (`get_pearson_corrs_generator`) reduced as :330-333 do.  segment: host pointer to float16
 * (channels, n) row-major, n >= 1535; jumps: n_jumps distances in [1, 512); negative != 0 when the output is longer
 * than the input.  loc[n / 512][n_jumps] (int16) = position inside the window with the largest 512-sample Pearson
 * correlation, best[n / 512][n_jumps] (float64) = that correlation; bit-identical to the reference's float64 running
 * sums (same pieces, same epsilon, same order).  Host buffers; the copies happen inside the call.
 * --------------------------------------------------------------------------------------------------------- */
/* The drift dynamic programme over (window, drift) of `stretch` and its traceback (describealign.py:320-371), host code.
 * loc / best as dab_stretch_best_jumps returns them; out_at / out_dist: room for n_in / 512 entries, *count jumps in input
 * order with unsigned distances.  DAB_E_ARG where the reference's index arithmetic would leave its arrays. */
int dab_host_stretch_plan(int64_t n_in, int64_t n_out, const int32_t *jumps, int32_t n_jumps, const int16_t *loc,
                          const double *best, int64_t *out_at, int64_t *out_dist, int64_t *count);
int dab_stretch_best_jumps(dab_ctx *ctx, const void *segment_f16, int32_t channels, int64_t n, int32_t negative,
                           const int32_t *jumps, int32_t n_jumps, int16_t *loc, double *best);

#ifdef __cplusplus
}
#endif
#endif /* DESCRIBEALIGN_B200_H */
