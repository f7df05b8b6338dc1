// Device stage B of align() (reference describealign.py:895-993):
//   corridor scoring  every audio row inside a cluster's +-30 s corridor gets one point on the
//                     cluster's line; qual from the linearly interpolated video features and the
//                     energy gates; first cluster to claim (i, int(j)) wins          (:931-944)
//   dp2               second frontier DP with global / same-cluster / local steps    (:946-983)
//   trace             traceback (traceback.cu), rows (j, i, cluster, qual, cum)      (:985-990)
//
// The reference keys its frontier by the float video coordinate j.  Here every point gets
// rank(j) = 1 + number of corridor rows (over all corridors) whose coordinate is < j, found by
// one binary search per corridor on the same float expression; equal j share a rank and the
// order is preserved, so the frontier becomes a prefix-max tree over ranks with no sort.
#include "common.cuh"

namespace {

constexpr int MAXC = 32;   // corridors that may overlap one audio row

struct __align__(16) P2Rec {     // one pass-2 point, as the DP walks it
  double j, q;
  int32_t i;
  int32_t kf;      // corridor index | P2_* flags
  int32_t cell;    // int(j)
  int32_t ro;      // row offset inside its corridor
};

// static facts about a point, worked out by the (parallel) scoring kernel so that the serial DP
// does not have to:
constexpr int P2_NEAR = 1 << 8;    // a point of another corridor may share its prev_cache cells
constexpr int P2_VIS1 = 1 << 9;    // the corridor's previous point is a prev_cache candidate
constexpr int P2_VIS2 = 1 << 10;   // ... and so is the one before it
constexpr int P2_GAP = 1 << 11;    // the corridor has no point on row i - 1 (its cell was claimed)
constexpr int P2_MAYQ = 1 << 12;   // another corridor has processed rows to the right of j

struct ScoreBArgs {
  const float *a_scaled;   // (n_a, 3)
  const float *v_scaled;   // (n_v, 3)
  int64_t n_a, n_v;
  const dab_corridor *cor;
  int32_t n_cor;
  const float *maxes;      // np.max of the audio / video energy columns (dab_enqueue_column_maxes)
  int32_t *row_count;
  const int32_t *row_off;
  int32_t *p_i, *p_c, *p_rank;
  P2Rec *rec;
  double *p_j, *p_q;
  int32_t *overflow;
  int32_t want_rank;       // the generic DP needs rank(j); the corridor-state DP does not
  int64_t q_lo, q_hi;      // quals are computed for audio rows q_lo <= i < q_hi only (long-pair sharding); others get 0
};

__device__ __forceinline__ double line_at(const dab_corridor &c, int64_t i) {
  // numpy: slope * x + offset on an int64 arange -> f64 multiply, then add (no fma)
  return __dadd_rn(__dmul_rn(c.slope, (double)i), c.offset);
}

// corridors holding a point on row r, in cluster order, with the cells they claimed (:937-941)
__device__ __forceinline__ int claim_row(const ScoreBArgs &s, int64_t r, int *ks, long long *cells) {
  int n = 0;
  if (r < 0 || r >= s.n_a) return 0;
  for (int k = 0; k < s.n_cor; ++k) {
    const dab_corridor c = s.cor[k];
    if (r < c.lo || r >= c.hi) continue;
    const long long cell = (long long)line_at(c, r);
    bool dup = false;
    for (int m = 0; m < n; ++m) dup = dup || (cells[m] == cell);
    if (dup || n == MAXC) continue;
    ks[n] = k; cells[n] = cell; ++n;
  }
  return n;
}

template <bool FILL>
__global__ void corridor_kernel(ScoreBArgs s) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= s.n_a) return;
  double js[MAXC];
  int cs[MAXC], ks[MAXC];
  int n = 0;
  for (int k = 0; k < s.n_cor; ++k) {
    const dab_corridor c = s.cor[k];
    if (i < c.lo || i >= c.hi) continue;
    const double j = line_at(c, i);
    const long long cell = (long long)j;
    bool dup = false;
    for (int m = 0; m < n; ++m) dup = dup || ((long long)js[m] == cell);
    if (dup) continue;     // an earlier (lower-index) cluster already claimed (i, int(j))
    if (n == MAXC) { atomicOr(s.overflow, DAB_OVF_ROWCOR); break; }
    js[n] = j; cs[n] = c.cluster; ks[n] = k; ++n;
  }
  if (!FILL) { s.row_count[i] = n; return; }
  // insertion sort by j (cells are unique within the row, hence so are the j)
  for (int a = 1; a < n; ++a) {
    double j = js[a]; int c = cs[a]; int kk = ks[a]; int b = a - 1;
    while (b >= 0 && js[b] > j) { js[b + 1] = js[b]; cs[b + 1] = cs[b]; ks[b + 1] = ks[b]; --b; }
    js[b + 1] = j; cs[b + 1] = c; ks[b + 1] = kk;
  }
  const int64_t off = s.row_off[i];
  const float a0 = s.a_scaled[i * 3 + 0], a1 = s.a_scaled[i * 3 + 1], a2 = s.a_scaled[i * 3 + 2];
  // which corridors had a point on the two rows before (for the prev_cache visibility flags)
  int ks1[MAXC], ks2[MAXC];
  long long cells1[MAXC], cells2[MAXC];
  const int n1 = claim_row(s, i - 1, ks1, cells1), n2 = claim_row(s, i - 2, ks2, cells2);
  for (int m = 0; m < n; ++m) {
    const double j = js[m];
    const double fl = floor(j);
    const int64_t f = (int64_t)fl;
    const double t = j - fl;
    const double omt = 1.0 - t;
    const float *v0 = s.v_scaled + f * 3, *v1 = v0 + 3;
    const double vl0 = (double)v0[0] * omt + (double)v1[0] * t;
    const double vl1 = (double)v0[1] * omt + (double)v1[1] * t;
    const double vl2 = (double)v0[2] * omt + (double)v1[2] * t;
    double q = 0.0;
    if (i >= s.q_lo && i < s.q_hi) {
      const double t0 = -.5 - log10(1e-4 + fabs((double)a0 - vl0));
      const double t1 = -.5 - log10(1e-4 + fabs((double)a1 - vl1));
      const double t2 = -.5 - log10(1e-4 + fabs((double)a2 - vl2));
      q = (t0 + t1) + t2;
      const float v_max = s.maxes[1], a_max = s.maxes[0];
      q = q * fmin(fmax((vl0 + 2.5) - (double)v_max, 0.0), 1.0);
      // the audio gate is evaluated in float32 by numpy (f32 array, weak Python scalars)
      float ag = (a0 + 2.5f) - a_max;
      ag = fminf(fmaxf(ag, 0.0f), 1.0f) * 0.1f;
      q = q + (double)ag;
    }
    // rank of j over all corridor rows
    int rank = 1;
    if (s.want_rank) {
      for (int k = 0; k < s.n_cor; ++k) {
        const dab_corridor c = s.cor[k];
        int lo = c.lo, hi = c.hi;        // first row in [lo, hi) whose coordinate is >= j
        while (lo < hi) {
          const int mid = lo + ((hi - lo) >> 1);
          if (line_at(c, mid) < j) lo = mid + 1; else hi = mid;
        }
        rank += lo - c.lo;
      }
    }
    // neighbourhood flag for the corridor-state DP: could a point of another corridor have
    // written one of the prev_cache cells int(j)-2 .. int(j) during rows i-2 .. i?  (A superset
    // test on the lines themselves: it ignores which duplicates were dropped.)
    int near = 0;
    const long long cell = (long long)j;
    for (int k = 0; k < s.n_cor; ++k) {
      if (k == ks[m]) continue;
      const dab_corridor c = s.cor[k];
      for (int64_t r = i - 2; r <= i; ++r) {
        if (r < c.lo || r >= c.hi) continue;
        const long long oc = (long long)line_at(c, r);
        near |= (oc >= cell - 2 && oc <= cell);
      }
    }
    s.p_i[off + m] = (int32_t)i;
    s.p_j[off + m] = j;
    s.p_c[off + m] = cs[m];
    s.p_q[off + m] = q;
    s.p_rank[off + m] = rank;
    // own-corridor prev_cache candidates (describealign.py:966-973): the corridor's points on rows
    // i-1 / i-2, as long as their cell is within two of this one and was not overwritten
    bool has1 = false, has2 = false;
    long long cell_a = 0, cell_b = 0;
    for (int e = 0; e < n1; ++e) if (ks1[e] == ks[m]) { has1 = true; cell_a = cells1[e]; }
    for (int e = 0; e < n2; ++e) if (ks2[e] == ks[m]) { has2 = true; cell_b = cells2[e]; }
    const bool vis1 = has1 ? cell_a >= cell - 2 : (has2 && cell_b >= cell - 2);
    const bool vis2 = has1 && has2 && cell_b >= cell - 2 && cell_b != cell_a;
    const int ro = (int)(i - s.cor[ks[m]].lo);
    const bool gap = !has1 && ro > 0;
    // can the frontier's best entry lie to the right of this point?  Only if another corridor has
    // processed rows (< i) with a larger coordinate.
    bool mayq = false;
    for (int k = 0; k < s.n_cor; ++k) {
      if (k == ks[m]) continue;
      const dab_corridor c = s.cor[k];
      if (c.hi <= c.lo || c.lo > i - 1) continue;
      const int64_t r = i - 1 < c.hi - 1 ? i - 1 : c.hi - 1;
      mayq = mayq || line_at(c, r) > j;
    }
    P2Rec rc;
    rc.j = j; rc.q = q; rc.i = (int32_t)i; rc.cell = (int32_t)cell; rc.ro = ro;
    rc.kf = ks[m] | (near ? P2_NEAR : 0) | (vis1 ? P2_VIS1 : 0) | (vis2 ? P2_VIS2 : 0) | (gap ? P2_GAP : 0) |
            (mayq ? P2_MAYQ : 0);
    s.rec[off + m] = rc;
  }
}

// ------------------------------------------------------------------------------------------
// DP #2 (SURVEY.md A.7).  One warp walks the points in (i, j) order.
// ------------------------------------------------------------------------------------------
struct __align__(16) Node2 {
  double val;     // cum - 1000 of the best point in the subtree, -inf = empty
  int32_t id;     // point id, -1 = the seed (0, 0, -1, 0, 0)
  int32_t rank;
};

struct __align__(16) Cell2 {   // prev_cache row
  double j, q, cum;
  int32_t i, c, id, pad;       // id -2 = never written
};

constexpr int L2N = 5;          // 32^5 ranks

struct Dp2Args {
  const int32_t *p_i, *p_c, *p_rank;
  const double *p_j, *p_q;
  const int32_t *n_points;   // device count
  Node2 *level[L2N];
  Cell2 *cache;
  double *cb_val;     // per cluster: cum - 50 of its best point
  int32_t *cb_id;
  BackRec *back;
  int32_t *result;    // [0] end id ; double result_val at +2
};

__device__ __forceinline__ unsigned long long order_bits(double v) {
  unsigned long long b = (unsigned long long)__double_as_longlong(v);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}

__device__ __forceinline__ bool key2_better(double va, int ra, double vb, int rb) {
  return va > vb || (va == vb && ra < rb);
}

__global__ void __launch_bounds__(32, 1) dp2_kernel(Dp2Args a) {
  const int lane = threadIdx.x;
  const int n = *a.n_points;
  // the overall best frontier entry: starts as the seed (val 0 at rank 0)
  double top_val = 0.0;
  int top_id = -1, top_rank = 0;
  for (int p = 0; p < n; ++p) {
    const int r = a.p_rank[p];
    const int i = a.p_i[p], c = a.p_c[p];
    const double j = a.p_j[p], q = a.p_q[p];
    Node2 nd[L2N];
    int pos[L2N];
#pragma unroll
    for (int k = 0; k < L2N; ++k) {
      const int g = r >> (5 * k);
      pos[k] = g & 31;
      nd[k] = a.level[k][(g & ~31) + lane];
    }
    const long long ij = (long long)j;
    const long long c_lo = ij - 2 > 0 ? ij - 2 : 0;
    // prev_cache cells ij-2 .. ij and the cluster's best, fetched alongside the tree rows
    Cell2 cell[3];
#pragma unroll
    for (int m = 0; m < 3; ++m) {
      const long long idx = ij - 2 + m;
      if (idx >= c_lo) cell[m] = a.cache[idx]; else cell[m].id = -2;
    }
    const double cl_val = a.cb_val[c];
    const int cl_id = a.cb_id[c];

    // (1) global frontier: best val among ranks <= r ; ties -> smaller rank
    double bv = -INFINITY;
    int bid = -2, brank = 0x7fffffff;
#pragma unroll
    for (int k = L2N - 1; k >= 0; --k) {
      const bool elig = (k == 0) ? (lane <= pos[0]) : (lane < pos[k]);
      if (elig && key2_better(nd[k].val, nd[k].rank, bv, brank)) { bv = nd[k].val; bid = nd[k].id; brank = nd[k].rank; }
    }
    const unsigned long long bits = order_bits(bv);
    const unsigned hi = (unsigned)(bits >> 32), lo = (unsigned)bits;
    const unsigned mhi = __reduce_max_sync(0xffffffffu, hi);
    bool alive = hi == mhi;
    const unsigned mlo = __reduce_max_sync(0xffffffffu, alive ? lo : 0u);
    alive = alive && lo == mlo;
    const unsigned mr = __reduce_min_sync(0xffffffffu, alive ? (unsigned)brank : 0xffffffffu);
    alive = alive && (unsigned)brank == mr;
    const int src = __ffs(__ballot_sync(0xffffffffu, alive)) - 1;
    const double front_val = __shfl_sync(0xffffffffu, bv, src);
    const int front_id = __shfl_sync(0xffffffffu, bid, src);

    double best = front_val;
    int pred = front_id;
    // (2) same-cluster jump
    if (cl_val >= best) { best = cl_val; pred = cl_id; }
    // (3) local steps
#pragma unroll
    for (int m = 0; m < 3; ++m) {
      if (cell[m].id == -2) continue;
      double cum = cell[m].cum;
      if (c != cell[m].c) {
        const double d = (j - cell[m].j) - (double)(i - cell[m].i);
        cum = cum - (100.0 + 100.0 * (d * d));
      }
      if (cell[m].i >= i - 2 && cell[m].j <= j && cum >= best) { best = cum; pred = cell[m].id; }
    }
    const double cum = best + q;
    if (lane == 0) {
      Cell2 me; me.j = j; me.q = q; me.cum = cum; me.i = i; me.c = c; me.id = p; me.pad = 0;
      a.cache[ij] = me;
      // the BackRec {best, pred, 0} as one double2: a struct copy here costs this kernel 12 more registers
      *reinterpret_cast<double2 *>(a.back + p) = make_double2(best, __hiloint2double(0, pred));
      if (cl_val < cum - 50.0) { a.cb_val[c] = cum - 50.0; a.cb_id[c] = p; }
    }
    const double jump = cum - 1000.0;
    if (front_val < jump) {
      // leaf: keep the earlier entry on equal val (strictly greater replaces)
      if (lane == pos[0] && jump > nd[0].val) {
        Node2 me; me.val = jump; me.id = p; me.rank = r;
        a.level[0][r] = me;
      }
#pragma unroll
      for (int k = 1; k < L2N; ++k) {
        if (lane == pos[k] && key2_better(jump, r, nd[k].val, nd[k].rank)) {
          Node2 me; me.val = jump; me.id = p; me.rank = r;
          a.level[k][r >> (5 * k)] = me;
        }
      }
      if (key2_better(jump, r, top_val, top_rank)) { top_val = jump; top_id = p; top_rank = r; }
    }
    __syncwarp();
  }
  if (lane == 0) {
    a.result[0] = top_id;
    *reinterpret_cast<double *>(a.result + 2) = top_val;
  }
}

__global__ void init_dp2_kernel(Node2 *nodes, int64_t n_nodes, Cell2 *cache, int64_t n_cells, double *cb_val,
                                int32_t *cb_id, int32_t n_clusters, const int64_t *level_off) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n_nodes) {
    Node2 z; z.val = -INFINITY; z.id = -2; z.rank = 0x7fffffff;
    // rank 0 of every level lies on the seed's path: the seed (0, 0, -1, 0, 0) has val 0
    bool seed = false;
#pragma unroll
    for (int k = 0; k < L2N; ++k) seed = seed || (t == level_off[k]);
    if (seed) { z.val = 0.0; z.id = -1; z.rank = 0; }
    nodes[t] = z;
  }
  if (t < n_cells) {
    Cell2 e; e.j = 0; e.q = 0; e.cum = 0; e.i = 0; e.c = -1; e.id = (t == 0) ? -1 : -2; e.pad = 0;
    cache[t] = e;
  }
  if (t < n_clusters) { cb_val[t] = -1000.0; cb_id[t] = -1; }
}

// ------------------------------------------------------------------------------------------
// DP #2, corridor-state formulation (the fast path; the tree kernel above stays as the generic
// fallback for > 32 corridors or lines with non-positive slope).
//
// Every point lies on one of <= 32 corridor lines j = slope * i + offset with slope > 0, so
//   * prev_cache (describealign.py:956, 966-973) only ever yields points of rows i-2 .. i: the
//     last three points of each corridor are enough state ("history");
//   * the frontier (describealign.py:946, 961-962, 976-981) seen from (i, j) is
//         F(j) = max over corridors c' of PM_c'[ #rows of c' processed so far with j' <= j ]
//     where PM_c' is the running maximum of cum - 1000 along corridor c' (ties: earliest row),
//     because j' grows with the row inside a corridor.  PM_c' is append-only, lives in HBM,
//     its last 16 rows in shared memory;
//   * when the frontier's top entry lies at j' <= j it IS F(j): no query at all.  A query is
//     only needed for points below the top's coordinate whose own candidates do not already
//     beat the top value; then lane c' looks PM_c' up (head / recent ring / a small per-lane
//     window cache of older rows, refilled 16 rows at a time) and the warp arg-max-reduces.
// One warp walks the points in (i, j) order; the state of the corridor being extended lives in
// registers (uniform across lanes), the other corridors' state in shared memory.  The dependent
// chain per point is compare + select + one f64 add.  cum values are bit-identical to the
// reference because every cum is still "chosen predecessor value + qual".
// ------------------------------------------------------------------------------------------
struct __align__(16) PmEntry {
  double val;
  int32_t id;
  int32_t pad;
};

struct Dp2LArgs {
  const P2Rec *rec;
  const double *p_j;
  const int32_t *n_points;   // device count
  const dab_corridor *cor;
  int32_t n_cor;
  int64_t pm_off[32];        // first PM row of each corridor
  PmEntry *pm;
  BackRec *back;
  int32_t *result;           // [0] end id ; double top value at +2
  unsigned long long *counters;   // [0] frontier queries, [1] window refills, [2] neighbour points
};

#include "dp2_scan.cuh"
#include "refine.cuh"

}  // namespace

// The corridor-state DP needs: at most 32 corridors, positive slopes, every coordinate >= 3 (so the
// seeded prev_cache cell 0 is never in reach; x_limits keeps lines >= 4, describealign.py:898).
static bool corridor_dp_eligible(const StageBPlan &b, int dp2_impl) {
  if (dp2_impl == 2 || b.cor.size() > 32) return false;   // dp2_impl 2: the tree DP (cross-checks)
  for (const dab_corridor &c : b.cor) {
    if (!(c.slope > 0.0)) return false;
    // (device-planned corridors: the host holds row ranges that contain the planned ones; the planned lines
    // start at coordinate >= 4 by construction, describealign.py:898)
    if (!b.device_planned && c.hi > c.lo && !(c.slope * (double)c.lo + c.offset >= 3.0)) return false;
  }
  return true;
}

void dab_set_stage_b_plan(dab_pair *pr, int64_t n_audio, int64_t n_video, std::vector<dab_corridor> cor, int32_t n_clusters,
                          bool device_planned) {
  StageBPlan b;
  b.n_audio = n_audio;
  b.n_video = n_video;
  b.cor = std::move(cor);
  b.n_clusters = n_clusters;
  b.device_planned = device_planned;
  for (size_t k = 0; k < b.cor.size(); ++k) {
    if (k < 32) b.pm_off[k] = b.rows;
    b.rows += b.cor[k].hi > b.cor[k].lo ? b.cor[k].hi - b.cor[k].lo : 0;
  }
  b.scan_dp = corridor_dp_eligible(b, pr->ctx->opt_dp2_impl);
  pr->plan_b = std::move(b);
  pr->stats.n_audio_frames = n_audio;
  pr->stats.n_video_frames = n_video;
}

// describealign.py:737-741 on the device: audio_scaled = audio / std(audio), video_scaled =
// video * gain / std(audio), float32 with numpy's roundings (one division; one multiply then one
// division), stacked as (n, 3).  The feature vectors are the pair's own device copies.
__global__ void scale_features_kernel(const float *f0, const float *f1, const float *f2, int64_t n, float g0, float g1,
                                      float g2, float s0, float s1, float s2, int with_gain, float *out) {
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  float x0 = f0[k], x1 = f1[k], x2 = f2[k];
  if (with_gain) { x0 = __fmul_rn(x0, g0); x1 = __fmul_rn(x1, g1); x2 = __fmul_rn(x2, g2); }
  out[3 * k + 0] = __fdiv_rn(x0, s0);
  out[3 * k + 1] = __fdiv_rn(x1, s1);
  out[3 * k + 2] = __fdiv_rn(x2, s2);
}

static int enqueue_scaling(dab_pair *pr, const float gain[3], const float audio_std[3], int64_t n_audio, int64_t n_video) {
  dab_ctx *ctx = pr->ctx;
  if (!gain || !audio_std || n_audio <= 0 || n_video <= 8) {
    dab_set_err(ctx, "stage B: invalid argument");
    return DAB_E_ARG;
  }
  Track &V = pr->trk[DAB_TRACK_VIDEO], &A = pr->trk[DAB_TRACK_AUDIO];
  if (!V.have_features || !A.have_features) { dab_set_err(ctx, "stage B: the pair holds no features"); return DAB_E_STATE; }
  // np.stack truncates to the shortest of the three vectors (energy may be one longer)
  const int64_t na = A.L < A.Le ? A.L : A.Le, nv = V.L < V.Le ? V.L : V.Le;
  if (n_audio != na || n_video != nv) { dab_set_err(ctx, "stage B: lengths differ from the pair's features"); return DAB_E_ARG; }
  DAB_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = pr->stream;
  DAB_TRY(dab_ensure(ctx, pr->a_scaled, sizeof(float) * 3 * (size_t)n_audio));
  DAB_TRY(dab_ensure(ctx, pr->v_scaled, sizeof(float) * 3 * (size_t)n_video));
  scale_features_kernel<<<(unsigned)cdiv(n_audio, 256), 256, 0, st>>>(A.energy.as<float>(), A.zc.as<float>(), A.b0.as<float>(),
      n_audio, 1.f, 1.f, 1.f, audio_std[0], audio_std[1], audio_std[2], 0, pr->a_scaled.as<float>());
  scale_features_kernel<<<(unsigned)cdiv(n_video, 256), 256, 0, st>>>(V.energy.as<float>(), V.zc.as<float>(), V.b0.as<float>(),
      n_video, gain[0], gain[1], gain[2], audio_std[0], audio_std[1], audio_std[2], 1, pr->v_scaled.as<float>());
  ctx->launches += 2;
  DAB_CUDA(cudaGetLastError());
  return DAB_OK;
}

// describealign.py:895-900 on the host, for buffer sizes only (the device computes the ranges it scores)
static void host_x_limits(double x_first, double x_last, double offset, double slope, int64_t n_a, int64_t n_v,
                          long long extend, long long &lo, long long &hi) {
  auto to_ll = [](double x) { return !(x > -9.0e15) ? -9000000000000000LL : (!(x < 9.0e15) ? 9000000000000000LL : (long long)x); };
  lo = to_ll(x_first) - extend;
  if (lo < 0) lo = 0;
  hi = to_ll(x_last) + extend;
  if (hi > n_a - 1) hi = n_a - 1;
  const long long l2 = to_ll(ceil((4.0 - offset) / slope));
  const long long h2 = to_ll(floor(((double)(n_v - 4) - offset) / slope));
  if (l2 > lo) lo = l2;
  if (h2 < hi) hi = h2;
}

// np.max of the energy columns of the scaled arrays (describealign.py:908-909) into pr->maxes[0] (audio),
// pr->maxes[1] (video); enqueued after the scaled arrays, before the corridor scoring that reads them.
int dab_enqueue_column_maxes(dab_pair *pr, int64_t n_a, int64_t n_v) {
  dab_ctx *ctx = pr->ctx;
  cudaStream_t st = pr->stream;
  DAB_TRY(dab_ensure(ctx, pr->maxes, sizeof(float) * 4));
  unsigned int *max_keys = reinterpret_cast<unsigned int *>(pr->maxes.as<float>() + 2);
  DAB_CUDA(cudaMemsetAsync(max_keys, 0, 2 * sizeof(unsigned int), st));
  column_max_kernel<<<dim3(64, 2), 256, 0, st>>>(pr->a_scaled.as<float>(), n_a, pr->v_scaled.as<float>(), n_v, max_keys);
  column_max_decode_kernel<<<1, 32, 0, st>>>(max_keys, pr->maxes.as<float>());
  ctx->launches += 2;
  return DAB_OK;
}

// Corridor planning on the device (refine.cuh).  `clusters` is read by an asynchronous copy: it must stay
// valid until the stream has consumed it.  The plan's host corridors are row ranges that CONTAIN the planned
// ones (the refined offset moves the limits by at most 2 / slope rows), for buffer sizes.
static int enqueue_plan_corridors(dab_pair *pr, const dab_cluster *clusters, int32_t n_clusters, int64_t n_a, int64_t n_v) {
  dab_ctx *ctx = pr->ctx;
  cudaStream_t st = pr->stream;
  std::vector<dab_corridor> cor;
  for (int k = 0; k < n_clusters; ++k) {
    const dab_cluster &c = clusters[k];
    if (c.cluster < 0 || (k > 0 && c.cluster <= clusters[k - 1].cluster) || !(c.slope == c.slope) || c.slope == 0.0) {
      dab_set_err(ctx, "dab_pair_stage_b_clusters: clusters must be in ascending cluster order with a non-zero slope");
      return DAB_E_ARG;
    }
    long long lo, hi;
    host_x_limits(c.x_first, c.x_last, c.offset, c.slope, n_a, n_v, 0, lo, hi);
    dab_corridor out;
    out.cluster = c.cluster; out.lo = 0; out.hi = 0; out.reserved = 0; out.slope = c.slope; out.offset = c.offset;
    if (!(hi < lo + 5)) {
      double xf = c.x_first, xl = c.x_last;
      if (hi > lo + 100) { xf = (double)lo; xl = (double)(hi - 1); }
      // widest range any |coef| < 2 can give: the audio-side limits only
      long long lo2 = (long long)xf - 6300, hi2 = (long long)xl + 6300;
      if (lo2 < 0) lo2 = 0;
      if (hi2 > n_a - 1) hi2 = n_a - 1;
      if (hi2 > lo2) { out.lo = (int32_t)lo2; out.hi = (int32_t)hi2; }
    }
    cor.push_back(out);
  }
  const int max_blocks = (int)cdiv(n_a > 0 ? n_a : 1, RF_CHUNK);
  DAB_TRY(dab_ensure(ctx, pr->clusters, sizeof(dab_cluster) * (size_t)(n_clusters + 1)));
  DAB_TRY(dab_ensure(ctx, pr->corridors, sizeof(dab_corridor) * (size_t)(n_clusters + 1)));
  DAB_TRY(dab_ensure(ctx, pr->refine_partial, sizeof(double) * 4 * (size_t)max_blocks * (size_t)(n_clusters + 1)));
  DAB_TRY(dab_enqueue_column_maxes(pr, n_a, n_v));
  if (n_clusters > 0) {
    DAB_CUDA(cudaMemcpyAsync(pr->clusters.p, clusters, sizeof(dab_cluster) * (size_t)n_clusters, cudaMemcpyHostToDevice, st));
    RefineArgs ra;
    ra.a_scaled = pr->a_scaled.as<float>(); ra.v_scaled = pr->v_scaled.as<float>();
    ra.n_a = n_a; ra.n_v = n_v;
    ra.cl = pr->clusters.as<dab_cluster>(); ra.n_cl = n_clusters; ra.max_blocks = max_blocks;
    ra.partial = pr->refine_partial.as<double>();
    ra.cor = pr->corridors.as<dab_corridor>();
    refine_partial_kernel<<<dim3((unsigned)max_blocks, (unsigned)n_clusters), RF_THREADS, 0, st>>>(ra);
    refine_plan_kernel<<<(unsigned)cdiv(n_clusters, 64), 64, 0, st>>>(ra);
    ctx->launches += 2;
  }
  DAB_CUDA(cudaGetLastError());
  dab_set_stage_b_plan(pr, n_a, n_v, std::move(cor), n_clusters > 0 ? clusters[n_clusters - 1].cluster + 1 : 0, true);
  return DAB_OK;
}

int dab_enqueue_stage_b_clusters(dab_pair *pr, const float gain[3], const float audio_std[3], int64_t n_audio, int64_t n_video,
                                 const dab_cluster *clusters, int32_t n_clusters, int64_t row_lo, int64_t row_hi, bool with_dp,
                                 const char *who) {
  if (n_clusters < 0 || (n_clusters > 0 && !clusters) || row_lo < 0 || row_hi < row_lo) {
    dab_set_err(pr->ctx, std::string(who) + ": invalid argument");
    return DAB_E_ARG;
  }
  DAB_TRY(enqueue_scaling(pr, gain, audio_std, n_audio, n_video));
  DAB_TRY(enqueue_plan_corridors(pr, clusters, n_clusters, n_audio, n_video));
  return dab_enqueue_stage_b(pr, row_lo, row_hi, with_dp);
}

// corridor scoring: the sorted point list with flags; quals only for audio rows [q_lo, q_hi)
static int enqueue_points(dab_pair *pr, int64_t q_lo, int64_t q_hi) {
  dab_ctx *ctx = pr->ctx;
  cudaStream_t st = pr->stream;
  const StageBPlan &b = pr->plan_b;
  const int64_t n_a = b.n_audio, n_v = b.n_video, rows = b.rows;
  const int32_t n_cor = (int32_t)b.cor.size();
  pr->n_points2 = pr->n_path2 = 0;
  const int64_t cap = rows > 0 ? rows : 1;
  DAB_TRY(dab_ensure(ctx, pr->counters, sizeof(int32_t) * DC_WORDS));
  int32_t *dc = pr->counters.as<int32_t>();
  DAB_CUDA(cudaMemsetAsync(dc + DC_N_PTS2, 0, sizeof(int32_t) * (DC_WORDS - DC_N_PTS2), st));
  ScoreBArgs sb;
  sb.a_scaled = pr->a_scaled.as<float>(); sb.v_scaled = pr->v_scaled.as<float>();
  sb.n_a = n_a; sb.n_v = n_v;
  sb.cor = pr->corridors.as<dab_corridor>(); sb.n_cor = n_cor;
  sb.maxes = pr->maxes.as<float>();
  sb.want_rank = b.scan_dp ? 0 : 1;
  sb.q_lo = q_lo; sb.q_hi = q_hi;
  DAB_TRY(dab_ensure(ctx, pr->row2_count, sizeof(int32_t) * (size_t)(n_a + 2)));
  DAB_TRY(dab_ensure(ctx, pr->row2_off, sizeof(int32_t) * (size_t)(n_a + 2)));
  DAB_TRY(dab_ensure(ctx, pr->p2_i, sizeof(int32_t) * (size_t)(cap + 1)));
  DAB_TRY(dab_ensure(ctx, pr->p2_c, sizeof(int32_t) * (size_t)(cap + 1)));
  DAB_TRY(dab_ensure(ctx, pr->p2_rank, sizeof(int32_t) * (size_t)(cap + 1)));
  DAB_TRY(dab_ensure(ctx, pr->p2_k, sizeof(P2Rec) * (size_t)(cap + 1)));
  DAB_TRY(dab_ensure(ctx, pr->p2_j, sizeof(double) * (size_t)(cap + 1)));
  DAB_TRY(dab_ensure(ctx, pr->p2_q, sizeof(double) * (size_t)(cap + 1)));
  DAB_TRY(dab_ensure(ctx, pr->path2, sizeof(double) * 5 * (size_t)(cap + 1)));
  sb.row_count = pr->row2_count.as<int32_t>(); sb.row_off = pr->row2_off.as<int32_t>();
  sb.p_i = pr->p2_i.as<int32_t>(); sb.p_c = pr->p2_c.as<int32_t>(); sb.p_rank = pr->p2_rank.as<int32_t>();
  sb.rec = pr->p2_k.as<P2Rec>();
  sb.p_j = pr->p2_j.as<double>(); sb.p_q = pr->p2_q.as<double>();
  sb.overflow = dc + DC_OVERFLOW_B;
  DAB_CUDA(cudaEventRecord(pr->ev[14], st));
  if (n_a > 0 && n_cor > 0 && rows > 0) {
    const unsigned gb = (unsigned)cdiv(n_a, 128);
    corridor_kernel<false><<<gb, 128, 0, st>>>(sb);
    DAB_TRY(dab_exclusive_scan(pr, sb.row_count, pr->row2_off.as<int32_t>(), n_a, nullptr, dc + DC_N_PTS2));
    corridor_kernel<true><<<gb, 128, 0, st>>>(sb);
    ctx->launches += 2;
  }
  DAB_CUDA(cudaEventRecord(pr->ev[15], st));
  pr->ev_used[7] = true;
  DAB_CUDA(cudaGetLastError());
  return DAB_OK;
}

// DP #2 + traceback over the pair's pass-2 points
int dab_enqueue_stage_b_dp(dab_pair *pr) {
  dab_ctx *ctx = pr->ctx;
  cudaStream_t st = pr->stream;
  const StageBPlan &b = pr->plan_b;
  const int64_t n_v = b.n_video, rows = b.rows;
  const int32_t n_cor = (int32_t)b.cor.size(), n_clusters = b.n_clusters;
  const int64_t cap = rows > 0 ? rows : 1;
  int32_t *dc = pr->counters.as<int32_t>();
  DAB_CUDA(cudaEventRecord(pr->ev[16], st));
  if (rows > 0) DAB_TRY(dab_ensure(ctx, pr->back2, sizeof(BackRec) * (size_t)(cap + 2)));
  if (rows > 0 && b.scan_dp) {
    DAB_TRY(dab_ensure(ctx, pr->pm2, sizeof(PmEntry) * (size_t)(rows + 1)));
    Dp2LArgs la;
    la.rec = pr->p2_k.as<P2Rec>(); la.p_j = pr->p2_j.as<double>();
    la.n_points = dc + DC_N_PTS2;
    la.cor = pr->corridors.as<dab_corridor>(); la.n_cor = n_cor;
    for (int k = 0; k < 32; ++k) la.pm_off[k] = b.pm_off[k];
    la.pm = pr->pm2.as<PmEntry>();
    la.back = pr->back2.as<BackRec>();
    la.result = dc + DC_DP2_END;
    la.counters = reinterpret_cast<unsigned long long *>(dc + DC_DP2_CNT);
    {
      static std::atomic<int> attr_set[64];
      if (ctx->device < 64 && !attr_set[ctx->device].load()) {
        DAB_CUDA(cudaFuncSetAttribute(dp2_scan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(ScanShared)));
        attr_set[ctx->device].store(1);
      }
      dp2_scan_kernel<<<1, SC_T, sizeof(ScanShared), st>>>(la);
    }
    ctx->launches += 1;
  } else if (rows > 0) {
    // ---- generic tree DP (more than 32 corridors, or a line with non-positive slope) ----
    const int64_t dom = 1 + rows;        // rank domain: 1 + total corridor rows
    if (dom > (1LL << (5 * L2N))) { dab_set_err(ctx, "pass-2 rank domain too large"); return DAB_E_CAPACITY; }
    int64_t lv[L2N], loff[L2N], tot = 0, m = dom;
    for (int k = 0; k < L2N; ++k) { lv[k] = cdiv(m > 0 ? m : 1, 32) * 32; loff[k] = tot; tot += lv[k]; m = cdiv(m, 32); }
    DAB_TRY(dab_ensure(ctx, pr->tree2, sizeof(Node2) * (size_t)tot + sizeof(int64_t) * L2N));
    DAB_TRY(dab_ensure(ctx, pr->cache2, sizeof(Cell2) * (size_t)(n_v + 1)));
    DAB_TRY(dab_ensure(ctx, pr->cluster_best2, (sizeof(double) + sizeof(int32_t)) * (size_t)(n_clusters + 1)));
    Node2 *nodes = pr->tree2.as<Node2>();
    int64_t *d_loff = reinterpret_cast<int64_t *>(nodes + tot);
    DAB_CUDA(cudaMemcpyAsync(d_loff, loff, sizeof(int64_t) * L2N, cudaMemcpyHostToDevice, st));
    double *cb_val = pr->cluster_best2.as<double>();
    int32_t *cb_id = reinterpret_cast<int32_t *>(cb_val + (n_clusters + 1));
    int64_t span = tot > n_v ? tot : n_v;
    if (n_clusters > span) span = n_clusters;
    init_dp2_kernel<<<(unsigned)cdiv(span, 256), 256, 0, st>>>(nodes, tot, pr->cache2.as<Cell2>(), n_v, cb_val, cb_id,
                                                              n_clusters, d_loff);
    Dp2Args da;
    da.p_i = pr->p2_i.as<int32_t>(); da.p_c = pr->p2_c.as<int32_t>(); da.p_rank = pr->p2_rank.as<int32_t>();
    da.p_j = pr->p2_j.as<double>(); da.p_q = pr->p2_q.as<double>();
    da.n_points = dc + DC_N_PTS2;
    for (int k = 0; k < L2N; ++k) da.level[k] = nodes + loff[k];
    da.cache = pr->cache2.as<Cell2>(); da.cb_val = cb_val; da.cb_id = cb_id;
    da.back = pr->back2.as<BackRec>(); da.result = dc + DC_DP2_END;
    dp2_kernel<<<1, 32, 0, st>>>(da);
    ctx->launches += 2;
  }
  DAB_CUDA(cudaEventRecord(pr->ev[18], st));
  if (rows > 0) {
    Path2Out out;
    out.p_i = pr->p2_i.as<int32_t>(); out.p_c = pr->p2_c.as<int32_t>();
    out.p_j = pr->p2_j.as<double>(); out.p_q = pr->p2_q.as<double>(); out.rows = pr->path2.as<double>();
    DAB_TRY(dab_enqueue_traceback(pr, pr->back2.as<BackRec>(), dc + DC_N_PTS2, dc + DC_DP2_END, cap, dc + DC_N_PATH2, out));
  }
  DAB_CUDA(cudaEventRecord(pr->ev[17], st));
  pr->ev_used[8] = true;
  DAB_CUDA(cudaGetLastError());
  return DAB_OK;
}

// Stage B enqueued on the pair's stream without a host round trip: every (corridor, row) yields at most
// one point, so the sum of the corridor rows (known to the host) bounds all buffers; the actual point
// count stays on the device and every later kernel reads it from there.
int dab_enqueue_stage_b(dab_pair *pr, int64_t row_lo, int64_t row_hi, bool with_dp) {
  DAB_TRY(enqueue_points(pr, row_lo, row_hi));
  if (with_dp) DAB_TRY(dab_enqueue_stage_b_dp(pr));
  return dab_enqueue_counts(pr);
}

// quals of all pass-2 points replaced by `q_all` (device memory): the exchange step of a long pair whose
// corridor rows were scored on several GPUs
static __global__ void set_quals_kernel(const double *q_all, const int32_t *n_dev, P2Rec *rec, double *p_q) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= *n_dev) return;
  const double q = q_all[p];
  rec[p].q = q;
  p_q[p] = q;
}

int dab_enqueue_set_quals2(dab_pair *pr, const double *d_q_all) {
  dab_ctx *ctx = pr->ctx;
  const int64_t cap = pr->plan_b.rows > 0 ? pr->plan_b.rows : 1;
  set_quals_kernel<<<(unsigned)cdiv(cap, 256), 256, 0, pr->stream>>>(d_q_all, pr->counters.as<int32_t>() + DC_N_PTS2,
                                                                    pr->p2_k.as<P2Rec>(), pr->p2_q.as<double>());
  ctx->launches += 1;
  DAB_CUDA(cudaGetLastError());
  return DAB_OK;
}

// first point and number of points of the audio rows [lo, hi) (needs a finished dab_enqueue_stage_b)
int dab_row_range_points2(dab_pair *pr, int64_t lo, int64_t hi, int64_t *first, int64_t *count) {
  dab_ctx *ctx = pr->ctx;
  const int64_t n_a = pr->plan_b.n_audio;
  lo = lo < 0 ? 0 : (lo > n_a ? n_a : lo);
  hi = hi < lo ? lo : (hi > n_a ? n_a : hi);
  int32_t off[2] = {0, 0};
  DAB_CUDA(cudaMemcpyAsync(&off[0], pr->row2_off.as<int32_t>() + lo, sizeof(int32_t), cudaMemcpyDeviceToHost, pr->stream));
  DAB_CUDA(cudaMemcpyAsync(&off[1], pr->row2_off.as<int32_t>() + hi, sizeof(int32_t), cudaMemcpyDeviceToHost, pr->stream));
  DAB_CUDA(dab_wait_stream(pr->stream));
  *first = off[0];
  *count = off[1] - off[0];
  return DAB_OK;
}

int dab_collect_stage_b(dab_pair *pr, bool with_dp) {
  dab_ctx *ctx = pr->ctx;
  const int32_t *hc = reinterpret_cast<const int32_t *>(pr->h_counters);
  if (hc[DC_OVERFLOW_B] & DAB_OVF_ROWCOR) { dab_set_err(ctx, "more than 32 corridors overlap one audio row"); return DAB_E_CAPACITY; }
  pr->n_points2 = hc[DC_N_PTS2];
  pr->stats.n_points2 = pr->n_points2;
  if (!with_dp) return DAB_OK;
  pr->n_path2 = (pr->n_points2 > 0 && hc[DC_DP2_END] >= 0) ? hc[DC_N_PATH2] : 0;
  pr->stats.n_path2 = pr->n_path2;
  const int64_t *cnt = reinterpret_cast<const int64_t *>(hc + DC_DP2_CNT);
  pr->stats.n_dp2_queries = cnt[0];
  pr->stats.n_dp2_refills = cnt[1];
  pr->stats.n_dp2_neighbour = cnt[2];
  pr->stats.n_dp2_run_points = cnt[3];
  return DAB_OK;
}
