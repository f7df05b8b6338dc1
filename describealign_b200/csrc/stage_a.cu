// Device stage A of align() (reference describealign.py:596-700):
//   prep      41-tap Hann local-mean subtraction, 41-frame sliding L2 norm   (:599-608)
//   codes     7 quantised samples per feature -> packed digits + flags       (:622-628, 638-644)
//   select    not-quiet frames; video keeps every 4th of that list           (:629-630, 657-658)
//   tables    5 direct-address tables over the 7^7 codes, video frames stored under every
//             code reachable through their flagged digits                     (:615-633)
//   gate      per audio query: (>= 2 of tables 0-2) and (table 3 or 4)         (:649-660)
//   score     3 x 41-tap normalised correlation -> prob -> qual                (:662-673)
//   dp1       frontier DP as a prefix-max over video rank, with back pointers  (:654-656, 674-682)
//   trace     chunked traceback of the back pointers (traceback.cu)            (:690-697)
//
// Layout: every per-frame array is structure-of-arrays in HBM (feature-major) so that a warp
// touching consecutive frames reads consecutive addresses.  The hash "dict of sets" of the
// reference becomes a counting-sort CSR (start[code], items[]) per table: 7^7 = 823 543
// codes x 5 tables x 4 B = 16.5 MB of starts, L2 resident.  The gate is evaluated as an
// integer predicate on packed 3-bit digits, so a bucket entry costs five 4-byte loads.
//
// The video's prep, select and tables make up a VideoSide (common.cuh).  dab_enqueue_stage_a builds the pair's own
// in the same run, or runs against a shared index, built once by dab_enqueue_index; gate, scoring and DP 1 only
// read the side they are given.
#include "common.cuh"
#include "hann_tables.h"

namespace {

__constant__ double c_hflip[41];   // flipped 41-tap Hann (np.convolve flips; the window is not bit-symmetric)

// ------------------------------------------------------------------------------------------
// prep: ms = feat - conv_same(feat, hann41)   (f64, OpenBLAS ddot order incl. shorter edge dots)
// ------------------------------------------------------------------------------------------
struct PrepArgs {
  const float *f32[4];
  const double *f64;
  int64_t len[5];     // per-feature length (energy may be one longer)
  int64_t Lp;         // frames kept for ms / nrm storage (min length)
  double *ms;         // [5][Lms]  Lms = max len (stride)
  int64_t stride;
};

__device__ __forceinline__ double feat_at(const PrepArgs &a, int f, int64_t t) {
  return f < 4 ? (double)a.f32[f][t] : a.f64[t];
}

// A block walks MS_TILES consecutive tiles of 256 outputs of one feature; the 296 inputs a tile reads are converted to
// float64 once and staged in shared memory (every input is used by 41 outputs).  The next tile's inputs are fetched
// into registers before the current tile is computed, so the global-load latency (ncu: 6 of 13 stall cycles per
// issue were the long scoreboard with one tile per block) hides behind the 76 FP64 operations per output.
constexpr int MS_TILES = 4;

__global__ void __launch_bounds__(256, 3) meansub_kernel(PrepArgs a) {
  __shared__ double tile[2][256 + 40];
  const int f = blockIdx.y;
  const int64_t n = a.len[f];
  const int64_t first = (int64_t)blockIdx.x * (256 * MS_TILES);
  if (first >= n) return;
  const int tid = threadIdx.x;
  auto fetch = [&](int64_t t0, double &r0, double &r1) {
    const int64_t g0 = t0 - 20 + tid, g1 = g0 + 256;
    r0 = (g0 >= 0 && g0 < n) ? feat_at(a, f, g0) : 0.0;
    r1 = (tid < 40 && g1 >= 0 && g1 < n) ? feat_at(a, f, g1) : 0.0;
  };
  double r0, r1;
  fetch(first, r0, r1);
  tile[0][tid] = r0;
  if (tid < 40) tile[0][256 + tid] = r1;
  __syncthreads();
#pragma unroll 1
  for (int k = 0; k < MS_TILES; ++k) {
    const int64_t t0 = first + 256 * k;
    if (t0 >= n) break;
    const bool has_next = k + 1 < MS_TILES && t0 + 256 < n;
    if (has_next) fetch(t0 + 256, r0, r1);
    const double *cur = tile[k & 1];
    const int64_t base = t0 - 20;
    const int64_t t = t0 + tid;
    if (t < n) {
      int64_t lo = t - 20, hi = t + 21, klo = 0;
      if (lo < 0) { klo = -lo; lo = 0; }
      if (hi > n) hi = n;
      const int m = (int)(hi - lo);
      const double *src = cur + (lo - base);
      auto X = [&](int i) { return src[i]; };
      auto Y = [&](int i) { return c_hflip[klo + i]; };
      // interior outputs (m == 41 implies klo == 0): the window taps are compile-time constant-bank operands
      auto Y0 = [&](int i) { return c_hflip[i]; };
      const double mean = (m == 41) ? ddot41_skx(X, Y0) : ddot_skx(X, Y, m);
      a.ms[(int64_t)f * a.stride + t] = cur[t - base] - mean;
    }
    if (has_next) {
      tile[(k + 1) & 1][tid] = r0;
      if (tid < 40) tile[(k + 1) & 1][256 + tid] = r1;
    }
    __syncthreads();
  }
}

// nrm[t] = max(1e-3, sqrt(sum_{k<41} ms[t+k]^2)) and the digit codes of frame t.
struct CodeArgs {
  const double *ms;     // [5][stride]
  int64_t stride;
  int64_t len[5];
  double *nrm;          // [3][nstride] (features 0..2 only are stored)
  int64_t nstride;
  uint32_t *pack;       // [5][nstride]
  int32_t *code;        // [5][nstride]
  int is_video;
};

__global__ void norm_codes_kernel(CodeArgs a) {
  const int f = blockIdx.y;
  const int64_t ncodes = a.len[f] - 40;
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= ncodes) return;
  const double *m = a.ms + (int64_t)f * a.stride + t;
  auto X = [&](int i) { double v = m[i]; return v * v; };
  auto Y = [&](int) { return 1.0; };
  double nr = sqrt(ddot41_skx(X, Y));
  if (nr < 0.001) nr = 0.001;
  if (f < 3) a.nrm[(int64_t)f * a.nstride + t] = nr;
  uint32_t pk = 0;
  int32_t code = 0, p7 = 1;
  // The digits are floor(8 * (m / nr) + offset) and the flags compare its fraction with .6: integers.  The
  // quotient is first taken as m * (1 / nr) - within 2 ulp of the true quotient - and only a value that
  // lands within 1e-9 of a boundary (an integer, an integer + .6, the clip limits) is divided exactly, so
  // the digits are those of the exact arithmetic with one division per frame instead of seven.
  const double inv = 1.0 / nr;
#pragma unroll
  for (int k = 0; k < 7; ++k) {
    const double mk = m[2 + 6 * k];
    double d = 8.0 * (mk * inv) + (a.is_video ? 3.3 : 3.5);
    {
      const double fr = d - floor(d);
      const bool risky = fr < 1e-9 || fr > 1.0 - 1e-9 || (a.is_video && fabs(fr - 0.6) < 1e-9) || !(fabs(d) < 1e6);
      if (risky) {
        d = mk / nr;
        d = 8.0 * d;
        d = d + (a.is_video ? 3.3 : 3.5);
      }
    }
    int dig;
    if (a.is_video) {
      d = fmin(fmax(d, 0.0), 6.0);
      double fl = floor(d);
      if (d - fl > 0.6) pk |= 8u << (4 * k);
      dig = (int)fl;
    } else {
      double fl = floor(d);
      fl = fmin(fmax(fl, 0.0), 6.0);
      dig = (int)fl;
    }
    pk |= (uint32_t)dig << (4 * k);
    code += dig * p7;
    p7 *= 7;
  }
  a.pack[(int64_t)f * a.nstride + t] = pk;
  a.code[(int64_t)f * a.nstride + t] = code;
}

// ------------------------------------------------------------------------------------------
// scans / compaction
// ------------------------------------------------------------------------------------------
constexpr int SCAN_THREADS = 512;
constexpr int SCAN_ITEMS = 8;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

template <typename T> struct PlainAdd {
  __device__ static T add(T a, T b) { return a + b; }
};

// exclusive scan over the block; Op::add is the (associative) sum
template <typename T, typename Op = PlainAdd<T>>
__device__ __forceinline__ T block_exclusive_scan(T v, T *total, T *smem /* >= 33 */) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  T inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const T y = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc = Op::add(inc, y);
  }
  if (lane == 31) smem[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    T winc = (lane < (int)(blockDim.x >> 5)) ? smem[lane] : T(0);
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const T y = __shfl_up_sync(0xffffffffu, winc, o);
      if (lane >= o) winc = Op::add(winc, y);
    }
    const T wex = __shfl_up_sync(0xffffffffu, winc, 1);
    smem[lane] = lane ? wex : T(0);
    if (lane == 31) smem[32] = winc;
  }
  __syncthreads();
  // exclusive within the warp (a shuffle, not inc - v: a saturated sum cannot be undone), then the warps before it
  T wex = __shfl_up_sync(0xffffffffu, inc, 1);
  if (lane == 0) wex = 0;
  const T res = Op::add(wex, smem[warp]);
  *total = smem[32];
  __syncthreads();
  return res;
}

// n_dev (optional): the number of valid elements lives in device memory (a count produced earlier in
// the same stream); launches are sized for the capacity n and elements past *n_dev count as zero.
__device__ __forceinline__ int64_t scan_len(int64_t n, const int32_t *n_dev) {
  if (!n_dev) return n;
  const int64_t m = *n_dev;
  return m < n ? (m < 0 ? 0 : m) : n;
}

// Single-pass exclusive scan (decoupled look-back): one launch per scan.  Tiles take their index from an
// atomic ticket, so a tile's predecessors have always started; a tile publishes its aggregate, then walks
// back over its predecessors' published (aggregate | inclusive prefix) words until it meets an inclusive
// prefix.  Status words carry the epoch of the scan call, so the array needs no clearing between calls;
// the last tile to finish resets the ticket counter.
//   status[t] = epoch << 34 | kind << 32 | value      kind 1 = aggregate, 2 = inclusive prefix
// The input is int32; the sums are T.  T = int32_t (list offsets, row counts, keep flags) adds with saturation at
// INT32_MAX, which is associative over non-negative values: a total that does not fit reads INT32_MAX instead of
// wrapping.  T = int64_t (the gate's entry prefix) spends two status words per tile, the low and the high half of the
// value, each under the same epoch and kind.  A reader takes a pair only when both words carry this call's epoch and
// the same kind: a tile publishes each kind once per call, so the two halves are of one publication, and a word left
// by an earlier call (other epoch) or a half-updated pair (kinds differ) is read again.  The words are 64-bit
// aligned stores, so each half is seen whole.
template <typename T> struct ScanOps;
template <> struct ScanOps<int32_t> {
  static constexpr int WORDS = 1;
  __device__ static int32_t add(int32_t a, int32_t b) { return (int32_t)min((uint32_t)a + (uint32_t)b, 0x7fffffffu); }
};
template <> struct ScanOps<int64_t> : PlainAdd<int64_t> {
  static constexpr int WORDS = 2;
};

template <typename T>
struct ScanArgs {
  const int32_t *in;
  T *out;
  int64_t n;
  const int32_t *n_dev;
  unsigned long long *status;      // [tiles * ScanOps<T>::WORDS]
  unsigned int *ticket;            // [0] next tile, [1] tiles finished
  unsigned int epoch;              // 1 .. 2^30 - 1, different from the previous call's on this array
  int32_t *total_out;              // the total's int32 words, low word first
};

template <typename T>
__device__ __forceinline__ void scan_publish(volatile unsigned long long *st, unsigned int tile, unsigned long long tag,
                                             unsigned long long kind, T value) {
  const unsigned long long hdr = tag | (kind << 32);
  if constexpr (ScanOps<T>::WORDS == 1) {
    st[tile] = hdr | (uint32_t)value;
  } else {
    st[2 * (size_t)tile] = hdr | (uint32_t)(uint64_t)value;
    st[2 * (size_t)tile + 1] = hdr | (uint32_t)((uint64_t)value >> 32);
  }
}

// tile t's status in this call, waited for: its kind (1 aggregate, 2 inclusive prefix) and value
template <typename T>
__device__ __forceinline__ unsigned scan_wait(volatile unsigned long long *st, int t, unsigned int epoch, T &value) {
  if constexpr (ScanOps<T>::WORDS == 1) {
    unsigned long long w;
    do { w = st[t]; } while ((w >> 34) != epoch);
    value = (int32_t)(uint32_t)w;
    return (unsigned)(w >> 32) & 3u;
  } else {
    unsigned long long lo, hi;
    do {
      lo = st[2 * (size_t)t];
      hi = st[2 * (size_t)t + 1];
    } while ((lo >> 34) != epoch || (hi >> 34) != epoch || ((lo ^ hi) >> 32) != 0ull);
    value = (int64_t)(((hi & 0xffffffffull) << 32) | (lo & 0xffffffffull));
    return (unsigned)(lo >> 32) & 3u;
  }
}

template <typename T>
__global__ void __launch_bounds__(SCAN_THREADS) scan_onepass_kernel(ScanArgs<T> a) {
  using Op = ScanOps<T>;
  __shared__ T sm[33];
  __shared__ unsigned int s_tile;
  __shared__ T s_prefix;
  const int64_t n = scan_len(a.n, a.n_dev);
  if (threadIdx.x == 0) s_tile = atomicAdd(a.ticket, 1u);
  __syncthreads();
  const unsigned int tile = s_tile;
  if ((int64_t)tile > n / SCAN_TILE) {
    // past the tile that holds position n (a device-side count far below the capacity): nobody looks back here
    if (threadIdx.x == 0) {
      const unsigned int done = atomicAdd(a.ticket + 1, 1u);
      if (done == gridDim.x - 1) { a.ticket[0] = 0u; a.ticket[1] = 0u; __threadfence(); }
    }
    return;
  }
  const int64_t base = (int64_t)tile * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
  int32_t v[SCAN_ITEMS];
  T s = 0;
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k) {
    v[k] = (base + k < n) ? a.in[base + k] : 0;
    s = Op::add(s, (T)v[k]);
  }
  T total;
  const T ex = block_exclusive_scan<T, Op>(s, &total, sm);
  if (threadIdx.x < 32) {
    // warp 0 publishes the tile's aggregate, then looks back 32 predecessors at a time
    const int lane = threadIdx.x;
    const unsigned long long tag = (unsigned long long)a.epoch << 34;
    volatile unsigned long long *st = a.status;
    T prefix = 0;
    if (tile > 0) {
      if (lane == 0) { scan_publish<T>(st, tile, tag, 1ull, total); __threadfence(); }
      int end = (int)tile;                      // tiles [.., end) are still to be accounted for
      while (end > 0) {
        const int t = end - 1 - lane;           // lane 0 = nearest predecessor
        T w = 0;
        const unsigned kind = t >= 0 ? scan_wait<T>(st, t, a.epoch, w) : 0u;
        const bool is_prefix = kind == 2u;
        const unsigned pm = __ballot_sync(0xffffffffu, is_prefix);
        const int stop = pm ? __ffs(pm) - 1 : 32;             // nearest lane holding an inclusive prefix
        T x = (t >= 0 && lane <= stop) ? w : T(0);
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) x = Op::add(x, __shfl_xor_sync(0xffffffffu, x, o));
        prefix = Op::add(prefix, x);
        if (pm) break;
        end -= 32;
      }
    }
    if (lane == 0) {
      scan_publish<T>(st, tile, tag, 2ull, Op::add(prefix, total));
      __threadfence();
      s_prefix = prefix;
    }
  }
  __syncthreads();
  T run = Op::add(ex, s_prefix);
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k) {
    if (base + k < n) a.out[base + k] = run;
    run = Op::add(run, (T)v[k]);
  }
  // the tile that holds position n (or the last tile) writes the total
  const int64_t last_tile = n / SCAN_TILE;
  if ((int64_t)tile == last_tile && threadIdx.x == 0) {
    // total of all elements = prefix of this tile + its own total (elements past n are zero)
    const T all = Op::add(s_prefix, total);
    a.out[n] = all;
    if (a.total_out) {
      a.total_out[0] = (int32_t)(uint32_t)(uint64_t)all;
      if constexpr (ScanOps<T>::WORDS == 2) a.total_out[1] = (int32_t)(uint32_t)((uint64_t)all >> 32);
    }
  }
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned int done = atomicAdd(a.ticket + 1, 1u);
    if (done == gridDim.x - 1) { a.ticket[0] = 0u; a.ticket[1] = 0u; __threadfence(); }
  }
}

__global__ void notquiet_flag_kernel(const float *energy, int64_t n, int32_t *flag) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) flag[t] = energy[t] > 0.5f ? 1 : 0;
}

// list[rank / every] = t for flagged t whose rank % every == 0
__global__ void compact_kernel(const int32_t *flag, const int32_t *off, int64_t n, int every, int32_t *list) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n && flag[t]) {
    int r = off[t];
    if (r % every == 0) list[r / every] = (int32_t)t;
  }
}

// ------------------------------------------------------------------------------------------
// tables: a two-level counting sort of the expanded entries by slot f * 7^7 + code
// ------------------------------------------------------------------------------------------
// A hashed video frame is stored under every code reachable through its flagged digits (2^flags codes per table,
// :630-633).  A C2 pair expands 5 x 69 k frames to 3.7 M entries over 4.1 M slots, 88 % of which stay empty, so
// the slots are cut into super-buckets of TB_SB: entries are first sorted by super-bucket (high bits of the slot),
// then every super-bucket sorts its own entries by local slot (low bits) in shared memory.  Nothing touches all
// 4.1 M slots except the coalesced write of start[], and no global atomic is issued per entry.
//   table_count_kernel    thread per hashed frame: its record (below) and a shared-memory histogram of the
//                         super-buckets of its entries; one global add per non-zero bin and CTA
//   table_scan_kernel     one CTA: offsets of the super-buckets; the entry total against the capacity
//   table_scatter_kernel  the same CTAs again: one range per (CTA, super-bucket) reserved by one atomic, the
//                         entries written into it as (local slot, rank)
//   table_sort_kernel     CTA per super-bucket: TB_SB counters in shared memory, start[] of its slots, items[] in
//                         its own range.  The order of the ranks inside a bucket is free (the gate orders what it
//                         finds by rank).
constexpr int TB_SB_BITS = 12, TB_SB = 1 << TB_SB_BITS;
constexpr int64_t TB_NSLOTS = 5LL * DAB_NCODE;
constexpr int TB_NSB = (int)((TB_NSLOTS + TB_SB - 1) / TB_SB);     // 1006, the last one partial
constexpr int TB_THREADS = 256;                                   // count / scatter: one hashed frame per thread
constexpr int TS_THREADS = 512, TS_UNROLL = 4;                    // sort: entries in chunks of TS_THREADS x TS_UNROLL
constexpr int TB_SCAN_THREADS = 1024;
static_assert(TB_NSB <= TB_SCAN_THREADS, "one super-bucket count per thread of the scan");
static_assert(TB_SB == TS_THREADS * 8, "the sort's block scan gives every thread 8 consecutive counters");

__device__ __forceinline__ int32_t pack_to_code(uint32_t pk) {
  int32_t c = 0, p7 = 1;
#pragma unroll
  for (int k = 0; k < 7; ++k) {
    c += (int32_t)((pk >> (4 * k)) & 7u) * p7;
    p7 *= 7;
  }
  return c;
}

// fn(slot) for every slot f * 7^7 + code the digit word pk of table f is stored under
template <typename F>
__device__ __forceinline__ void for_each_slot(int f, uint32_t pk, F &&fn) {
  const int32_t P7[7] = {1, 7, 49, 343, 2401, 16807, 117649};
  const uint32_t fl = pk & 0x8888888u;             // flag bits, one per nibble
  const int32_t base = f * DAB_NCODE + pack_to_code(pk);
  uint32_t sub = fl;
  while (true) {
    int32_t c = base;
#pragma unroll
    for (int k = 0; k < 7; ++k)
      if (sub & (8u << (4 * k))) c += P7[k];
    fn(c);
    if (sub == 0) break;
    sub = (sub - 1) & fl;
  }
}

// The five digit words (one digit per nibble, see digits_match) of every hashed video frame side by side (32 bytes
// per frame, indexed by the frame's rank in the hashed list): a bucket entry then costs the gate ONE 32-byte sector
// instead of a rank -> frame look-up plus five gathers from five arrays.  The count pass writes them; the scatter
// pass reads its digit words back from them.
__global__ void __launch_bounds__(TB_THREADS) table_count_kernel(const uint32_t *pack, int64_t nstride, const int32_t *sel,
                                                                  const int32_t *dc, uint4 *rec, int32_t *sb_count) {
  __shared__ int hist[TB_NSB];
  for (int b = threadIdx.x; b < TB_NSB; b += TB_THREADS) hist[b] = 0;
  __syncthreads();
  const int64_t s = (int64_t)blockIdx.x * TB_THREADS + threadIdx.x;
  if (s < dc[DC_N_VSEL]) {
    const int32_t v = sel[s];
    uint32_t p[5];
#pragma unroll
    for (int f = 0; f < 5; ++f) p[f] = pack[(int64_t)f * nstride + v];
    rec[2 * s] = make_uint4(p[0], p[1], p[2], p[3]);
    rec[2 * s + 1] = make_uint4(p[4], (uint32_t)v, 0u, 0u);
#pragma unroll
    for (int f = 0; f < 5; ++f) for_each_slot(f, p[f], [&](int32_t slot) { atomicAdd(&hist[slot >> TB_SB_BITS], 1); });
  }
  __syncthreads();
  for (int b = threadIdx.x; b < TB_NSB; b += TB_THREADS) {
    const int n = hist[b];
    if (n) atomicAdd(&sb_count[b], n);
  }
}

// sb_off[b] = first entry of super-bucket b (sb_off[TB_NSB] = total), the scatter's cursors = the same; the total
// goes to DC_NEED_ENTRIES and, unless it exceeds the capacity (overflow bit, count 0), to DC_N_ENTRIES
__global__ void __launch_bounds__(TB_SCAN_THREADS) table_scan_kernel(int32_t *dc, int64_t cap, const int32_t *sb_count,
                                                                      int32_t *sb_off, int32_t *sb_cursor) {
  __shared__ int sm[33];
  const int b = threadIdx.x;
  int total;
  const int ex = block_exclusive_scan(b < TB_NSB ? sb_count[b] : 0, &total, sm);
  if (b < TB_NSB) { sb_off[b] = ex; sb_cursor[b] = ex; }
  if (b == 0) {
    sb_off[TB_NSB] = total;
    dc[DC_NEED_ENTRIES] = total;
    if ((int64_t)total > cap) { dc[DC_N_ENTRIES] = 0; atomicOr(&dc[DC_OVERFLOW], DAB_OVF_ENTRIES); }
    else dc[DC_N_ENTRIES] = total;
  }
}

// ent[] = (local slot, rank) of every entry, grouped by super-bucket (any order inside one)
__global__ void __launch_bounds__(TB_THREADS) table_scatter_kernel(const uint4 *rec, const int32_t *dc, int32_t *sb_cursor,
                                                                    uint2 *ent) {
  __shared__ int pos[TB_NSB];
  if (dc[DC_OVERFLOW] & DAB_OVF_ENTRIES) return;
  for (int b = threadIdx.x; b < TB_NSB; b += TB_THREADS) pos[b] = 0;
  __syncthreads();
  const int64_t s = (int64_t)blockIdx.x * TB_THREADS + threadIdx.x;
  const bool live = s < dc[DC_N_VSEL];
  uint32_t p[5] = {0u, 0u, 0u, 0u, 0u};
  if (live) {
    const uint4 r0 = rec[2 * s], r1 = rec[2 * s + 1];
    p[0] = r0.x; p[1] = r0.y; p[2] = r0.z; p[3] = r0.w; p[4] = r1.x;
#pragma unroll
    for (int f = 0; f < 5; ++f) for_each_slot(f, p[f], [&](int32_t slot) { atomicAdd(&pos[slot >> TB_SB_BITS], 1); });
  }
  __syncthreads();
  // this CTA's range in every super-bucket it reaches; pos[] then holds the next free entry of each range
  for (int b = threadIdx.x; b < TB_NSB; b += TB_THREADS) {
    const int n = pos[b];
    if (n) pos[b] = atomicAdd(&sb_cursor[b], n);
  }
  __syncthreads();
  if (live) {
#pragma unroll
    for (int f = 0; f < 5; ++f)
      for_each_slot(f, p[f], [&](int32_t slot) {
        const int at = atomicAdd(&pos[slot >> TB_SB_BITS], 1);
        ent[at] = make_uint2((uint32_t)slot & (TB_SB - 1), (uint32_t)s);
      });
  }
}

// start[] of the super-bucket's TB_SB slots and its entries' ranks in items[].  Its entries are read twice (count,
// then place), TS_THREADS x TS_UNROLL at a time, so a super-bucket of any size is sorted in the same shared memory.
// After an entries overflow every start is 0 (empty tables), as the gate expects.
__global__ void __launch_bounds__(TS_THREADS) table_sort_kernel(const int32_t *dc, const int32_t *sb_off, const uint2 *ent,
                                                                 int32_t *start, int32_t *items) {
  __shared__ __align__(16) int cnt[TB_SB];
  __shared__ int sm[33];
  const int tid = threadIdx.x;
  const int sb = blockIdx.x;
  const bool ovf = (dc[DC_OVERFLOW] & DAB_OVF_ENTRIES) != 0;
  const int lo = ovf ? 0 : sb_off[sb], hi = ovf ? 0 : sb_off[sb + 1];
  for (int j = tid; j < TB_SB; j += TS_THREADS) cnt[j] = 0;
  __syncthreads();
  for (int e0 = lo + tid; e0 < hi; e0 += TS_THREADS * TS_UNROLL) {
    uint32_t key[TS_UNROLL];
#pragma unroll
    for (int u = 0; u < TS_UNROLL; ++u) {
      const int e = e0 + u * TS_THREADS;
      key[u] = e < hi ? ent[e].x : (uint32_t)TB_SB;
    }
#pragma unroll
    for (int u = 0; u < TS_UNROLL; ++u)
      if (key[u] < (uint32_t)TB_SB) atomicAdd(&cnt[key[u]], 1);
  }
  __syncthreads();
  // exclusive scan of the counters, 8 consecutive ones per thread: the slots' starts, written coalesced
  const int4 c0 = *reinterpret_cast<const int4 *>(&cnt[tid * 8]);
  const int4 c1 = *reinterpret_cast<const int4 *>(&cnt[tid * 8 + 4]);
  const int v[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
  int total;
  const int ex = block_exclusive_scan(v[0] + v[1] + v[2] + v[3] + v[4] + v[5] + v[6] + v[7], &total, sm);
  int st[8];
  st[0] = lo + ex;
#pragma unroll
  for (int k = 1; k < 8; ++k) st[k] = st[k - 1] + v[k - 1];
  const int64_t slot0 = (int64_t)sb * TB_SB + tid * 8;
  if (slot0 + 8 <= TB_NSLOTS) {
    reinterpret_cast<int4 *>(start + slot0)[0] = make_int4(st[0], st[1], st[2], st[3]);
    reinterpret_cast<int4 *>(start + slot0)[1] = make_int4(st[4], st[5], st[6], st[7]);
  } else {
#pragma unroll
    for (int k = 0; k < 8; ++k)
      if (slot0 + k < TB_NSLOTS) start[slot0 + k] = st[k];
  }
  if (sb == TB_NSB - 1 && tid == 0) start[TB_NSLOTS] = hi;    // the total (0 after an overflow)
  // counters become the slots' cursors (block_exclusive_scan's barriers order every read of cnt before this)
  *reinterpret_cast<int4 *>(&cnt[tid * 8]) = make_int4(st[0], st[1], st[2], st[3]);
  *reinterpret_cast<int4 *>(&cnt[tid * 8 + 4]) = make_int4(st[4], st[5], st[6], st[7]);
  __syncthreads();
  for (int e0 = lo + tid; e0 < hi; e0 += TS_THREADS * TS_UNROLL) {
    uint2 x[TS_UNROLL];
#pragma unroll
    for (int u = 0; u < TS_UNROLL; ++u) {
      const int e = e0 + u * TS_THREADS;
      x[u] = e < hi ? ent[e] : make_uint2((uint32_t)TB_SB, 0u);
    }
#pragma unroll
    for (int u = 0; u < TS_UNROLL; ++u)
      if (x[u].x < (uint32_t)TB_SB) items[atomicAdd(&cnt[x[u].x], 1)] = (int32_t)x[u].y;
  }
}

// ------------------------------------------------------------------------------------------
// gate
// ------------------------------------------------------------------------------------------
// The gate compares the 7 quantised digits of an audio frame with those of a video frame, per feature
// (SURVEY.md A.4): the frames match in a feature when every audio digit equals the video digit, or the
// video digit + 1 where that digit is flagged (fraction > .6, stored under both codes, :622-633).
// Digits live one per nibble (the format norm_codes_kernel writes): bits 0-2 the digit (0..6), bit 3 the
// flag (video) / a guard bit set by the gate (audio).
//   d = (audio | 0x8888888) - (video digits)         per nibble 8 + a - v, no borrow between nibbles
//   d ^ 0x8888888                                    a - v for a >= v (0..6), >= 10 for a < v
//   ... & ~flags                                     0 exactly when a - v is 0, or 1 on a flagged digit
// i.e. five integer instructions per feature instead of a per-digit loop.
__device__ __forceinline__ bool digits_match(uint32_t a_guarded, uint32_t v) {
  const uint32_t d = (a_guarded - (v & 0x7777777u)) ^ 0x8888888u;
  return (d & ~((v >> 3) & 0x1111111u)) == 0u;
}

constexpr int GATE_STASH = 4;   // rows with at most this many candidates (nearly all) are not enumerated a second time

struct GateArgs {
  const int32_t *a_code;    // [5][a_nstride]
  const uint32_t *a_pack;
  int64_t a_nstride;
  const int32_t *a_list;    // not-quiet audio frames
  const int32_t *dc;        // device counts: query range [DC_Q_LO, DC_Q_HI) of the list
  int64_t q_cap;            // launch size (rows)
  const uint4 *v_rec;       // per hashed video frame (rank): its five digit packs, 32 bytes = one sector
  const int32_t *start;     // [5*NCODE + 1]
  const int32_t *items;
  int32_t *row_count;       // count pass output
  const int32_t *row_off;   // fill pass input
  int32_t *cand_tmp, *cand_s, *cand_i;
  int64_t cand_cap;
  int32_t *stash;           // [q_cap][GATE_STASH]: the first candidates of every row, kept by the count pass
  int32_t *big_list;        // rows with more than GATE_STASH candidates (fill pass work list)
  int32_t *big_count;
};

// Fill pass, rows of up to GATE_STASH candidates (nearly all): thread per query; the candidates the count pass
// stashed are ordered by video rank and written out.  Larger rows go to a work list for gate_fill_big_kernel.
__global__ void gate_fill_small_kernel(GateArgs g) {
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= g.q_cap || q >= g.dc[DC_N_Q]) return;
  if (g.dc[DC_OVERFLOW] & DAB_OVF_CAND) return;
  const int64_t off0 = g.row_off[q];
  const int n_row = g.row_off[q + 1] - (int)off0;
  if (n_row == 0) return;
  if (n_row > GATE_STASH) {
    g.big_list[atomicAdd(g.big_count, 1)] = (int32_t)q;
    return;
  }
  if (off0 + n_row > g.cand_cap) return;
  const int32_t i = g.a_list[g.dc[DC_Q_LO] + q];
  const int4 st = *reinterpret_cast<const int4 *>(g.stash + q * GATE_STASH);
  static_assert(GATE_STASH == 4, "the stash is read as one int4");
  int32_t x[4] = {st.x, n_row > 1 ? st.y : 0x7fffffff, n_row > 2 ? st.z : 0x7fffffff, n_row > 3 ? st.w : 0x7fffffff};
  // sorting network of four
  auto cswap = [&](int a, int b) { if (x[b] < x[a]) { const int32_t t = x[a]; x[a] = x[b]; x[b] = t; } };
  cswap(0, 1); cswap(2, 3); cswap(0, 2); cswap(1, 3); cswap(1, 2);
#pragma unroll
  for (int k = 0; k < 4; ++k)
    if (k < n_row) { g.cand_s[off0 + k] = x[k]; g.cand_i[off0 + k] = i; }
}

// Fill pass, rows with more than GATE_STASH candidates (false-match clusters; a few hundred per pair): a warp per
// row of the work list enumerates the row's two buckets again and orders what it finds by video rank.
__global__ void gate_fill_big_kernel(GateArgs g) {
  const int lane = threadIdx.x & 31;
  const int n_big = *g.big_count;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < n_big; w += n_warps) {
    const int64_t q = g.big_list[w];
    const int32_t i = g.a_list[g.dc[DC_Q_LO] + q];
    // lanes 0-4 fetch the query's five digit words and bucket ranges, one feature each; then broadcast
    uint32_t my_ap = 0u;
    int32_t my_st = 0, my_en = 0;
    if (lane < 5) {
      my_ap = g.a_pack[(int64_t)lane * g.a_nstride + i] | 0x8888888u;
      const int64_t slot = (int64_t)lane * DAB_NCODE + g.a_code[(int64_t)lane * g.a_nstride + i];
      my_st = g.start[slot];
      my_en = g.start[slot + 1];
    }
    uint32_t ap[5];
    int32_t st[5], nb[5];
#pragma unroll
    for (int f = 0; f < 5; ++f) {
      ap[f] = __shfl_sync(0xffffffffu, my_ap, f);
      st[f] = __shfl_sync(0xffffffffu, my_st, f);
      nb[f] = __shfl_sync(0xffffffffu, my_en, f) - st[f];
    }
    // every candidate lies in at least one bucket of any pair out of {0,1,2}, and in bucket 3 or 4
    int fa = 0, fb = 1, best = nb[0] + nb[1];
    if (nb[0] + nb[2] < best) { best = nb[0] + nb[2]; fa = 0; fb = 2; }
    if (nb[1] + nb[2] < best) { best = nb[1] + nb[2]; fa = 1; fb = 2; }
    if (nb[3] + nb[4] < best) { best = nb[3] + nb[4]; fa = 3; fb = 4; }
    int found = 0;
    const int64_t off = g.row_off[q];
    // the two buckets are walked as one list of `best` entries, 32 per step
    const int sa = st[fa], ca = nb[fa], sb = st[fb];
    for (int base = 0; base < best; base += 32) {
      const int e = base + lane;
      bool ok = false;
      int32_t s = 0;
      if (e < best) {
        const bool second = e >= ca;
        s = g.items[second ? sb + (e - ca) : sa + e];
        const uint4 r0 = __ldg(g.v_rec + 2 * (int64_t)s), r1 = __ldg(g.v_rec + 2 * (int64_t)s + 1);
        const uint32_t vp[5] = {r0.x, r0.y, r0.z, r0.w, r1.x};
        bool m[5];
#pragma unroll
        for (int f = 0; f < 5; ++f) m[f] = digits_match(ap[f], vp[f]);
        ok = ((int)m[0] + (int)m[1] + (int)m[2] >= 2) && (m[3] || m[4]);
        if (second && m[fa]) ok = false;   // already enumerated from the first bucket
      }
      const unsigned bal = __ballot_sync(0xffffffffu, ok);
      if (ok) {
        const int64_t pos = off + found + __popc(bal & ((1u << lane) - 1u));
        if (pos < g.cand_cap) g.cand_tmp[pos] = s;
      }
      found += __popc(bal);
    }
    if (off + found > g.cand_cap) continue;
    __syncwarp();
    // order the row's candidates by video rank: position = number of smaller entries
    if (found <= 32) {
      // one candidate per lane, ranks by 32 register shuffles instead of found^2 memory reads
      const int32_t x = lane < found ? g.cand_tmp[off + lane] : 0x7fffffff;
      int r = 0;
#pragma unroll
      for (int j = 0; j < 32; ++j) r += (__shfl_sync(0xffffffffu, x, j) < x);
      if (lane < found) { g.cand_s[off + r] = x; g.cand_i[off + r] = i; }
      continue;
    }
    for (int k = lane; k < found; k += 32) {
      const int32_t x = g.cand_tmp[off + k];
      int r = 0;
      for (int j = 0; j < found; ++j) r += (g.cand_tmp[off + j] < x);
      g.cand_s[off + r] = x;
      g.cand_i[off + r] = i;
    }
  }
}

// ------------------------------------------------------------------------------------------
// gate, count pass, balanced over bucket ENTRIES instead of queries.  A query visits the entries of its two
// cheapest buckets; their number ranges from none to several hundred, so a warp per query leaves most lanes
// idle (ncu: 380 warp instructions per query for 33 entries on average).  Three steps:
//   gate_plan_kernel      thread per query: digit words, the two buckets, their joint length `best`
//   scan                  P = exclusive scan of best in 64 bits; its total is the number of entries to test
//   gate_entries_kernel   tiles of 2048 consecutive entries of the concatenated bucket lists; the tile finds
//                         the queries it spans by a warp-wide 32-ary search in P, marks where each one starts,
//                         spreads the owners by a max-scan, and every thread tests 8 consecutive entries.
//                         Matches are appended to the query's stash through an atomic row counter.
// The fill pass takes rows of up to GATE_STASH candidates from the stash (gate_fill_small_kernel; in any
// order - it sorts them by video rank), larger rows are enumerated again by a warp.
// ------------------------------------------------------------------------------------------
struct __align__(16) GateQ {
  uint32_t ap[5];     // guarded digit words of the query
  int32_t sa, sb;     // bucket starts in items[]
  uint32_t ca_fa;     // entries in the first bucket | first bucket's feature << 28
};

__global__ void gate_plan_kernel(GateArgs g, GateQ *rec, int32_t *best_out) {
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= g.q_cap) return;
  g.row_count[q] = 0;
  if (q >= g.dc[DC_N_Q]) { best_out[q] = 0; return; }
  const int32_t i = g.a_list[g.dc[DC_Q_LO] + q];
  uint32_t ap[5];
  int32_t st[5], nb[5];
#pragma unroll
  for (int f = 0; f < 5; ++f) {
    ap[f] = g.a_pack[(int64_t)f * g.a_nstride + i] | 0x8888888u;
    const int64_t slot = (int64_t)f * DAB_NCODE + g.a_code[(int64_t)f * g.a_nstride + i];
    st[f] = g.start[slot];
    nb[f] = g.start[slot + 1] - st[f];
  }
  // every candidate lies in at least one bucket of any pair out of {0,1,2}, and in bucket 3 or 4
  int fa = 0, fb = 1, best = nb[0] + nb[1];
  if (nb[0] + nb[2] < best) { best = nb[0] + nb[2]; fa = 0; fb = 2; }
  if (nb[1] + nb[2] < best) { best = nb[1] + nb[2]; fa = 1; fb = 2; }
  if (nb[3] + nb[4] < best) { best = nb[3] + nb[4]; fa = 3; fb = 4; }
  GateQ r;
#pragma unroll
  for (int f = 0; f < 5; ++f) r.ap[f] = ap[f];
  int32_t sa = 0, sb = 0, ca = 0;
#pragma unroll
  for (int f = 0; f < 5; ++f) {
    if (f == fa) { sa = st[f]; ca = nb[f]; }
    if (f == fb) sb = st[f];
  }
  r.sa = sa; r.sb = sb; r.ca_fa = (uint32_t)ca | ((uint32_t)fa << 28);
  rec[q] = r;
  best_out[q] = best;
}

constexpr int GE_THREADS = 256, GE_PER = 8, GE_TILE = GE_THREADS * GE_PER;

// last index q in [0, n] with P[q] <= x (P non-decreasing, P[0] = 0 <= x), found by one warp: 32 probes per round
__device__ __forceinline__ int warp_last_le(const int64_t *P, int n, int64_t x, int lane) {
  int lo = 0, hi = n + 1;                 // P[lo] <= x; hi == n + 1 or P[hi] > x
  while (hi - lo > 1) {
    const int step = (hi - lo + 31) / 32;
    const int idx = lo + (lane + 1) * step;
    const bool le = idx < hi && P[idx] <= x;
    const int cnt = __popc(__ballot_sync(0xffffffffu, le));     // monotone: the lanes with le form a prefix
    const int nlo = lo + cnt * step;
    const int nhi = lo + (cnt + 1) * step;
    lo = nlo;
    if (nhi < hi) hi = nhi;
  }
  return lo;
}

// Entry positions are 64-bit (a long pair's queries visit more than 2^31 entries in all); the position of an entry
// inside its query's two buckets is below that query's count, an int32.
__global__ void __launch_bounds__(GE_THREADS) gate_entries_kernel(GateArgs g, const GateQ *rec, const int64_t *P) {
  __shared__ __align__(16) int owner[GE_TILE];
  __shared__ int s_q[2];
  __shared__ int s_wmax[GE_THREADS / 32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nq = g.dc[DC_N_Q];
  const int64_t total = (int64_t)(((uint64_t)(uint32_t)g.dc[DC_ENUM_HI] << 32) | (uint32_t)g.dc[DC_ENUM_LO]);
  if (g.dc[DC_OVERFLOW] & DAB_OVF_ENTRIES) return;
  for (int64_t E0 = (int64_t)blockIdx.x * GE_TILE; E0 < total; E0 += (int64_t)gridDim.x * GE_TILE) {
    const int64_t E1 = E0 + GE_TILE < total ? E0 + GE_TILE : total;
    // the queries this tile spans: q0 owns entry E0, q1 owns entry E1 - 1 (both non-empty rows)
    if (warp < 2) {
      const int r = warp_last_le(P, nq, warp == 0 ? E0 : E1 - 1, lane);
      if (lane == 0) s_q[warp] = r;
    }
#pragma unroll
    for (int j = 0; j < GE_PER; ++j) owner[tid + j * GE_THREADS] = 0;
    __syncthreads();
    const int q0 = s_q[0], q1 = s_q[1];
    // every later query that starts inside the tile marks its first entry (empty rows share a position with the
    // non-empty row that follows them: the largest index wins)
    for (int q = q0 + 1 + tid; q <= q1; q += GE_THREADS) {
      const int64_t pos = P[q] - E0;
      if (pos > 0 && pos < GE_TILE) atomicMax(&owner[(int)pos], q - q0);
    }
    __syncthreads();
    // inclusive max-scan: slot e belongs to the last marked query at or before it
    int m[GE_PER];
    {
      const int4 a = *reinterpret_cast<const int4 *>(&owner[tid * GE_PER]);
      const int4 b = *reinterpret_cast<const int4 *>(&owner[tid * GE_PER + 4]);
      m[0] = a.x; m[1] = a.y; m[2] = a.z; m[3] = a.w; m[4] = b.x; m[5] = b.y; m[6] = b.z; m[7] = b.w;
    }
#pragma unroll
    for (int j = 1; j < GE_PER; ++j) m[j] = max(m[j], m[j - 1]);
    int inc = m[GE_PER - 1];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc = max(inc, y);
    }
    if (lane == 31) s_wmax[warp] = inc;
    int before = __shfl_up_sync(0xffffffffu, inc, 1);
    if (lane == 0) before = 0;
    __syncthreads();
    for (int w = 0; w < warp; ++w) before = max(before, s_wmax[w]);
    // owners back to shared memory, then entries interleaved over the threads: consecutive lanes read consecutive
    // bucket items (coalesced) and mostly share a query, whose record is then one broadcast load
    __syncthreads();
#pragma unroll
    for (int j = 0; j < GE_PER; ++j) owner[tid * GE_PER + j] = max(before, m[j]);
    __syncthreads();
#pragma unroll
    for (int j = 0; j < GE_PER; ++j) {
      const int64_t e = E0 + j * GE_THREADS + tid;
      if (e < E1) {
        const int q = q0 + owner[j * GE_THREADS + tid];
        const uint4 *rp = reinterpret_cast<const uint4 *>(rec + q);
        const uint4 x0 = __ldg(rp), x1 = __ldg(rp + 1);
        const int el = (int)(e - P[q]);
        const int ca = (int)(x1.w & 0x0fffffffu), fa = (int)(x1.w >> 28);
        const bool second = el >= ca;
        const int32_t s = g.items[second ? (int32_t)x1.z + (el - ca) : (int32_t)x1.y + el];
        // features 0-3 are the first 16 bytes of the frame's record; feature 4 is only fetched when it decides
        const uint4 v0 = __ldg(g.v_rec + 2 * (int64_t)s);
        const bool m0 = digits_match(x0.x, v0.x), m1 = digits_match(x0.y, v0.y), m2 = digits_match(x0.z, v0.z),
                   m3 = digits_match(x0.w, v0.w);
        bool ok = (int)m0 + (int)m1 + (int)m2 >= 2;
        if (ok && second) {
          // already enumerated from the first bucket
          const bool mfa = fa == 0 ? m0 : (fa == 1 ? m1 : m3);
          if (mfa) ok = false;
        }
        if (ok && !m3) ok = digits_match(x1.x, __ldg(reinterpret_cast<const uint32_t *>(g.v_rec + 2 * (int64_t)s + 1)));
        if (ok) {
          const int idx = atomicAdd(&g.row_count[q], 1);
          if (idx < GATE_STASH) g.stash[(int64_t)q * GATE_STASH + idx] = s;
        }
      }
    }
    __syncthreads();     // owner[] and s_q[] are rewritten by the next tile
  }
}

// ------------------------------------------------------------------------------------------
// scoring: thread per candidate
// ------------------------------------------------------------------------------------------
struct ScoreArgs {
  const int32_t *cand_s, *cand_i;
  const int32_t *dc;             // n_cand = dc[DC_N_CAND]
  const int32_t *v_sel;
  const double *a_ms, *v_ms;     // [5][stride]
  int64_t a_stride, v_stride;
  const double *a_nrm, *v_nrm;   // [3][nstride]
  int64_t a_nstride, v_nstride;
  double *qual;                  // < 0: rejected
  int32_t *keep;
};

__global__ void score_kernel(ScoreArgs s) {
  // the launch is a fixed number of blocks (the candidate count is only known to the device): grid stride
  const int64_t n_cand = s.dc[DC_N_CAND];
  for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < n_cand; c += (int64_t)gridDim.x * blockDim.x) {
  const int32_t i = s.cand_i[c];
  const int32_t v = s.v_sel[s.cand_s[c]];
  double prob = 1.0;
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    const double *am = s.a_ms + (int64_t)j * s.a_stride + i;
    const double *vm = s.v_ms + (int64_t)j * s.v_stride + v;
    auto X = [&](int k) { return am[k]; };
    auto Y = [&](int k) { return vm[k]; };
    double corr = ddot41_skx(X, Y);
    corr = corr / (s.a_nrm[(int64_t)j * s.a_nstride + i] * s.v_nrm[(int64_t)j * s.v_nstride + v]);
    prob = prob * fmax(1e-8, 1.0 - corr);
  }
  prob = pow(prob, 2.9);
  double qual = -1.0;
  if (!(prob > 1e-8)) qual = fmin(50.0, pow(prob / 1e-12, -1.0 / 3));
  s.qual[c] = qual;
  s.keep[c] = qual >= 0.0 ? 1 : 0;
  }
}

__global__ void gather_points_kernel(const int32_t *keep, const int32_t *off, const int32_t *dc,
                                     const int32_t *cand_i, const int32_t *cand_s, const double *qual,
                                     int32_t *pt_i, int32_t *pt_s, double *pt_q) {
  const int64_t n_cand = dc[DC_N_CAND];
  for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < n_cand; c += (int64_t)gridDim.x * blockDim.x) {
    if (!keep[c]) continue;
    const int o = off[c];
    pt_i[o] = cand_i[c];
    pt_s[o] = cand_s[c];
    pt_q[o] = qual[c];
  }
}

// ------------------------------------------------------------------------------------------
// frontier DP #1 (SURVEY.md A.5): cum(p) = q(p) + max{cum(p') : p' earlier, rank' <= rank},
// ties to the smallest rank; the seed has cum 0.  One warp walks the points in (i, v) order;
// the prefix maximum lives in a 32-ary max tree over the video ranks (HBM/L2 resident).
// ------------------------------------------------------------------------------------------
struct __align__(16) Node1 {
  double cum;     // 0 = empty / seed
  int32_t id;     // point id, -1 = seed
  int32_t rank;
};

constexpr int DP_LEVELS = 4;

struct Dp1Args {
  const int32_t *pt_s;
  const double *pt_q;
  const int32_t *n_points;       // device count
  Node1 *level[DP_LEVELS];
  BackRec *back;                 // per point (predecessor's cum, predecessor)
  int32_t *result;               // [0] end id, -1: no path
};

__device__ __forceinline__ bool key_better(double ca, int ra, double cb, int rb) {
  return ca > cb || (ca == cb && ra < rb);
}

__device__ __forceinline__ Node1 load_node_cg(const Node1 *p) {
  // L2 read (bypasses L1): the node may have been rewritten by another lane's fire-and-forget store
  const int4 v = __ldcg(reinterpret_cast<const int4 *>(p));
  Node1 n;
  n.cum = __hiloint2double(v.y, v.x);
  n.id = v.z;
  n.rank = v.w;
  return n;
}

// The walk keeps the frontier's top entry (largest cum; ties -> smallest rank) in registers.
// A point whose rank is >= the top's rank has the top as its predecessor and becomes the new
// top (quals are > 0): no tree loads, one f64 add on the dependent chain; the leaf, the back
// record and the old top's level-k ancestors (written only when the top leaves that ancestor's
// block - the ancestors of the current top are implied by the registers; every other node is
// exact) are stored lane-parallel for a whole run of such points at a time.  Only points left
// of the top (false matches, backward jumps) run the full prefix-max query: one 32-node row per
// level (512 B, coalesced), lanes left of the path feed the query and the lane on the path keeps
// the old node for the conditional update.
__global__ void __launch_bounds__(32, 1) dp1_kernel(Dp1Args a) {
  __shared__ int s_r[2][32];
  __shared__ double s_q[2][32];
  const int lane = threadIdx.x;
  const int n = *a.n_points;
  double top_cum = 0.0;
  int top_id = -1, top_rank = -1;
  const int role = lane < DP_LEVELS ? lane : 0;
  int4 *const my_level = reinterpret_cast<int4 *>(a.level[role]);
  const int my_shift = 5 * role;
  int rr = lane < n ? a.pt_s[lane] : 0;
  double qq = lane < n ? a.pt_q[lane] : 0.0;
  for (int base = 0; base < n; base += 32) {
    const int buf = (base >> 5) & 1;
    s_r[buf][lane] = rr;
    s_q[buf][lane] = qq;
    __syncwarp();
    if (base + 32 + lane < n) { rr = a.pt_s[base + 32 + lane]; qq = a.pt_q[base + 32 + lane]; }
    const int cnt = n - base < 32 ? n - base : 32;
    // ---- runs of points that each extend the top (rank >= the rank before it) are handled 32 at
    //      a time: the cums are one sequential chain of f64 adds (exactly the reference's order),
    //      everything else - back records, leaves, ancestor flushes - is lane-parallel ----------
    const int my_r = s_r[buf][lane];
    const int prev_r = lane > 0 ? s_r[buf][lane - 1] : 0;
    const int next_r = lane + 1 < cnt ? s_r[buf][lane + 1] : -1;
    const unsigned inc = __ballot_sync(0xffffffffu, lane < cnt && (lane == 0 || my_r >= prev_r));
    int t = 0;
    while (t < cnt) {
      const int p = base + t;
      const int r = s_r[buf][t];
      const double q = s_q[buf][t];
      if (r >= top_rank) {
        int len = 1;
        if (t + 1 < 32) {
          const unsigned stop = (~inc) >> (t + 1);
          len += stop ? __ffs(stop) - 1 : 31 - t;
        }
        if (len > cnt - t) len = cnt - t;
        const bool in_run = lane >= t && lane < t + len;
        // The cums of the run are top_cum + q, + q, ... added one after the other in float64 (the
        // reference's order).  While the sums stay inside the binade of top_cum every such add is exact
        // arithmetic on multiples of that binade's unit once q is rounded to it (fl(x + q) = x + rn_u(q),
        // ties aside), so a warp prefix sum gives all of them in five steps; each lane then checks its
        // value against the one rounded add the reference performs, and only a run that fails the check
        // (binade crossing, rounding tie) is added up serially.
        double my_cum = 0.0;
        {
          const double my_q = in_run ? s_q[buf][lane] : 0.0;
          const unsigned long long tb = (unsigned long long)__double_as_longlong(top_cum);
          const double big = __longlong_as_double((long long)((tb & 0x7ff0000000000000ull) | 0x0008000000000000ull));  // 1.5 * 2^e
          double ps = in_run ? __dadd_rn(__dadd_rn(my_q, big), -big) : 0.0;       // q rounded to the unit of top_cum's binade
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            const double y = __shfl_up_sync(0xffffffffu, ps, o);
            if (lane >= t + o) ps = ps + y;
          }
          const double spec = top_cum + ps;
          double prev = __shfl_up_sync(0xffffffffu, spec, 1);
          if (lane == t) prev = top_cum;
          const bool ok = !in_run || (top_cum > 0.0 && __double_as_longlong(prev + my_q) == __double_as_longlong(spec));
          if (__all_sync(0xffffffffu, ok)) {
            my_cum = spec;
          } else {
            double c = top_cum;
            for (int u = 0; u < len; ++u) {
              c = c + s_q[buf][t + u];
              if (lane == t + u) my_cum = c;
            }
          }
        }
        const bool first = lane == t;
        double old_cum = __shfl_up_sync(0xffffffffu, my_cum, 1);
        int old_id = base + lane - 1, old_rank = prev_r;
        if (first) { old_cum = top_cum; old_id = top_id; old_rank = top_rank; }
        if (in_run) {
          BackRec b; b.best = old_cum; b.pred = old_id; b.pad = 0;
          a.back[base + lane] = b;
          if (lane == t + len - 1 || next_r != my_r) {       // the last point on a rank owns its leaf
            Node1 me; me.cum = my_cum; me.id = base + lane; me.rank = my_r;
            a.level[0][my_r] = me;
          }
          if (old_id >= 0) {                                  // the old top leaves ancestor blocks
#pragma unroll
            for (int k = 1; k < DP_LEVELS; ++k) {
              if ((my_r >> (5 * k)) != (old_rank >> (5 * k))) {
                Node1 me; me.cum = old_cum; me.id = old_id; me.rank = old_rank;
                a.level[k][old_rank >> (5 * k)] = me;
              }
            }
          }
        }
        const int last = t + len - 1;
        top_cum = __shfl_sync(0xffffffffu, my_cum, last);
        top_rank = __shfl_sync(0xffffffffu, my_r, last);
        top_id = base + last;
        t += len;
        continue;
      }
      ++t;
      __syncwarp();   // orders the stores above before the loads below
      Node1 nd[DP_LEVELS];
      int pos[DP_LEVELS];
#pragma unroll
      for (int k = 0; k < DP_LEVELS; ++k) {
        const int g = r >> (5 * k);
        pos[k] = g & 31;
        nd[k] = load_node_cg(&a.level[k][(g & ~31) + lane]);
      }
      // lane-local best over eligible nodes; higher levels hold smaller ranks
      double bc = 0.0;
      int bid = -1, brank = 0x7fffffff;
#pragma unroll
      for (int k = DP_LEVELS - 1; k >= 0; --k) {
        const bool elig = (k == 0) ? (lane <= pos[0]) : (lane < pos[k]);
        if (elig && key_better(nd[k].cum, nd[k].rank, bc, brank)) { bc = nd[k].cum; bid = nd[k].id; brank = nd[k].rank; }
      }
      // warp arg-max on (cum desc, rank asc); all cum >= 0 so the bit patterns order like integers
      const unsigned long long bits = (unsigned long long)__double_as_longlong(bc);
      const unsigned hi = (unsigned)(bits >> 32), lo = (unsigned)bits;
      const unsigned mhi = __reduce_max_sync(0xffffffffu, hi);
      bool alive = hi == mhi;
      const unsigned mlo = __reduce_max_sync(0xffffffffu, alive ? lo : 0u);
      alive = alive && lo == mlo;
      const unsigned mr = __reduce_min_sync(0xffffffffu, alive ? (unsigned)brank : 0xffffffffu);
      alive = alive && (unsigned)brank == mr;
      const int src = __ffs(__ballot_sync(0xffffffffu, alive)) - 1;
      const double pc = __shfl_sync(0xffffffffu, bc, src);
      const int pid = __shfl_sync(0xffffffffu, bid, src);
      const double cum = pc + q;
      // updates: leaf always (a later point on the same rank chains from the earlier one), upper
      // levels when the new key wins.  (A node on the current top's path may be stale-low; the
      // top is written over it when it leaves the block, and it is >= everything in that block.)
      if (lane == pos[0]) {
        Node1 me; me.cum = cum; me.id = p; me.rank = r;
        a.level[0][r] = me;
      }
#pragma unroll
      for (int k = 1; k < DP_LEVELS; ++k) {
        if (lane == pos[k] && key_better(cum, r, nd[k].cum, nd[k].rank)) {
          Node1 me; me.cum = cum; me.id = p; me.rank = r;
          a.level[k][r >> (5 * k)] = me;
        }
      }
      if (lane == 0) { BackRec b; b.best = pc; b.pred = pid; b.pad = 0; a.back[p] = b; }
      if (key_better(cum, r, top_cum, top_rank)) {
        // the old top's ancestors are flushed where the new top lies in another block
        if (lane >= 1 && lane < DP_LEVELS && top_id >= 0 && (r >> my_shift) != (top_rank >> my_shift)) {
          int4 val;
          val.x = __double2loint(top_cum); val.y = __double2hiint(top_cum); val.z = top_id; val.w = top_rank;
          my_level[top_rank >> my_shift] = val;
        }
        top_cum = cum; top_id = p; top_rank = r;
      }
      __syncwarp();
    }
    __syncwarp();
  }
  if (lane == 0) a.result[0] = top_id;
}

__global__ void fill_nodes_kernel(Node1 *p, int64_t n) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) { Node1 z; z.cum = 0.0; z.id = -1; z.rank = 0x7fffffff; p[i] = z; }
}

}  // namespace

// ------------------------------------------------------------------------------------------
// host drivers
// ------------------------------------------------------------------------------------------
template <typename T>
static int exclusive_scan(dab_pair *pr, const int32_t *in, T *out, int64_t n, const int32_t *n_dev, int32_t *total_out) {
  dab_ctx *ctx = pr->ctx;
  // tiles cover positions 0 .. n inclusive, so that the tile holding position n exists and writes the total
  const int nblocks = (int)(n / SCAN_TILE) + 1;
  const size_t need = sizeof(unsigned long long) * (size_t)(ScanOps<T>::WORDS * nblocks + 2);
  if (need > pr->scan_tmp.cap || !pr->scan_tmp.p) {
    DAB_TRY(dab_ensure(ctx, pr->scan_tmp, need + 4096));
    DAB_CUDA(cudaMemsetAsync(pr->scan_tmp.p, 0, pr->scan_tmp.cap, pr->stream));   // epoch 0 = never written; ticket = 0
    pr->scan_epoch = 0;
  }
  ScanArgs<T> sa;
  sa.in = in; sa.out = out; sa.n = n; sa.n_dev = n_dev; sa.total_out = total_out;
  sa.ticket = pr->scan_tmp.as<unsigned int>();
  sa.status = pr->scan_tmp.as<unsigned long long>() + 1;
  pr->scan_epoch = pr->scan_epoch >= 0x3ffffffe ? 1 : pr->scan_epoch + 1;
  sa.epoch = pr->scan_epoch;
  scan_onepass_kernel<T><<<nblocks, SCAN_THREADS, 0, pr->stream>>>(sa);
  pr->ctx->launches += 1;
  DAB_CUDA(cudaGetLastError());
  return DAB_OK;
}

int dab_exclusive_scan(dab_pair *pr, const int32_t *in, int32_t *out, int64_t n, const int32_t *n_dev,
                       int32_t *total_out) {
  return exclusive_scan(pr, in, out, n, n_dev, total_out);
}

int dab_exclusive_scan(dab_pair *pr, const int32_t *in, int64_t *out, int64_t n, const int32_t *n_dev,
                       int32_t *total_out) {
  return exclusive_scan(pr, in, out, n, n_dev, total_out);
}

// derived counts after both tracks' not-quiet scans: hashed video frames, this shard's query range
static __global__ void counts_lists_kernel(int32_t *dc, const int32_t *v_off, int64_t v_n, const int32_t *a_off, int64_t a_n,
                                    int64_t row_lo, int64_t row_hi) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const int32_t n_vnq = v_off[v_n];
  dc[DC_N_VNQ] = n_vnq;
  dc[DC_N_VSEL] = (n_vnq + 3) / 4;
  dc[DC_N_AQ_ALL] = a_off[a_n];
  const int64_t lo = row_lo < 0 ? 0 : (row_lo > a_n ? a_n : row_lo);
  const int64_t hi = row_hi < lo ? lo : (row_hi > a_n ? a_n : row_hi);
  dc[DC_Q_LO] = a_off[lo];
  dc[DC_Q_HI] = a_off[hi];
  dc[DC_N_Q] = a_off[hi] - a_off[lo];
}

// a scan total against the capacity of the buffer it sizes: keeps the total in need_word, then clamps the count and
// raises the overflow bit
static __global__ void check_capacity_kernel(int32_t *dc, int word, int need_word, int64_t cap, int bit) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  dc[need_word] = dc[word];
  if ((int64_t)dc[word] > cap) { dc[word] = 0; atomicOr(&dc[DC_OVERFLOW], bit); }
}

// Prep of one track's features `in` into `out` (the pair's audio prep, or the prep of a video side).
static int prep_track(dab_pair *pr, const Track &in, Prep &out, bool is_video) {
  dab_ctx *ctx = pr->ctx;
  const Track &tk = in;
  const int64_t Lmax = tk.Le > tk.L ? tk.Le : tk.L;
  const int64_t Lmin = tk.Le < tk.L ? tk.Le : tk.L;
  const int64_t nc = Lmax - 40;     // stride of the code arrays (energy may have one more)
  out.L = tk.L; out.Le = tk.Le;
  DAB_TRY(dab_ensure(ctx, out.ms, sizeof(double) * (size_t)(5 * Lmax)));
  DAB_TRY(dab_ensure(ctx, out.nrm, sizeof(double) * (size_t)(3 * nc)));
  DAB_TRY(dab_ensure(ctx, out.pack, sizeof(uint32_t) * (size_t)(5 * nc)));
  DAB_TRY(dab_ensure(ctx, out.code, sizeof(int32_t) * (size_t)(5 * nc)));
  PrepArgs pa;
  pa.f32[0] = tk.energy.as<float>(); pa.f32[1] = tk.zc.as<float>();
  pa.f32[2] = tk.b0.as<float>(); pa.f32[3] = tk.b1.as<float>();
  pa.f64 = tk.b2.as<double>();
  pa.len[0] = tk.Le; pa.len[1] = pa.len[2] = pa.len[3] = pa.len[4] = tk.L;
  pa.Lp = Lmin; pa.ms = out.ms.as<double>(); pa.stride = Lmax;
  dim3 g1((unsigned)cdiv(Lmax, 256 * MS_TILES), 5);
  meansub_kernel<<<g1, 256, 0, pr->stream>>>(pa);
  CodeArgs ca;
  ca.ms = out.ms.as<double>(); ca.stride = Lmax;
  for (int f = 0; f < 5; ++f) ca.len[f] = pa.len[f];
  ca.nrm = out.nrm.as<double>(); ca.nstride = nc;
  ca.pack = out.pack.as<uint32_t>(); ca.code = out.code.as<int32_t>();
  ca.is_video = is_video;
  dim3 g2((unsigned)cdiv(nc, 256), 5);
  norm_codes_kernel<<<g2, 256, 0, pr->stream>>>(ca);
  ctx->launches += 2;
  // not-quiet selection: t < len(energy) - 41 with energy[t] > .5
  const int64_t nqn = tk.Le - 41;
  DAB_TRY(dab_ensure(ctx, out.nq_flag, sizeof(int32_t) * (size_t)(2 * (nqn + 2))));
  DAB_TRY(dab_ensure(ctx, out.nq_list, sizeof(int32_t) * (size_t)(nqn + 2)));
  int32_t *flag = out.nq_flag.as<int32_t>();
  int32_t *off = flag + (nqn + 1);
  notquiet_flag_kernel<<<(unsigned)cdiv(nqn, 256), 256, 0, pr->stream>>>(tk.have_gate ? tk.gate.as<float>() : tk.energy.as<float>(), nqn, flag);
  ctx->launches += 1;
  DAB_TRY(dab_exclusive_scan(pr, flag, off, nqn));
  compact_kernel<<<(unsigned)cdiv(nqn, 256), 256, 0, pr->stream>>>(flag, off, nqn, is_video ? 4 : 1,
                                                                  out.nq_list.as<int32_t>());
  ctx->launches += 1;
  DAB_CUDA(cudaGetLastError());
  return DAB_OK;
}

// counts_lists_kernel over the not-quiet scans of the video prep V and the audio prep A
static void enqueue_counts_lists(dab_pair *pr, int32_t *dc, const Prep &V, const Prep &A, int64_t row_lo, int64_t row_hi) {
  const int64_t v_nq = V.Le - 41, a_nq = A.Le - 41;
  counts_lists_kernel<<<1, 32, 0, pr->stream>>>(dc, V.nq_flag.as<int32_t>() + (v_nq + 1), v_nq, A.nq_flag.as<int32_t>() + (a_nq + 1),
                                                a_nq, row_lo, row_hi);
  pr->ctx->launches += 1;
}

static int ensure_hann(dab_ctx *ctx) {
  static std::atomic<int> ready[64];
  int dev = 0;
  DAB_CUDA(cudaGetDevice(&dev));
  if (dev < 64 && ready[dev].load(std::memory_order_acquire)) return DAB_OK;
  static std::mutex mu;
  std::lock_guard<std::mutex> g(mu);
  if (dev < 64 && ready[dev].load(std::memory_order_acquire)) return DAB_OK;
  double hf[41];
  for (int k = 0; k < 41; ++k) hf[k] = DAB_HANN41_F64[40 - k];
  DAB_CUDA(cudaMemcpyToSymbol(c_hflip, hf, sizeof(hf)));
  if (dev < 64) ready[dev].store(1, std::memory_order_release);
  return DAB_OK;
}

// Capacities of the buffers whose fill level only the device knows (table entries, candidates).  They
// start from what pairs of this size normally need and double when a run overflows (the overflow bit
// comes back with the counts; the stage is then run again - rare, and only ever during the first pairs).
static int64_t video_sel_ub(int64_t v_Le) { return (v_Le - 41 + 3) / 4 + 1; }
static int64_t first_entries_cap(int64_t v_Le) {
  return 5 * 16 * video_sel_ub(v_Le) + 4096;            // ~10 expanded entries per frame and table (SURVEY.md D)
}
static int64_t first_cand_cap(int64_t a_Le) {
  return 2 * (a_Le - 41) + 4096;                         // < 1 candidate per query on matching tracks
}

// tables over the hashed video frames (dc[DC_N_VSEL] of them) of the side's prep, and the frames' records; the
// pair's table scratch holds the super-bucket counts and the entries between the passes
static int enqueue_tables(dab_pair *pr, VideoSide &vs, int32_t *dc) {
  dab_ctx *ctx = pr->ctx;
  cudaStream_t st = pr->stream;
  const Prep &V = vs.prep;
  const int64_t vsel_ub = video_sel_ub(V.Le);
  const int64_t v_nstride = (V.Le > V.L ? V.Le : V.L) - 40;
  vs.cap_entries = std::max<int64_t>(vs.cap_entries, first_entries_cap(V.Le));
  const int64_t cap_e = vs.cap_entries;
  DAB_TRY(dab_ensure(ctx, vs.tbl_start, sizeof(int32_t) * (size_t)(TB_NSLOTS + 2)));
  DAB_TRY(dab_ensure(ctx, vs.tbl_items, sizeof(int32_t) * (size_t)(cap_e + 1)));
  DAB_TRY(dab_ensure(ctx, vs.v_rec, sizeof(uint4) * 2 * (size_t)(vsel_ub + 1)));
  DAB_TRY(dab_ensure(ctx, pr->tbl_sb, sizeof(int32_t) * (size_t)(3 * TB_NSB + 1)));
  DAB_TRY(dab_ensure(ctx, pr->tbl_ent, sizeof(uint2) * (size_t)(cap_e + 1)));
  int32_t *sb_count = pr->tbl_sb.as<int32_t>(), *sb_off = sb_count + TB_NSB, *sb_cursor = sb_off + (TB_NSB + 1);
  uint4 *rec = vs.v_rec.as<uint4>();
  DAB_CUDA(cudaMemsetAsync(sb_count, 0, sizeof(int32_t) * TB_NSB, st));
  const unsigned nb = (unsigned)cdiv(vsel_ub, TB_THREADS);
  table_count_kernel<<<nb, TB_THREADS, 0, st>>>(V.pack.as<uint32_t>(), v_nstride, V.nq_list.as<int32_t>(), dc, rec, sb_count);
  table_scan_kernel<<<1, TB_SCAN_THREADS, 0, st>>>(dc, cap_e, sb_count, sb_off, sb_cursor);
  table_scatter_kernel<<<nb, TB_THREADS, 0, st>>>(rec, dc, sb_cursor, pr->tbl_ent.as<uint2>());
  table_sort_kernel<<<TB_NSB, TS_THREADS, 0, st>>>(dc, sb_off, pr->tbl_ent.as<uint2>(), vs.tbl_start.as<int32_t>(),
                                                   vs.tbl_items.as<int32_t>());
  ctx->launches += 4;
  DAB_CUDA(cudaGetLastError());
  return DAB_OK;
}

// The counts of a video side built in this run.  False after an entries overflow: the tables are empty and their
// capacity has grown to at least the total the run needed.
static bool collect_tables(VideoSide &vs, const int32_t *hc) {
  vs.n_vsel = hc[DC_N_VSEL];
  vs.n_entries = hc[DC_N_ENTRIES];
  if (!(hc[DC_OVERFLOW] & DAB_OVF_ENTRIES)) return true;
  vs.cap_entries = std::max<int64_t>(2 * vs.cap_entries, hc[DC_NEED_ENTRIES]);
  return false;
}

// gate + scoring + compaction of the pair's audio queries against `vs`: the points go to pr->pt_*
static int enqueue_gate_score(dab_pair *pr, const VideoSide &vs, int32_t *dc) {
  dab_ctx *ctx = pr->ctx;
  const Prep &V = vs.prep, &A = pr->prep_a;
  cudaStream_t st = pr->stream;
  const int64_t a_nq = A.Le - 41;
  const int64_t q_ub = a_nq > 0 ? a_nq : 1;
  const int64_t cap_c = pr->cap_cand;
  const int64_t v_nstride = (V.Le > V.L ? V.Le : V.L) - 40;
  const int64_t a_nstride = (A.Le > A.L ? A.Le : A.L) - 40;

  // ---- gate: count, scan, fill ----
  DAB_TRY(dab_ensure(ctx, pr->row_count, sizeof(int32_t) * (size_t)(q_ub + 2)));
  DAB_TRY(dab_ensure(ctx, pr->row_off, sizeof(int32_t) * (size_t)(q_ub + 2)));
  DAB_TRY(dab_ensure(ctx, pr->cand_tmp, sizeof(int32_t) * (size_t)(cap_c + 1)));
  DAB_TRY(dab_ensure(ctx, pr->cand_s, sizeof(int32_t) * (size_t)(cap_c + 1)));
  DAB_TRY(dab_ensure(ctx, pr->cand_i, sizeof(int32_t) * (size_t)(cap_c + 1)));
  GateArgs ga;
  ga.a_code = A.code.as<int32_t>(); ga.a_pack = A.pack.as<uint32_t>(); ga.a_nstride = a_nstride;
  ga.a_list = A.nq_list.as<int32_t>(); ga.dc = dc; ga.q_cap = q_ub;
  ga.v_rec = vs.v_rec.as<uint4>();
  ga.start = vs.tbl_start.as<int32_t>(); ga.items = vs.tbl_items.as<int32_t>();
  ga.row_count = pr->row_count.as<int32_t>(); ga.row_off = pr->row_off.as<int32_t>();
  ga.cand_tmp = pr->cand_tmp.as<int32_t>(); ga.cand_s = pr->cand_s.as<int32_t>(); ga.cand_i = pr->cand_i.as<int32_t>();
  ga.cand_cap = cap_c;
  DAB_TRY(dab_ensure(ctx, pr->row_stash, sizeof(int32_t) * GATE_STASH * (size_t)(q_ub + 1)));
  ga.stash = pr->row_stash.as<int32_t>();
  DAB_TRY(dab_ensure(ctx, pr->gate_big, sizeof(int32_t) * (size_t)(q_ub + 1)));
  ga.big_list = pr->gate_big.as<int32_t>();
  ga.big_count = dc + DC_N_BIGROWS;
  DAB_CUDA(cudaEventRecord(pr->ev[8], st));
  // count pass, balanced over bucket entries (see gate_entries_kernel)
  DAB_TRY(dab_ensure(ctx, pr->gate_rec, sizeof(GateQ) * (size_t)(q_ub + 1)));
  DAB_TRY(dab_ensure(ctx, pr->gate_best, (sizeof(int64_t) + sizeof(int32_t)) * (size_t)(q_ub + 2)));
  int64_t *g_P = pr->gate_best.as<int64_t>();
  int32_t *g_best = reinterpret_cast<int32_t *>(g_P + (q_ub + 2));
  gate_plan_kernel<<<(unsigned)cdiv(q_ub, 128), 128, 0, st>>>(ga, pr->gate_rec.as<GateQ>(), g_best);
  // 64-bit entry prefix; its total (the entries the gate visits) goes to DC_ENUM_LO / DC_ENUM_HI
  DAB_TRY(dab_exclusive_scan(pr, g_best, g_P, q_ub, nullptr, dc + DC_ENUM_LO));
  gate_entries_kernel<<<(unsigned)(8 * ctx->sm_count), GE_THREADS, 0, st>>>(ga, pr->gate_rec.as<GateQ>(), g_P);
  ctx->launches += 2;
  // the candidate total saturates at INT32_MAX (int32 scan): a run that needs that many is refused by the collect
  DAB_TRY(dab_exclusive_scan(pr, pr->row_count.as<int32_t>(), pr->row_off.as<int32_t>(), q_ub, nullptr, dc + DC_N_CAND));
  check_capacity_kernel<<<1, 32, 0, st>>>(dc, DC_N_CAND, DC_NEED_CAND, cap_c, DAB_OVF_CAND);
  gate_fill_small_kernel<<<(unsigned)cdiv(q_ub, 256), 256, 0, st>>>(ga);
  gate_fill_big_kernel<<<(unsigned)(2 * ctx->sm_count), 256, 0, st>>>(ga);
  ctx->launches += 4;
  DAB_CUDA(cudaEventRecord(pr->ev[9], st));

  // ---- scoring + compaction ----
  DAB_CUDA(cudaEventRecord(pr->ev[10], st));
  DAB_TRY(dab_ensure(ctx, pr->cand_q, sizeof(double) * (size_t)(cap_c + 1)));
  DAB_TRY(dab_ensure(ctx, pr->keep_flag, sizeof(int32_t) * (size_t)(cap_c + 2)));
  DAB_TRY(dab_ensure(ctx, pr->keep_off, sizeof(int32_t) * (size_t)(cap_c + 2)));
  DAB_TRY(dab_ensure(ctx, pr->pt_i, sizeof(int32_t) * (size_t)(cap_c + 1)));
  DAB_TRY(dab_ensure(ctx, pr->pt_s, sizeof(int32_t) * (size_t)(cap_c + 1)));
  DAB_TRY(dab_ensure(ctx, pr->pt_q, sizeof(double) * (size_t)(cap_c + 1)));
  ScoreArgs sa;
  sa.cand_s = pr->cand_s.as<int32_t>(); sa.cand_i = pr->cand_i.as<int32_t>(); sa.dc = dc;
  sa.v_sel = V.nq_list.as<int32_t>();
  sa.a_ms = A.ms.as<double>(); sa.v_ms = V.ms.as<double>();
  sa.a_stride = (A.Le > A.L ? A.Le : A.L); sa.v_stride = (V.Le > V.L ? V.Le : V.L);
  sa.a_nrm = A.nrm.as<double>(); sa.v_nrm = V.nrm.as<double>();
  sa.a_nstride = a_nstride; sa.v_nstride = v_nstride;
  sa.qual = pr->cand_q.as<double>(); sa.keep = pr->keep_flag.as<int32_t>();
  const unsigned n_fixed = (unsigned)(4 * ctx->sm_count);     // grid-stride kernels over a device-side count
  score_kernel<<<n_fixed, 128, 0, st>>>(sa);
  DAB_TRY(dab_exclusive_scan(pr, pr->keep_flag.as<int32_t>(), pr->keep_off.as<int32_t>(), cap_c, dc + DC_N_CAND, dc + DC_N_PTS1));
  gather_points_kernel<<<n_fixed, 256, 0, st>>>(
      pr->keep_flag.as<int32_t>(), pr->keep_off.as<int32_t>(), dc, pr->cand_i.as<int32_t>(),
      pr->cand_s.as<int32_t>(), pr->cand_q.as<double>(), pr->pt_i.as<int32_t>(), pr->pt_s.as<int32_t>(),
      pr->pt_q.as<double>());
  ctx->launches += 2;
  DAB_CUDA(cudaEventRecord(pr->ev[11], st));
  pr->cap_points1 = cap_c;
  return DAB_OK;
}

// ---- DP #1 + traceback over pr->pt_* (dc[DC_N_PTS1] points sorted by (audio frame, rank in vs's hashed frames)) ----
static int enqueue_dp1(dab_pair *pr, const VideoSide &vs) {
  dab_ctx *ctx = pr->ctx;
  cudaStream_t st = pr->stream;
  int32_t *dc = pr->counters.as<int32_t>();
  const int64_t cap_p = pr->cap_points1 > 0 ? pr->cap_points1 : 1;
  const int64_t vsel_ub = video_sel_ub(vs.prep.Le);
  DAB_CUDA(cudaEventRecord(pr->ev[12], st));
  if (vsel_ub > (1LL << (5 * DP_LEVELS))) { dab_set_err(ctx, "too many hashed video frames for the DP tree"); return DAB_E_CAPACITY; }
  int64_t lv[DP_LEVELS], tot = 0;
  int64_t m = vsel_ub;
  for (int k = 0; k < DP_LEVELS; ++k) { lv[k] = cdiv(m > 0 ? m : 1, 32) * 32; tot += lv[k]; m = cdiv(m, 32); }
  DAB_TRY(dab_ensure(ctx, pr->tree1, sizeof(Node1) * (size_t)tot));
  fill_nodes_kernel<<<(unsigned)cdiv(tot, 256), 256, 0, st>>>(pr->tree1.as<Node1>(), tot);
  DAB_TRY(dab_ensure(ctx, pr->back1, sizeof(BackRec) * (size_t)(cap_p + 1)));
  DAB_TRY(dab_ensure(ctx, pr->path1_x, sizeof(int32_t) * (size_t)(cap_p + 1)));
  DAB_TRY(dab_ensure(ctx, pr->path1_y, sizeof(int32_t) * (size_t)(cap_p + 1)));
  Dp1Args da;
  da.pt_s = pr->pt_s.as<int32_t>(); da.pt_q = pr->pt_q.as<double>();
  da.n_points = dc + DC_N_PTS1;
  Node1 *base = pr->tree1.as<Node1>();
  for (int k = 0; k < DP_LEVELS; ++k) { da.level[k] = base; base += lv[k]; }
  da.back = pr->back1.as<BackRec>();
  da.result = dc + DC_DP1_END;
  dp1_kernel<<<1, 32, 0, st>>>(da);
  ctx->launches += 2;
  Path1Out out;
  out.pt_i = pr->pt_i.as<int32_t>(); out.pt_s = da.pt_s; out.v_sel = vs.prep.nq_list.as<int32_t>();
  out.x = pr->path1_x.as<int32_t>(); out.y = pr->path1_y.as<int32_t>();
  DAB_TRY(dab_enqueue_traceback(pr, da.back, da.n_points, da.result, cap_p, dc + DC_N_PATH1, out));
  DAB_CUDA(cudaEventRecord(pr->ev[13], st));
  pr->ev_used[6] = true;
  DAB_CUDA(cudaGetLastError());
  return DAB_OK;
}

int dab_enqueue_stage_a_dp(dab_pair *pr) { return enqueue_dp1(pr, pr->video); }

// ---- stage A, enqueued without a host round trip: prep, codes, lists, tables (own video side only), gate,
// scoring, then DP 1 + traceback if with_dp, then the counts ----
static const char *const kTooManyCandidates =
    "stage A: the gate found 2147483647 or more candidates; the candidate arrays hold at most 2147483646";

int dab_enqueue_stage_a(dab_pair *pr, const dab_index *ix, int64_t row_lo, int64_t row_hi, bool with_dp) {
  dab_ctx *ctx = pr->ctx;
  if (pr->cap_cand > DAB_MAX_CANDIDATES) {
    // the last run needed more candidates than the arrays can index (dab_collect_stage_a): not run again; the next
    // call starts from the first guess
    pr->cap_cand = 0;
    dab_set_err(ctx, kTooManyCandidates);
    return DAB_E_CAPACITY;
  }
  DAB_TRY(ensure_hann(ctx));
  const Track &A = pr->trk[DAB_TRACK_AUDIO];
  const VideoSide &vs = ix ? ix->side : pr->video;
  cudaStream_t st = pr->stream;
  pr->n_points1 = pr->n_path1 = 0;
  pr->points_side = nullptr;
  pr->cap_cand = std::max<int64_t>(pr->cap_cand, first_cand_cap(A.Le));

  DAB_TRY(dab_ensure(ctx, pr->counters, sizeof(int32_t) * DC_WORDS));
  int32_t *dc = pr->counters.as<int32_t>();
  if (ix) DAB_CUDA(cudaStreamWaitEvent(st, ix->ready, 0));
  DAB_CUDA(cudaEventRecord(pr->ev[4], st));
  DAB_CUDA(cudaMemsetAsync(dc, 0, sizeof(int32_t) * DC_WORDS, st));
  if (!ix) DAB_TRY(prep_track(pr, pr->trk[DAB_TRACK_VIDEO], pr->video.prep, true));
  DAB_TRY(prep_track(pr, A, pr->prep_a, false));
  enqueue_counts_lists(pr, dc, vs.prep, pr->prep_a, row_lo, row_hi);
  DAB_CUDA(cudaEventRecord(pr->ev[5], st));
  pr->stats.n_video_frames = vs.prep.L; pr->stats.n_audio_frames = A.L;
  if (!ix) {
    DAB_CUDA(cudaEventRecord(pr->ev[6], st));
    DAB_TRY(enqueue_tables(pr, pr->video, dc));
    DAB_CUDA(cudaEventRecord(pr->ev[7], st));
  }
  DAB_TRY(enqueue_gate_score(pr, vs, dc));
  pr->ev_used[2] = pr->ev_used[4] = pr->ev_used[5] = true;
  pr->ev_used[3] = !ix;             // timing slot of the table build
  if (with_dp) DAB_TRY(enqueue_dp1(pr, vs));
  DAB_CUDA(cudaGetLastError());
  return dab_enqueue_counts(pr);
}

int dab_enqueue_counts(dab_pair *pr) {
  dab_ctx *ctx = pr->ctx;
  DAB_CUDA(dab_readback(pr, pr->h_counters, pr->counters.as<int32_t>(), sizeof(int32_t) * DC_WORDS));
  return DAB_OK;
}

int dab_check_stage_a_inputs(dab_pair *pr, const char *who) {
  dab_ctx *ctx = pr->ctx;
  for (int t = 0; t < 2; ++t) {
    if (!pr->trk[t].have_features) { dab_set_err(ctx, std::string(who) + ": features of both tracks are required first"); return DAB_E_STATE; }
    const int64_t lmin = pr->trk[t].Le < pr->trk[t].L ? pr->trk[t].Le : pr->trk[t].L;
    if (lmin < 2 * DAB_WIN) { dab_set_err(ctx, std::string(who) + ": track shorter than 82 frames"); return DAB_E_TOO_SHORT; }
  }
  return DAB_OK;
}

// dp1_kernel ends with DC_DP1_END = -1 when there is no path (also when there are no points)
void dab_collect_stage_a_dp(dab_pair *pr) {
  const int32_t *hc = reinterpret_cast<const int32_t *>(pr->h_counters);
  pr->n_path1 = hc[DC_DP1_END] < 0 ? 0 : hc[DC_N_PATH1];
  pr->stats.n_path1 = pr->n_path1;
}

// the counts of a stage-A run against the same video side as dab_enqueue_stage_a
int dab_collect_stage_a(dab_pair *pr, const dab_index *ix, bool with_dp) {
  dab_ctx *ctx = pr->ctx;
  const int32_t *hc = reinterpret_cast<const int32_t *>(pr->h_counters);
  const bool tables_ok = ix || collect_tables(pr->video, hc);   // the pair's own side was built in this run
  const VideoSide &vs = ix ? ix->side : pr->video;
  pr->points_side = &vs;
  pr->stats.n_video_selected = hc[DC_N_VSEL];
  pr->stats.n_audio_queries = hc[DC_N_Q];
  pr->stats.n_table_entries = vs.n_entries;
  pr->stats.n_enumerated = (int64_t)(((uint64_t)(uint32_t)hc[DC_ENUM_HI] << 32) | (uint32_t)hc[DC_ENUM_LO]);
  pr->stats.n_candidates = hc[DC_N_CAND];
  if (!tables_ok || (hc[DC_OVERFLOW] & DAB_OVF_CAND)) {
    if ((hc[DC_OVERFLOW] & DAB_OVF_CAND) && hc[DC_NEED_CAND] > DAB_MAX_CANDIDATES) {
      pr->cap_cand = DAB_MAX_CANDIDATES + 1;     // over the limit: the next enqueue refuses instead of running again
      dab_set_err(ctx, kTooManyCandidates);
      return DAB_E_CAPACITY;
    }
    // doubled, and at least the total this run needed: repeated audio (a shared tone, a looped bed) can need
    // hundreds of times the first guess, more than doubling reaches within DAB_STAGE_A_ATTEMPTS runs
    if (hc[DC_OVERFLOW] & DAB_OVF_CAND)
      pr->cap_cand = std::min(std::max<int64_t>(2 * pr->cap_cand, hc[DC_NEED_CAND]), DAB_MAX_CANDIDATES);
    dab_set_err(ctx, "stage A: a device buffer overflowed, capacity doubled");
    return DAB_E_CAPACITY;
  }
  pr->n_points1 = hc[DC_N_PTS1];
  pr->stats.n_points1 = pr->n_points1;
  if (with_dp) dab_collect_stage_a_dp(pr);
  return DAB_OK;
}

// ---- shared video index: the video side of the match stage, built once, read by any number of pairs --------
int dab_enqueue_index(dab_pair *src, dab_index *ix) {
  dab_ctx *ctx = src->ctx;
  DAB_TRY(ensure_hann(ctx));
  VideoSide &vs = ix->side;
  DAB_TRY(dab_ensure(ctx, ix->counters, sizeof(int32_t) * DC_WORDS));
  int32_t *dc = ix->counters.as<int32_t>();
  DAB_CUDA(cudaMemsetAsync(dc, 0, sizeof(int32_t) * DC_WORDS, src->stream));
  DAB_TRY(prep_track(src, src->trk[DAB_TRACK_VIDEO], vs.prep, true));
  // DC_N_VNQ and DC_N_VSEL; the audio words it also writes are never read from the index's block
  enqueue_counts_lists(src, dc, vs.prep, vs.prep, 0, 0);
  DAB_TRY(enqueue_tables(src, vs, dc));
  DAB_CUDA(dab_readback(src, src->h_counters, dc, sizeof(int32_t) * DC_WORDS));
  return DAB_OK;
}

int dab_collect_index(dab_pair *src, dab_index *ix) {
  dab_ctx *ctx = src->ctx;
  if (!collect_tables(ix->side, reinterpret_cast<const int32_t *>(src->h_counters))) return DAB_E_CAPACITY;
  DAB_CUDA(cudaEventRecord(ix->ready, src->stream));
  DAB_CUDA(cudaGetLastError());
  return DAB_OK;
}

// ---- row-sharded match stage: exchange of match points -----------------------------------
namespace {
// video frame -> rank in the selected-frame list (binary search; every frame of a point is in the list).
// Also checks what dp1_kernel relies on: points sorted by (audio frame, video frame) and quals > 0.
__global__ void frames_to_ranks_kernel(const int32_t *i_audio, const int32_t *v_frame, const double *qual, int64_t n,
                                       const int32_t *v_sel, int32_t n_sel, int32_t *rank, int32_t *bad) {
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int32_t v = v_frame[k];
  int lo = 0, hi = n_sel;
  while (lo < hi) {
    const int mid = lo + ((hi - lo) >> 1);
    if (v_sel[mid] < v) lo = mid + 1; else hi = mid;
  }
  if (lo >= n_sel || v_sel[lo] != v) { atomicOr(bad, 1); lo = 0; }
  if (!(qual[k] > 0.0)) atomicOr(bad, 2);
  if (k > 0) {
    const int32_t ip = i_audio[k - 1], ic = i_audio[k];
    if (ip > ic || (ip == ic && v_frame[k - 1] >= v)) atomicOr(bad, 4);
  }
  rank[k] = lo;
}
}  // namespace

static __global__ void set_word_kernel(int32_t *dc, int word, int32_t value) {
  if (threadIdx.x == 0 && blockIdx.x == 0) dc[word] = value;
}

int dab_run_import_points1(dab_pair *pr, const int32_t *i_audio, const int32_t *v_video, const double *qual,
                           int64_t n, int src_on_device) {
  dab_ctx *ctx = pr->ctx;
  const VideoSide &V = pr->video;
  cudaStream_t st = pr->stream;
  const cudaMemcpyKind kind = src_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
  DAB_TRY(dab_ensure(ctx, pr->pt_i, sizeof(int32_t) * (size_t)(n + 1)));
  DAB_TRY(dab_ensure(ctx, pr->pt_s, sizeof(int32_t) * (size_t)(n + 1)));
  DAB_TRY(dab_ensure(ctx, pr->pt_q, sizeof(double) * (size_t)(n + 1)));
  DAB_TRY(dab_ensure(ctx, pr->cand_tmp, sizeof(int32_t) * (size_t)(n + 1)));
  DAB_TRY(dab_ensure(ctx, pr->dpres, sizeof(int32_t) * 16));
  if (n > 0) {
    DAB_CUDA(cudaMemcpyAsync(pr->pt_i.p, i_audio, sizeof(int32_t) * (size_t)n, kind, st));
    DAB_CUDA(cudaMemcpyAsync(pr->cand_tmp.p, v_video, sizeof(int32_t) * (size_t)n, kind, st));
    DAB_CUDA(cudaMemcpyAsync(pr->pt_q.p, qual, sizeof(double) * (size_t)n, kind, st));
    DAB_CUDA(cudaMemsetAsync(pr->dpres.as<int32_t>() + 8, 0, sizeof(int32_t), st));
    frames_to_ranks_kernel<<<(unsigned)cdiv(n, 256), 256, 0, st>>>(pr->pt_i.as<int32_t>(), pr->cand_tmp.as<int32_t>(), pr->pt_q.as<double>(), n,
                                                                    V.prep.nq_list.as<int32_t>(), (int32_t)V.n_vsel, pr->pt_s.as<int32_t>(),
                                                                    pr->dpres.as<int32_t>() + 8);
    ctx->launches += 1;
    DAB_CUDA(dab_readback(pr, &pr->h_counters[22], pr->dpres.as<int32_t>() + 8, sizeof(int32_t)));
    DAB_CUDA(dab_wait_stream(st));
    const int32_t badbits = (int32_t)pr->h_counters[22];
    if (badbits != 0) {
      dab_set_err(ctx, badbits & 1 ? "import_points1: a point's video frame is not one of this pair's hashed video frames"
                        : (badbits & 2 ? "import_points1: match qualities must be > 0"
                                       : "import_points1: points must be sorted by (audio frame, video frame), without duplicates"));
      return DAB_E_ARG;
    }
  }
  set_word_kernel<<<1, 32, 0, st>>>(pr->counters.as<int32_t>(), DC_N_PTS1, (int32_t)n);
  ctx->launches += 1;
  DAB_CUDA(cudaGetLastError());
  pr->n_points1 = n;
  pr->stats.n_points1 = n;
  pr->n_path1 = 0;
  if (pr->cap_points1 < n) pr->cap_points1 = n;   // DP 1 sizes its buffers from it
  return DAB_OK;
}
