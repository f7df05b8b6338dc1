// Traceback of both frontier DPs (reference describealign.py:690-697 and :985-990) in five launches.
//
// The path is the chain of predecessor ids from the DP's end point; ids are in processing order, so a
// predecessor always has a smaller id and the path is sorted by id.  Points are cut into chunks of
// 1024 consecutive ids:
//   tb_exit_kernel    per chunk, in shared memory: pointer jumping (10 doublings) takes every point to its
//                     first ancestor in an EARLIER chunk (its exit)
//   tb_chain_kernel   one thread follows the exits from the end point: one hop per chunk the path visits,
//                     and notes where the path enters each chunk
//   tb_mark_kernel    per chunk: the in-chunk ancestors of the entry point, by the same doubling tables;
//                     their number
//   tb_offsets_kernel exclusive scan of the chunk counts (one block): first path position of every chunk
//   tb_emit_kernel    every marked point writes its path entry at offset + rank (Path1Out / Path2Out)
// instead of the 2 log2(n) full-size launches of plain list ranking.
#include "common.cuh"

namespace {

constexpr int TB_CHUNK = 1024;
constexpr int TB_THREADS = 256;
constexpr int TB_PER = TB_CHUNK / TB_THREADS;
constexpr int TB_LEVELS = 10;          // 2^10 = TB_CHUNK

struct TbArgs {
  const BackRec *back;
  const int32_t *n_dev;          // number of points
  const int32_t *result;         // [0] end id (-1: the seed, empty path); pass 2: double frontier value at +2
  int32_t *exit_id;              // [cap] first ancestor in an earlier chunk (-1 = seed)
  int32_t *entry;                // [chunks] id where the path enters the chunk, -1 = not visited (preset)
  int32_t *count;                // [chunks + 1] path points per chunk, then their exclusive scan
  unsigned char *mark;           // [cap]
  int32_t *n_path;
  int32_t chunks;                // launch size (from the capacity)
};

__global__ void __launch_bounds__(TB_THREADS) tb_exit_kernel(TbArgs a) {
  __shared__ int32_t up[2][TB_CHUNK];
  const int n = *a.n_dev;
  const int cs = blockIdx.x * TB_CHUNK;
  if (cs >= n) return;
#pragma unroll
  for (int u = 0; u < TB_PER; ++u) {
    const int l = threadIdx.x + u * TB_THREADS;
    up[0][l] = cs + l < n ? a.back[cs + l].pred : -1;
  }
  __syncthreads();
  int cur = 0;
  for (int k = 0; k < TB_LEVELS; ++k) {
#pragma unroll
    for (int u = 0; u < TB_PER; ++u) {
      const int l = threadIdx.x + u * TB_THREADS;
      const int p = up[cur][l];
      up[cur ^ 1][l] = p >= cs ? up[cur][p - cs] : p;
    }
    cur ^= 1;
    __syncthreads();
  }
#pragma unroll
  for (int u = 0; u < TB_PER; ++u) {
    const int l = threadIdx.x + u * TB_THREADS;
    if (cs + l < n) a.exit_id[cs + l] = up[cur][l];
  }
}

__global__ void tb_chain_kernel(TbArgs a) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  int cur = *a.n_dev > 0 ? a.result[0] : -1;
  while (cur >= 0) {
    a.entry[cur / TB_CHUNK] = cur;
    cur = a.exit_id[cur];
  }
}

__global__ void __launch_bounds__(TB_THREADS) tb_mark_kernel(TbArgs a) {
  __shared__ unsigned short up[TB_LEVELS][TB_CHUNK];     // 2^k-th in-chunk ancestor, TB_CHUNK = leaves the chunk
  __shared__ unsigned char mk[TB_CHUNK];
  __shared__ int s_cnt[TB_THREADS / 32];
  const int n = *a.n_dev;
  const int c = blockIdx.x;
  const int cs = c * TB_CHUNK;
  if (cs >= n) { if (threadIdx.x == 0) a.count[c] = 0; return; }
  const int e = a.entry[c];
  if (e < 0) {
#pragma unroll
    for (int u = 0; u < TB_PER; ++u) {
      const int l = threadIdx.x + u * TB_THREADS;
      if (cs + l < n) a.mark[cs + l] = 0;
    }
    if (threadIdx.x == 0) a.count[c] = 0;
    return;
  }
#pragma unroll
  for (int u = 0; u < TB_PER; ++u) {
    const int l = threadIdx.x + u * TB_THREADS;
    const int p = cs + l < n ? a.back[cs + l].pred : -1;
    up[0][l] = (unsigned short)(p >= cs ? p - cs : TB_CHUNK);
    mk[l] = (cs + l == e) ? 1 : 0;
  }
  __syncthreads();
  for (int k = 1; k < TB_LEVELS; ++k) {
#pragma unroll
    for (int u = 0; u < TB_PER; ++u) {
      const int l = threadIdx.x + u * TB_THREADS;
      const int p = up[k - 1][l];
      up[k][l] = p < TB_CHUNK ? up[k - 1][p] : (unsigned short)TB_CHUNK;
    }
    __syncthreads();
  }
  // ancestors of e: after processing level k (from the top), all ancestors at distances whose binary
  // expansion uses the levels seen so far are marked.  Within one level a thread may already see a mark another
  // thread set in the same pass (compute-sanitizer's racecheck reports it): that only marks a further TRUE ancestor
  // early - marks travel along predecessor links from e and are idempotent byte stores of 1 - so the final set,
  // all in-chunk ancestors of e, does not depend on the interleaving.
  for (int k = TB_LEVELS - 1; k >= 0; --k) {
#pragma unroll
    for (int u = 0; u < TB_PER; ++u) {
      const int l = threadIdx.x + u * TB_THREADS;
      if (mk[l]) {
        const int p = up[k][l];
        if (p < TB_CHUNK) mk[p] = 1;
      }
    }
    __syncthreads();
  }
  int cnt = 0;
#pragma unroll
  for (int u = 0; u < TB_PER; ++u) {
    const int l = threadIdx.x + u * TB_THREADS;
    if (cs + l < n) { a.mark[cs + l] = mk[l]; cnt += mk[l]; }
  }
  cnt = __reduce_add_sync(0xffffffffu, cnt);
  if ((threadIdx.x & 31) == 0) s_cnt[threadIdx.x >> 5] = cnt;
  __syncthreads();
  if (threadIdx.x == 0) {
    int t = 0;
    for (int x = 0; x < TB_THREADS / 32; ++x) t += s_cnt[x];
    a.count[c] = t;
  }
}

// exclusive scan of count[0 .. chunks) in place, total to count[chunks] and *n_path
__global__ void __launch_bounds__(1024) tb_offsets_kernel(TbArgs a) {
  __shared__ int s_w[32];
  __shared__ int s_carry;
  if (threadIdx.x == 0) s_carry = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int base = 0; base < a.chunks; base += 1024) {
    const int i = base + threadIdx.x;
    const int v = i < a.chunks ? a.count[i] : 0;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += y;
    }
    if (lane == 31) s_w[w] = inc;
    __syncthreads();
    if (w == 0) {
      int x = s_w[lane], xi = x;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, xi, o);
        if (lane >= o) xi += y;
      }
      s_w[lane] = xi - x;
    }
    __syncthreads();
    const int carry = s_carry;
    if (i < a.chunks) a.count[i] = carry + s_w[w] + inc - v;
    __syncthreads();
    if (threadIdx.x == 1023) s_carry = carry + s_w[w] + inc;
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    a.count[a.chunks] = s_carry;
    *a.n_path = (*a.n_dev > 0 && a.result[0] >= 0) ? s_carry : 0;
  }
}

// pass 1: audio frame and video frame of the point
__device__ __forceinline__ void emit_point(const Path1Out &o, const TbArgs &, int pos, int p) {
  o.x[pos] = o.pt_i[p];
  o.y[pos] = o.v_sel[o.pt_s[p]];
}

// pass 2: the row (j, i, cluster, qual, cum)
__device__ __forceinline__ void emit_point(const Path2Out &o, const TbArgs &a, int pos, int p) {
  double *row = o.rows + (int64_t)pos * 5;
  row[0] = o.p_j[p]; row[1] = (double)o.p_i[p]; row[2] = (double)o.p_c[p]; row[3] = o.p_q[p];
  // 5th column of a row = the (penalised) value its successor started from (describealign.py:983);
  // the end row carries the frontier value of the end point
  if (pos > 0) o.rows[(int64_t)(pos - 1) * 5 + 4] = a.back[p].best;
  if (p == a.result[0]) row[4] = *reinterpret_cast<const double *>(a.result + 2);
}

template <class Out>
__global__ void __launch_bounds__(TB_THREADS) tb_emit_kernel(TbArgs a, Out out) {
  __shared__ int s_w[TB_THREADS / 32];
  const int n = *a.n_dev;
  const int c = blockIdx.x;
  const int cs = c * TB_CHUNK;
  if (cs >= n || a.entry[c] < 0) return;
  // rank of every marked point among the chunk's marked points: thread-contiguous items
  int m[TB_PER], loc = 0;
#pragma unroll
  for (int u = 0; u < TB_PER; ++u) {
    const int l = threadIdx.x * TB_PER + u;
    m[u] = cs + l < n ? a.mark[cs + l] : 0;
    loc += m[u];
  }
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int inc = loc;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += y;
  }
  if (lane == 31) s_w[w] = inc;
  __syncthreads();
  int before = a.count[c] + inc - loc;
  for (int x = 0; x < w; ++x) before += s_w[x];
#pragma unroll
  for (int u = 0; u < TB_PER; ++u) {
    if (m[u]) emit_point(out, a, before++, cs + threadIdx.x * TB_PER + u);
  }
}

template <class Out>
int enqueue_traceback(dab_pair *pr, const BackRec *back, const int32_t *n_dev, const int32_t *result, int64_t cap,
                      int32_t *n_path, const Out &out) {
  dab_ctx *ctx = pr->ctx;
  cudaStream_t st = pr->stream;
  if (cap < 1) cap = 1;
  const int chunks = (int)cdiv(cap, TB_CHUNK);
  DAB_TRY(dab_ensure(ctx, pr->tb_up, sizeof(int32_t) * (size_t)(cap + 2 * chunks + 8)));
  DAB_TRY(dab_ensure(ctx, pr->tb_mark, (size_t)cap + 16));
  TbArgs a;
  a.back = back; a.n_dev = n_dev; a.result = result;
  a.exit_id = pr->tb_up.as<int32_t>();
  a.entry = a.exit_id + cap;
  a.count = a.entry + chunks;
  a.mark = pr->tb_mark.as<unsigned char>();
  a.n_path = n_path; a.chunks = chunks;
  DAB_CUDA(cudaMemsetAsync(a.entry, 0xff, sizeof(int32_t) * (size_t)chunks, st));
  tb_exit_kernel<<<chunks, TB_THREADS, 0, st>>>(a);
  tb_chain_kernel<<<1, 32, 0, st>>>(a);
  tb_mark_kernel<<<chunks, TB_THREADS, 0, st>>>(a);
  tb_offsets_kernel<<<1, 1024, 0, st>>>(a);
  tb_emit_kernel<<<chunks, TB_THREADS, 0, st>>>(a, out);
  ctx->launches += 5;
  return DAB_OK;
}

}  // namespace

int dab_enqueue_traceback(dab_pair *pr, const BackRec *back, const int32_t *n_dev, const int32_t *result, int64_t cap,
                          int32_t *n_path, const Path1Out &out) {
  return enqueue_traceback(pr, back, n_dev, result, cap, n_path, out);
}

int dab_enqueue_traceback(dab_pair *pr, const BackRec *back, const int32_t *n_dev, const int32_t *result, int64_t cap,
                          int32_t *n_path, const Path2Out &out) {
  return enqueue_traceback(pr, back, n_dev, result, cap, n_path, out);
}
