// Feature extraction for one track: the five 210 Hz feature vectors of the reference
// (get_energy describealign.py:545-555, get_zero_crossings :557-566, downsample_blur
// :568-573, get_freq_bands :575-593) in two kernels.
//
// features_kernel makes one pass over the PCM.  One CTA produces the per-frame intermediates of FT consecutive
// frames.  It stages the samples of frames [t0-8, t0+FT+8) plus 40 samples of filter halo in shared memory as float16
// (the reference's own sample type, :156) with 16-byte loads, derives lp1 @8820 Hz and lp2 @1260 Hz of the polyphase
// filter bank in shared memory, and writes per frame the 42 + 6 residual band energies, the band-2 frame energy, the
// two 105-sample block energies and the zero-crossing count (212 B) to a per-track scratch buffer.
// bands_kernel reads that scratch back and runs the 42 + 6 polyphase 15-tap filters at 210 Hz and the five outputs
// (24 B per frame).  The split sits where the least data crosses: the 210 Hz stage is bound by the f32->f64
// converts of the XU pipe, the 8820 Hz stage by the FMA / ALU / LSU pipes, and in one CTA each waited on the other
// at the barriers of every tile.  Apart, the small 210 Hz CTAs share SMs with other pairs' ALU-bound kernels.
// The Hann tables of features_kernel live in shared memory: they are indexed by the phase, which differs between the
// threads of a warp, and divergent __constant__ reads serialise.
//
// Bit-exactness (SURVEY.md B.1-B.3): every sum is evaluated in the order numpy / OpenBLAS
// use in the reference - parallelism is across outputs, never across the taps of one
// output - with separately rounded multiplies and adds (-fmad=false), f32 products
// accumulated in f64 where numpy does, and glibc's log10f restated in IEEE operations.
// The arithmetic cost of those fixed orders (about 6 500 instructions per frame, of which
// 630 f32->f64 conversions) is what bounds these kernels, not HBM.
#include <cuda_fp16.h>

#include <atomic>
#include <mutex>

#include "common.cuh"
#include "hann_tables.h"

namespace {

constexpr int FH = 8;             // halo frames each side (7 needed; 8 keeps tiles 16-byte aligned)
constexpr int PADS = 40;          // halo samples each side (lp2 needs lp1 +-7, lp1 needs +-5 samples)
constexpr int THREADS = 512;
constexpr int NTAB = 772;         // 630 + 90 + 21 + 15 + 13 = 769 floats, padded

template <int CH> struct Tile {
  static constexpr int FT = CH == 1 ? 100 : 48;      // output frames per tile
  static constexpr int NF = FT + 2 * FH;              // frames staged
  static constexpr int NS = NF * 210 + 2 * PADS;      // samples staged (multiple of 8)
  static constexpr int N1 = NF * 42 + 14;             // lp1 entries staged (+-7)
  // shared memory carve-up, in bytes, every section 16-byte aligned
  static constexpr int O_TAB = 0;
  static constexpr int O_SIG = O_TAB + NTAB * 4;
  static constexpr int O_RAW = O_SIG + (NS + 16) * 2;                           // stereo only: half2 per sample
  static constexpr int O_LP1 = O_RAW + (CH == 2 ? NF * 210 * 4 : 0);
  static constexpr int O_ZI = O_LP1 + ((N1 * 4 + 15) & ~15);
  static constexpr int BYTES = O_ZI + NF * 4;
  static_assert(NS % 8 == 0 && N1 % 2 == 0 && (NS * 2) % 16 == 0 && O_SIG % 16 == 0, "tile layout");
};

// bands_kernel: FR output frames per CTA, one thread per (phase, run of TC frames), 48 phases
constexpr int FR = 32;
constexpr int TC = 8;
constexpr int THREADS2 = 48 * FR / TC;

__device__ float g_tables[NTAB];   // w630 | w90 | w21 | w15 | w13
// "native numpy" mode (SURVEY.md B.4): numpy's SIMD log10 differs from glibc's log10f by up to 2 ulp on about
// half of the float32 inputs when the host CPU has AVX-512.  The host evaluates ITS np.log10 over every
// float32 in [1, 2^34) once and uploads the difference to the formula below as one nibble per input
// (value + 8); with the table set the feature kernel reproduces the host's numpy bit for bit.
__device__ const unsigned char *g_log10f_fix = nullptr;
__device__ unsigned int g_log10f_fix_count = 0;
__constant__ double c_logf_invc[16];
__constant__ double c_logf_logc[16];

const double h_logf_invc[16] = {
    0x1.661ec79f8f3bep+0, 0x1.571ed4aaf883dp+0, 0x1.49539f0f010bp+0,  0x1.3c995b0b80385p+0,
    0x1.30d190c8864a5p+0, 0x1.25e227b0b8eap+0,  0x1.1bb4a4a1a343fp+0, 0x1.12358f08ae5bap+0,
    0x1.0953f419900a7p+0, 0x1p+0,               0x1.e608cfd9a47acp-1, 0x1.ca4b31f026aap-1,
    0x1.b2036576afce6p-1, 0x1.9c2d163a1aa2dp-1, 0x1.886e6037841edp-1, 0x1.767dcf5534862p-1};
const double h_logf_logc[16] = {
    -0x1.57bf7808caadep-2, -0x1.2bef0a7c06ddbp-2, -0x1.01eae7f513a67p-2, -0x1.b31d8a68224e9p-3,
    -0x1.6574f0ac07758p-3, -0x1.1aa2bc79c81p-3,   -0x1.a4e76ce8c0e5ep-4, -0x1.1973c5a611cccp-4,
    -0x1.252f438e10c1ep-5, 0x0p+0,                0x1.aa5aa5df25984p-5,  0x1.c5e53aa362eb4p-4,
    0x1.526e57720db08p-3,  0x1.bc2860d22477p-3,   0x1.1058bc8a07ee1p-2,  0x1.4043057b6ee09p-2};

// glibc 2.39 logf / log10f for x >= 1 in plain IEEE operations (SURVEY.md B.3).
__device__ __forceinline__ float glibc_logf(float x) {
  uint32_t ix = __float_as_uint(x);
  if (ix == 0x3f800000u) return 0.0f;
  uint32_t tmp = ix - 0x3f330000u;
  int i = (tmp >> 19) & 15;
  int k = (int)tmp >> 23;
  uint32_t iz = ix - (tmp & 0xff800000u);
  double z = (double)__uint_as_float(iz);
  double r = z * c_logf_invc[i] - 1.0;
  double y0 = c_logf_logc[i] + (double)k * 0x1.62e42fefa39efp-1;
  double r2 = r * r;
  double p = 0x1.5575b0be00b6ap-2 * r + -0x1.ffffef20a4123p-2;
  p = -0x1.00ea348b88334p-2 * r2 + p;
  p = p * r2 + (y0 + r);
  return (float)p;
}

__device__ __forceinline__ float glibc_log10f(float x) {
  uint32_t hx = __float_as_uint(x);
  int k = (int)(hx >> 23) - 127;
  uint32_t i = ((uint32_t)k & 0x80000000u) >> 31;
  hx = (hx & 0x007fffffu) | ((0x7fu - i) << 23);
  float y = (float)(k + (int)i);
  float m = __uint_as_float(hx);
  float z = y * 7.9034151668e-07f + 4.3429449201e-01f * glibc_logf(m);
  return z + y * 3.0102920532e-01f;
}

// log10f as the reference's host computes it: glibc's formula, plus the host-specific correction if one was uploaded
__device__ __forceinline__ float host_log10f(float x) {
  float r = glibc_log10f(x);
  const unsigned char *fix = g_log10f_fix;
  if (fix) {
    const unsigned int idx = __float_as_uint(x) - 0x3f800000u;       // x >= 1: index of x among the floats from 1.0f up
    if (idx < g_log10f_fix_count) {
      const int nib = (fix[idx >> 1] >> ((idx & 1u) * 4u)) & 15;
      r = __int_as_float(__float_as_int(r) + (nib - 8));                // r >= 0: consecutive floats are consecutive ints
    }
  }
  return r;
}

// one PCM element as float16: int16 -> float16 (RNE) as describealign.py:156, or the half itself
template <int FMT>
__device__ __forceinline__ __half elem_half(const void *pcm, int64_t idx) {
  if (FMT == DAB_PCM_S16) return __short2half_rn(reinterpret_cast<const short *>(pcm)[idx]);
  return reinterpret_cast<const __half *>(pcm)[idx];
}

template <int FMT>
__device__ __forceinline__ __half bits_half(unsigned short b) {
  if (FMT == DAB_PCM_S16) return __short2half_rn((short)b);
  return __ushort_as_half(b);
}

// np.mean over the two float16 channels: float32 accumulate, divide, round to float16 (:576)
__device__ __forceinline__ __half mid_half(__half l, __half r) {
  const float s = __half2float(l) + __half2float(r);
  return __float2half_rn(s / 2.0f);
}

// Per-frame intermediates of a track, frames [0, L) (eb: blocks [0, 2 Le)), written by features_kernel and read by
// bands_kernel.  Frame-major: a warp over consecutive phases of one frame reads consecutive addresses.
struct FeatMid {
  float *be0;     // [L][42] band-0 residual energies at 8820 Hz
  float *be1;     // [L][6]  band-1 residual energies at 1260 Hz
  double *be2;    // [L]     band-2 frame energies
  float *eb;      // [2 Le]  105-sample block energies (0 past the last block)
  int *zi;        // [L]     zero crossings
};

struct FeatArgs {
  const void *pcm;
  int64_t S;      // samples per channel
  int64_t L;      // S / 210
  int64_t nb;     // S / 105
  int64_t Le;     // ceil(nb / 2)
  int vec_ok;     // pcm is 16-byte aligned
  int64_t tiles;  // tiles of FT output frames
  unsigned int *ticket;   // next tile (zeroed before the launch)
  FeatMid mid;
};

// 210 Hz kernel: the scratch written by features_kernel in, the five features out
struct BandArgs {
  FeatMid mid;
  int64_t L, Le;
  float *energy, *zc, *b0, *b1;
  double *b2;
};

// einsum('ijk,ijk->j') lane l of one 105 * CH element block (SURVEY.md B.2 i): elements
// l, l+4, ... accumulated in steps of 16 elements visiting the four 4-wide chunks in the order
// 3, 2, 1, 0, then the tail in increasing order.  X(e) returns element e of the block as float.
template <int CNT, typename FX>
__device__ __forceinline__ float energy_lane(FX X, int l) {
  float acc = 0.0f;
  int q = 0;
#pragma unroll 2
  for (; q + 16 <= CNT; q += 16) {
#pragma unroll
    for (int c4 = 3; c4 >= 0; --c4) {
      const float x = X(q + 4 * c4 + l);
      acc = acc + x * x;
    }
  }
#pragma unroll
  for (; q < CNT; q += 4) {
    if (q + l < CNT) {
      const float x = X(q + l);
      acc = acc + x * x;
    }
  }
  return acc;
}

// acc + a * b per lane with the product rounded on its own.  ptxas contracts mul.rn.f32x2 followed by
// add.rn.f32x2 into one FFMA2 (a single rounding) even under -fmad=false, which it never does for the
// scalar .rn forms; so the multiply is packed and the two adds are scalar.
__device__ __forceinline__ float2 mul2_then_add(float2 acc, float2 a, float2 b) {
  const float2 p = __fmul2_rn(a, b);
  return make_float2(__fadd_rn(acc.x, p.x), __fadd_rn(acc.y, p.y));
}

// lanes l and l + 1 (l even) of the same block as one packed accumulator.  (Here the contraction into
// FFMA2 is harmless and wanted: the samples are float16 values, so x * x is exact in float32 and
// fma(x, x, acc) rounds exactly what acc + x * x rounds.)
template <int CNT, typename FX>
__device__ __forceinline__ float2 energy_lanes2(FX X, int l) {
  float2 acc = make_float2(0.0f, 0.0f);
  int q = 0;
#pragma unroll 1
  for (; q + 16 <= CNT; q += 16) {
#pragma unroll
    for (int c4 = 3; c4 >= 0; --c4) {
      const float2 x = make_float2(X(q + 4 * c4 + l), X(q + 4 * c4 + l + 1));
      acc = __fadd2_rn(acc, __fmul2_rn(x, x));
    }
  }
#pragma unroll
  for (; q < CNT; q += 4) {
    // tail: lanes past the end of the block add nothing (they are skipped, not zero-filled, in the scalar form;
    // x = 0 adds +0, which leaves a non-negative accumulator unchanged)
    const float2 x = make_float2(q + l < CNT ? X(q + l) : 0.0f, q + l + 1 < CNT ? X(q + l + 1) : 0.0f);
    if (q + l < CNT) acc = __fadd2_rn(acc, __fmul2_rn(x, x));
  }
  return acc;
}

// ---- mbarrier / 1-D bulk copy (TMA) helpers: the raw PCM of the next tile is fetched by the copy engine into
//      the shared-memory signal buffer while the current tile's filter stages run ------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_load(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
  // the buffer was last touched through the generic proxy (all threads, before the CTA barrier that precedes this call)
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// Persistent kernel: 2 CTAs per SM, each taking tiles of FT frames from an atomic ticket.  Per tile:
//   S0   the staged signal arrives (bulk copy issued during the previous tile, converted int16 -> float16 in place;
//        edge tiles and stereo tracks are staged by the threads themselves)
//   S1   lp1 = downsample_blur(m, 5, 3) and, from the same register window, the band-0 residual energies
//   S2a  block energies, S2b zero crossings: like S1 they read only the signal, so the three share one phase; the
//        signal buffer is dead after it: the next tile's bulk copy is issued here and overlaps S2c
//   S2c  lp2 = downsample_blur(lp1, 7, 3) with the band-1 residual energies from the same window and the band-2
//        frame energies by warp shuffles
// The halo frames [t0-8, t0) and [t0+FT, t0+FT+8) are computed (lp2 needs them) but only the FT frames of the tile
// itself are written to the scratch.
template <int FMT, int CH>
__global__ void __launch_bounds__(THREADS, 2) features_kernel(FeatArgs a) {
  using T = Tile<CH>;
  constexpr int FT = T::FT, NF = T::NF, NS = T::NS, N1 = T::N1;
  extern __shared__ __align__(16) unsigned char smem[];
  __shared__ __align__(8) uint64_t s_bar;
  __shared__ int s_next;
  float *tab = reinterpret_cast<float *>(smem + T::O_TAB);
  const float *w21 = tab + 720, *w15 = tab + 741;
  __half *sig = reinterpret_cast<__half *>(smem + T::O_SIG);
  __half2 *raw = reinterpret_cast<__half2 *>(smem + T::O_RAW);   // stereo: (left, right) of frame samples
  float *lp1 = reinterpret_cast<float *>(smem + T::O_LP1);
  int *zi = reinterpret_cast<int *>(smem + T::O_ZI);

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t Sb = a.L * 210;                         // band signal length (:577)
  const int64_t len1 = a.L * 42, len2 = a.L * 6;

  // a tile whose staged window lies inside the band signal is fetched by the copy engine (mono tracks)
  auto bulk_ok = [&](int64_t tile) {
    if (CH != 1 || !a.vec_ok || tile >= a.tiles) return false;
    const int64_t s = (tile * FT - FH) * 210 - PADS;
    return s >= 0 && s + NS <= Sb;
  };
  auto bulk_issue = [&](int64_t tile) {
    const int64_t s = (tile * FT - FH) * 210 - PADS;
    mbar_expect_tx(&s_bar, NS * 2);
    bulk_load(sig, reinterpret_cast<const unsigned short *>(a.pcm) + s, NS * 2, &s_bar);
  };

  // ---- once per CTA: tables, the pad behind the signal, the first tile ------------------------------------
  for (int k = tid; k < NTAB; k += THREADS) tab[k] = g_tables[k];
  if (tid < 16) sig[NS + tid] = __float2half_rn(0.0f);      // read (never used) by the last lp1 task
  if (tid == 0) {
    mbar_init(&s_bar, 1);
    s_next = (int)atomicAdd(a.ticket, 1u);
  }
  __syncthreads();
  int64_t tile = s_next;
  if (tid == 0 && bulk_ok(tile)) bulk_issue(tile);
  uint32_t parity = 0;

  while (tile < a.tiles) {
    const int64_t t0 = tile * FT;                         // first output frame of this tile
    const int64_t f0 = t0 - FH;                           // first staged frame (may be < 0)
    const int64_t s0 = f0 * 210 - PADS;                   // first staged sample (may be < 0)

    // ---- S0: the mono / mid signal as float16, zero outside [0, Sb); the zero-crossing counts cleared ---------
    if (bulk_ok(tile)) {
      mbar_wait(&s_bar, parity);
      parity ^= 1u;
      if (FMT == DAB_PCM_S16) {
        // int16 -> float16 (RNE, describealign.py:156) in place, 8 samples per step
        for (int v = tid; v < NS / 8; v += THREADS) {
          const uint4 w = *reinterpret_cast<const uint4 *>(sig + 8 * v);
          const unsigned u[4] = {w.x, w.y, w.z, w.w};
          __align__(16) __half h[8];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            h[2 * e] = __short2half_rn((short)(u[e] & 0xffffu));
            h[2 * e + 1] = __short2half_rn((short)(u[e] >> 16));
          }
          *reinterpret_cast<uint4 *>(sig + 8 * v) = *reinterpret_cast<const uint4 *>(h);
        }
      }
    } else {
      // 8 samples per step; s0 is a multiple of 8 samples, so a 16-byte aligned source stays aligned
      for (int v = tid; v < NS / 8; v += THREADS) {
        const int64_t g = s0 + 8 * (int64_t)v;
        __align__(16) __half h[8];
        if (a.vec_ok && g >= 0 && g + 8 <= Sb) {
          if (CH == 1) {
            const uint4 w = __ldg(reinterpret_cast<const uint4 *>(reinterpret_cast<const unsigned short *>(a.pcm) + g));
            const unsigned u[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              h[2 * e] = bits_half<FMT>((unsigned short)(u[e] & 0xffffu));
              h[2 * e + 1] = bits_half<FMT>((unsigned short)(u[e] >> 16));
            }
          } else {
            const uint4 *src = reinterpret_cast<const uint4 *>(reinterpret_cast<const unsigned short *>(a.pcm) + 2 * g);
            const uint4 w0 = __ldg(src), w1 = __ldg(src + 1);
            const unsigned u[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
            const int fr = 8 * v - PADS;                      // index into raw (frame samples only)
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              const __half l = bits_half<FMT>((unsigned short)(u[e] & 0xffffu));
              const __half r = bits_half<FMT>((unsigned short)(u[e] >> 16));
              h[e] = mid_half(l, r);
              if (fr + e >= 0 && fr + e < NF * 210) raw[fr + e] = __halves2half2(l, r);
            }
          }
        } else {
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const int64_t ge = g + e;
            __half x = __float2half_rn(0.0f), l = x, r = x;
            if (ge >= 0 && ge < Sb) {
              if (CH == 1) x = elem_half<FMT>(a.pcm, ge);
              else { l = elem_half<FMT>(a.pcm, 2 * ge); r = elem_half<FMT>(a.pcm, 2 * ge + 1); x = mid_half(l, r); }
            }
            h[e] = x;
            if (CH == 2) {
              const int fr = 8 * v - PADS + e;
              if (fr >= 0 && fr < NF * 210) raw[fr] = __halves2half2(l, r);
            }
          }
        }
        *reinterpret_cast<uint4 *>(sig + 8 * v) = *reinterpret_cast<const uint4 *>(h);
      }
    }
    for (int k = tid; k < NF; k += THREADS) zi[k] = 0;     // the previous tile copied its counts out before its last barrier
    __syncthreads();

    // ---- S1: lp1 = downsample_blur(m, 5, 3): 5 phases x 3 taps, f32 accumulators (B.2 ii).  Two adjacent
    //      outputs per thread: their windows overlap (20 samples instead of 30 are loaded and converted) and
    //      their multiplies are one packed FMUL2.  The band-0 residual energy at 8820 Hz of lp1 entry k sums
    //      (x - lp1[k])^2 over the MIDDLE five samples of the very window lp1[k] was filtered from, so it is
    //      formed here from the registers ---------------------------------------------------------------------
    const int64_t n1_first = f0 * 42 - 7;          // global lp1 index of lp1[0]
    // the next tile; every thread has read s_next of this one before the barrier above, and reads this after S2b
    if (tid == 0) s_next = (int)atomicAdd(a.ticket, 1u);
    {
    const float w15r[15] = {w15[0], w15[1], w15[2], w15[3], w15[4], w15[5], w15[6], w15[7],
                            w15[8], w15[9], w15[10], w15[11], w15[12], w15[13], w15[14]};
    for (int u = tid; u < N1 / 2; u += THREADS) {
      const int k = 2 * u;
      // lp1[k] reads the staged samples 5k .. 5k+14 (samples outside [0, Sb) are staged as zero, which is
      // exactly the zero padding of the phase signals); 5k is a multiple of 10 halves: 4-byte aligned
      const __half2 *src = reinterpret_cast<const __half2 *>(sig + 5 * k);
      float x[20];
#pragma unroll
      for (int e = 0; e < 10; ++e) { const float2 v = __half22float2(src[e]); x[2 * e] = v.x; x[2 * e + 1] = v.y; }
      float2 tot = make_float2(0.0f, 0.0f);
#pragma unroll
      for (int p = 0; p < 5; ++p) {
        float2 acc = make_float2(0.0f, 0.0f);
#pragma unroll
        for (int j = 0; j < 3; ++j) {
          const float wv = w15r[p + (2 - j) * 5];
          acc = mul2_then_add(acc, make_float2(x[j * 5 + p], x[j * 5 + p + 5]), make_float2(wv, wv));
        }
        tot = __fadd2_rn(tot, acc);
      }
      const int64_t n = n1_first + k;
      const bool in0 = n >= 0 && n < len1, in1 = n + 1 >= 0 && n + 1 < len1;
      const float lo0 = in0 ? tot.x : 0.0f, lo1 = in1 ? tot.y : 0.0f;
      lp1[k] = lo0;
      lp1[k + 1] = lo1;
      // band-0 residuals of the same two entries: staged be0 index = k - 7 (be0[0] <-> lp1 entry f0 * 42)
      const float2 nlo = make_float2(-lo0, -lo1);
      float2 acc = make_float2(0.0f, 0.0f);
#pragma unroll
      for (int i = 0; i < 5; ++i) {
        const float2 d = __fadd2_rn(make_float2(x[5 + i], x[10 + i]), nlo);        // x - lo
        acc = (i == 0) ? __fmul2_rn(d, d) : mul2_then_add(acc, d, d);
      }
      // staged frame of lp1 entry k is (k - 7) / 42; the scratch takes the tile's own frames FH .. FH + FT - 1
      const int kb = k - 7;
      if (in0 && kb >= FH * 42 && kb < (FH + FT) * 42) a.mid.be0[n] = acc.x;
      if (in1 && kb + 1 >= FH * 42 && kb + 1 < (FH + FT) * 42) a.mid.be0[n + 1] = acc.y;
    }
    }

    // ---- S2a (no barrier before it: it reads only the signal): block energies (einsum order), 2 threads per
    //      105-sample block, each running two of the four lane accumulators as one packed f32x2 -----------------
    for (int k0 = 0; k0 < 2 * NF * 2; k0 += THREADS) {     // whole warps stay in the loop: it ends in a shuffle
      const int k = k0 + tid;
      const bool on = k < 2 * NF * 2;
      const int kb = k >> 1, l = (k & 1) * 2;           // lanes l, l + 1
      const int64_t b = 2 * f0 + kb;
      float2 acc = make_float2(0.0f, 0.0f);
      const bool valid = on && b >= 0 && b < a.nb;
      if (valid) {
        if ((b + 1) * 105 <= Sb) {
          if (CH == 1) {
            const __half *src = sig + PADS + kb * 105;
            acc = energy_lanes2<105>([&](int e) { return __half2float(src[e]); }, l);
          } else {
            const __half *src = reinterpret_cast<const __half *>(raw + kb * 105);
            acc = energy_lanes2<210>([&](int e) { return __half2float(src[e]); }, l);
          }
        } else {
          // the one block past the band signal (S mod 210 >= 105) is not staged: read it from HBM
          const int64_t base = b * 105 * CH;
          acc = energy_lanes2<105 * CH>([&](int e) { return __half2float(elem_half<FMT>(a.pcm, base + e)); }, l);
        }
      }
      const float s01 = acc.x + acc.y;                          // l0 + l1  /  l2 + l3
      const float o2 = __shfl_xor_sync(0xffffffffu, s01, 1);
      if (on && l == 0 && kb >= 2 * FH && kb < 2 * (FH + FT) && b < 2 * a.Le) a.mid.eb[b] = valid ? (s01 + o2) / (float)(105 * CH) : 0.0f;
    }

    // ---- S2b: zero crossings.  Sign changes between neighbouring samples, two samples (mono) or both
    //      channels of one sample (stereo) per 32-bit word: xor with the word shifted by one sample, keep the
    //      two sign bits, add them into two 16-bit counters.  Four chunks per frame ---------------------------
    for (int k = tid; k < NF * 4; k += THREADS) {
      const int kf = k >> 2, c = k & 3;
      const int64_t f = f0 + kf;
      if (f >= 0 && f < a.L) {
        constexpr int NW = CH == 1 ? 105 : 210;          // words per frame
        const int wlo = (NW * c) / 4, whi = (NW * (c + 1)) / 4;
        uint32_t acc = 0u;
        if (CH == 1) {
          // frame kf starts at half PADS + 210 kf: word 20 + 105 kf of the signal buffer
          const uint32_t *W = reinterpret_cast<const uint32_t *>(sig) + (PADS / 2 + 105 * kf);
          uint32_t prev = W[wlo - 1];                   // the staged zero (+0) in front of sample 0: np.diff prepend=False
#pragma unroll 9
          for (int e = wlo; e < whi; ++e) {
            const uint32_t w = W[e];
            const uint32_t y = __funnelshift_l(prev, w, 16);      // (sample 2e-1, sample 2e)
            acc += ((w ^ y) & 0x80008000u) >> 15;
            prev = w;
          }
        } else {
          const uint32_t *W = reinterpret_cast<const uint32_t *>(raw) + 210 * kf;
          uint32_t prev;
          if (kf == 0 && c == 0) {
            const int64_t n = f * 210;
            prev = n == 0 ? 0u
                          : ((uint32_t)__half_as_ushort(elem_half<FMT>(a.pcm, (n - 1) * 2)) |
                             ((uint32_t)__half_as_ushort(elem_half<FMT>(a.pcm, (n - 1) * 2 + 1)) << 16));
          } else {
            prev = W[wlo - 1];
          }
#pragma unroll 8
          for (int e = wlo; e < whi; ++e) {
            const uint32_t w = W[e];
            acc += ((w ^ prev) & 0x80008000u) >> 15;
            prev = w;
          }
        }
        atomicAdd(&zi[kf], (int)((acc & 0xffffu) + (acc >> 16)));
      }
    }

    __syncthreads();   // sig is dead from here on: it receives the next tile while S2c runs
    const int64_t next = s_next;
    if (tid == 0 && bulk_ok(next)) bulk_issue(next);
    for (int k = tid; k < FT; k += THREADS) {
      const int64_t f = t0 + k;
      if (f < a.L) a.mid.zi[f] = zi[FH + k];
    }

    // ---- S2c: lp2 = downsample_blur(lp1, 7, 3), 7 phases x 3 taps (f32), the band-1 residual energy at
    //      1260 Hz from the middle seven entries of the same window, and the band-2 energy of a frame
    //      (f64, :583/:588) from its six lp2 values by shuffles: a warp takes five frames (30 lanes) ----------
    {
      float w21r[21];
#pragma unroll
      for (int e = 0; e < 21; ++e) w21r[e] = w21[e];
      constexpr int NG = (NF + 4) / 5;
      for (int g = warp; g < NG; g += THREADS / 32) {
        const int fr = lane / 6, i6 = lane - fr * 6;
        const int kf = 5 * g + fr;
        const bool act = lane < 30 && kf < NF;
        const int k = kf * 6 + i6;
        const int64_t n2 = f0 * 6 + k;
        float total = 0.0f, r1 = 0.0f;
        if (act && n2 >= 0 && n2 < len2) {
          const float *src = lp1 + 7 * k;                 // lp1 entries (n2 - 1) * 7 .. + 20; lp1 is zero outside [0, len1)
          float r[21];
#pragma unroll
          for (int e = 0; e < 21; ++e) r[e] = src[e];
#pragma unroll
          for (int p = 0; p < 7; ++p) {
            float acc = 0.0f;
#pragma unroll
            for (int j = 0; j < 3; ++j) acc = acc + r[j * 7 + p] * w21r[p + (2 - j) * 7];
            total = total + acc;
          }
#pragma unroll
          for (int i = 0; i < 7; ++i) {
            const float d = r[7 + i] - total;
            const float sq = d * d;
            r1 = (i == 0) ? sq : r1 + sq;
          }
        }
        const bool own = act && kf >= FH && kf < FH + FT;
        if (own && n2 >= 0 && n2 < len2) a.mid.be1[n2] = r1;
        double acc2 = 0.0;
#pragma unroll
        for (int i = 0; i < 6; ++i) {
          const double x = (double)__shfl_sync(0xffffffffu, total, (lane - i6 + i) & 31);
          const double sq = x * x;
          acc2 = (i == 0) ? sq : acc2 + sq;
        }
        if (own && i6 == 0) {
          const int64_t f = f0 + kf;
          if (f >= 0 && f < a.L) a.mid.be2[f] = acc2;
        }
      }
    }
    __syncthreads();   // lp1 and zi are dead from here on
    tile = next;
  }
}

// The 210 Hz stage: a plain grid, one CTA per FR output frames.
//   S3   band 0: 42 phases x 15 taps and band 1: 6 phases x 15 taps; each phase = f32 products accumulated in f64
//        (B.2 iii).  One thread per (phase, run of TC frames), its window read from the scratch into registers
//   S4   the five outputs, four thread roles per frame (one role per warp)
// Scratch frames outside [0, L) (blocks outside [0, 2 Le)) read as zero, as the reference's zero padding does.
template <int CH>
__global__ void __launch_bounds__(THREADS2, 6) bands_kernel(BandArgs a) {
  __shared__ float ph[FR * 42];
  __shared__ float p1[FR * 6];
  const float *w630 = g_tables, *w90 = g_tables + 630, *w15 = g_tables + 741, *w13 = g_tables + 756;
  const int tid = threadIdx.x;
  const int64_t t0 = (int64_t)blockIdx.x * FR;      // first output frame of this CTA

  {
    const int ch = tid / 48, pp = tid - ch * 48;
    const bool b0 = pp < 42;
    const int p = b0 ? pp : pp - 42;
    const int np = b0 ? 42 : 6;
    const float *src = (b0 ? a.mid.be0 : a.mid.be1) + p;
    const float *w = (b0 ? w630 : w90) + p;
    float *dst = (b0 ? ph : p1) + p;
    const int tb = ch * TC;
    // output frame t0 + tb + t uses frames t0 + tb + t - 7 .. + 7 (tap j <-> window entry t + j)
    const int64_t fw = t0 + tb - 7;
    float win[14 + TC], wr[15];
    if (fw >= 0 && fw + 14 + TC <= a.L) {
      const float *s = src + fw * np;
#pragma unroll
      for (int e = 0; e < 14 + TC; ++e) win[e] = __ldg(s + e * np);
    } else {
#pragma unroll
      for (int e = 0; e < 14 + TC; ++e) win[e] = (fw + e >= 0 && fw + e < a.L) ? __ldg(src + (fw + e) * np) : 0.0f;
    }
#pragma unroll
    for (int j = 0; j < 15; ++j) wr[j] = __ldg(w + (14 - j) * np);
#pragma unroll
    for (int t = 0; t < TC; ++t) {
      if (t0 + tb + t < a.L) {
        double acc = 0.0;
#pragma unroll
        for (int j = 0; j < 15; ++j) {
          const float prod = win[t + j] * wr[j];
          acc += (double)prod;
        }
        dst[(tb + t) * np] = (float)acc;
      }
    }
  }
  __syncthreads();

  if (tid < 4 * FR) {
    const int role = tid / FR, t = tid - role * FR;
    const int64_t f = t0 + t;
    if (role == 0) {
      if (f < a.L) {
        // band 0: phases added sequentially in f32 (B.2 v), /210, log10(1+x)/2
        float tot = 0.0f;
#pragma unroll 6
        for (int p = 0; p < 42; ++p) tot = tot + ph[t * 42 + p];
        a.b0[f] = host_log10f(1.0f + tot / 210.0f) / 2.0f;
      }
    } else if (role == 1) {
      if (f < a.L) {
        float tot = 0.0f;
#pragma unroll
        for (int p = 0; p < 6; ++p) tot = tot + p1[t * 6 + p];
        a.b1[f] = host_log10f(1.0f + tot / 210.0f) / 2.0f;
        // zero crossings: 13-tap Hann over frames f-6 .. f+6
        double acc = 0.0;
#pragma unroll
        for (int j = 0; j < 13; ++j) {
          const int64_t g = f - 6 + j;
          float z = (g >= 0 && g < a.L) ? (float)a.mid.zi[g] : 0.0f;
          if (CH == 1) z = z * 2.0f;
          const float prod = z * w13[12 - j];
          acc += (double)prod;
        }
        a.zc[f] = (float)acc;
      }
    } else if (role == 2) {
      if (f < a.L) {
        // band 2: one 15-tap f64 filter = OpenBLAS ddot tail, a sequential FMA chain (B.2 iv)
        double acc = 0.0;
#pragma unroll
        for (int j = 0; j < 15; ++j) {
          const int64_t g = f - 7 + j;
          acc = fma((double)w15[14 - j], (g >= 0 && g < a.L) ? a.mid.be2[g] : 0.0, acc);
        }
        a.b2[f] = log10(1.0 + acc / 210.0) / 2.0;
      }
    } else {
      if (f < a.Le) {
        // energy: 13-tap Hann over blocks 2f-6 .. 2f+6, log10(1+x)/2, every second block (:553-555)
        double acc = 0.0;
#pragma unroll
        for (int j = 0; j < 13; ++j) {
          const int64_t b = 2 * f - 6 + j;
          const float prod = ((b >= 0 && b < 2 * a.Le) ? a.mid.eb[b] : 0.0f) * w13[12 - j];
          acc += (double)prod;
        }
        a.energy[f] = host_log10f(1.0f + (float)acc) / 2.0f;
      }
    }
  }
}

std::atomic<bool> g_const_ready[64];
std::mutex g_const_mu;

// the tables are the same for every pair: uploaded once per device, by whichever host thread comes first
int upload_constants(dab_ctx *ctx) {
  int dev = 0;
  DAB_CUDA(cudaGetDevice(&dev));
  if (dev < 64 && g_const_ready[dev].load(std::memory_order_acquire)) return DAB_OK;
  std::lock_guard<std::mutex> lock(g_const_mu);
  if (dev < 64 && g_const_ready[dev].load(std::memory_order_acquire)) return DAB_OK;
  float tab[NTAB] = {};
  memcpy(tab, DAB_HANN630_F32, sizeof(DAB_HANN630_F32));
  memcpy(tab + 630, DAB_HANN90_F32, sizeof(DAB_HANN90_F32));
  memcpy(tab + 720, DAB_HANN21_F32, sizeof(DAB_HANN21_F32));
  memcpy(tab + 741, DAB_HANN15_F32, sizeof(DAB_HANN15_F32));
  memcpy(tab + 756, DAB_HANN13_F32, sizeof(DAB_HANN13_F32));
  DAB_CUDA(cudaMemcpyToSymbol(g_tables, tab, sizeof(tab)));
  DAB_CUDA(cudaMemcpyToSymbol(c_logf_invc, h_logf_invc, sizeof(h_logf_invc)));
  DAB_CUDA(cudaMemcpyToSymbol(c_logf_logc, h_logf_logc, sizeof(h_logf_logc)));
  if (dev < 64) g_const_ready[dev].store(true, std::memory_order_release);
  return DAB_OK;
}

__global__ void eval_log10f_kernel(const float *x, float *y, int64_t n) {
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k < n) y[k] = x[k] >= 1.0f ? host_log10f(x[k]) : 0.0f;
}

std::mutex g_fix_mu;
void *g_fix_buf[64] = {};      // per device: the uploaded correction table

template <int FMT, int CH>
int launch(dab_pair *pr, const FeatArgs &fa_in, const BandArgs &ba, int64_t frames) {
  dab_ctx *ctx = pr->ctx;
  const int64_t tiles = cdiv(frames, Tile<CH>::FT);
  if (tiles <= 0) return DAB_OK;
  FeatArgs fa = fa_in;
  fa.tiles = tiles;
  const size_t smem = Tile<CH>::BYTES;
  DAB_CUDA(cudaFuncSetAttribute(features_kernel<FMT, CH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  // persistent: two CTAs per SM take tiles from the ticket
  DAB_CUDA(cudaMemsetAsync(fa.ticket, 0, sizeof(unsigned int), pr->stream));
  const int64_t grid = tiles < 2 * (int64_t)ctx->sm_count ? tiles : 2 * (int64_t)ctx->sm_count;
  features_kernel<FMT, CH><<<(unsigned)grid, THREADS, smem, pr->stream>>>(fa);
  DAB_LAUNCHED(pr);
  DAB_CUDA(cudaGetLastError());
  bands_kernel<CH><<<(unsigned)cdiv(frames, FR), THREADS2, 0, pr->stream>>>(ba);
  DAB_LAUNCHED(pr);
  DAB_CUDA(cudaGetLastError());
  return DAB_OK;
}

}  // namespace

extern "C" {

int dab_set_log10f_correction(dab_ctx *ctx, const unsigned char *nibbles, uint64_t count) {
  if (!ctx || (count > 0 && !nibbles) || count > 0xffffffffull) return DAB_E_ARG;
  DAB_CUDA(cudaSetDevice(ctx->device));
  DAB_TRY(upload_constants(ctx));
  std::lock_guard<std::mutex> lock(g_fix_mu);
  DAB_CUDA(cudaDeviceSynchronize());       // no feature kernel may be reading the old table
  const unsigned char *none = nullptr;
  const unsigned int zero = 0;
  DAB_CUDA(cudaMemcpyToSymbol(g_log10f_fix, &none, sizeof(none)));
  DAB_CUDA(cudaMemcpyToSymbol(g_log10f_fix_count, &zero, sizeof(zero)));
  const int dev = ctx->device;
  if (dev < 64 && g_fix_buf[dev]) { cudaFree(g_fix_buf[dev]); g_fix_buf[dev] = nullptr; }
  if (count == 0) return DAB_OK;
  void *buf = nullptr;
  const size_t bytes = (size_t)((count + 1) / 2);
  DAB_CUDA(cudaMalloc(&buf, bytes));
  DAB_CUDA(cudaMemcpy(buf, nibbles, bytes, cudaMemcpyHostToDevice));
  const unsigned int cnt = (unsigned int)count;
  DAB_CUDA(cudaMemcpyToSymbol(g_log10f_fix, &buf, sizeof(buf)));
  DAB_CUDA(cudaMemcpyToSymbol(g_log10f_fix_count, &cnt, sizeof(cnt)));
  if (dev < 64) g_fix_buf[dev] = buf;
  return DAB_OK;
}

int dab_eval_log10f(dab_ctx *ctx, const float *x, float *y, int64_t n) {
  if (!ctx || n < 0 || (n > 0 && (!x || !y))) return DAB_E_ARG;
  if (n == 0) return DAB_OK;
  DAB_CUDA(cudaSetDevice(ctx->device));
  DAB_TRY(upload_constants(ctx));
  float *dx = nullptr, *dy = nullptr;
  DAB_CUDA(cudaMalloc(&dx, sizeof(float) * (size_t)n));
  if (cudaMalloc(&dy, sizeof(float) * (size_t)n) != cudaSuccess) { cudaFree(dx); dab_set_err(ctx, "dab_eval_log10f: out of device memory"); return DAB_E_CUDA; }
  cudaError_t e = cudaMemcpy(dx, x, sizeof(float) * (size_t)n, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) {
    eval_log10f_kernel<<<(unsigned)cdiv(n, 256), 256>>>(dx, dy, n);
    ctx->launches += 1;
    e = cudaMemcpy(y, dy, sizeof(float) * (size_t)n, cudaMemcpyDeviceToHost);
  }
  cudaFree(dx); cudaFree(dy);
  if (e != cudaSuccess) { dab_set_err(ctx, std::string("dab_eval_log10f: ") + cudaGetErrorString(e)); return DAB_E_CUDA; }
  return DAB_OK;
}

}  // extern "C"

int dab_run_features(dab_pair *pr, int track, const void *d_pcm, int format) {
  dab_ctx *ctx = pr->ctx;
  Track &tk = pr->trk[track];
  DAB_TRY(upload_constants(ctx));
  const int64_t L = tk.S / 210, nb = tk.S / 105, Le = (nb + 1) / 2;
  tk.L = L;
  tk.Le = Le;
  DAB_TRY(dab_ensure(ctx, tk.energy, sizeof(float) * (size_t)(Le + 1)));
  DAB_TRY(dab_ensure(ctx, tk.zc, sizeof(float) * (size_t)(L + 1)));
  DAB_TRY(dab_ensure(ctx, tk.b0, sizeof(float) * (size_t)(L + 1)));
  DAB_TRY(dab_ensure(ctx, tk.b1, sizeof(float) * (size_t)(L + 1)));
  DAB_TRY(dab_ensure(ctx, tk.b2, sizeof(double) * (size_t)(L + 1)));
  DAB_TRY(dab_ensure(ctx, tk.feat_ticket, 64));
  // the scratch between the two kernels: 212 B per frame, each section 256-byte aligned
  size_t off = 0;
  auto section = [&](size_t bytes) { const size_t o = off; off += (bytes + 255) & ~(size_t)255; return o; };
  const size_t o_be2 = section(sizeof(double) * (size_t)L), o_be0 = section(sizeof(float) * 42 * (size_t)L),
               o_be1 = section(sizeof(float) * 6 * (size_t)L), o_eb = section(sizeof(float) * 2 * (size_t)Le),
               o_zi = section(sizeof(int) * (size_t)L);
  DAB_TRY(dab_ensure(ctx, tk.feat_mid, off + 256));
  unsigned char *mid = tk.feat_mid.as<unsigned char>();
  FeatMid fm;
  fm.be0 = reinterpret_cast<float *>(mid + o_be0); fm.be1 = reinterpret_cast<float *>(mid + o_be1);
  fm.be2 = reinterpret_cast<double *>(mid + o_be2); fm.eb = reinterpret_cast<float *>(mid + o_eb);
  fm.zi = reinterpret_cast<int *>(mid + o_zi);
  FeatArgs fa;
  fa.tiles = 0;
  fa.ticket = tk.feat_ticket.as<unsigned int>();
  fa.pcm = d_pcm; fa.S = tk.S; fa.L = L; fa.nb = nb; fa.Le = Le;
  fa.vec_ok = (reinterpret_cast<uintptr_t>(d_pcm) & 15u) == 0;
  fa.mid = fm;
  BandArgs ba;
  ba.mid = fm; ba.L = L; ba.Le = Le;
  ba.energy = tk.energy.as<float>(); ba.zc = tk.zc.as<float>();
  ba.b0 = tk.b0.as<float>(); ba.b1 = tk.b1.as<float>(); ba.b2 = tk.b2.as<double>();
  const int64_t frames = Le > L ? Le : L;
  if (format == DAB_PCM_S16 && tk.ch == 1) DAB_TRY((launch<DAB_PCM_S16, 1>(pr, fa, ba, frames)));
  else if (format == DAB_PCM_S16 && tk.ch == 2) DAB_TRY((launch<DAB_PCM_S16, 2>(pr, fa, ba, frames)));
  else if (format == DAB_PCM_F16 && tk.ch == 1) DAB_TRY((launch<DAB_PCM_F16, 1>(pr, fa, ba, frames)));
  else if (format == DAB_PCM_F16 && tk.ch == 2) DAB_TRY((launch<DAB_PCM_F16, 2>(pr, fa, ba, frames)));
  else { dab_set_err(ctx, "unsupported PCM format / channel count"); return DAB_E_ARG; }
  tk.have_features = true;
  return DAB_OK;
}
