// Temporal reductions and scans over the band axis
// (raster/temporal.py:722-768 TemporalAggregate, :959-1005 Cumulative).
//
// Consecutive threads own consecutive pixels, so every frame is read with fully coalesced
// accesses and the whole (T, H, W) stack is streamed once (twice for std / var).  The streaming
// kernels give a thread VEC pixels: VEC = 16 / sizeof(S) when every frame is whole 16-byte
// pixel groups from a 16-byte aligned base (one 128-bit load per frame), else VEC = 1.
// Accumulation is sequential in t in the reference's working dtype W (float32 or float64 =
// result_type(float32, out dtype)), which is what NumPy's axis-0 reductions do, so sums are
// bit-identical.  Each per-pixel rule of NumPy's semantics is stated once, in the helpers below.
#include "gm_common.cuh"
#include "gm_sort_networks.cuh"
#include <type_traits>
#include <cfloat>
#include <limits>

namespace gm {

constexpr int TMP_MAX_SORT = 1024;  // frames per bin for median / percentile
constexpr int TMP_SORT_SMEM = 160 * 1024;  // shared-memory sort columns per block
constexpr int GM_STAT_ANY = -1;     // temporal_stream_kernel reads the statistic at run time

template <typename W> __device__ __forceinline__ W nan_();
template <> __device__ __forceinline__ float nan_<float>() { return __int_as_float(0x7fc00000); }
template <> __device__ __forceinline__ double nan_<double>() { return __longlong_as_double(0x7ff8000000000000LL); }

template <typename D> struct DMax { static __host__ __device__ D value() { return std::numeric_limits<D>::max(); } };

// A sample counts unless it is the source's no-data value or NaN in the working dtype.
template <typename W, typename S>
__device__ __forceinline__ bool sample_counts(S v, S nodata, int has_nodata) {
  const W w = (W)v;
  return !(has_nodata && v == nodata) && w == w;
}

// A result is stored when it is finite in the working dtype (and the bin has frames), else the
// fill value.
template <typename W, typename D>
__device__ __forceinline__ D finite_or(W result, D fill, bool has_frames = true) {
  const bool finite = (result == result) && (fabs((double)result) <= (sizeof(W) == 4 ? (double)FLT_MAX : DBL_MAX));
  return (has_frames && finite) ? (D)result : fill;
}

// Median and np.nanpercentile(method="linear") of n sorted samples: the ranks lo, hi of the two
// samples a, b it reads and the weight t; then the value from a and b.  Percentiles take q / 100,
// the virtual index (n - 1) * q, t and the lerp all in W arithmetic
// (numpy/lib/_function_base_impl.py: percentile, _quantile, _lerp).
template <typename W> struct OrderRanks { int lo, hi; W t; };

template <typename W>
__device__ __forceinline__ OrderRanks<W> order_ranks(int n, int stat, double q) {
  if (stat == GM_STAT_MEDIAN) return {(n - 1) / 2, n / 2, (W)0};
  const W qw = (W)q / (W)100;
  const W virt = (W)(n - 1) * qw;
  int lo = (int)floor((double)virt);
  if (lo < 0) lo = 0;
  if (lo > n - 1) lo = n - 1;
  return {lo, lo + 1 < n ? lo + 1 : n - 1, virt - (W)lo};
}

template <typename W>
__device__ __forceinline__ W order_value(W a, W b, W t, int n, int stat) {
  if (stat == GM_STAT_MEDIAN) return (n & 1) ? a : (a + b) / (W)2;
  const W diff = b - a;
  return t >= (W)0.5 ? b - diff * ((W)1 - t) : a + diff * t;
}

// np.nanvar / np.nanstd from the sum of squared deviations from the mean and the sample count.
template <typename W>
__device__ __forceinline__ W var_or_std(W ss, int cnt, int stat) {
  const W var = cnt > 0 ? (W)((double)ss / (double)cnt) : nan_<W>();
  if (stat != GM_STAT_STD) return var;
  return sizeof(W) == 4 ? (W)sqrtf((float)var) : (W)sqrt((double)var);
}

// VEC consecutive pixels of one frame: one 128-bit streaming load, or one element when VEC = 1.
template <typename S, int VEC> struct alignas(sizeof(S) * VEC) PixelVec { S v[VEC]; };

template <int VEC, typename S>
__device__ __forceinline__ PixelVec<S, VEC> load_pixels(const S* p) {
  PixelVec<S, VEC> x;
  if constexpr (VEC == 1) {
    x.v[0] = __ldcs(p);
  } else {
    static_assert(sizeof(PixelVec<S, VEC>) == 16, "16-byte pixel groups");
    union { uint4 raw; PixelVec<S, VEC> vec; } u;
    u.raw = ::__ldcs(reinterpret_cast<const uint4*>(p));
    x = u.vec;
  }
  return x;
}

// The frame walk of the streaming kernels over the frames f0..f1 of a bin: UNROLL frames of the
// thread's VEC pixels are loaded before any is used, then step(x, f) takes frame f's pixels x in
// order of t, and round_end() runs after every round (UNROLL frames, or one frame of the tail).
template <int VEC, int UNROLL, typename S, typename Step, typename RoundEnd>
__device__ __forceinline__ void walk_frames(const S* __restrict__ src, const int* __restrict__ frame_index,
                                            int f0, int f1, int64_t plane, int64_t pix, Step step,
                                            RoundEnd round_end) {
  int f = f0;
  for (; f + UNROLL <= f1; f += UNROLL) {
    PixelVec<S, VEC> x[UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) x[u] = load_pixels<VEC>(src + (int64_t)frame_index[f + u] * plane + pix);
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) step(x[u], f + u);
    round_end();
  }
  for (; f < f1; ++f) {
    step(load_pixels<VEC>(src + (int64_t)frame_index[f] * plane + pix), f);
    round_end();
  }
}

// Median / percentile: every thread sorts the valid samples of its pixel in its own
// shared-memory column (column-major, so the lanes of a warp touch consecutive words: no
// bank conflicts) with a bitonic network.  The network is data independent -- all threads run
// the same compare-exchange sequence, no divergence -- and costs n log^2 n / 4 exchanges.
// Invalid samples are padded with +inf behind the valid ones.
template <typename S, typename W, typename D>
__global__ void temporal_sort_kernel(const S* __restrict__ src, D* __restrict__ dst, S nodata, int has_nodata,
                                     int stat, double q, const int* __restrict__ bin_offsets,
                                     const int* __restrict__ frame_index, int n_bins, int64_t plane) {
  extern __shared__ __align__(16) unsigned char sort_smem[];
  W* col = reinterpret_cast<W*>(sort_smem) + threadIdx.x;
  const int BD = blockDim.x;
  const int64_t pix = blockIdx.x * (int64_t)BD + threadIdx.x;
  if (pix >= plane) return;
  const D fill = DMax<D>::value();
  const W inf = (W)INFINITY;
  for (int g = 0; g < n_bins; ++g) {
    const int f0 = bin_offsets[g], f1 = bin_offsets[g + 1];
    int n = 0;
    for (int f = f0; f < f1; ++f) {
      const S v = __ldcs(src + (int64_t)frame_index[f] * plane + pix);
      if (sample_counts<W>(v, nodata, has_nodata)) { col[n * BD] = (W)v; ++n; }
    }
    int p2 = 1;
    while (p2 < f1 - f0) p2 <<= 1;
    for (int i = n; i < p2; ++i) col[i * BD] = inf;
    for (int k = 2; k <= p2; k <<= 1)
      for (int j = k >> 1; j > 0; j >>= 1)
        for (int idx = 0; idx < (p2 >> 1); ++idx) {
          const int i = ((idx & ~(j - 1)) << 1) | (idx & (j - 1)), l = i | j;
          const W a = col[i * BD], b = col[l * BD];
          const bool up = (i & k) == 0;
          const W lo = a < b ? a : b, hi = a < b ? b : a;
          col[i * BD] = up ? lo : hi;
          col[l * BD] = up ? hi : lo;
        }
    D out = fill;
    if (n > 0) {
      const OrderRanks<W> r = order_ranks<W>(n, stat, q);
      out = finite_or(order_value(col[r.lo * BD], col[r.hi * BD], r.t, n, stat), fill);
    }
    dst[(int64_t)g * plane + pix] = out;
  }
}

// Median / percentile of bins of at most 64 frames: the samples of a pixel live in REGISTERS
// (P = 16, 32 or 64 slots, invalid ones = +inf) and the sorting network is fully unrolled --
// every compare-exchange is two FMNMX on registers instead of two loads, two stores and the
// selects of the shared-memory version (543 exchanges at P = 64: 1.1 k instead of 6.7 k
// instructions per pixel).  The two order statistics are picked with unrolled predicated moves
// (a dynamically indexed register array would go to local memory).
template <typename W> __device__ __forceinline__ W wmin(W a, W b) { return a < b ? a : b; }
template <typename W> __device__ __forceinline__ W wmax(W a, W b) { return a < b ? b : a; }
template <> __device__ __forceinline__ float wmin<float>(float a, float b) { return fminf(a, b); }
template <> __device__ __forceinline__ float wmax<float>(float a, float b) { return fmaxf(a, b); }
template <> __device__ __forceinline__ double wmin<double>(double a, double b) { return fmin(a, b); }
template <> __device__ __forceinline__ double wmax<double>(double a, double b) { return fmax(a, b); }

template <typename S, typename W, typename D, int P>
__global__ void __launch_bounds__(128)
temporal_sort_reg_kernel(const S* __restrict__ src, D* __restrict__ dst, S nodata, int has_nodata,
                         int stat, double q, const int* __restrict__ bin_offsets,
                         const int* __restrict__ frame_index, int n_bins, int64_t plane) {
  const int64_t pix = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (pix >= plane) return;
  const D fill = DMax<D>::value();
  const W inf = (W)INFINITY;
  for (int g = 0; g < n_bins; ++g) {
    const int f0 = bin_offsets[g], len = bin_offsets[g + 1] - f0;
    W w[P];
    int n = 0;
#pragma unroll
    for (int i = 0; i < P; ++i) {
      w[i] = inf;
      if (i < len) {
        const S v = __ldcs(src + (int64_t)frame_index[f0 + i] * plane + pix);
        const bool ok = sample_counts<W>(v, nodata, has_nodata);
        w[i] = ok ? (W)v : inf;
        n += ok ? 1 : 0;
      }
    }
    // +inf never is a NaN, so fmin / fmax order the slots like the `a < b` exchange.
    // Batcher's odd-even merge sort: 543 exchanges at P = 64 (191 at 32) against the bitonic
    // network's 672 (240), as a flat generated list (gm_sort_networks.cuh) so that every slot is
    // a register name (nested loops with data-dependent bounds left the array in local memory).
#define GM_CE(I, J) { const W a_ = w[I], b_ = w[J]; w[I] = wmin<W>(a_, b_); w[J] = wmax<W>(a_, b_); }
    if constexpr (P == 64) { GM_SORT_NETWORK_64(GM_CE) }
    else if constexpr (P == 32) { GM_SORT_NETWORK_32(GM_CE) }
    else { static_assert(P == 16, "sorting networks exist for 16, 32 and 64 slots"); GM_SORT_NETWORK_16(GM_CE) }
#undef GM_CE
    D out = fill;
    if (n > 0) {
      const OrderRanks<W> r = order_ranks<W>(n, stat, q);
      W a = (W)0, b = (W)0;
#pragma unroll
      for (int i = 0; i < P; ++i) {
        a = i == r.lo ? w[i] : a;
        b = i == r.hi ? w[i] : b;
      }
      out = finite_or(order_value(a, b, r.t, n, stat), fill);
    }
    dst[(int64_t)g * plane + pix] = out;
  }
}

// Sum / count / min / max / mean, streaming.  With STAT a statistic, only the accumulators it
// needs exist; with STAT = GM_STAT_ANY (the VEC = 1 form) the kernel keeps the sum, count,
// minimum and maximum and picks the statistic `stat` at the end.  UNROLL = 4 frames in flight
// per thread (64 B at VEC = 16 / sizeof(S)).
template <typename S, typename W, typename D, int VEC, int STAT>
__global__ void __launch_bounds__(256)
temporal_stream_kernel(const S* __restrict__ src, D* __restrict__ dst, S nodata, int has_nodata,
                       int stat_arg, const int* __restrict__ bin_offsets, const int* __restrict__ frame_index,
                       int n_bins, int64_t plane) {
  constexpr bool ANY = STAT == GM_STAT_ANY;
  const int stat = ANY ? stat_arg : STAT;
  const int64_t grp = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (grp >= plane / VEC) return;
  const int64_t pix = grp * VEC;
  const D fill = (stat == GM_STAT_SUM || stat == GM_STAT_COUNT) ? (D)0 : DMax<D>::value();
  // Integer sources: minima / maxima are taken in the source dtype, and sums of sources of at
  // most 4 bytes that the reference accumulates in float64 are accumulated in int64 -- both
  // exact, hence identical to the sequential float arithmetic, without one int -> float
  // conversion per sample.  (Sums of int64 sources are rounded in float64 as the reference does.)
  constexpr bool INT_EXACT = std::is_integral<S>::value &&
      (STAT == GM_STAT_MIN || STAT == GM_STAT_MAX ||
       (STAT == GM_STAT_SUM && std::is_same<W, double>::value && sizeof(S) <= 4));
  // sources of at most 16 bits: the samples of a round add up in 32 bits, one 64-bit add per round
  constexpr bool SUM16 = INT_EXACT && STAT == GM_STAT_SUM && sizeof(S) <= 2;
  // sums in int64; extremes in int (sources below 4 bytes) or the source dtype itself
  typedef typename std::conditional<(sizeof(S) < 4), int, S>::type Extreme;
  typedef typename std::conditional<STAT == GM_STAT_SUM, long long, Extreme>::type IntAcc;
  typedef typename std::conditional<INT_EXACT, IntAcc, W>::type A;
  for (int g = 0; g < n_bins; ++g) {
    const int f0 = bin_offsets[g], f1 = bin_offsets[g + 1];
    A acc[VEC];         // the sum, or the extreme of an INT_EXACT minimum / maximum
    W lo[VEC], hi[VEC];  // the float minimum / maximum
    int cnt[VEC], part[VEC];
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      if constexpr (INT_EXACT)
        acc[i] = STAT == GM_STAT_MIN ? std::numeric_limits<A>::max()
                                     : STAT == GM_STAT_MAX ? std::numeric_limits<A>::lowest() : (A)0;
      else acc[i] = (W)0;
      lo[i] = hi[i] = nan_<W>();
      cnt[i] = part[i] = 0;
    }
    auto take = [&](const PixelVec<S, VEC>& x, int) {
#pragma unroll
      for (int i = 0; i < VEC; ++i) {
        const S v = x.v[i];
        const bool valid = sample_counts<W>(v, nodata, has_nodata);
        if constexpr (SUM16) {
          part[i] += valid ? (int)v : 0;
        } else if constexpr (INT_EXACT) {
          const A a = (A)v;
          if (STAT == GM_STAT_SUM) acc[i] += valid ? a : (A)0;
          if (STAT == GM_STAT_MIN) acc[i] = valid ? (a < acc[i] ? a : acc[i]) : acc[i];
          if (STAT == GM_STAT_MAX) acc[i] = valid ? (a > acc[i] ? a : acc[i]) : acc[i];
          if (STAT != GM_STAT_SUM) cnt[i] += valid ? 1 : 0;
        } else {
          const W w = (W)v;
          if (ANY || STAT == GM_STAT_SUM || STAT == GM_STAT_MEAN) acc[i] = valid ? acc[i] + w : acc[i];
          if (ANY || STAT == GM_STAT_MIN) lo[i] = (valid && (lo[i] != lo[i] || w < lo[i])) ? w : lo[i];
          if (ANY || STAT == GM_STAT_MAX) hi[i] = (valid && (hi[i] != hi[i] || w > hi[i])) ? w : hi[i];
          if (ANY || STAT == GM_STAT_COUNT || STAT == GM_STAT_MEAN) cnt[i] += valid ? 1 : 0;
        }
      }
    };
    walk_frames<VEC, 4>(src, frame_index, f0, f1, plane, pix, take, [&] {
      if constexpr (SUM16) {
#pragma unroll
        for (int i = 0; i < VEC; ++i) { acc[i] += part[i]; part[i] = 0; }
      }
    });
    D* o = dst + (int64_t)g * plane + pix;
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      W result;
      if (stat == GM_STAT_COUNT) result = (W)(int64_t)cnt[i];
      else if (stat == GM_STAT_MEAN) result = (W)((double)acc[i] / (double)(int64_t)cnt[i]);
      else if (INT_EXACT && STAT != GM_STAT_SUM) result = cnt[i] == 0 ? nan_<W>() : (W)acc[i];  // no valid sample
      else if (stat == GM_STAT_MIN) result = lo[i];
      else if (stat == GM_STAT_MAX) result = hi[i];
      else result = (W)acc[i];
      o[i] = finite_or(result, fill, f1 > f0);
    }
  }
}

// std / var, streaming: np.nanvar's two passes over t (mean, then the squared deviations from it)
// in the same order, four frames in flight per thread.
// Algorithmic bytes: 2 * T * itemsize in + itemsize out per pixel.
template <typename S, typename W, typename D, int VEC>
// (float64 at VEC = 1: without the minimum of one block, ptxas holds 32 registers and spills around
// the division / square-root calls; float32 fits 32 registers and keeps full occupancy)
__global__ void __launch_bounds__(256, (VEC == 1 && sizeof(W) == 8) ? 1 : 0)
temporal_moments_stream_kernel(const S* __restrict__ src, D* __restrict__ dst, S nodata, int has_nodata,
                               int stat, const int* __restrict__ bin_offsets,
                               const int* __restrict__ frame_index, int n_bins, int64_t plane) {
  const int64_t grp = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (grp >= plane / VEC) return;
  const int64_t pix = grp * VEC;
  const D fill = DMax<D>::value();
  for (int g = 0; g < n_bins; ++g) {
    const int f0 = bin_offsets[g], f1 = bin_offsets[g + 1];
    W acc[VEC], avg[VEC], ss[VEC];
    int cnt[VEC];
#pragma unroll
    for (int i = 0; i < VEC; ++i) { acc[i] = (W)0; ss[i] = (W)0; cnt[i] = 0; }
    for (int pass = 0; pass < 2; ++pass) {
      auto take = [&](const PixelVec<S, VEC>& x, int) {
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
          const S v = x.v[i];
          const W w = (W)v;
          const bool valid = sample_counts<W>(v, nodata, has_nodata);
          if (pass == 0) {
            acc[i] = valid ? acc[i] + w : acc[i];
            cnt[i] += valid ? 1 : 0;
          } else {
            const W d = w - avg[i];
            ss[i] = valid ? ss[i] + d * d : ss[i];
          }
        }
      };
      walk_frames<VEC, 4>(src, frame_index, f0, f1, plane, pix, take, [] {});
      if (pass == 0) {
#pragma unroll
        for (int i = 0; i < VEC; ++i) avg[i] = (W)((double)acc[i] / (double)(int64_t)cnt[i]);
      }
    }
    D* o = dst + (int64_t)g * plane + pix;
#pragma unroll
    for (int i = 0; i < VEC; ++i) o[i] = finite_or(var_or_std(ss[i], cnt[i], stat), fill, f1 > f0);
  }
}

// Cumulative sum / count, streaming: every frame is read once (eight frames in flight) and every
// running total is written once, with 16-byte streaming stores where VEC pixels of D make whole
// 16-byte groups.  Algorithmic bytes: T * (itemsize in + itemsize out) per pixel.
template <typename S, typename W, typename D, int VEC>
__global__ void __launch_bounds__(256)
temporal_cumulative_stream_kernel(const S* __restrict__ src, D* __restrict__ dst, S nodata, int has_nodata,
                                  int stat, const int* __restrict__ bin_offsets,
                                  const int* __restrict__ frame_index, const int* __restrict__ out_frame,
                                  int n_bins, int64_t plane) {
  const int64_t grp = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (grp >= plane / VEC) return;
  const int64_t pix = grp * VEC;
  for (int g = 0; g < n_bins; ++g) {
    W acc[VEC];
    int cnt[VEC];
#pragma unroll
    for (int i = 0; i < VEC; ++i) { acc[i] = (W)0; cnt[i] = 0; }
    auto step = [&](const PixelVec<S, VEC>& x, int f) {
      D outv[VEC];
#pragma unroll
      for (int i = 0; i < VEC; ++i) {
        const S v = x.v[i];
        const W w = (W)v;
        const bool valid = sample_counts<W>(v, nodata, has_nodata);
        acc[i] = valid ? acc[i] + w : acc[i];
        cnt[i] += valid ? 1 : 0;
        if (stat == GM_STAT_COUNT) outv[i] = (D)cnt[i];
        else outv[i] = finite_or(acc[i], (D)0);
      }
      const int o = out_frame[f];
      if (o >= 0) {
        D* at = dst + (int64_t)o * plane + pix;
        if constexpr ((VEC * sizeof(D)) % 16 == 0) {
          uint4 raw[VEC * sizeof(D) / 16];
          memcpy(raw, outv, sizeof(raw));
#pragma unroll
          for (int k = 0; k < (int)(VEC * sizeof(D) / 16); ++k) __stcs(reinterpret_cast<uint4*>(at) + k, raw[k]);
        } else {
#pragma unroll
          for (int i = 0; i < VEC; ++i) at[i] = outv[i];
        }
      }
    };
    walk_frames<VEC, 8>(src, frame_index, bin_offsets[g], bin_offsets[g + 1], plane, pix, step, [] {});
  }
}

struct TemporalArgs {
  const void* nodata; int has_nodata; int stat; double q;
  const int* bins; const int* frames; const int* out_frame; int n_bins; int64_t plane;
  int sort_slots = 0;     // power of two >= longest bin (median / percentile)
  int sort_threads = 0;   // threads per block of temporal_sort_kernel
};

// VEC = 16 / sizeof(S) needs every frame to be whole 16-byte pixel groups from a 16-byte aligned base.
template <typename S>
static bool whole_groups(int64_t plane, const void* base) {
  return plane % (16 / (int64_t)sizeof(S)) == 0 && (uintptr_t)base % 16 == 0;
}

template <typename S, typename W, typename D, int VEC>
static void launch_reduction(const S* src, D* dst, S nd, const TemporalArgs& a, cudaStream_t s) {
  const unsigned nb = (unsigned)((a.plane / VEC + 255) / 256);
#define GM_ARGS src, dst, nd, a.has_nodata, a.stat, a.bins, a.frames, a.n_bins, a.plane
  if (a.stat == GM_STAT_STD || a.stat == GM_STAT_VAR)
    temporal_moments_stream_kernel<S, W, D, VEC><<<nb, 256, 0, s>>>(GM_ARGS);
  else if constexpr (VEC == 1)
    temporal_stream_kernel<S, W, D, 1, GM_STAT_ANY><<<nb, 256, 0, s>>>(GM_ARGS);
  else switch (a.stat) {
    case GM_STAT_SUM: temporal_stream_kernel<S, W, D, VEC, GM_STAT_SUM><<<nb, 256, 0, s>>>(GM_ARGS); break;
    case GM_STAT_COUNT: temporal_stream_kernel<S, W, D, VEC, GM_STAT_COUNT><<<nb, 256, 0, s>>>(GM_ARGS); break;
    case GM_STAT_MIN: temporal_stream_kernel<S, W, D, VEC, GM_STAT_MIN><<<nb, 256, 0, s>>>(GM_ARGS); break;
    case GM_STAT_MAX: temporal_stream_kernel<S, W, D, VEC, GM_STAT_MAX><<<nb, 256, 0, s>>>(GM_ARGS); break;
    default: temporal_stream_kernel<S, W, D, VEC, GM_STAT_MEAN><<<nb, 256, 0, s>>>(GM_ARGS); break;
  }
#undef GM_ARGS
}

template <typename S, typename W, typename D>
static int launch_aggregate(const Staged& in, Staged& out, const TemporalArgs& a, cudaStream_t s) {
  S nd = S(0);
  if (a.has_nodata) memcpy(&nd, a.nodata, sizeof(S));
  const S* src = (const S*)in.dev;
  D* dst = (D*)out.dev;
  constexpr int VEC = 16 / (int)sizeof(S);
  if (a.stat != GM_STAT_MEDIAN && a.stat != GM_STAT_PERCENTILE) {
    if (whole_groups<S>(a.plane, src)) launch_reduction<S, W, D, VEC>(src, dst, nd, a, s);
    else launch_reduction<S, W, D, 1>(src, dst, nd, a, s);
    GM_LAUNCH_CHECK();
    return 0;
  }
  // register-resident network: float32 working dtype over the usual source dtypes (the fully
  // unrolled networks are expensive to compile, so only these are instantiated)
  if constexpr (std::is_same<W, float>::value && std::is_same<D, float>::value &&
                (std::is_same<S, float>::value || std::is_same<S, int16_t>::value ||
                 std::is_same<S, uint8_t>::value)) {
    if (a.sort_slots <= 64) {
      const unsigned nb = (unsigned)((a.plane + 127) / 128);
#define GM_SORT_REG(P)                                                                         \
      temporal_sort_reg_kernel<S, W, D, P><<<nb, 128, 0, s>>>(                                  \
          src, dst, nd, a.has_nodata, a.stat, a.q, a.bins, a.frames, a.n_bins, a.plane)
      if (a.sort_slots <= 32) GM_SORT_REG(32);
      else GM_SORT_REG(64);
#undef GM_SORT_REG
      GM_LAUNCH_CHECK();
      return 0;
    }
  }
  auto kernel = temporal_sort_kernel<S, W, D>;
  const size_t smem = (size_t)a.sort_slots * a.sort_threads * sizeof(W);
  if (smem > 48 * 1024)
    GM_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const unsigned nb = (unsigned)((a.plane + a.sort_threads - 1) / a.sort_threads);
  kernel<<<nb, a.sort_threads, smem, s>>>(src, dst, nd, a.has_nodata, a.stat, a.q, a.bins, a.frames,
                                          a.n_bins, a.plane);
  GM_LAUNCH_CHECK();
  return 0;
}

template <typename S, typename W, typename D>
static int launch_cumulative(const Staged& in, Staged& out, const TemporalArgs& a, cudaStream_t s) {
  S nd = S(0);
  if (a.has_nodata) memcpy(&nd, a.nodata, sizeof(S));
  const S* src = (const S*)in.dev;
  D* dst = (D*)out.dev;
  constexpr int VEC = 16 / (int)sizeof(S);
#define GM_CUMULATIVE(V)                                                                               \
  temporal_cumulative_stream_kernel<S, W, D, V><<<(unsigned)((a.plane / (V) + 255) / 256), 256, 0, s>>>( \
      src, dst, nd, a.has_nodata, a.stat, a.bins, a.frames, a.out_frame, a.n_bins, a.plane)
  if (whole_groups<S>(a.plane, src) && (uintptr_t)dst % 16 == 0) GM_CUMULATIVE(VEC);
  else GM_CUMULATIVE(1);
#undef GM_CUMULATIVE
  GM_LAUNCH_CHECK();
  return 0;
}

static bool work_is_double(int out_dtype) {
  // np.result_type(np.float32, out dtype)
  return out_dtype == GM_F64 || out_dtype == GM_I32 || out_dtype == GM_U32 || out_dtype == GM_I64;
}

template <typename S, bool CUMULATIVE>
static int dispatch_out(int out_dtype, const Staged& in, Staged& out, const TemporalArgs& a, cudaStream_t s) {
#define GM_GO(W, D) (CUMULATIVE ? launch_cumulative<S, W, D>(in, out, a, s) : launch_aggregate<S, W, D>(in, out, a, s))
  switch (out_dtype) {
    case GM_U8: case GM_BOOL: return GM_GO(float, uint8_t);
    case GM_I8: return GM_GO(float, int8_t);
    case GM_U16: return GM_GO(float, uint16_t);
    case GM_I16: return GM_GO(float, int16_t);
    case GM_F32: return GM_GO(float, float);
    case GM_U32: return GM_GO(double, uint32_t);
    case GM_I32: return GM_GO(double, int32_t);
    case GM_I64: return GM_GO(double, int64_t);
    case GM_F64: return GM_GO(double, double);
  }
#undef GM_GO
  return fail("temporal: unsupported output dtype");
}

template <bool CUMULATIVE>
static int dispatch_src(int src_dtype, int out_dtype, const Staged& in, Staged& out,
                        const TemporalArgs& a, cudaStream_t s) {
  switch (src_dtype) {
    case GM_U8: case GM_BOOL: return dispatch_out<uint8_t, CUMULATIVE>(out_dtype, in, out, a, s);
    case GM_I8: return dispatch_out<int8_t, CUMULATIVE>(out_dtype, in, out, a, s);
    case GM_U16: return dispatch_out<uint16_t, CUMULATIVE>(out_dtype, in, out, a, s);
    case GM_I16: return dispatch_out<int16_t, CUMULATIVE>(out_dtype, in, out, a, s);
    case GM_U32: return dispatch_out<uint32_t, CUMULATIVE>(out_dtype, in, out, a, s);
    case GM_I32: return dispatch_out<int32_t, CUMULATIVE>(out_dtype, in, out, a, s);
    case GM_I64: return dispatch_out<int64_t, CUMULATIVE>(out_dtype, in, out, a, s);
    case GM_F32: return dispatch_out<float, CUMULATIVE>(out_dtype, in, out, a, s);
    case GM_F64: return dispatch_out<double, CUMULATIVE>(out_dtype, in, out, a, s);
  }
  return fail("temporal: unsupported source dtype");
}

template <bool CUMULATIVE>
static int run_temporal(const GmArray* src, GmArray* dst, const void* nodata, int has_nodata,
                        int stat, double q, const int32_t* bin_offsets, const int32_t* frame_index,
                        const int32_t* out_frame, int n_bins, void* stream) {
  if (ensure_init()) return 1;
  if (!src || !dst || !bin_offsets || (n_bins > 0 && !frame_index)) return fail("temporal: null argument");
  if (src->shape[1] != dst->shape[1] || src->shape[2] != dst->shape[2])
    return fail("temporal: spatial shapes differ");
  if (stat < GM_STAT_SUM || stat > GM_STAT_PERCENTILE) return fail("temporal: unknown statistic");
  cudaStream_t s = resolve_stream(stream);
  const int n_frames = bin_offsets[n_bins];
  int longest = 0;
  for (int g = 0; g < n_bins; ++g) {
    const int len = bin_offsets[g + 1] - bin_offsets[g];
    if (len > longest) longest = len;
  }
  for (int i = 0; i < n_frames; ++i)
    if (frame_index[i] < 0 || frame_index[i] >= src->shape[0]) return fail("temporal: frame index out of range");
  if (!CUMULATIVE && dst->shape[0] != n_bins) return fail("temporal: one output frame per bin expected");
  const bool needs_sort = !CUMULATIVE && (stat == GM_STAT_MEDIAN || stat == GM_STAT_PERCENTILE);
  if (needs_sort && longest > TMP_MAX_SORT) return fail("temporal: more than 1024 frames per bin for median/percentile");

  TemporalArgs a;
  a.nodata = nodata; a.has_nodata = has_nodata; a.stat = stat; a.q = q; a.n_bins = n_bins;
  a.plane = src->shape[1] * src->shape[2];
  if (needs_sort) {
    // shared-memory sort: one column of `slots` working-dtype values per thread; whole warps
    // while 32 columns fit, else as many threads as fit (20 at 1024 float64 slots)
    const size_t w = work_is_double(dst->dtype) ? 8 : 4;
    int slots = 1;
    while (slots < longest) slots <<= 1;
    int threads = (int)(TMP_SORT_SMEM / ((size_t)slots * w));
    if (threads > 128) threads = 128;
    if (threads >= 32) threads = threads / 32 * 32;
    a.sort_slots = slots; a.sort_threads = threads;
  }
  Staged in, out;
  void *dbins = nullptr, *dframes = nullptr, *dout = nullptr;
  int rc = in.open_input(*src, s);
  if (!rc) rc = out.open_output(*dst, s);
  if (!rc) rc = upload(&dbins, bin_offsets, sizeof(int32_t) * (n_bins + 1), s);
  if (!rc) rc = upload(&dframes, frame_index, sizeof(int32_t) * (n_frames > 0 ? n_frames : 1), s);
  if (!rc && CUMULATIVE) rc = upload(&dout, out_frame, sizeof(int32_t) * (n_frames > 0 ? n_frames : 1), s);
  a.bins = (const int*)dbins; a.frames = (const int*)dframes; a.out_frame = (const int*)dout;
  if (!rc && a.plane > 0 && array_count(*dst) > 0) {
    if (CUMULATIVE) {
      // output frames that no bin writes keep the (extensive) fill 0; the others are written in
      // full by the kernel (clearing all T frames first cost as much as half the kernel)
      std::vector<char> written((size_t)dst->shape[0], 0);
      for (int i = 0; i < n_frames; ++i)
        if (out_frame[i] >= 0 && out_frame[i] < dst->shape[0]) written[out_frame[i]] = 1;
      const size_t frame_bytes = out.bytes / (size_t)dst->shape[0];
      for (int64_t f = 0; f < dst->shape[0] && !rc; ++f)
        if (!written[f] &&
            cudaMemsetAsync((char*)out.dev + (size_t)f * frame_bytes, 0, frame_bytes, s) != cudaSuccess)
          rc = fail("temporal: memset failed");
    }
    if (!rc) rc = dispatch_src<CUMULATIVE>(src->dtype, dst->dtype, in, out, a, s);
  }
  if (!rc) rc = out.finish_output();
  const bool sync = out.owned;
  in.release(); out.release();
  if (dbins) cudaFreeAsync(dbins, s);
  if (dframes) cudaFreeAsync(dframes, s);
  if (dout) cudaFreeAsync(dout, s);
  if (!rc && sync) GM_CUDA(cudaStreamSynchronize(s));
  return rc;
}

}  // namespace gm

using namespace gm;

extern "C" int gm_temporal_aggregate(const GmArray* src, GmArray* dst, const void* nodata,
                                     int has_nodata, int stat, double q, const int32_t* bin_offsets,
                                     const int32_t* frame_index, int n_bins, void* stream) {
  return run_temporal<false>(src, dst, nodata, has_nodata, stat, q, bin_offsets, frame_index,
                             nullptr, n_bins, stream);
}

extern "C" int gm_temporal_cumulative(const GmArray* src, GmArray* dst, const void* nodata,
                                      int has_nodata, int stat, const int32_t* bin_offsets,
                                      const int32_t* frame_index, const int32_t* out_frame,
                                      int n_bins, void* stream) {
  if (!out_frame) return fail("gm_temporal_cumulative: null out_frame");
  return run_temporal<true>(src, dst, nodata, has_nodata, stat, 0.0, bin_offsets, frame_index,
                            out_frame, n_bins, stream);
}
