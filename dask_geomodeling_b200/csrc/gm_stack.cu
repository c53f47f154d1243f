// Stacks of any length: reduce_rasters in one pass (gm_reduce_stack) and Place at any number of
// coordinates without per-coordinate copies (gm_place).
//
// Both fold every raster (copy) into a register accumulator with overlay() from gm_eval_ops.cuh,
// the step the evaluator's OVERLAY instruction executes, and finish with the evaluator's reduce
// epilogue, so that for stacks the evaluator can take the results are the same bytes.
//
//   - gm_reduce_stack: a thread owns PIX consecutive pixels.  The raster descriptors go to the
//     device in one copy; a block stages them through shared memory, so the dispatch on
//     (dtype, class, flags) is a broadcast read, uniform across the block.  The loads of BATCH
//     rasters are issued before any of them is folded.  A raster is read with vector loads when its
//     pointer allows (Group hands in frame views at any byte offset), with scalar loads otherwise.
//   - gm_place: the output is cut into TILE_H x TILE_W tiles.  The (tile, copy) pairs of every copy
//     footprint are listed on the device (count, scan, fill, radix sort by tile then copy), and one
//     block per tile and band walks its list in copy order, reading the small source through L1/L2.
//     Every output cell is written once.
//   - gm_reduce_stack_stat / gm_place_stat: mean, var, std, argmin and argmax over the same walks
//     (walk_stack, walk_tile), keeping a StatAcc per pixel instead of one accumulator; var and std
//     walk the stack a second time in the same launch.  For argmin / argmax gm_place_stat first
//     ranks the copies on the device (summed-area table of the source's has-data mask, one window
//     sum per copy, exclusive scan).
//
// Reference: raster/reduction.py:38-119, raster/spatial.py:657-731.
#include "gm_common.cuh"
#include <cuda_fp16.h>
#include <type_traits>
#include <cub/block/block_scan.cuh>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

// internal linkage: gm_eval.cu defines the same out-of-line helpers (none of them is used here)
#define GM_OUTLINE static __device__ __forceinline__
#include "gm_eval_ops.cuh"

namespace gm {
namespace {

constexpr int THREADS = 256;
constexpr int PIX = 4;    // consecutive pixels of one thread (gm_reduce_stack)
constexpr int BATCH = 4;  // rasters whose loads are in flight before the first of them is folded
constexpr int TILE_W = 64, TILE_H = 32;
constexpr int ROWS = TILE_H / (THREADS / TILE_W);  // output rows of one thread in a tile (gm_place)

// (natural class of the storage, test class) of a raster: the conversions has_data_test produces
enum TestPair { P_I32, P_I64, P_F32, P_F32_F64, P_F64, P_INVALID };

__host__ __device__ inline int test_pair(int dtype, int cls) {
  const int from = natural_class(dtype);
  if (from == cls) return from == GM_C_I32 ? P_I32 : from == GM_C_I64 ? P_I64 : from == GM_C_F32 ? P_F32 : P_F64;
  return from == GM_C_F32 && cls == GM_C_F64 ? P_F32_F64 : P_INVALID;
}

template <int P> struct Pair;
template <> struct Pair<P_I32> { typedef int32_t From; typedef int32_t T; };
template <> struct Pair<P_I64> { typedef int64_t From; typedef int64_t T; };
template <> struct Pair<P_F32> { typedef float From; typedef float T; };
template <> struct Pair<P_F32_F64> { typedef float From; typedef double T; };
template <> struct Pair<P_F64> { typedef double From; typedef double T; };

struct Desc {
  const unsigned char* data;
  uint64_t k2, k4;
  int32_t dtype;
  uint8_t pair, flags, isz, vec;
};

__device__ __forceinline__ Desc make_desc(const GmStackInput& g) {
  Desc d;
  d.data = reinterpret_cast<const unsigned char*>(g.data);
  d.k2 = g.k2;
  d.k4 = g.k4;
  d.dtype = g.dtype;
  d.pair = (uint8_t)test_pair(g.dtype, g.cls);
  d.flags = g.flags;
  d.isz = (uint8_t)dtype_size(g.dtype);
  const int need = d.isz * PIX < 16 ? d.isz * PIX : 16;
  d.vec = ((uintptr_t)g.data & (uintptr_t)(need - 1)) == 0;
  return d;
}

template <typename F> __device__ __forceinline__ void with_class(int cls, F&& f) {
  if (cls == GM_C_I32) f(int32_t(0));
  else if (cls == GM_C_F32) f(float(0));
  else if (cls == GM_C_I64) f(int64_t(0));
  else f(double(0));
}

// one stored element (raw bits, zero-extended) -> slot bits of the dtype's natural class, as the
// evaluator's read_loop makes them
__device__ __forceinline__ uint64_t natural_bits(int dtype, uint64_t raw) {
  switch (dtype) {
    case GM_I8: return (uint64_t)(uint32_t)(int32_t)(int8_t)raw;
    case GM_I16: return (uint64_t)(uint32_t)(int32_t)(int16_t)raw;
    default: return raw;
  }
}

__device__ __forceinline__ uint64_t load_one(const unsigned char* p, int isz) {
  switch (isz) {
    case 1: return *p;
    case 2: return *reinterpret_cast<const uint16_t*>(p);
    case 4: return *reinterpret_cast<const uint32_t*>(p);
    default: return *reinterpret_cast<const uint64_t*>(p);
  }
}

// PIX elements of an isz-byte dtype -> the layout of load_raw (constant indices only: w stays in
// registers)
__device__ __forceinline__ void pack(uint32_t (&w)[2 * PIX], const uint64_t (&v)[PIX], int isz) {
  switch (isz) {
    case 1:
      w[0] = (uint32_t)(v[0] & 0xff) | (uint32_t)(v[1] & 0xff) << 8 | (uint32_t)(v[2] & 0xff) << 16 |
             (uint32_t)(v[3] & 0xff) << 24;
      break;
    case 2:
      w[0] = (uint32_t)(v[0] & 0xffff) | (uint32_t)(v[1] & 0xffff) << 16;
      w[1] = (uint32_t)(v[2] & 0xffff) | (uint32_t)(v[3] & 0xffff) << 16;
      break;
    case 4:
#pragma unroll
      for (int i = 0; i < PIX; ++i) w[i] = (uint32_t)v[i];
      break;
    default:
#pragma unroll
      for (int i = 0; i < PIX; ++i) { w[2 * i] = (uint32_t)v[i]; w[2 * i + 1] = (uint32_t)(v[i] >> 32); }
      break;
  }
}

// raw words of pixels [base, base + PIX) of one raster: element p of an isz-byte dtype sits at
// byte p * isz of w
__device__ __forceinline__ void load_raw(const Desc& d, int64_t base, int64_t n, uint32_t (&w)[2 * PIX]) {
  static_assert(PIX == 4, "the vector paths below load 4 pixels");
  const unsigned char* p = d.data + base * d.isz;
  if (d.vec && base + PIX <= n) {
    if (d.isz == 1) {
      w[0] = __ldcs(reinterpret_cast<const unsigned int*>(p));
    } else if (d.isz == 2) {
      const uint2 v = __ldcs(reinterpret_cast<const uint2*>(p));
      w[0] = v.x; w[1] = v.y;
    } else {
      const uint4 v = __ldcs(reinterpret_cast<const uint4*>(p));
      w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
      if (d.isz == 8) {
        const uint4 u = __ldcs(reinterpret_cast<const uint4*>(p) + 1);
        w[4] = u.x; w[5] = u.y; w[6] = u.z; w[7] = u.w;
      }
    }
  } else {
    uint64_t v[PIX];
#pragma unroll
    for (int i = 0; i < PIX; ++i) v[i] = base + i < n ? load_one(p + i * d.isz, d.isz) : 0;
    pack(w, v, d.isz);
  }
}

__device__ __forceinline__ uint64_t element(const uint32_t (&w)[2 * PIX], int isz, int i) {
  switch (isz) {
    case 1: return (w[i >> 2] >> ((i & 3) * 8)) & 0xffu;
    case 2: return (w[i >> 1] >> ((i & 1) * 16)) & 0xffffu;
    case 4: return w[i];
    default: return (uint64_t)w[2 * i] | ((uint64_t)w[2 * i + 1] << 32);
  }
}

// acc[i] = overlay(acc[i], x[i]): x holds slot bits of class From (the natural class of the
// storage), tested and reduced in class T (the OVERLAY step the evaluator runs for this raster)
template <typename From, typename T, typename A, int KIND, int Q>
__device__ __forceinline__ void fold_typed(uint64_t (&acc)[Q], const uint64_t (&x)[Q], const Desc& d) {
  const bool has = d.flags & GM_F_ND_T, cl = d.flags & GM_F_CLOSE, fin = d.flags & GM_F_ND_FINITE;
#pragma unroll
  for (int i = 0; i < Q; ++i)
    acc[i] = overlay<T, A>(acc[i], cvt<From, T>(x[i], false, 0), has, cl, fin, KIND, d.k2, d.k4);
}

// f(From(), T()) with the class pair of a raster (TestPair; block-uniform)
template <typename F> __device__ __forceinline__ void with_pair(int pair, F&& f) {
  switch (pair) {
    case P_I32: f(int32_t(0), int32_t(0)); break;
    case P_I64: f(int64_t(0), int64_t(0)); break;
    case P_F32: f(float(0), float(0)); break;
    case P_F32_F64: f(float(0), double(0)); break;
    default: f(double(0), double(0)); break;
  }
}

// fold_typed with the class pair chosen per raster
template <typename A, int KIND, int Q>
__device__ __forceinline__ void fold(uint64_t (&acc)[Q], const uint64_t (&x)[Q], const Desc& d) {
  with_pair(d.pair, [&](auto from, auto t) { fold_typed<decltype(from), decltype(t), A, KIND>(acc, x, d); });
}

// the has-data test of an OVERLAY step on slot bits y of class T: Mask's (1 = data, 0 = no data)
template <typename T> __device__ __forceinline__ bool has_data(uint64_t y, const Desc& d) {
  const bool has = d.flags & GM_F_ND_T, cl = d.flags & GM_F_CLOSE, fin = d.flags & GM_F_ND_FINITE;
  return mask<T, T>(y, has, cl, fin, 1, d.k2, 0, d.k4) != 0;
}

// ---- the statistics of GmStackStat ---------------------------------------------------------------
template <int WB> struct Work { typedef float V; };  // a float16 W is held in a float (exact)
template <> struct Work<8> { typedef double V; };

// a value of class T in the working dtype W, as NumPy's astype rounds it.  An integer goes to
// float16 through float: exact below 2^24, and beyond half's range above it.
template <int WB, typename T> __device__ __forceinline__ typename Work<WB>::V to_work(T y) {
  if constexpr (WB == 8) return (double)y;
  else if constexpr (WB == 4) return (float)y;
  else if constexpr (std::is_same<T, double>::value) return __half2float(__double2half(y));
  else return __half2float(__float2half_rn((float)y));
}

// one slot of the stacked array: x = slot bits of class From (the natural class of the storage),
// tested in class T; v = the value in W.  False for a NaN slot (no data, or a NaN value).
template <typename From, typename T, int WB>
__device__ __forceinline__ bool stacked(uint64_t x, const Desc& d, typename Work<WB>::V& v) {
  const T y = Raw<T>::get(cvt<From, T>(x, false, 0));
  v = to_work<WB>(y);
  return has_data<T>(Raw<T>::put(y), d) && v == v;
}

// Per-pixel state of a statistic.  mean / var / std: v = the sum of the data slots in stack order
// (pass 1), then that of their squared deviations (pass 2), m = the mean between the passes,
// n = data slots.  argmin / argmax: v = the extreme so far, n = the first index reaching it, -1 while
// no slot had data; a NaN slot counts as +inf / -inf, so an extreme of -inf under argmax (+inf under
// argmin) is first reached at index 0.
template <int STAT, int WB> struct StatAcc {
  typedef typename Work<WB>::V V;
  static constexpr bool ARG = STAT == GM_STACK_ARGMIN || STAT == GM_STACK_ARGMAX;
  static constexpr bool TWO_PASS = STAT == GM_STACK_VAR || STAT == GM_STACK_STD;
  V v, m;
  int32_t n;

  __device__ __forceinline__ StatAcc()
      : v(STAT == GM_STACK_ARGMIN ? V(INFINITY) : STAT == GM_STACK_ARGMAX ? V(-INFINITY) : V(0)),
        m(0), n(ARG ? -1 : 0) {}
  // pass 1: data slot k holds x
  __device__ __forceinline__ void add(V x, int32_t k) {
    if constexpr (ARG) {
      const bool better = STAT == GM_STACK_ARGMAX ? x > v : x < v;
      n = better ? k : (n < 0 ? 0 : n);
      v = better ? x : v;
    } else {
      v = v + x;
      ++n;
    }
  }
  // np.nan* divide by the count in float64 (np.divide(W, intp)), then round to W
  __device__ __forceinline__ V per_slot(V s) const { return V((double)s / (double)n); }
  __device__ __forceinline__ void start_pass2() { m = per_slot(v); v = V(0); }
  __device__ __forceinline__ void add2(V x) {
    const V d = x - m;
    v = v + d * d;
  }
  // raw bits of the result in the output dtype (class out_cls); `fill` where no slot had data
  __device__ __forceinline__ uint64_t result(int out_dtype, uint64_t fill) const {
    if (n <= (ARG ? -1 : 0)) return fill;
    if constexpr (ARG) {
      if (out_dtype == GM_BOOL) return n != 0;
      uint64_t r = 0;
      with_class(natural_class(out_dtype), [&](auto ot) { r = cvt<int64_t, decltype(ot)>((uint64_t)(int64_t)n, false, 0); });
      return r;
    } else if constexpr (STAT != GM_STACK_STD) {
      return Raw<V>::put(per_slot(v));  // mean, var
    } else {
      return Raw<V>::put(sqrt(per_slot(v)));
    }
  }
};

// the evaluator's reduce epilogue, then the store in the output dtype
template <typename A, int KIND>
__device__ __forceinline__ uint64_t finish(uint64_t acc, int out_cls, uint64_t fill) {
  if constexpr (KIND == GM_RED_REPLACE || KIND == GM_RED_COUNT) {
    return acc;
  } else {
    const A v = Raw<A>::get(acc);
    uint64_t r = fill;
    with_class(out_cls, [&](auto ot) {
      typedef decltype(ot) To;
      r = v != v ? fill : cvt<A, To>(acc, false, 0);
    });
    return r;
  }
}

__device__ __forceinline__ void store_one(unsigned char* p, int isz, uint64_t v) {
  switch (isz) {
    case 1: *p = (uint8_t)v; break;
    case 2: *reinterpret_cast<uint16_t*>(p) = (uint16_t)v; break;
    case 4: *reinterpret_cast<uint32_t*>(p) = (uint32_t)v; break;
    default: *reinterpret_cast<uint64_t*>(p) = v; break;
  }
}

// f(d, k, x) for the rasters k = 0 .. n_inputs - 1 of the stack in order: d = the descriptor of
// raster k, x = slot bits of its natural class at pixels [base, base + PIX).  The descriptors pass
// through `desc` THREADS at a time; every thread of the block takes part in that, also one past n.
template <typename F>
__device__ __forceinline__ void walk_stack(const GmStackInput* __restrict__ inputs, int64_t n_inputs,
                                           Desc (&desc)[THREADS], int64_t base, int64_t n, F&& f) {
  for (int64_t c0 = 0; c0 < n_inputs; c0 += THREADS) {
    const int m = (int)(n_inputs - c0 < THREADS ? n_inputs - c0 : THREADS);
    __syncthreads();
    if (threadIdx.x < m) desc[threadIdx.x] = make_desc(inputs[c0 + threadIdx.x]);
    __syncthreads();
    if (base >= n) continue;
#pragma unroll 1
    for (int r = 0; r < m; r += BATCH) {
      uint32_t w[BATCH][2 * PIX];
#pragma unroll
      for (int u = 0; u < BATCH; ++u)
        if (r + u < m) load_raw(desc[r + u], base, n, w[u]);
#pragma unroll
      for (int u = 0; u < BATCH; ++u) {
        if (r + u < m) {
          const Desc& d = desc[r + u];
          uint64_t x[PIX];
#pragma unroll
          for (int i = 0; i < PIX; ++i) x[i] = natural_bits(d.dtype, element(w[u], d.isz, i));
          f(d, c0 + r + u, x);
        }
      }
    }
  }
}

// v (slot bits) -> pixels [base, base + PIX) of the output, vector stores where aligned
__device__ __forceinline__ void store_pixels(unsigned char* __restrict__ out, int out_dtype, int64_t base, int64_t n,
                                             const uint64_t (&v)[PIX]) {
  const int osz = dtype_size(out_dtype);
  uint32_t w[2 * PIX];
  pack(w, v, osz);
  unsigned char* p = out + base * osz;
  const int need = osz * PIX < 16 ? osz * PIX : 16;
  if (((uintptr_t)p & (uintptr_t)(need - 1)) == 0 && base + PIX <= n) {
    if (osz == 1) *reinterpret_cast<unsigned int*>(p) = w[0];
    else if (osz == 2) *reinterpret_cast<uint2*>(p) = make_uint2(w[0], w[1]);
    else {
      reinterpret_cast<uint4*>(p)[0] = make_uint4(w[0], w[1], w[2], w[3]);
      if (osz == 8) reinterpret_cast<uint4*>(p)[1] = make_uint4(w[4], w[5], w[6], w[7]);
    }
  } else {
    for (int i = 0; i < PIX && base + i < n; ++i) store_one(p + i * osz, osz, v[i]);
  }
}

template <typename A, int KIND>
__global__ void __launch_bounds__(THREADS, 3)
reduce_stack_kernel(const GmStackInput* __restrict__ inputs, int64_t n_inputs, uint64_t init, uint64_t fill,
                    unsigned char* __restrict__ out, int out_dtype, int64_t n) {
  __shared__ Desc desc[THREADS];
  const int64_t base = ((int64_t)blockIdx.x * THREADS + threadIdx.x) * PIX;
  uint64_t acc[PIX];
#pragma unroll
  for (int i = 0; i < PIX; ++i) acc[i] = init;
  walk_stack(inputs, n_inputs, desc, base, n,
             [&](const Desc& d, int64_t, const uint64_t (&x)[PIX]) { fold<A, KIND>(acc, x, d); });
  if (base >= n) return;
  const int out_cls = natural_class(out_dtype);
  uint64_t v[PIX];
#pragma unroll
  for (int i = 0; i < PIX; ++i) v[i] = finish<A, KIND>(acc[i], out_cls, fill);
  store_pixels(out, out_dtype, base, n, v);
}

// GmStackStat `STAT` in working dtype W (WB bytes); var and std walk the stack twice
template <int STAT, int WB>
__global__ void __launch_bounds__(THREADS, 3)
stack_stat_kernel(const GmStackInput* __restrict__ inputs, int64_t n_inputs, uint64_t fill,
                  unsigned char* __restrict__ out, int out_dtype, int64_t n) {
  typedef StatAcc<STAT, WB> Acc;
  typedef typename Acc::V V;
  __shared__ Desc desc[THREADS];
  const int64_t base = ((int64_t)blockIdx.x * THREADS + threadIdx.x) * PIX;
  Acc acc[PIX];
  walk_stack(inputs, n_inputs, desc, base, n, [&](const Desc& d, int64_t k, const uint64_t (&x)[PIX]) {
    with_pair(d.pair, [&](auto from, auto t) {
#pragma unroll
      for (int i = 0; i < PIX; ++i) {
        V v;
        if (stacked<decltype(from), decltype(t), WB>(x[i], d, v)) acc[i].add(v, (int32_t)k);
      }
    });
  });
  if constexpr (Acc::TWO_PASS) {
#pragma unroll
    for (int i = 0; i < PIX; ++i) acc[i].start_pass2();
    walk_stack(inputs, n_inputs, desc, base, n, [&](const Desc& d, int64_t, const uint64_t (&x)[PIX]) {
      with_pair(d.pair, [&](auto from, auto t) {
#pragma unroll
        for (int i = 0; i < PIX; ++i) {
          V v;
          if (stacked<decltype(from), decltype(t), WB>(x[i], d, v)) acc[i].add2(v);
        }
      });
    });
  }
  if (base >= n) return;
  uint64_t v[PIX];
#pragma unroll
  for (int i = 0; i < PIX; ++i) v[i] = acc[i].result(out_dtype, fill);
  store_pixels(out, out_dtype, base, n, v);
}

// ---- Place: tile lists ----------------------------------------------------------------------
struct TileRange { int64_t r0, r1, c0, c1; };  // tile rows / columns a copy meets (inclusive)

__host__ __device__ inline TileRange tiles_met(int2 o, int sh, int sw, int dh, int dw) {
  const int64_t j0 = o.y > 0 ? o.y : 0, j1 = ((int64_t)o.y + sh < dh ? (int64_t)o.y + sh : dh) - 1;
  const int64_t i0 = o.x > 0 ? o.x : 0, i1 = ((int64_t)o.x + sw < dw ? (int64_t)o.x + sw : dw) - 1;
  TileRange t{0, -1, 0, -1};
  if (j0 <= j1 && i0 <= i1) t = TileRange{j0 / TILE_H, j1 / TILE_H, i0 / TILE_W, i1 / TILE_W};
  return t;
}

// counts[c] = tiles met by copy c.  *walk_all = 1 when a copy changes cells outside its footprint,
// where it holds the fill value `pad`: under last / first / count when the pad tests as data (a NaN
// or None no data value), under max / min / sum / product when it is a value rather than NaN (a
// NaN operand leaves those accumulators as they are).  Then every tile visits every copy.
__global__ void place_count_kernel(const int2* __restrict__ off, int64_t n, int sh, int sw, int dh, int dw,
                                   int64_t* __restrict__ counts, GmStackInput test, uint64_t pad, int kind,
                                   int acc_cls, int* __restrict__ walk_all) {
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c == 0 && walk_all) {
    const Desc d = make_desc(test);
    const uint64_t x[1] = {natural_bits(test.dtype, pad)};
    if (kind == GM_RED_REPLACE || kind == GM_RED_COUNT) {
      uint64_t acc[1] = {0};
      fold<int32_t, GM_RED_COUNT>(acc, x, d);
      *walk_all = acc[0] != 0;
    } else if (acc_cls == GM_C_F32) {
      uint64_t acc[1] = {Raw<float>::put(quiet_nan<float>())};
      fold<float, GM_RED_MAX>(acc, x, d);
      *walk_all = Raw<float>::get(acc[0]) == Raw<float>::get(acc[0]);
    } else {
      uint64_t acc[1] = {Raw<double>::put(quiet_nan<double>())};
      fold<double, GM_RED_MAX>(acc, x, d);
      *walk_all = Raw<double>::get(acc[0]) == Raw<double>::get(acc[0]);
    }
  }
  if (c >= n) return;
  const TileRange t = tiles_met(off[c], sh, sw, dh, dw);
  counts[c] = (t.r1 - t.r0 + 1) * (t.c1 - t.c0 + 1);
}

// keys of copy blockIdx.x: tile << 32 | copy, at [incl[c] - counts[c], incl[c])
__global__ void place_fill_kernel(const int2* __restrict__ off, int sh, int sw, int dh, int dw, int tiles_x,
                                  const int64_t* __restrict__ counts, const int64_t* __restrict__ incl,
                                  uint64_t* __restrict__ keys) {
  const int c = blockIdx.x;
  const TileRange t = tiles_met(off[c], sh, sw, dh, dw);
  const int cols = (int)(t.c1 - t.c0 + 1), count = (int)counts[c];
  const int64_t start = incl[c] - count;
  for (int k = threadIdx.x; k < count; k += blockDim.x) {
    const int tile = ((int)t.r0 + k / cols) * tiles_x + (int)t.c0 + k % cols;
    keys[start + k] = (uint64_t)tile << 32 | (uint32_t)c;
  }
}

// first[t] = first sorted entry of tile t (t = 0 .. tiles)
__global__ void place_bounds_kernel(const uint64_t* __restrict__ keys, int64_t total, int tiles,
                                    int64_t* __restrict__ first) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t > tiles) return;
  const uint64_t key = (uint64_t)t << 32;
  int64_t lo = 0, hi = total;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (keys[mid] < key) lo = mid + 1; else hi = mid;
  }
  first[t] = lo;
}

constexpr int JSTEP = THREADS / TILE_W;  // rows between the cells of one thread in a tile

// f(o, c) for the entries [begin, end) of a tile's list in order: o = offset of copy c (with `all`,
// entry e is copy e).  The offsets pass through shared memory THREADS at a time.
template <typename F>
__device__ __forceinline__ void walk_tile(const int2* __restrict__ off, const uint64_t* __restrict__ keys,
                                          int begin, int end, bool all, F&& f) {
  __shared__ int2 list[THREADS];
  __shared__ int ids[THREADS];
  for (int e0 = begin; e0 < end; e0 += THREADS) {
    const int m = end - e0 < THREADS ? end - e0 : THREADS;
    __syncthreads();
    if (threadIdx.x < m) {
      const int e = e0 + threadIdx.x, c = all ? e : (int)(uint32_t)keys[e];
      list[threadIdx.x] = off[c];
      ids[threadIdx.x] = c;
    }
    __syncthreads();
#pragma unroll 1
    for (int q = 0; q < m; ++q) f(list[q], ids[q]);
  }
}

// the ROWS cells (column i, rows j0 + k * JSTEP) of copy o as slot bits of the natural class of the
// storage: `pad` outside the source and, gm_resample_nn's rule, at a non-finite float.  Bit k of
// the result is set when cell k lies inside the copy's footprint.
template <typename From>
__device__ __forceinline__ unsigned gather(const unsigned char* __restrict__ plane, const Desc& d, int2 o, int i,
                                           int j0, int sh, int sw, uint64_t pad, uint64_t (&x)[ROWS]) {
  const int si = i - o.x;
  unsigned inside = 0;
#pragma unroll
  for (int k = 0; k < ROWS; ++k) {
    const int sj = j0 + k * JSTEP - o.y;
    uint64_t v = pad;
    if ((unsigned)si < (unsigned)sw && (unsigned)sj < (unsigned)sh) {
      v = load_one(plane + ((int64_t)sj * sw + si) * d.isz, d.isz);
      inside |= 1u << k;
    }
    x[k] = v;
  }
#pragma unroll
  for (int k = 0; k < ROWS; ++k) {
    if constexpr (IsFloat<From>::value) x[k] = finite_(Raw<From>::get(x[k])) ? x[k] : pad;
    x[k] = natural_bits(d.dtype, x[k]);
  }
  return inside;
}

// one block per (tile, band): out = reduction over the tile's copies, in copy order, or over every
// copy when *walk_all (see place_count_kernel).  Source class pair P is fixed for the call.
template <typename A, int KIND, int P>
__global__ void __launch_bounds__(THREADS, 4)
place_kernel(const unsigned char* __restrict__ src, GmStackInput test, int sh, int sw, uint64_t pad,
             const int2* __restrict__ off, int64_t n, const uint64_t* __restrict__ keys,
             const int64_t* __restrict__ first, const int* __restrict__ walk_all, int tiles_x,
             uint64_t init, uint64_t fill,
             unsigned char* __restrict__ out, int out_dtype, int dh, int dw) {
  const Desc d = make_desc(test);
  const int tile = blockIdx.x, band = blockIdx.y;
  const int i = (tile % tiles_x) * TILE_W + (int)(threadIdx.x % TILE_W);
  const int j0 = (tile / tiles_x) * TILE_H + (int)(threadIdx.x / TILE_W);
  const unsigned char* plane = src + band * (int64_t)sh * sw * d.isz;
  typedef typename Pair<P>::From From;
  uint64_t acc[ROWS];
#pragma unroll
  for (int k = 0; k < ROWS; ++k) acc[k] = init;
  const bool all = *walk_all;
  const int begin = all ? 0 : (int)first[tile], end = all ? (int)n : (int)first[tile + 1];
  walk_tile(off, keys, begin, end, all, [&](int2 o, int) {
    uint64_t x[ROWS];
    gather<From>(plane, d, o, i, j0, sh, sw, pad, x);
    fold_typed<From, typename Pair<P>::T, A, KIND>(acc, x, d);
  });
  const int osz = dtype_size(out_dtype), out_cls = natural_class(out_dtype);
  unsigned char* dst = out + band * (int64_t)dh * dw * osz;
#pragma unroll
  for (int k = 0; k < ROWS; ++k) {
    const int j = j0 + k * JSTEP;
    if (i < dw && j < dh) store_one(dst + ((int64_t)j * dw + i) * osz, osz, finish<A, KIND>(acc[k], out_cls, fill));
  }
}

// ---- Place with a GmStackStat --------------------------------------------------------------------
// The reference stacks a copy only when it puts a data cell of some band inside the request, and a
// cell outside a copy's footprint is NaN in its stack: every tile walks just its own list, and a
// copy's argmin / argmax index is its rank among the stacked copies (place_rank_kernel).  "Data"
// is the has-data test alone there, as the reference decides (a non-finite value counts).

// sat[(j + 1) * (sw + 1) + i + 1] = data cells of source row j in columns <= i (any band); one
// block per row; sat[(j + 1) * (sw + 1)] = 0
__global__ void __launch_bounds__(THREADS)
place_sat_rows_kernel(const unsigned char* __restrict__ src, GmStackInput test, int bands, int sh, int sw,
                      uint32_t* __restrict__ sat) {
  typedef cub::BlockScan<uint32_t, THREADS> Scan;
  __shared__ typename Scan::TempStorage temp;
  const Desc d = make_desc(test);
  const int j = blockIdx.x;
  uint32_t* row = sat + (int64_t)(j + 1) * (sw + 1);
  if (threadIdx.x == 0) row[0] = 0;
  uint32_t carry = 0;
  for (int i0 = 0; i0 < sw; i0 += THREADS) {
    const int i = i0 + (int)threadIdx.x;
    uint32_t data = 0;
    if (i < sw) {
      for (int b = 0; b < bands && !data; ++b) {
        const uint64_t x = natural_bits(d.dtype, load_one(src + (((int64_t)b * sh + j) * sw + i) * d.isz, d.isz));
        with_pair(d.pair, [&](auto from, auto t) {
          data = has_data<decltype(t)>(cvt<decltype(from), decltype(t)>(x, false, 0), d);
        });
      }
    }
    uint32_t sum, total;
    Scan(temp).InclusiveSum(data, sum, total);
    if (i < sw) row[i + 1] = carry + sum;
    carry += total;
    __syncthreads();  // temp is reused
  }
}

// column sums of the row prefixes: sat becomes the summed-area table (row 0 zero)
__global__ void place_sat_cols_kernel(int sh, int sw, uint32_t* __restrict__ sat) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i > sw) return;
  uint32_t run = 0;
  sat[i] = 0;
  for (int j = 1; j <= sh; ++j) {
    uint32_t* p = sat + (int64_t)j * (sw + 1) + i;
    run += *p;
    *p = run;
  }
}

// stacked[c] = 1 when copy c puts a data cell inside the dh x dw request (a window sum of sat;
// uint32 wrap-around is exact for sh * sw < 2^32)
__global__ void place_stacked_kernel(const int2* __restrict__ off, int64_t n, int sh, int sw, int dh, int dw,
                                     const uint32_t* __restrict__ sat, int* __restrict__ stacked) {
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n) return;
  const int2 o = off[c];
  const int i0 = max(0, -o.x), i1 = (int)min((int64_t)sw, (int64_t)dw - o.x);
  const int j0 = max(0, -o.y), j1 = (int)min((int64_t)sh, (int64_t)dh - o.y);
  uint32_t cells = 0;
  if (i0 < i1 && j0 < j1) {
    const int64_t w = sw + 1;
    cells = sat[j1 * w + i1] - sat[j0 * w + i1] - sat[j1 * w + i0] + sat[j0 * w + i0];
  }
  stacked[c] = cells != 0;
}

// one block per (tile, band): out = statistic STAT over the tile's copies in working dtype W (WB
// bytes); argmin / argmax index copy c by rank[c] (null for the other statistics)
template <int STAT, int WB, int P>
__global__ void __launch_bounds__(THREADS, 2)
place_stat_kernel(const unsigned char* __restrict__ src, GmStackInput test, int sh, int sw, uint64_t pad,
                  const int2* __restrict__ off, const int* __restrict__ rank, const uint64_t* __restrict__ keys,
                  const int64_t* __restrict__ first, int tiles_x, uint64_t fill,
                  unsigned char* __restrict__ out, int out_dtype, int dh, int dw) {
  typedef StatAcc<STAT, WB> Acc;
  typedef typename Acc::V V;
  typedef typename Pair<P>::From From;
  typedef typename Pair<P>::T T;
  const Desc d = make_desc(test);
  const int tile = blockIdx.x, band = blockIdx.y;
  const int i = (tile % tiles_x) * TILE_W + (int)(threadIdx.x % TILE_W);
  const int j0 = (tile / tiles_x) * TILE_H + (int)(threadIdx.x / TILE_W);
  const unsigned char* plane = src + band * (int64_t)sh * sw * d.isz;
  const int begin = (int)first[tile], end = (int)first[tile + 1];
  Acc acc[ROWS];
  walk_tile(off, keys, begin, end, false, [&](int2 o, int c) {
    uint64_t x[ROWS];
    const unsigned inside = gather<From>(plane, d, o, i, j0, sh, sw, pad, x);
    const int32_t k = Acc::ARG ? rank[c] : 0;
#pragma unroll
    for (int r = 0; r < ROWS; ++r) {
      V v;
      if (((inside >> r) & 1u) && stacked<From, T, WB>(x[r], d, v)) acc[r].add(v, k);
    }
  });
  if constexpr (Acc::TWO_PASS) {
#pragma unroll
    for (int r = 0; r < ROWS; ++r) acc[r].start_pass2();
    walk_tile(off, keys, begin, end, false, [&](int2 o, int) {
      uint64_t x[ROWS];
      const unsigned inside = gather<From>(plane, d, o, i, j0, sh, sw, pad, x);
#pragma unroll
      for (int r = 0; r < ROWS; ++r) {
        V v;
        if (((inside >> r) & 1u) && stacked<From, T, WB>(x[r], d, v)) acc[r].add2(v);
      }
    });
  }
  const int osz = dtype_size(out_dtype);
  unsigned char* dst = out + band * (int64_t)dh * dw * osz;
#pragma unroll
  for (int r = 0; r < ROWS; ++r) {
    const int j = j0 + r * JSTEP;
    if (i < dw && j < dh) store_one(dst + ((int64_t)j * dw + i) * osz, osz, acc[r].result(out_dtype, fill));
  }
}

// ---- dispatch over (accumulator class, kind) -------------------------------------------------
template <template <typename, int> class K, typename F>
int with_kernel(int acc_cls, int kind, F&& f) {
  auto by_kind = [&](auto at) -> int {
    typedef decltype(at) A;
    switch (kind) {
      case GM_RED_REPLACE: return f(K<A, GM_RED_REPLACE>::get());
      case GM_RED_COUNT: return f(K<A, GM_RED_COUNT>::get());
      default: break;
    }
    if constexpr (IsFloat<A>::value) {
      switch (kind) {
        case GM_RED_MAX: return f(K<A, GM_RED_MAX>::get());
        case GM_RED_MIN: return f(K<A, GM_RED_MIN>::get());
        case GM_RED_SUM: return f(K<A, GM_RED_SUM>::get());
        case GM_RED_PRODUCT: return f(K<A, GM_RED_PRODUCT>::get());
        default: break;
      }
    }
    return fail("stack reduction: max / min / sum / product need a float accumulator, kind "
                + std::to_string(kind));
  };
  switch (acc_cls) {
    case GM_C_I32: return by_kind(int32_t(0));
    case GM_C_I64: return by_kind(int64_t(0));
    case GM_C_F32: return by_kind(float(0));
    case GM_C_F64: return by_kind(double(0));
  }
  return fail("stack reduction: bad accumulator class");
}

template <typename A, int KIND> struct StackKernel {
  static auto get() { return reduce_stack_kernel<A, KIND>; }
};
template <int P> struct PlaceKernel {
  template <typename A, int KIND> struct Of {
    static auto get() { return place_kernel<A, KIND, P>; }
  };
};

// ---- dispatch over (statistic, working dtype) ----------------------------------------------------
template <template <int, int> class K, typename F>
int with_stat(int stat, int work_bytes, F&& f) {
  auto by_stat = [&](auto wb) -> int {
    constexpr int WB = decltype(wb)::value;
    switch (stat) {
      case GM_STACK_ARGMIN: return f(K<GM_STACK_ARGMIN, WB>::get());
      case GM_STACK_ARGMAX: return f(K<GM_STACK_ARGMAX, WB>::get());
      default: break;
    }
    if constexpr (WB != 2) {
      switch (stat) {
        case GM_STACK_MEAN: return f(K<GM_STACK_MEAN, WB>::get());
        case GM_STACK_VAR: return f(K<GM_STACK_VAR, WB>::get());
        case GM_STACK_STD: return f(K<GM_STACK_STD, WB>::get());
        default: break;
      }
    }
    return fail("stack statistic: bad statistic " + std::to_string(stat) + " for a float" + std::to_string(8 * WB) +
                " working dtype");
  };
  switch (work_bytes) {
    case 2: return by_stat(std::integral_constant<int, 2>());
    case 4: return by_stat(std::integral_constant<int, 4>());
    case 8: return by_stat(std::integral_constant<int, 8>());
  }
  return fail("stack statistic: the working dtype is float16, float32 or float64 (2, 4 or 8 bytes)");
}

template <int STAT, int WB> struct StackStatKernel {
  static auto get() { return stack_stat_kernel<STAT, WB>; }
};
template <int P> struct PlaceStatKernel {
  template <int STAT, int WB> struct Of {
    static auto get() { return place_stat_kernel<STAT, WB, P>; }
  };
};

int check_input(const GmStackInput& g, const char* who) {
  if (!dtype_size(g.dtype)) return fail(std::string(who) + ": bad input dtype");
  if (g.cls > GM_C_F64 || test_pair(g.dtype, g.cls) == P_INVALID)
    return fail(std::string(who) + ": the test class does not fit the dtype");
  return 0;
}

// mean / var / std are stored in W itself
int check_stat(int stat, int work_bytes, int out_dtype, const char* who) {
  if (stat < GM_STACK_MEAN || stat > GM_STACK_ARGMAX) return fail(std::string(who) + ": bad statistic");
  if (stat <= GM_STACK_STD && !((work_bytes == 4 && out_dtype == GM_F32) || (work_bytes == 8 && out_dtype == GM_F64)))
    return fail(std::string(who) + ": mean / var / std are stored in their float32 or float64 working dtype");
  return 0;
}

// What gm_place and gm_place_stat share: the checks, the offsets on the device, the tile lists
// (keys `sorted` = tile << 32 | copy by tile, then copy; first[t] = first entry of tile t) and the
// scratch memory of the call, freed in stream order when the call ends.
struct PlaceCall {
  cudaStream_t s = nullptr;
  std::vector<void*> scratch;
  int64_t bands = 0, tiles = 0, tiles_x = 0;
  int sh = 0, sw = 0, dh = 0, dw = 0;
  uint64_t pad = 0;
  bool empty = false;  // nothing to write
  int2* off = nullptr;
  int* walk_all = nullptr;
  uint64_t* sorted = nullptr;
  int64_t* first = nullptr;

  ~PlaceCall() {
    for (void* p : scratch) cudaFreeAsync(p, s);
  }
  int alloc(void** p, size_t bytes) {
    GM_CUDA(cudaMallocAsync(p, bytes > 0 ? bytes : 16, s));
    scratch.push_back(*p);
    return 0;
  }

  int open(const char* who, const GmArray* src, const GmArray* dst, const void* nodata, const int32_t* offsets,
           int64_t n_copies, const GmStackInput* test, void* stream) {
    const std::string w(who);
    if (ensure_init()) return 1;
    if (!src || !dst || !nodata || !test || (n_copies > 0 && !offsets)) return fail(w + ": null argument");
    if (src->space != GM_DEVICE || dst->space != GM_DEVICE) return fail(w + ": operands must be device resident");
    if (src->shape[0] != dst->shape[0]) return fail(w + ": band count mismatch");
    if (test->dtype != src->dtype) return fail(w + ": the test must be that of the source dtype");
    if (check_input(*test, who) || !dtype_size(dst->dtype)) return 1;
    if (n_copies < 0) return fail(w + ": negative copy count");
    bands = src->shape[0];
    sh = (int)src->shape[1], sw = (int)src->shape[2], dh = (int)dst->shape[1], dw = (int)dst->shape[2];
    empty = bands == 0 || dh == 0 || dw == 0;
    if (empty) return 0;
    if (bands > 65535) return fail(w + ": too many bands");
    s = resolve_stream(stream);
    memcpy(&pad, nodata, dtype_size(src->dtype));
    tiles_x = (dw + TILE_W - 1) / TILE_W;
    tiles = tiles_x * ((dh + TILE_H - 1) / TILE_H);
    if (tiles >= ((int64_t)1 << 31) || n_copies >= ((int64_t)1 << 31)) return fail(w + ": too many tiles or copies");
    void* dev = nullptr;
    if (upload(&dev, offsets, n_copies * 8, s)) return 1;
    scratch.push_back(dev);
    off = (int2*)dev;
    return 0;
  }

  // the tile lists, their length from the offsets on the host, so that nothing waits for the device;
  // with `kind` >= 0 also *walk_all (place_count_kernel)
  int list(const char* who, const int32_t* offsets, int64_t n_copies, const GmStackInput* test, int kind,
           int acc_cls) {
    const std::string w(who);
    int64_t total = 0;
    for (int64_t c = 0; c < n_copies; ++c) {
      const TileRange t = tiles_met(make_int2(offsets[2 * c], offsets[2 * c + 1]), sh, sw, dh, dw);
      total += (t.r1 - t.r0 + 1) * (t.c1 - t.c0 + 1);
    }
    if (total >= ((int64_t)1 << 31)) return fail(w + ": too many (tile, copy) pairs");
    int64_t* counts = nullptr; int64_t* incl = nullptr; uint64_t* keys = nullptr;
    if (alloc((void**)&counts, n_copies * 8) || alloc((void**)&incl, n_copies * 8) ||
        (kind >= 0 && alloc((void**)&walk_all, 4)) || alloc((void**)&keys, total * 8) ||
        alloc((void**)&sorted, total * 8) || alloc((void**)&first, (tiles + 1) * 8))
      return 1;
    place_count_kernel<<<(unsigned)(n_copies > 0 ? (n_copies + THREADS - 1) / THREADS : 1), THREADS, 0, s>>>(
        off, n_copies, sh, sw, dh, dw, counts, *test, pad, kind, acc_cls, walk_all);
    if (cudaGetLastError() != cudaSuccess) return fail(w + ": count launch failed");
    count_launch();
    if (total > 0) {
      size_t scan_bytes = 0, sort_bytes = 0;
      int end_bit = 33;  // keys are tile << 32 | copy
      while (((int64_t)1 << (end_bit - 32)) <= tiles) ++end_bit;
      cub::DeviceScan::InclusiveSum(nullptr, scan_bytes, counts, incl, n_copies, s);
      cub::DeviceRadixSort::SortKeys(nullptr, sort_bytes, keys, sorted, total, 0, end_bit, s);
      void* temp = nullptr;
      if (alloc(&temp, scan_bytes > sort_bytes ? scan_bytes : sort_bytes)) return 1;
      if (cub::DeviceScan::InclusiveSum(temp, scan_bytes, counts, incl, n_copies, s) != cudaSuccess)
        return fail(w + ": scan failed");
      count_launch();
      place_fill_kernel<<<(unsigned)n_copies, THREADS, 0, s>>>(off, sh, sw, dh, dw, (int)tiles_x, counts, incl, keys);
      if (cudaGetLastError() != cudaSuccess) return fail(w + ": fill launch failed");
      count_launch();
      if (cub::DeviceRadixSort::SortKeys(temp, sort_bytes, keys, sorted, total, 0, end_bit, s) != cudaSuccess)
        return fail(w + ": sort failed");
      count_launch();
    }
    place_bounds_kernel<<<(unsigned)((tiles + 1 + THREADS - 1) / THREADS), THREADS, 0, s>>>(sorted, total, (int)tiles,
                                                                                           first);
    if (cudaGetLastError() != cudaSuccess) return fail(w + ": bounds launch failed");
    count_launch();
    return 0;
  }

  // rank[c] = copies before c that put a data cell inside the request (gm_place_stat's argmin / argmax)
  int rank_copies(const GmArray* src, const GmStackInput* test, int64_t n_copies, int** rank) {
    uint32_t* sat = nullptr; int* stacked = nullptr;
    if ((int64_t)sh * sw >= ((int64_t)1 << 32)) return fail("gm_place_stat: source too large to rank copies");
    if (alloc((void**)rank, n_copies * 4) || alloc((void**)&stacked, n_copies * 4) ||
        alloc((void**)&sat, ((int64_t)sh + 1) * (sw + 1) * 4))
      return 1;
    if (n_copies == 0) return 0;
    if (sh > 0 && sw > 0) {
      place_sat_rows_kernel<<<(unsigned)sh, THREADS, 0, s>>>((const unsigned char*)src->data, *test, (int)bands, sh, sw,
                                                            sat);
      GM_LAUNCH_CHECK();
    }
    place_sat_cols_kernel<<<(unsigned)((sw + THREADS) / THREADS), THREADS, 0, s>>>(sh, sw, sat);
    GM_LAUNCH_CHECK();
    place_stacked_kernel<<<(unsigned)((n_copies + THREADS - 1) / THREADS), THREADS, 0, s>>>(off, n_copies, sh, sw, dh,
                                                                                           dw, sat, stacked);
    GM_LAUNCH_CHECK();
    size_t scan_bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, stacked, *rank, n_copies, s);
    void* temp = nullptr;
    if (alloc(&temp, scan_bytes)) return 1;
    if (cub::DeviceScan::ExclusiveSum(temp, scan_bytes, stacked, *rank, n_copies, s) != cudaSuccess)
      return fail("gm_place_stat: rank scan failed");
    count_launch();
    return 0;
  }
};

// f(std::integral_constant<int, P>) with the class pair P of the source (TestPair)
template <typename F>
int with_place_pair(const GmStackInput& test, F&& f) {
  switch (test_pair(test.dtype, test.cls)) {
    case P_I32: return f(std::integral_constant<int, P_I32>());
    case P_I64: return f(std::integral_constant<int, P_I64>());
    case P_F32: return f(std::integral_constant<int, P_F32>());
    case P_F32_F64: return f(std::integral_constant<int, P_F32_F64>());
    default: return f(std::integral_constant<int, P_F64>());
  }
}

}  // namespace
}  // namespace gm

using namespace gm;

extern "C" int gm_reduce_stack(const GmStackInput* inputs, int64_t n_inputs, int kind, int acc_cls,
                               uint64_t init, uint64_t fill, GmArray* out, void* stream) {
  if (ensure_init()) return 1;
  if (!out || (n_inputs > 0 && !inputs)) return fail("gm_reduce_stack: null argument");
  if (n_inputs < 1) return fail("gm_reduce_stack: empty stack");
  if (out->space != GM_DEVICE) return fail("gm_reduce_stack: the output must be device resident");
  if (!dtype_size(out->dtype)) return fail("gm_reduce_stack: bad output dtype");
  for (int64_t k = 0; k < n_inputs; ++k) {
    if (check_input(inputs[k], "gm_reduce_stack")) return 1;
    if (!inputs[k].data) return fail("gm_reduce_stack: null input");
  }
  const int64_t n = array_count(*out);
  if (n == 0) return 0;
  cudaStream_t s = resolve_stream(stream);
  void* dev = nullptr;
  if (upload(&dev, inputs, n_inputs * (int64_t)sizeof(GmStackInput), s)) return 1;
  const int64_t blocks = (n + (int64_t)THREADS * PIX - 1) / ((int64_t)THREADS * PIX);
  const int rc = with_kernel<StackKernel>(acc_cls, kind, [&](auto kernel) -> int {
    kernel<<<(unsigned)blocks, THREADS, 0, s>>>((const GmStackInput*)dev, n_inputs, init, fill,
                                                (unsigned char*)out->data, out->dtype, n);
    GM_LAUNCH_CHECK();
    return 0;
  });
  cudaFreeAsync(dev, s);
  return rc;
}

extern "C" int gm_place(const GmArray* src, GmArray* dst, const void* nodata, const int32_t* offsets,
                        int64_t n_copies, const GmStackInput* test, int kind, int acc_cls, uint64_t init,
                        uint64_t fill, void* stream) {
  PlaceCall call;
  if (call.open("gm_place", src, dst, nodata, offsets, n_copies, test, stream)) return 1;
  if (call.empty) return 0;
  if (call.list("gm_place", offsets, n_copies, test, kind, acc_cls)) return 1;
  auto launch = [&](auto kernel) -> int {
    kernel<<<dim3((unsigned)call.tiles, (unsigned)call.bands), THREADS, 0, call.s>>>(
        (const unsigned char*)src->data, *test, call.sh, call.sw, call.pad, call.off, n_copies, call.sorted,
        call.first, call.walk_all, (int)call.tiles_x, init, fill, (unsigned char*)dst->data, dst->dtype, call.dh,
        call.dw);
    GM_LAUNCH_CHECK();
    return 0;
  };
  return with_place_pair(*test, [&](auto p) -> int {
    return with_kernel<PlaceKernel<decltype(p)::value>::template Of>(acc_cls, kind, launch);
  });
}

extern "C" int gm_reduce_stack_stat(const GmStackInput* inputs, int64_t n_inputs, int stat, int work_bytes,
                                    uint64_t fill, GmArray* out, void* stream) {
  if (ensure_init()) return 1;
  if (!out || (n_inputs > 0 && !inputs)) return fail("gm_reduce_stack_stat: null argument");
  if (n_inputs < 1) return fail("gm_reduce_stack_stat: empty stack");
  if (n_inputs >= ((int64_t)1 << 31)) return fail("gm_reduce_stack_stat: too many rasters");
  if (out->space != GM_DEVICE) return fail("gm_reduce_stack_stat: the output must be device resident");
  if (!dtype_size(out->dtype)) return fail("gm_reduce_stack_stat: bad output dtype");
  if (check_stat(stat, work_bytes, out->dtype, "gm_reduce_stack_stat")) return 1;
  for (int64_t k = 0; k < n_inputs; ++k) {
    if (check_input(inputs[k], "gm_reduce_stack_stat")) return 1;
    if (!inputs[k].data) return fail("gm_reduce_stack_stat: null input");
  }
  const int64_t n = array_count(*out);
  if (n == 0) return 0;
  cudaStream_t s = resolve_stream(stream);
  void* dev = nullptr;
  if (upload(&dev, inputs, n_inputs * (int64_t)sizeof(GmStackInput), s)) return 1;
  const int64_t blocks = (n + (int64_t)THREADS * PIX - 1) / ((int64_t)THREADS * PIX);
  const int rc = with_stat<StackStatKernel>(stat, work_bytes, [&](auto kernel) -> int {
    kernel<<<(unsigned)blocks, THREADS, 0, s>>>((const GmStackInput*)dev, n_inputs, fill, (unsigned char*)out->data,
                                                out->dtype, n);
    GM_LAUNCH_CHECK();
    return 0;
  });
  cudaFreeAsync(dev, s);
  return rc;
}

extern "C" int gm_place_stat(const GmArray* src, GmArray* dst, const void* nodata, const int32_t* offsets,
                             int64_t n_copies, const GmStackInput* test, int stat, int work_bytes, uint64_t fill,
                             void* stream) {
  PlaceCall call;
  if (call.open("gm_place_stat", src, dst, nodata, offsets, n_copies, test, stream)) return 1;
  if (check_stat(stat, work_bytes, dst->dtype, "gm_place_stat")) return 1;
  if (call.empty) return 0;
  if (call.list("gm_place_stat", offsets, n_copies, test, -1, 0)) return 1;
  int* rank = nullptr;
  if ((stat == GM_STACK_ARGMIN || stat == GM_STACK_ARGMAX) && call.rank_copies(src, test, n_copies, &rank)) return 1;
  auto launch = [&](auto kernel) -> int {
    kernel<<<dim3((unsigned)call.tiles, (unsigned)call.bands), THREADS, 0, call.s>>>(
        (const unsigned char*)src->data, *test, call.sh, call.sw, call.pad, call.off, rank, call.sorted, call.first,
        (int)call.tiles_x, fill, (unsigned char*)dst->data, dst->dtype, call.dh, call.dw);
    GM_LAUNCH_CHECK();
    return 0;
  };
  return with_place_pair(*test, [&](auto p) -> int {
    return with_stat<PlaceStatKernel<decltype(p)::value>::template Of>(stat, work_bytes, launch);
  });
}
