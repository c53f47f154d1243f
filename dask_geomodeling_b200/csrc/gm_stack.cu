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
//
// Reference: raster/reduction.py:38-119, raster/spatial.py:657-731.
#include "gm_common.cuh"
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

// the same with the class pair chosen per raster (block-uniform)
template <typename A, int KIND, int Q>
__device__ __forceinline__ void fold(uint64_t (&acc)[Q], const uint64_t (&x)[Q], const Desc& d) {
  switch (d.pair) {
    case P_I32: fold_typed<int32_t, int32_t, A, KIND>(acc, x, d); break;
    case P_I64: fold_typed<int64_t, int64_t, A, KIND>(acc, x, d); break;
    case P_F32: fold_typed<float, float, A, KIND>(acc, x, d); break;
    case P_F32_F64: fold_typed<float, double, A, KIND>(acc, x, d); break;
    default: fold_typed<double, double, A, KIND>(acc, x, d); break;
  }
}

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

template <typename A, int KIND>
__global__ void __launch_bounds__(THREADS, 3)
reduce_stack_kernel(const GmStackInput* __restrict__ inputs, int64_t n_inputs, uint64_t init, uint64_t fill,
                    unsigned char* __restrict__ out, int out_dtype, int64_t n) {
  __shared__ Desc desc[THREADS];
  const int64_t base = ((int64_t)blockIdx.x * THREADS + threadIdx.x) * PIX;
  uint64_t acc[PIX];
#pragma unroll
  for (int i = 0; i < PIX; ++i) acc[i] = init;
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
          fold<A, KIND>(acc, x, d);
        }
      }
    }
  }
  if (base >= n) return;
  const int osz = dtype_size(out_dtype), out_cls = natural_class(out_dtype);
  uint64_t v[PIX];
#pragma unroll
  for (int i = 0; i < PIX; ++i) v[i] = finish<A, KIND>(acc[i], out_cls, fill);
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
  if (c == 0) {
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

// one block per (tile, band): out = reduction over the tile's copies, in copy order, or over every
// copy when *walk_all (see place_count_kernel).  Source class pair P is fixed for the call.
template <typename A, int KIND, int P>
__global__ void __launch_bounds__(THREADS, 4)
place_kernel(const unsigned char* __restrict__ src, GmStackInput test, int sh, int sw, uint64_t pad,
             const int2* __restrict__ off, int64_t n, const uint64_t* __restrict__ keys,
             const int64_t* __restrict__ first, const int* __restrict__ walk_all, int tiles_x,
             uint64_t init, uint64_t fill,
             unsigned char* __restrict__ out, int out_dtype, int dh, int dw) {
  __shared__ int2 list[THREADS];
  const Desc d = make_desc(test);
  const int tile = blockIdx.x, band = blockIdx.y;
  const int i = (tile % tiles_x) * TILE_W + (int)(threadIdx.x % TILE_W);
  const int j0 = (tile / tiles_x) * TILE_H + (int)(threadIdx.x / TILE_W);
  constexpr int JSTEP = THREADS / TILE_W;
  const unsigned char* plane = src + band * (int64_t)sh * sw * d.isz;
  typedef typename Pair<P>::From From;
  uint64_t acc[ROWS];
#pragma unroll
  for (int k = 0; k < ROWS; ++k) acc[k] = init;
  const bool all = *walk_all;
  const int begin = all ? 0 : (int)first[tile], end = all ? (int)n : (int)first[tile + 1];
  for (int e0 = begin; e0 < end; e0 += THREADS) {
    const int m = end - e0 < THREADS ? end - e0 : THREADS;
    __syncthreads();
    if (threadIdx.x < m) {
      const int e = e0 + threadIdx.x;
      list[threadIdx.x] = off[all ? e : (int)(uint32_t)keys[e]];
    }
    __syncthreads();
#pragma unroll 1
    for (int q = 0; q < m; ++q) {
      const int2 o = list[q];
      const int si = i - o.x;
      uint64_t x[ROWS];
#pragma unroll
      for (int k = 0; k < ROWS; ++k) {
        const int sj = j0 + k * JSTEP - o.y;
        uint64_t v = pad;
        if ((unsigned)si < (unsigned)sw && (unsigned)sj < (unsigned)sh)
          v = load_one(plane + ((int64_t)sj * sw + si) * d.isz, d.isz);
        x[k] = v;
      }
#pragma unroll
      for (int k = 0; k < ROWS; ++k) {
        // gm_resample_nn's rule: a non-finite source value is no data
        if constexpr (IsFloat<From>::value) x[k] = finite_(Raw<From>::get(x[k])) ? x[k] : pad;
        x[k] = natural_bits(d.dtype, x[k]);
      }
      fold_typed<From, typename Pair<P>::T, A, KIND>(acc, x, d);
    }
  }
  const int osz = dtype_size(out_dtype), out_cls = natural_class(out_dtype);
  unsigned char* dst = out + band * (int64_t)dh * dw * osz;
#pragma unroll
  for (int k = 0; k < ROWS; ++k) {
    const int j = j0 + k * JSTEP;
    if (i < dw && j < dh) store_one(dst + ((int64_t)j * dw + i) * osz, osz, finish<A, KIND>(acc[k], out_cls, fill));
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

int check_input(const GmStackInput& g, const char* who) {
  if (!dtype_size(g.dtype)) return fail(std::string(who) + ": bad input dtype");
  if (g.cls > GM_C_F64 || test_pair(g.dtype, g.cls) == P_INVALID)
    return fail(std::string(who) + ": the test class does not fit the dtype");
  return 0;
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
  if (ensure_init()) return 1;
  if (!src || !dst || !nodata || !test || (n_copies > 0 && !offsets)) return fail("gm_place: null argument");
  if (src->space != GM_DEVICE || dst->space != GM_DEVICE) return fail("gm_place: operands must be device resident");
  if (src->shape[0] != dst->shape[0]) return fail("gm_place: band count mismatch");
  if (test->dtype != src->dtype) return fail("gm_place: the test must be that of the source dtype");
  if (check_input(*test, "gm_place") || !dtype_size(dst->dtype)) return 1;
  if (n_copies < 0) return fail("gm_place: negative copy count");
  const int64_t bands = src->shape[0];
  const int sh = (int)src->shape[1], sw = (int)src->shape[2], dh = (int)dst->shape[1], dw = (int)dst->shape[2];
  if (bands == 0 || dh == 0 || dw == 0) return 0;
  if (bands > 65535) return fail("gm_place: too many bands");
  cudaStream_t s = resolve_stream(stream);
  uint64_t pad = 0;
  memcpy(&pad, nodata, dtype_size(src->dtype));
  const int64_t tiles_x = (dw + TILE_W - 1) / TILE_W, tiles_y = (dh + TILE_H - 1) / TILE_H;
  const int64_t tiles = tiles_x * tiles_y;
  if (tiles >= ((int64_t)1 << 31) || n_copies >= ((int64_t)1 << 31)) return fail("gm_place: too many tiles or copies");

  std::vector<void*> scratch;
  auto cleanup = [&]() { for (void* p : scratch) cudaFreeAsync(p, s); };
  auto alloc = [&](void** p, size_t bytes) -> int {
    GM_CUDA(cudaMallocAsync(p, bytes > 0 ? bytes : 16, s));
    scratch.push_back(*p);
    return 0;
  };
  void* off = nullptr;
  if (upload(&off, offsets, n_copies * 8, s)) return 1;
  scratch.push_back(off);

  // tile lists: (tile, copy) keys sorted by tile, then copy; their length from the offsets on the
  // host, so that nothing waits for the device
  int64_t total = 0;
  for (int64_t c = 0; c < n_copies; ++c) {
    const TileRange t = tiles_met(make_int2(offsets[2 * c], offsets[2 * c + 1]), sh, sw, dh, dw);
    total += (t.r1 - t.r0 + 1) * (t.c1 - t.c0 + 1);
  }
  if (total >= ((int64_t)1 << 31)) { cleanup(); return fail("gm_place: too many (tile, copy) pairs"); }
  int64_t* counts = nullptr; int64_t* incl = nullptr; int* walk_all = nullptr;
  uint64_t* keys = nullptr; uint64_t* sorted = nullptr; int64_t* first = nullptr;
  int rc = alloc((void**)&counts, n_copies * 8) || alloc((void**)&incl, n_copies * 8) ||
           alloc((void**)&walk_all, 4) || alloc((void**)&keys, total * 8) || alloc((void**)&sorted, total * 8) ||
           alloc((void**)&first, (tiles + 1) * 8);
  if (rc) { cleanup(); return 1; }
  place_count_kernel<<<(unsigned)(n_copies > 0 ? (n_copies + THREADS - 1) / THREADS : 1), THREADS, 0, s>>>(
      (const int2*)off, n_copies, sh, sw, dh, dw, counts, *test, pad, kind, acc_cls, walk_all);
  if (cudaGetLastError() != cudaSuccess) { cleanup(); return fail("gm_place: count launch failed"); }
  count_launch();
  if (total > 0) {
    size_t scan_bytes = 0, sort_bytes = 0;
    int end_bit = 33;  // keys are tile << 32 | copy
    while (((int64_t)1 << (end_bit - 32)) <= tiles) ++end_bit;
    cub::DeviceScan::InclusiveSum(nullptr, scan_bytes, counts, incl, n_copies, s);
    cub::DeviceRadixSort::SortKeys(nullptr, sort_bytes, keys, sorted, total, 0, end_bit, s);
    void* temp = nullptr;
    if (alloc(&temp, scan_bytes > sort_bytes ? scan_bytes : sort_bytes)) { cleanup(); return 1; }
    if (cub::DeviceScan::InclusiveSum(temp, scan_bytes, counts, incl, n_copies, s) != cudaSuccess) {
      cleanup(); return fail("gm_place: scan failed");
    }
    count_launch();
    place_fill_kernel<<<(unsigned)n_copies, THREADS, 0, s>>>((const int2*)off, sh, sw, dh, dw, (int)tiles_x,
                                                             counts, incl, keys);
    if (cudaGetLastError() != cudaSuccess) { cleanup(); return fail("gm_place: fill launch failed"); }
    count_launch();
    if (cub::DeviceRadixSort::SortKeys(temp, sort_bytes, keys, sorted, total, 0, end_bit, s) != cudaSuccess) {
      cleanup(); return fail("gm_place: sort failed");
    }
    count_launch();
  }
  place_bounds_kernel<<<(unsigned)((tiles + 1 + THREADS - 1) / THREADS), THREADS, 0, s>>>(
      sorted, total, (int)tiles, first);
  if (cudaGetLastError() != cudaSuccess) { cleanup(); return fail("gm_place: bounds launch failed"); }
  count_launch();
  auto launch = [&](auto kernel) -> int {
    kernel<<<dim3((unsigned)tiles, (unsigned)bands), THREADS, 0, s>>>(
        (const unsigned char*)src->data, *test, sh, sw, pad, (const int2*)off, n_copies, sorted, first, walk_all,
        (int)tiles_x, init, fill, (unsigned char*)dst->data, dst->dtype, dh, dw);
    GM_LAUNCH_CHECK();
    return 0;
  };
  switch (test_pair(test->dtype, test->cls)) {
    case P_I32: rc = with_kernel<PlaceKernel<P_I32>::Of>(acc_cls, kind, launch); break;
    case P_I64: rc = with_kernel<PlaceKernel<P_I64>::Of>(acc_cls, kind, launch); break;
    case P_F32: rc = with_kernel<PlaceKernel<P_F32>::Of>(acc_cls, kind, launch); break;
    case P_F32_F64: rc = with_kernel<PlaceKernel<P_F32_F64>::Of>(acc_cls, kind, launch); break;
    default: rc = with_kernel<PlaceKernel<P_F64>::Of>(acc_cls, kind, launch); break;
  }
  cleanup();
  return rc;
}
