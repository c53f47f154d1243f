// Polygon scanline rasteriser and zonal statistics.
//
//   gm_rasterize_polygons  utils.rasterize_geoseries (utils.py:638-756), i.e. GDAL's
//                          GDALRasterizeLayers without ALL_TOUCHED
//   gm_zonal_stats         geometry/aggregate.py:113-203 (aggregate_polygons) with
//                          scipy.ndimage sum/mean/minimum/maximum/median and
//                          measurements.percentile (measurements.py:18-137)
//
// The fill rule restates GDAL's alg/llrasterize.cpp::GDALdllImageFilledPolygon
// (see oracle/polyfill.c for the CPU restatement it is tested against): vertices in
// pixel space through the inverse geotransform, scanline at y + 0.5, crossing
// x = floor(intersect + 0.5), even-odd pairs over all rings of a feature, bottom
// horizontal edges filled on their own.  The per-edge part of the rule is written once,
// in edge_crossing; rows reach it through one of two routines:
//   generic_scanline  the whole warp on one row, any number of vertices and crossings
//   row_crossings     lane per row, for polygons of <= ZW_MAXV vertices staged in shared
//                     memory; a row it cannot describe (a bottom horizontal edge, more
//                     than ZW_MAXC crossings) goes to generic_scanline
// Zonal statistics read the raster directly under the spans; no label raster is ever
// materialised.  Which kernel takes which polygon:
//   - count / sum / mean / min / max: zonal_reduce_warp_kernel, one warp per polygon, for
//     polygons of <= ZW_MAXV vertices, <= ZW_BIG_ROWS rows and a bounding box of <= ZW_BIG_CELLS
//     cells; the rest is deferred to zonal_reduce_kernel, one block per polygon (scan_polygon).
//   - median / percentile of float32 and integer rasters up to 4 bytes without thresholds: the
//     streaming select, one warp per polygon in three kernels (bracket, main, final) under the
//     same limits; the polygons it defers, and every other raster, go to zonal_select_kernel,
//     one block per polygon with an MSD radix select over the polygon's values.
//   - rasterize: rasterize_tile_kernel, one block per tile of the output, one warp per polygon.
//   - stripes of the multi-GPU path: the reduce kernels above, or zonal_values_kernel for the
//     values that segment_select_kernel selects from.
#include "gm_common.cuh"
#include <cfloat>
#include <cstdlib>
#include <limits>
#include <memory>
#include <mutex>
#include <type_traits>
#include <vector>

namespace gm {

constexpr int PG_THREADS = 128;               // 4 warps per polygon
constexpr int PG_WARPS = PG_THREADS / 32;
constexpr int PG_MAX_CROSSINGS = 4096;        // per scanline
constexpr int PG_MAX_HSPANS = 8;
constexpr int SEL_THREADS = 256;
constexpr int ZW_MAXV = 64;                  // vertices of a polygon handled lane-per-scanline
constexpr int ZW_MAXC = 8;                   // crossings per scanline on that path
constexpr int PG_FAST_WARPS = SEL_THREADS / 32;
constexpr int PG_BATCH = 4;                 // single-span rows handed to a visitor at once

struct PolyDev {
  const double* px;             // pixel-space x of every vertex
  const double* py;
  const int64_t* ring_offsets;
  const int64_t* poly_offsets;
  const int* miny;              // per polygon, clamped to the raster and the stripe
  const int* maxy;              // inclusive
  int64_t n_polygons;
  int height, width;
  int cap;                      // crossing capacity per warp (power of two)
  int* error;                   // device flag: 1 = crossing overflow
  const int* active;            // stripe calls: ids of the polygons with rows here (else nullptr)
  const int* n_active;          // device scalar: length of `active`
};

// ---- preparation -------------------------------------------------------------------
__global__ void poly_transform_kernel(const double* __restrict__ xy, double* __restrict__ px,
                                      double* __restrict__ py, int64_t n, double inv0, double inv1,
                                      double inv3, double inv5) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double x = xy[2 * i], y = xy[2 * i + 1];
  // GDALApplyGeoTransform on GDALInvGeoTransform's output (rotation terms are 0)
  px[i] = (inv0 + x * inv1) + y * 0.0;
  py[i] = (inv3 + x * 0.0) + y * inv5;
}

__global__ void poly_rows_kernel(const double* __restrict__ py, const int64_t* __restrict__ ring_offsets,
                                 const int64_t* __restrict__ poly_offsets, int64_t n_polygons,
                                 int height, int row_begin, int row_end, int* __restrict__ miny,
                                 int* __restrict__ maxy) {
  const int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (p >= n_polygons) return;
  const int64_t v0 = ring_offsets[poly_offsets[p]], v1 = ring_offsets[poly_offsets[p + 1]];
  int lo = 1, hi = 0;
  if (v1 > v0) {
    double dmin = py[v0], dmax = py[v0];
    for (int64_t i = v0 + 1; i < v1; ++i) {
      dmin = fmin(dmin, py[i]);
      dmax = fmax(dmax, py[i]);
    }
    // static_cast<int>(dminy) / (dmaxy), then clamped to the raster
    dmin = fmin(fmax(dmin, -1.0e9), 1.0e9);
    dmax = fmin(fmax(dmax, -1.0e9), 1.0e9);
    lo = (int)dmin;
    hi = (int)dmax;
    if (v1 - v0 == 1) { lo = hi = (int)floor(dmin); }  // point feature: the cell that contains it
    if (lo < 0) lo = 0;
    if (hi >= height) hi = height - 1;
    if (lo < row_begin) lo = row_begin;
    if (hi >= row_end) hi = row_end - 1;
  }
  miny[p] = lo;
  maxy[p] = hi;
}

// Stripe calls: most polygons have no row in this stripe.  Their ids are compacted away once, so
// that the reduce kernel's work counter only hands out polygons that do something (every hand-out
// is an atomic on ONE address plus a dependent chain of offset loads: 87 000 of them cost more
// than the 12 500 polygons of a 1/8 stripe of configs[3]).  Order inside a warp is kept, so
// neighbouring polygons still travel together.
__global__ void poly_active_kernel(const int* __restrict__ miny, const int* __restrict__ maxy,
                                   const int64_t* __restrict__ ring_offsets,
                                   const int64_t* __restrict__ poly_offsets, int64_t n_polygons,
                                   int* __restrict__ active, int* __restrict__ n_active) {
  const int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  bool on = false;
  if (p < n_polygons)
    on = miny[p] <= maxy[p] && ring_offsets[poly_offsets[p + 1]] > ring_offsets[poly_offsets[p]];
  const unsigned mask = __ballot_sync(0xffffffffu, on);
  if (!mask) return;
  const int lane = threadIdx.x & 31;
  int base = 0;
  if (lane == __ffs(mask) - 1) base = atomicAdd(n_active, __popc(mask));
  base = __shfl_sync(0xffffffffu, base, __ffs(mask) - 1);
  if (on) active[base + __popc(mask & ((1u << lane) - 1u))] = (int)p;
}

// ---- warp-level scanline walk ---------------------------------------------------------
__device__ __forceinline__ int clamp_to_int(double v) {
  return (int)fmin(fmax(v, -2.0e9), 2.0e9);
}

// sort buf[0..n) ascending, warp cooperative
__device__ __forceinline__ void warp_sort(int* buf, int n, int lane) {
  __syncwarp();
  if (n <= 1) return;
  if (n <= 32) {
    const int v = lane < n ? buf[lane] : 0;
    int rank = 0;
    for (int j = 0; j < n; ++j) {
      const int o = __shfl_sync(0xffffffffu, v, j);
      rank += (o < v) || (o == v && j < lane);
    }
    __syncwarp();
    if (lane < n) buf[rank] = v;
    __syncwarp();
    return;
  }
  int m = 1;
  while (m < n) m <<= 1;
  for (int i = n + lane; i < m; i += 32) buf[i] = INT_MAX;
  __syncwarp();
  for (int k = 2; k <= m; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = lane; i < m; i += 32) {
        const int l = i ^ j;
        if (l > i) {
          const int a = buf[i], b = buf[l];
          const bool up = (i & k) == 0;
          if ((a > b) == up) { buf[i] = b; buf[l] = a; }
        }
      }
      __syncwarp();
    }
}

// is column x inside one of the sorted crossing pairs?
__device__ __forceinline__ bool in_pairs(int x, const int* buf, int count) {
  for (int i = 0; i + 1 < count; i += 2)
    if (x >= buf[i] && x <= buf[i + 1] - 1) return true;
  return false;
}

// default: one span at a time (visitors that gain from batching overload this)
template <class Visitor>
__device__ __forceinline__ void span_batch(Visitor& vis, int n, const int* ys, const int* x0, const int* x1) {
#pragma unroll
  for (int i = 0; i < PG_BATCH; ++i)   // entries >= n are empty spans
    if (x0[i] <= x1[i]) vis.span(ys[i], x0[i], x1[i]);
}
template <typename T> struct ReduceVisitor;
template <typename T> struct GatherVisitor;
template <typename T>
__device__ __forceinline__ void span_batch(GatherVisitor<T>& vis, int n, const int* ys, const int* x0, const int* x1);
template <typename T>
__device__ __forceinline__ void span_batch(ReduceVisitor<T>& vis, int n, const int* ys, const int* x0, const int* x1);

// The fill rule of GDALdllImageFilledPolygon for ONE edge, from vertex i1 (its predecessor on
// the ring) to vertex i2, against the scanline at dy = y + 0.5.  Every path that converts
// polygons to rows decides through this function.  Returns
//   EDGE_CROSS   the edge crosses the scanline at column *x = floor(intersect + 0.5)
//   EDGE_BOTTOM  the edge is a bottom horizontal edge on the scanline, columns [*x, *x2),
//                which GDAL fills on its own (not part of the even-odd pairs)
//   EDGE_NONE    neither
enum { EDGE_NONE = 0, EDGE_CROSS = 1, EDGE_BOTTOM = 2 };
template <typename I>
__device__ __forceinline__ int edge_crossing(const double* px, const double* py, I i1, I i2, double dy,
                                             int* x, int* x2) {
  double dy1 = py[i1], dy2 = py[i2];
  if ((dy1 < dy && dy2 < dy) || (dy1 > dy && dy2 > dy)) return EDGE_NONE;
  double dx1, dx2;
  if (dy1 < dy2) {
    dx1 = px[i1]; dx2 = px[i2];
  } else if (dy1 > dy2) {
    const double t = dy1; dy1 = dy2; dy2 = t;
    dx2 = px[i1]; dx1 = px[i2];
  } else {
    const double xa = px[i1], xb = px[i2];
    if (!(xa > xb)) return EDGE_NONE;
    *x = clamp_to_int(floor(xb + 0.5));
    *x2 = clamp_to_int(floor(xa + 0.5));
    return EDGE_BOTTOM;
  }
  if (!(dy < dy2 && dy >= dy1)) return EDGE_NONE;
  const double intersect = (dy - dy1) * (dx2 - dx1) / (dy2 - dy1) + dx1;
  *x = clamp_to_int(floor(intersect + 0.5));
  return EDGE_CROSS;
}

// Visitor interface (all calls are warp-uniform):
//   span(y, x0, x1)                       regular even-odd span, inclusive, clipped
//   hspan(y, x0, x1, buf, count)          bottom horizontal edge on the scanline
//
// Generic scanline: the whole warp works on ONE row of the feature made of rings r0..r1
// (any number of vertices / crossings, at most `cap` of which fit `buf`).
template <class Visitor>
__device__ __forceinline__ void generic_scanline(const PolyDev& P, int64_t r0, int64_t r1, int y, int cap,
                                                 int* buf, int* hbuf, Visitor& vis) {
  const int lane = threadIdx.x & 31;
  const int maxx = P.width - 1;
  const double dy = y + 0.5;
  int count = 0, hcount = 0;
  for (int64_t r = r0; r < r1; ++r) {
    const int64_t a = P.ring_offsets[r], b = P.ring_offsets[r + 1];
    for (int64_t base = a; base < b; base += 32) {
      const int64_t i = base + lane;
      bool cross = false, hs = false;
      int xi = 0, hx2 = 0;      // the crossing, or the bottom horizontal edge [xi, hx2)
      if (i < b) {
        const int e = edge_crossing(P.px, P.py, (i == a) ? b - 1 : i - 1, i, dy, &xi, &hx2);
        cross = e == EDGE_CROSS;
        hs = e == EDGE_BOTTOM && !(xi > maxx || hx2 <= 0);
      }
      const unsigned cm = __ballot_sync(0xffffffffu, cross);
      if (cross) {
        const int pos = count + __popc(cm & ((1u << lane) - 1u));
        if (pos < cap) buf[pos] = xi;
      }
      count += __popc(cm);
      const unsigned hm = __ballot_sync(0xffffffffu, hs);
      if (hs) {
        const int pos = hcount + __popc(hm & ((1u << lane) - 1u));
        if (pos < PG_MAX_HSPANS) { hbuf[2 * pos] = xi; hbuf[2 * pos + 1] = hx2; }
      }
      hcount += __popc(hm);
    }
  }
  if (count > cap || hcount > PG_MAX_HSPANS) {
    if (lane == 0) atomicExch(P.error, 1);
    count = count > cap ? cap : count;
    hcount = hcount > PG_MAX_HSPANS ? PG_MAX_HSPANS : hcount;
  }
  warp_sort(buf, count, lane);
  for (int i = 0; i + 1 < count; i += 2) {
    const int xa = buf[i], xb = buf[i + 1];
    if (xa <= maxx && xb > 0) {
      const int x0 = xa < 0 ? 0 : xa, x1 = xb - 1 > maxx ? maxx : xb - 1;
      if (x0 <= x1) vis.span(y, x0, x1);
    }
  }
  __syncwarp();
  for (int h = 0; h < hcount; ++h) {
    const int x0 = hbuf[2 * h] < 0 ? 0 : hbuf[2 * h];
    const int x1 = hbuf[2 * h + 1] - 1 > maxx ? maxx : hbuf[2 * h + 1] - 1;
    if (x0 <= x1) vis.hspan(y, x0, x1, buf, count);
  }
  __syncwarp();
}

// Lane per scanline, for polygons of at most ZW_MAXV vertices staged in shared memory: vertex i
// at (px[i], py[i]), its predecessor on its ring at prev[i].
//
// Vertex v0 + i of the polygon made of rings r0..r1 and its ring predecessor to shared memory;
// returns the vertex' x.
__device__ __forceinline__ double stage_vertex(const PolyDev& P, int64_t r0, int64_t r1, int64_t v0, int i,
                                               double* px, double* py, int* prev) {
  const double x = P.px[v0 + i];
  px[i] = x; py[i] = P.py[v0 + i];
  int pr = i - 1;
  for (int64_t r = r0; r < r1; ++r)
    if ((int64_t)i + v0 == P.ring_offsets[r]) pr = (int)(P.ring_offsets[r + 1] - v0) - 1;
  prev[i] = pr;
  return x;
}

// the nv vertices of a polygon to the warp's shared memory; returns the width of the bounding
// box clipped to the raster, fmin(xmax, width) - fmax(xmin, 0) (negative when it misses)
__device__ __forceinline__ double stage_polygon(const PolyDev& P, int64_t r0, int64_t r1, int64_t v0, int nv,
                                                double* px, double* py, int* prev, int lane) {
  double xmin = DBL_MAX, xmax = -DBL_MAX;
  __syncwarp();
  for (int i = lane; i < nv; i += 32) {
    const double x = stage_vertex(P, r0, r1, v0, i, px, py, prev);
    xmin = fmin(xmin, x); xmax = fmax(xmax, x);
  }
  for (int o = 16; o > 0; o >>= 1) {
    xmin = fmin(xmin, __shfl_xor_sync(0xffffffffu, xmin, o));
    xmax = fmax(xmax, __shfl_xor_sync(0xffffffffu, xmax, o));
  }
  __syncwarp();
  return fmin(xmax, (double)P.width) - fmax(xmin, 0.0);
}

// sorted crossings of row y with the staged polygon into column `lane` of `cross`; returns their
// number, or -1 for a row that needs the generic scanline (a bottom horizontal edge on the
// scanline, more than ZW_MAXC crossings).  Inlined into the reduce kernels; the select and
// rasterize kernels call row_crossings_call.
__device__ __forceinline__ int row_crossings(const double* px, const double* py, const int* prev, int nv,
                                             int y, int (*cross)[32], int lane) {
  const double dy = y + 0.5;
  int cnt = 0;
  bool complex_row = false;
  for (int i = 0; i < nv; ++i) {
    int x = 0, x2 = 0;
    const int e = edge_crossing(px, py, prev[i], i, dy, &x, &x2);
    if (e == EDGE_BOTTOM) complex_row = true;
    if (e == EDGE_CROSS) {
      if (cnt < ZW_MAXC) cross[cnt][lane] = x;
      ++cnt;
    }
  }
  if (cnt > ZW_MAXC || complex_row) return -1;
  for (int a = 1; a < cnt; ++a) {  // insertion sort of this lane's column
    const int v = cross[a][lane];
    int j = a - 1;
    while (j >= 0 && cross[j][lane] > v) { cross[j + 1][lane] = cross[j][lane]; --j; }
    cross[j + 1][lane] = v;
  }
  return cnt;
}

// Not inlined: the select kernels have to stay small enough for the instruction cache (32 warps
// per SM in different phases).
__device__ __noinline__ int row_crossings_call(const double* px, const double* py, const int* prev, int nv,
                                               int y, int (*cross)[32], int lane) {
  return row_crossings(px, py, prev, nv, y, cross, lane);
}

template <class Visitor>
__device__ __forceinline__ void scan_polygon(const PolyDev& P, int64_t p, int* buf, int* hbuf,
                                             Visitor& vis) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nwarps = blockDim.x >> 5;
  const int64_t r0 = P.poly_offsets[p], r1 = P.poly_offsets[p + 1];
  if (r1 <= r0) return;
  const int64_t v0 = P.ring_offsets[r0], v1 = P.ring_offsets[r1];
  const int miny = P.miny[p], maxy = P.maxy[p];
  const int maxx = P.width - 1;
  if (v1 - v0 == 1) {  // point feature (GDALdllImagePoint): burn floor(x), floor(y)
    if (warp == 0 && miny <= maxy) {
      const int x = clamp_to_int(floor(P.px[v0]));
      if (x >= 0 && x <= maxx) vis.span(miny, x, x);
    }
    return;
  }
  auto generic_row = [&](int y) { generic_scanline(P, r0, r1, y, P.cap, buf, hbuf, vis); };

  const int nv = (int)(v1 - v0);
  if (nv > ZW_MAXV) {
    for (int y = miny + warp; y <= maxy; y += nwarps) generic_row(y);
    return;
  }

  // Small polygons (<= ZW_MAXV vertices, the usual case): the vertices are staged in
  // shared memory once, then each warp takes 32 scanlines at a time -- lane = scanline --
  // so the edge tests of 32 rows run in parallel instead of one row per warp; the
  // crossings are sorted per lane in shared memory and the spans are then walked by the
  // whole warp row by row (coalesced raster reads).  Rows with more than ZW_MAXC crossings
  // or a horizontal bottom edge fall back to generic_row.
  __shared__ double s_px[ZW_MAXV], s_py[ZW_MAXV];
  __shared__ int s_prev[ZW_MAXV];
  __shared__ int s_cross[PG_FAST_WARPS][ZW_MAXC][32];
  __syncthreads();
  for (int i = threadIdx.x; i < nv; i += blockDim.x) stage_vertex(P, r0, r1, v0, i, s_px, s_py, s_prev);
  __syncthreads();
  for (int base = miny + 32 * warp; base <= maxy; base += 32 * nwarps) {
    const int y = base + lane;
    int cnt = 0;
    if (y <= maxy) cnt = row_crossings(s_px, s_py, s_prev, nv, y, s_cross[warp], lane);
    const bool complex_row = cnt < 0;
    __syncwarp();
    const unsigned complex_mask = __ballot_sync(0xffffffffu, complex_row);
    const int n_rows = min(32, maxy - base + 1);
    for (int r = 0; r < n_rows; ++r) {
      const int yy = base + r;
      if ((complex_mask >> r) & 1u) { generic_row(yy); continue; }
      const int c = __shfl_sync(0xffffffffu, cnt, r);
      if (c == 2) {
        // the usual case, one span per row: hand up to PG_BATCH consecutive such rows to the
        // visitor together so that it can keep the raster reads of all of them in flight
        // (fixed-index, fully unrolled: the batch stays in registers)
        int ys[PG_BATCH], xs0[PG_BATCH], xs1[PG_BATCH];
        int nb = 0;
        bool open = true;
#pragma unroll
        for (int e = 0; e < PG_BATCH; ++e) {
          const int rr = (r + e) & 31;
          const bool single = __shfl_sync(0xffffffffu, cnt, rr) == 2;
          open = open && r + e < n_rows && !((complex_mask >> rr) & 1u) && single;
          const int xa = s_cross[warp][0][rr], xb = s_cross[warp][1][rr];
          int x0 = 1, x1 = 0;  // empty unless the span touches the raster
          if (open && xa <= maxx && xb > 0) { x0 = xa < 0 ? 0 : xa; x1 = xb - 1 > maxx ? maxx : xb - 1; }
          ys[e] = open ? base + r + e : yy; xs0[e] = x0; xs1[e] = x1;
          nb += open ? 1 : 0;
        }
        span_batch(vis, nb, ys, xs0, xs1);
        r += nb - 1;
        continue;
      }
      for (int i = 0; i + 1 < c; i += 2) {
        const int xa = s_cross[warp][i][r], xb = s_cross[warp][i + 1][r];
        if (xa <= maxx && xb > 0) {
          const int x0 = xa < 0 ? 0 : xa, x1 = xb - 1 > maxx ? maxx : xb - 1;
          if (x0 <= x1) vis.span(yy, x0, x1);
        }
      }
    }
    __syncwarp();
  }
}

// ---- zonal statistics ------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long order_f64(double v) {
  unsigned long long b = (unsigned long long)__double_as_longlong(v);
  return (b & 0x8000000000000000ULL) ? ~b : (b | 0x8000000000000000ULL);
}
__device__ __forceinline__ double unorder_f64(unsigned long long k) {
  unsigned long long b = (k & 0x8000000000000000ULL) ? (k & 0x7fffffffffffffffULL) : ~k;
  return __longlong_as_double((long long)b);
}
__device__ __forceinline__ unsigned order_f32(float v) {
  unsigned b = __float_as_uint(v);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float unorder_f32(unsigned k) {
  unsigned b = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
  return __uint_as_float(b);
}

// sortable key of a raster value: 32 bit for float32, 64 bit otherwise
template <typename T> struct KeyOf {
  typedef unsigned long long type;
  static __device__ __forceinline__ type key(T v) { return order_f64((double)v); }
  static __device__ __forceinline__ T value(type k) { return (T)unorder_f64(k); }
};
template <> struct KeyOf<float> {
  typedef unsigned type;
  static __device__ __forceinline__ type key(float v) { return order_f32(v); }
  static __device__ __forceinline__ float value(type k) { return unorder_f32(k); }
};

struct AreaVisitor {
  long long area;
  __device__ __forceinline__ void span(int, int x0, int x1) {
    if ((threadIdx.x & 31) == 0) area += x1 - x0 + 1;
  }
  __device__ __forceinline__ void hspan(int, int x0, int x1, const int* buf, int count) {
    int n = 0;
    for (int x = x0 + (threadIdx.x & 31); x <= x1; x += 32) n += !in_pairs(x, buf, count);
    for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
    if ((threadIdx.x & 31) == 0) area += n;
  }
};

__global__ void __launch_bounds__(PG_THREADS)
zonal_area_kernel(const PolyDev P, long long* __restrict__ area, const int* __restrict__ work) {
  // work[0] polygons listed from work[2]
  extern __shared__ int pg_smem[];
  __shared__ long long warp_area[PG_WARPS];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int* buf = pg_smem + warp * P.cap;
  int* hbuf = pg_smem + PG_WARPS * P.cap + warp * 2 * PG_MAX_HSPANS;
  const int n_listed = work[0];
  for (int item = blockIdx.x; item < n_listed; item += gridDim.x) {
    const int64_t p = work[2 + item];
    AreaVisitor vis{0};
    scan_polygon(P, p, buf, hbuf, vis);
    if (lane == 0) warp_area[warp] = vis.area;
    __syncthreads();
    if (threadIdx.x == 0) {
      long long a = 0;
      for (int w = 0; w < PG_WARPS; ++w) a += warp_area[w];
      area[p] = a;
    }
    __syncthreads();
  }
}

template <typename T>
struct ActiveTest {
  T nodata; int has_nodata; int has_threshold; float threshold;
  __device__ __forceinline__ bool operator()(T v) const {
    if (has_nodata && v == nodata) return false;
    if (has_threshold) {
      if (threshold != threshold) return false;          // NaN threshold: no aggregation
      if (!((double)v >= (double)threshold)) return false;
    }
    return true;
  }
};
// the test for polygon p (thresholds: one per polygon, or nullptr)
template <typename T>
__device__ __forceinline__ ActiveTest<T> active_test(T nodata, int has_nodata, const float* thresholds, int64_t p) {
  return ActiveTest<T>{nodata, has_nodata, thresholds != nullptr, thresholds ? thresholds[p] : 0.0f};
}

// min / max are tracked in the raster dtype (one FMNMX / IMNMX per value; NaN never wins,
// as with the `d < vmin` form) and the count in 32 bits per lane; only the sum needs the
// widening to double.  Everything is widened when the lanes are combined.
template <typename T> __device__ __forceinline__ T tmin(T a, T b) { return a < b ? a : b; }
template <typename T> __device__ __forceinline__ T tmax(T a, T b) { return a > b ? a : b; }
template <> __device__ __forceinline__ float tmin<float>(float a, float b) { return fminf(a, b); }
template <> __device__ __forceinline__ float tmax<float>(float a, float b) { return fmaxf(a, b); }
template <> __device__ __forceinline__ double tmin<double>(double a, double b) { return fmin(a, b); }
template <> __device__ __forceinline__ double tmax<double>(double a, double b) { return fmax(a, b); }

template <typename T>
struct ReduceVisitor {
  const T* raster; int width; ActiveTest<T> active;
  int count; long long cells; double sum; T vmin, vmax;
  __device__ __forceinline__ void reset() {
    count = 0; cells = 0; sum = 0.0;
    vmin = std::numeric_limits<T>::max(); vmax = std::numeric_limits<T>::lowest();
  }
  __device__ __forceinline__ void take(T v) {
    if (active(v)) {
      ++count; sum += (double)v;
      vmin = tmin<T>(vmin, v);
      vmax = tmax<T>(vmax, v);
    }
  }
  __device__ __forceinline__ void span(int y, int x0, int x1) {
    const T* row = raster + (int64_t)y * width;
    const int lane = threadIdx.x & 31;
    if (lane == 0) cells += x1 - x0 + 1;
    int x = x0 + lane;
    for (; x + 96 <= x1; x += 128) {  // four independent 128-byte requests in flight
      const T a = __ldg(row + x), b = __ldg(row + x + 32), c = __ldg(row + x + 64), d = __ldg(row + x + 96);
      take(a); take(b); take(c); take(d);
    }
    for (; x <= x1; x += 32) take(__ldg(row + x));
  }
  __device__ __forceinline__ void hspan(int y, int x0, int x1, const int* buf, int n) {
    const T* row = raster + (int64_t)y * width;
    int extra = 0;
    for (int x = x0 + (threadIdx.x & 31); x <= x1; x += 32)
      if (!in_pairs(x, buf, n)) { take(__ldg(row + x)); ++extra; }
    cells += extra;   // per lane; summed over the warp with the other accumulators
  }
};

// PG_BATCH rows x 4 requests of 128 bytes are issued before the first value is consumed.
// Slots beyond the span (and the empty padding rows of the batch) are given the no-data
// value, so `take` drops them without any per-slot bookkeeping.
template <typename T>
__device__ __forceinline__ void span_batch(ReduceVisitor<T>& vis, int n, const int* ys, const int* x0, const int* x1) {
  const int lane = threadIdx.x & 31;
  if (!vis.active.has_nodata) {  // no sentinel to mark unused slots with: one span at a time
#pragma unroll
    for (int b = 0; b < PG_BATCH; ++b)
      if (x0[b] <= x1[b]) vis.span(ys[b], x0[b], x1[b]);
    return;
  }
  const T skip = vis.active.nodata;
  T v[PG_BATCH][4];
#pragma unroll
  for (int b = 0; b < PG_BATCH; ++b) {
    const T* row = vis.raster + (int64_t)ys[b] * vis.width + lane;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int x = x0[b] + 32 * k;
      v[b][k] = (x + lane <= x1[b]) ? __ldg(row + x) : skip;
    }
  }
#pragma unroll
  for (int b = 0; b < PG_BATCH; ++b) {
    if (lane == 0 && x0[b] <= x1[b]) vis.cells += x1[b] - x0[b] + 1;
#pragma unroll
    for (int k = 0; k < 4; ++k) vis.take(v[b][k]);
  }
#pragma unroll
  for (int b = 0; b < PG_BATCH; ++b) {  // rows longer than 128 cells: the rest
    const T* row = vis.raster + (int64_t)ys[b] * vis.width;
    for (int x = x0[b] + 128 + lane; x <= x1[b]; x += 32) vis.take(__ldg(row + x));
  }
}

template <typename T>
__global__ void __launch_bounds__(PG_THREADS, 8)
zonal_reduce_kernel(const PolyDev P, const T* __restrict__ raster, T nodata, int has_nodata,
                    const float* __restrict__ thresholds, GmZonalPartial* __restrict__ partial,
                    long long* __restrict__ cells, const int* __restrict__ work) {
  // the polygons zonal_reduce_warp_kernel deferred: work[0] of them, listed from work[2]
  extern __shared__ int pg_smem[];
  __shared__ long long s_count[PG_WARPS], s_cells[PG_WARPS];
  __shared__ double s_sum[PG_WARPS], s_min[PG_WARPS], s_max[PG_WARPS];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int* buf = pg_smem + warp * P.cap;
  int* hbuf = pg_smem + PG_WARPS * P.cap + warp * 2 * PG_MAX_HSPANS;
  const int n_listed = work[0];
  for (int item = blockIdx.x; item < n_listed; item += gridDim.x) {
    const int64_t p = work[2 + item];
    ReduceVisitor<T> vis;
    vis.raster = raster; vis.width = P.width;
    vis.active = active_test(nodata, has_nodata, thresholds, p);
    vis.reset();
    scan_polygon(P, p, buf, hbuf, vis);
    long long count = vis.count;
    // a lane that saw nothing must not contribute the dtype extremes
    double vmin = vis.count > 0 ? (double)vis.vmin : DBL_MAX, vmax = vis.count > 0 ? (double)vis.vmax : -DBL_MAX;
    for (int o = 16; o > 0; o >>= 1) {
      count += __shfl_xor_sync(0xffffffffu, count, o);
      vis.cells += __shfl_xor_sync(0xffffffffu, vis.cells, o);
      vis.sum += __shfl_xor_sync(0xffffffffu, vis.sum, o);
      vmin = fmin(vmin, __shfl_xor_sync(0xffffffffu, vmin, o));
      vmax = fmax(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
    }
    if (lane == 0) { s_count[warp] = count; s_cells[warp] = vis.cells; s_sum[warp] = vis.sum; s_min[warp] = vmin; s_max[warp] = vmax; }
    __syncthreads();
    if (threadIdx.x == 0) {
      GmZonalPartial r{0, 0.0, DBL_MAX, -DBL_MAX};
      long long c = 0;
      for (int w = 0; w < PG_WARPS; ++w) {
        r.count += s_count[w]; r.sum += s_sum[w]; c += s_cells[w];
        r.vmin = fmin(r.vmin, s_min[w]); r.vmax = fmax(r.vmax, s_max[w]);
      }
      partial[p] = r;
      cells[p] = c;
    }
    __syncthreads();
  }
}

// ---- zonal reduce, one WARP per polygon ----------------------------------------------------
// The usual polygon (<= ZW_MAXV vertices, <= ZW_BIG_ROWS rows, bounding box <= ZW_BIG_CELLS
// cells) is taken by a single warp: no block barrier, no idle warps while the last rows of a
// polygon finish, and warps fetch polygons from one atomic counter, so that neighbouring
// polygons are in flight together.  Rows are read with 16-byte loads aligned to the raster
// (VEC = 16 / itemsize cells per lane, one 512-byte request per row and warp), ZW_ROWS rows
// issued before the first value is consumed; cells of a quad outside the span are masked by
// one unsigned compare.  Everything else (many vertices, many rows, wide boxes) is appended to
// a list that zonal_reduce_kernel (one block per polygon) works off afterwards.
constexpr int ZW_WARPS = 8;
constexpr int ZW_ROWS = 4;
constexpr int ZW_MIN_BLOCKS = 4;
constexpr int ZW_BIG_ROWS = 256;
constexpr long long ZW_BIG_CELLS = 1 << 17;
constexpr int ZW_SUM = 1, ZW_MIN = 2, ZW_MAX = 4, ZW_ALL = 7;

template <typename T, int NEED>
struct WarpReduce {
  // a lane's load: 16 bytes of 4- and 8-byte cells, 8 bytes of 2-byte cells, 4 bytes of
  // 1-byte cells -- four cells per lane (two doubles), so that a row of ~100 cells is one
  // load per lane with at most 3 edge cells either side
  static constexpr int QBYTES = sizeof(T) >= 4 ? 16 : sizeof(T) == 2 ? 8 : 4;
  static constexpr int VEC = QBYTES / (int)sizeof(T);
  typedef typename std::conditional<QBYTES == 16, uint4,
          typename std::conditional<QBYTES == 8, uint2, unsigned>::type>::type Quad;
  // integer cells: the sum is exact in int64 (no int -> double conversion per cell)
  typedef typename std::conditional<std::is_integral<T>::value, long long, double>::type Sum;
  const T* raster; int width; ActiveTest<T> active;
  int count; long long cells; Sum sum; T vmin, vmax;
  __device__ __forceinline__ void reset() {
    count = 0; cells = 0; sum = 0;
    vmin = std::numeric_limits<T>::max(); vmax = std::numeric_limits<T>::lowest();
  }
  __device__ __forceinline__ void take(T v) {
    if (active(v)) {
      ++count;
      if (NEED & ZW_SUM) sum += (Sum)v;
      if (NEED & ZW_MIN) vmin = tmin<T>(vmin, v);
      if (NEED & ZW_MAX) vmax = tmax<T>(vmax, v);
    }
  }
  // scalar walk of one span (rows that are not plain single spans)
  __device__ __forceinline__ void span(int y, int x0, int x1) {
    const T* row = raster + (int64_t)y * width;
    const int lane = threadIdx.x & 31;
    if (lane == 0) cells += x1 - x0 + 1;
    for (int x = x0 + lane; x <= x1; x += 32) take(__ldg(row + x));
  }
  __device__ __forceinline__ void hspan(int y, int x0, int x1, const int* buf, int n) {
    const T* row = raster + (int64_t)y * width;
    int extra = 0;
    for (int x = x0 + (threadIdx.x & 31); x <= x1; x += 32)
      if (!in_pairs(x, buf, n)) { take(__ldg(row + x)); ++extra; }
    cells += extra;
  }
  // float32 rasters with a no-data value and no threshold (the usual case): the activity
  // test and the predicated updates spelled out -- FSETP + 2 (+ F2F/DADD for the sum) or
  // + 1 FMNMX per extreme; the compiler's own selection for `take` needs about twice that
  __device__ __forceinline__ void take_f32(float v) {
    const float nd = (float)active.nodata;
    float lo = (float)vmin, hi = (float)vmax, vm = 0.0f;
    if (NEED == ZW_SUM) {
      asm("{\n\t.reg .pred p;\n\t"
          "setp.neu.f32 p, %2, %3;\n\t"
          "selp.f32 %0, %2, 0f00000000, p;\n\t"
          "@p add.s32 %1, %1, 1;\n\t}"
          : "=f"(vm), "+r"(count) : "f"(v), "f"(nd));
    } else if (NEED == ZW_MIN) {
      asm("{\n\t.reg .pred p;\n\t"
          "setp.neu.f32 p, %2, %3;\n\t"
          "@p min.f32 %0, %0, %2;\n\t"
          "@p add.s32 %1, %1, 1;\n\t}"
          : "+f"(lo), "+r"(count) : "f"(v), "f"(nd));
    } else if (NEED == ZW_MAX) {
      asm("{\n\t.reg .pred p;\n\t"
          "setp.neu.f32 p, %2, %3;\n\t"
          "@p max.f32 %0, %0, %2;\n\t"
          "@p add.s32 %1, %1, 1;\n\t}"
          : "+f"(hi), "+r"(count) : "f"(v), "f"(nd));
    } else {
      asm("{\n\t.reg .pred p;\n\t"
          "setp.neu.f32 p, %4, %5;\n\t"
          "selp.f32 %0, %4, 0f00000000, p;\n\t"
          "@p min.f32 %1, %1, %4;\n\t"
          "@p max.f32 %2, %2, %4;\n\t"
          "@p add.s32 %3, %3, 1;\n\t}"
          : "=f"(vm), "+f"(lo), "+f"(hi), "+r"(count) : "f"(v), "f"(nd));
    }
    if (NEED & ZW_SUM) sum += (Sum)vm;
    if (NEED & ZW_MIN) vmin = (T)lo;
    if (NEED & ZW_MAX) vmax = (T)hi;
  }
  // ZW_ROWS consecutive single-span rows y0.. are walked as one batch.  `tab` is the warp's
  // shared row table (see the kernel): per row x0 / xe = the span [x0, xe) and xh / xt = its
  // part [xh, xt) made of whole, 16-byte aligned quads.  The quads are read with one 16-byte
  // load per lane and need no position test; the at most 2 (VEC - 1) cells per row in front
  // of and behind them are read by one lane each, in the same round of loads.  `issue` only
  // starts the loads of a batch, `consume` reduces them: the kernel issues batch i + 1
  // before it consumes batch i, so every warp computes under its own loads.
  static constexpr int PER = 2 * (VEC - 1);                     // edge cells per row at most
  struct Batch { Quad q[ZW_ROWS]; T edge; };
  __device__ __forceinline__ bool edge_cell(int y0, const int* tab, int i, int64_t* at) const {
    const int b = i / PER, c = i - b * PER;
    const bool head = c < VEC - 1;
    const int bb = b < ZW_ROWS ? b : 0;
    const int x0 = tab[bb], xe = tab[32 + bb], xh = tab[64 + bb], xt = tab[96 + bb];
    const int x = (head ? x0 + c : xt + c - (VEC - 1));
    *at = (int64_t)(y0 + bb) * width + x;
    return i < ZW_ROWS * PER && x < (head ? min(xh, xe) : xe);
  }
  __device__ __forceinline__ void issue(int y0, const int* tab, Batch& B) const {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int b = 0; b < ZW_ROWS; ++b) {
      const int x = tab[64 + b] + VEC * lane;
      B.q[b] = Quad();
      if (x < tab[96 + b])
        B.q[b] = __ldg(reinterpret_cast<const Quad*>(raster + (int64_t)(y0 + b) * width + x));
    }
    int64_t at;
    B.edge = T(0);
    if (edge_cell(y0, tab, lane, &at)) B.edge = __ldg(raster + at);
  }
  template <bool F32_FAST>
  __device__ __forceinline__ void consume(int y0, const int* tab, const Batch& B) {
    const int lane = threadIdx.x & 31;
    int longest = 0;
#pragma unroll
    for (int b = 0; b < ZW_ROWS; ++b) {
      const int x = tab[64 + b] + VEC * lane, xt = tab[96 + b];
      longest = max(longest, xt - tab[64 + b]);
      if (x < xt) {
        T e[VEC];
        memcpy(e, &B.q[b], QBYTES);
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
          if constexpr (F32_FAST && std::is_same<T, float>::value) take_f32(e[j]);
          else take(e[j]);
        }
      }
    }
    int64_t at;
    if (edge_cell(y0, tab, lane, &at)) take(B.edge);
    // what one round of loads does not cover: quads beyond the first 32 of a row, edge
    // cells beyond the first 32 of the batch (1-byte rasters)
    if (longest > 32 * VEC) {
      for (int k = 32 * VEC + VEC * lane; k - VEC * lane < longest; k += 32 * VEC) {
#pragma unroll
        for (int b = 0; b < ZW_ROWS; ++b) {
          const int x = tab[64 + b] + k;
          if (x < tab[96 + b]) {
            const Quad q = __ldg(reinterpret_cast<const Quad*>(raster + (int64_t)(y0 + b) * width + x));
            T e[VEC];
            memcpy(e, &q, QBYTES);
#pragma unroll
            for (int j = 0; j < VEC; ++j) take(e[j]);
          }
        }
      }
    }
#pragma unroll 1
    for (int i = 32 + lane; i < ZW_ROWS * PER; i += 32)
      if (edge_cell(y0, tab, i, &at)) take(__ldg(raster + at));
  }
};

// The row table of the batched walk (WarpReduce / WarpSelect issue + consume) for the 32 rows
// base + lane, one per lane, from their crossings (row_crossings: cnt of them in column `lane` of
// `cross`, -1 for a row that needs the generic scanline).  A row that is one span gets its span
// [x0, xe) clipped to the raster and its part [xh, xt) made of whole quads of VEC cells aligned to
// 16 bytes, in lines 0..3 of `cross`; its cells are added to `cells`.  Rows of more spans, and
// rows on the raster's first / last line when a quad could reach outside the array
// (edge_scalar), are handed to scalar.span(y, x0, x1) span by span first, while their raw
// crossings are still there.  Returns the ballot of the generic-scanline rows; *single = the
// ballot of the rows in the table.
template <int VEC, class Scalar>
__device__ __forceinline__ unsigned row_table(const PolyDev& P, int mis, int edge_scalar, int base, int cnt,
                                              int (*cross)[32], long long& cells, unsigned* single,
                                              Scalar& scalar) {
  const int lane = threadIdx.x & 31;
  const int maxx = P.width - 1;
  const int y = base + lane;
  const bool complex_row = cnt < 0;
  const bool edge = edge_scalar && (y == 0 || y == P.height - 1);
  const bool scalar_row = !complex_row && cnt >= 2 && (cnt > 2 || edge);
  int fx0 = 0, fxe = 0, xh = 0, xt = 0;
  if (!complex_row && !scalar_row && cnt == 2) {
    const int xa = cross[0][lane], xb = cross[1][lane];
    if (xa <= maxx && xb > 0 && (xa < 0 ? 0 : xa) < (xb > P.width ? P.width : xb)) {
      fx0 = xa < 0 ? 0 : xa; fxe = xb > P.width ? P.width : xb;
      cells += fxe - fx0;
      const int64_t off = (int64_t)y * P.width + mis;      // element offset from the 16-byte grid
      xh = fx0 + (int)((VEC - ((off + fx0) & (VEC - 1))) & (VEC - 1));
      xt = fxe - (int)((off + fxe) & (VEC - 1));
      if (xt < xh) xt = xh;
    }
  }
  __syncwarp();
  const unsigned complex_mask = __ballot_sync(0xffffffffu, complex_row);
  unsigned scalar_mask = __ballot_sync(0xffffffffu, scalar_row);
  *single = __ballot_sync(0xffffffffu, fx0 < fxe);
  while (scalar_mask) {
    const int r = __ffs(scalar_mask) - 1;
    scalar_mask &= scalar_mask - 1;
    const int c = __shfl_sync(0xffffffffu, cnt, r);
    for (int i = 0; i + 1 < c; i += 2) {
      const int xa = cross[i][r], xb = cross[i + 1][r];
      if (xa <= maxx && xb > 0) {
        const int x0 = xa < 0 ? 0 : xa, x1 = xb - 1 > maxx ? maxx : xb - 1;
        if (x0 <= x1) scalar.span(base + r, x0, x1);
      }
    }
  }
  __syncwarp();
  cross[0][lane] = fx0; cross[1][lane] = fxe; cross[2][lane] = xh; cross[3][lane] = xt;
  __syncwarp();
  return complex_mask;
}

template <typename T, int NEED>
__global__ void __launch_bounds__(32 * ZW_WARPS, ZW_MIN_BLOCKS)
zonal_reduce_warp_kernel(const PolyDev P, const T* __restrict__ raster, T nodata, int has_nodata,
                         const float* __restrict__ thresholds, int mis, int edge_scalar,
                         GmZonalPartial* __restrict__ partial, long long* __restrict__ cells,
                         int* __restrict__ work) {
  // work[0]: length of the deferred list, work[1]: polygon counter, work[2...]: the list
  __shared__ double s_px[ZW_WARPS][ZW_MAXV], s_py[ZW_WARPS][ZW_MAXV];
  __shared__ int s_prev[ZW_WARPS][ZW_MAXV];
  __shared__ __align__(16) int s_cross[ZW_WARPS][ZW_MAXC][32];
  __shared__ int s_buf[ZW_WARPS][ZW_MAXV + 2 * PG_MAX_HSPANS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int maxx = P.width - 1;
  double* px = s_px[warp];
  double* py = s_py[warp];
  int* prev = s_prev[warp];
  int* buf = s_buf[warp];
  int* hbuf = buf + ZW_MAXV;
  WarpReduce<T, NEED> vis;
  vis.raster = raster; vis.width = P.width;
  const bool f32_fast = std::is_same<T, float>::value && has_nodata && thresholds == nullptr;
  // (with an active list the partials of the other polygons were cleared by the caller)
  const int64_t n_work = P.active ? (int64_t)*P.n_active : P.n_polygons;
  for (;;) {
    int64_t p = 0;
    if (lane == 0) {
      p = atomicAdd(work + 1, 1);
      if (P.active && p < n_work) p = P.active[p];
      else if (p >= n_work) p = -1;
    }
    p = __shfl_sync(0xffffffffu, p, 0);
    if (p < 0) break;
    const int64_t r0 = P.poly_offsets[p], r1 = P.poly_offsets[p + 1];
    const int miny = P.miny[p], maxy = P.maxy[p];
    int64_t v0 = 0, v1 = 0;
    if (r1 > r0) { v0 = P.ring_offsets[r0]; v1 = P.ring_offsets[r1]; }
    const int nv = (int)min((int64_t)(ZW_MAXV + 1), v1 - v0);
    vis.active = active_test(nodata, has_nodata, thresholds, p);
    vis.reset();
    bool defer = nv > ZW_MAXV || maxy - miny >= ZW_BIG_ROWS;
    if (!defer && nv > 1 && miny <= maxy) {
      const double wide = stage_polygon(P, r0, r1, v0, nv, px, py, prev, lane);
      defer = wide * (double)(maxy - miny + 1) > (double)ZW_BIG_CELLS;
    }
    if (defer) {
      if (lane == 0) work[2 + atomicAdd(work, 1)] = (int)p;
      continue;
    }
    if (nv == 1) {  // point feature (GDALdllImagePoint): the cell that contains it
      if (miny <= maxy) {
        const int x = clamp_to_int(floor(P.px[v0]));
        if (x >= 0 && x <= maxx) vis.span(miny, x, x);
      }
    } else if (nv > 1) {
      for (int base = miny; base <= maxy; base += 32) {
        const int y = base + lane;
        int cnt = 0;
        if (y <= maxy) cnt = row_crossings(px, py, prev, nv, y, s_cross[warp], lane);
        unsigned single_mask;
        const unsigned complex_mask = row_table<WarpReduce<T, NEED>::VEC>(
            P, mis, edge_scalar, base, cnt, s_cross[warp], vis.cells, &single_mask, vis);
        {
          typename WarpReduce<T, NEED>::Batch A;
          const int* tab = &s_cross[warp][0][0];
          constexpr unsigned BM = (1u << ZW_ROWS) - 1u;
#pragma unroll 1
          for (int rb = 0; rb < 32; rb += ZW_ROWS) {
            if (((single_mask >> rb) & BM) == 0) continue;
            vis.issue(base + rb, tab + rb, A);
            if (f32_fast) vis.template consume<true>(base + rb, tab + rb, A);
            else vis.template consume<false>(base + rb, tab + rb, A);
          }
        }
        unsigned cm = complex_mask;
        while (cm) {
          const int r = __ffs(cm) - 1;
          cm &= cm - 1;
          generic_scanline(P, r0, r1, base + r, ZW_MAXV, buf, hbuf, vis);
        }
        __syncwarp();
      }
    }
    long long count = vis.count;
    double vmin = vis.count > 0 ? (double)vis.vmin : DBL_MAX, vmax = vis.count > 0 ? (double)vis.vmax : -DBL_MAX;
    for (int o = 16; o > 0; o >>= 1) {
      count += __shfl_xor_sync(0xffffffffu, count, o);
      vis.cells += __shfl_xor_sync(0xffffffffu, vis.cells, o);
      if (NEED & ZW_SUM) vis.sum += __shfl_xor_sync(0xffffffffu, vis.sum, o);
      if (NEED & ZW_MIN) vmin = fmin(vmin, __shfl_xor_sync(0xffffffffu, vmin, o));
      if (NEED & ZW_MAX) vmax = fmax(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
    }
    if (lane == 0) {
      partial[p] = GmZonalPartial{count, (double)vis.sum, vmin, vmax};
      cells[p] = vis.cells;
    }
  }
}

__global__ void zonal_finalize_kernel(const GmZonalPartial* __restrict__ partial, int stat,
                                      float* __restrict__ out, int64_t n) {
  const int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (p >= n) return;
  const GmZonalPartial r = partial[p];
  float v = __int_as_float(0x7fc00000);
  if (r.count > 0) {
    switch (stat) {
      case GM_STAT_COUNT: v = (float)(double)r.count; break;
      case GM_STAT_SUM: v = (float)r.sum; break;
      case GM_STAT_MEAN: v = (float)(r.sum / (double)r.count); break;
      case GM_STAT_MIN: v = (float)r.vmin; break;
      case GM_STAT_MAX: v = (float)r.vmax; break;
      default: break;
    }
  }
  out[p] = v;
}

// gather visitor: append the keys of active cells to the polygon's buffer
template <typename T>
struct GatherVisitor {
  typedef typename KeyOf<T>::type K;
  const T* raster; int width; ActiveTest<T> active;
  K* keys; int* cursor; long long capacity;
  __device__ __forceinline__ void put(bool ok, T v) {
    const unsigned m = __ballot_sync(0xffffffffu, ok);
    if (m == 0) return;
    const int lane = threadIdx.x & 31;
    int base = 0;
    if (lane == 0) base = atomicAdd(cursor, __popc(m));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (ok) {
      const long long pos = base + __popc(m & ((1u << lane) - 1u));
      if (pos < capacity) keys[pos] = KeyOf<T>::key(v);
    }
  }
  __device__ __forceinline__ void span(int y, int x0, int x1) {
    const T* row = raster + (int64_t)y * width;
    const int lane = threadIdx.x & 31;
    for (int xb = x0; xb <= x1; xb += 32) {
      const int x = xb + lane;
      T v = T(0);
      bool ok = false;
      if (x <= x1) { v = __ldg(row + x); ok = active(v); }
      put(ok, v);
    }
  }
  __device__ __forceinline__ void hspan(int y, int x0, int x1, const int* buf, int n) {
    const T* row = raster + (int64_t)y * width;
    const int lane = threadIdx.x & 31;
    for (int xb = x0; xb <= x1; xb += 32) {
      const int x = xb + lane;
      T v = T(0);
      bool ok = false;
      if (x <= x1 && !in_pairs(x, buf, n)) { v = __ldg(row + x); ok = active(v); }
      put(ok, v);
    }
  }
};

// PG_BATCH rows x 4 requests in flight, ONE cursor update for the whole batch
template <typename T>
__device__ __forceinline__ void span_batch(GatherVisitor<T>& vis, int n, const int* ys, const int* x0, const int* x1) {
  const int lane = threadIdx.x & 31;
  T v[PG_BATCH][4];
  bool ok[PG_BATCH][4];
#pragma unroll
  for (int b = 0; b < PG_BATCH; ++b) {
    const T* row = vis.raster + (int64_t)(b < n ? ys[b] : 0) * vis.width;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int x = (b < n ? x0[b] : 1) + lane + 32 * k;
      ok[b][k] = b < n && x <= x1[b];
      v[b][k] = ok[b][k] ? __ldg(row + x) : T(0);
    }
  }
  int total = 0, mine[PG_BATCH][4];
#pragma unroll
  for (int b = 0; b < PG_BATCH; ++b)
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      ok[b][k] = ok[b][k] && vis.active(v[b][k]);
      const unsigned m = __ballot_sync(0xffffffffu, ok[b][k]);
      mine[b][k] = total + __popc(m & ((1u << lane) - 1u));
      total += __popc(m);
    }
  int base = 0;
  if (lane == 0 && total > 0) base = atomicAdd(vis.cursor, total);
  base = __shfl_sync(0xffffffffu, base, 0);
#pragma unroll
  for (int b = 0; b < PG_BATCH; ++b)
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (ok[b][k]) {
        const long long pos = base + mine[b][k];
        if (pos < vis.capacity) vis.keys[pos] = KeyOf<T>::key(v[b][k]);
      }
#pragma unroll
  for (int b = 0; b < PG_BATCH; ++b)  // rows longer than 128 cells: the rest
    if (x0[b] + 128 <= x1[b]) vis.span(ys[b], x0[b] + 128, x1[b]);
}

// Keys of ranks rank_lo <= rank_hi <= rank_lo + 1 (0-based) among keys[0..n): MSD radix
// select, 8 bits per level, block-wide.  `keys` is consumed: after every level each warp
// compacts, in place and warp-synchronously, the candidates of its own slice that fall
// into the selected digit, so level L+1 only sweeps what survived level L (a polygon's
// values collapse from n to a few dozen after two levels).  When the two ranks part ways
// at some level, the upper one is the smallest key of the next occupied digit.
template <typename K> struct SelectScratch { int b_lo, b_hi; long long r_lo, r_hi; K min_key; };

__device__ __forceinline__ unsigned atomic_min_key(unsigned* a, unsigned v) { return atomicMin(a, v); }
__device__ __forceinline__ unsigned long long atomic_min_key(unsigned long long* a, unsigned long long v) {
  return atomicMin(a, v);
}

template <typename K>
__device__ void block_select2(K* keys, int n, long long rank_lo, long long rank_hi, K* out_lo, K* out_hi,
                              int* hist, SelectScratch<K>* sc) {
  constexpr int BITS = sizeof(K) * 8;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int slice = (n + nwarps - 1) / nwarps;
  const int begin = min(warp * slice, n);
  int cnt = min(begin + slice, n) - begin;   // candidates left in this warp's slice
  K* mine = keys + begin;
  K prefix = 0, khi = 0;
  bool diverged = false;                     // block-uniform: rank_hi already resolved
  for (int shift = BITS - 8; shift >= 0; shift -= 8) {
    for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0;
    if (threadIdx.x == 0) sc->min_key = ~(K)0;
    __syncthreads();
    for (int i0 = 0; i0 < cnt; i0 += 32) {
      const int i = i0 + lane;
      const bool live = i < cnt;
      const int digit = live ? (int)((mine[i] >> shift) & 0xff) : 256 + lane;
      if (shift == BITS - 8) {
        // first level: a handful of digits (exponents) hold everything -> one add per digit
        const unsigned peers = __match_any_sync(0xffffffffu, digit);
        if (live && lane == __ffs(peers) - 1) atomicAdd(&hist[digit], __popc(peers));
      } else if (live) {
        atomicAdd(&hist[digit], 1);
      }
    }
    __syncthreads();
    if (warp == 0) {  // which digit holds each rank: 8 bins per lane + warp scan
      int local[8], sum = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) { local[j] = hist[lane * 8 + j]; sum += local[j]; }
      int incl = sum;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
      }
      const int excl = incl - sum;
      if (rank_lo >= excl && rank_lo < incl) {
        long long r = rank_lo - excl;
        int j = 0;
        while (r >= local[j]) { r -= local[j]; ++j; }
        sc->b_lo = lane * 8 + j; sc->r_lo = r;
      }
      if (!diverged && rank_hi >= excl && rank_hi < incl) {
        long long r = rank_hi - excl;
        int j = 0;
        while (r >= local[j]) { r -= local[j]; ++j; }
        sc->b_hi = lane * 8 + j; sc->r_hi = r;
      }
    }
    __syncthreads();
    const int b_lo = sc->b_lo;
    rank_lo = sc->r_lo;
    if (!diverged) {
      const int b_hi = sc->b_hi;
      if (b_hi != b_lo) {  // the upper rank leaves the path: smallest key of digit b_hi
        K m = ~(K)0;
        for (int i = lane; i < cnt; i += 32) {
          const K k = mine[i];
          if ((int)((k >> shift) & 0xff) == b_hi && k < m) m = k;
        }
        for (int o = 16; o > 0; o >>= 1) {
          const K other = __shfl_xor_sync(0xffffffffu, m, o);
          m = other < m ? other : m;
        }
        if (lane == 0) atomic_min_key(&sc->min_key, m);
        __syncthreads();
        khi = sc->min_key;
        diverged = true;
      } else {
        rank_hi = sc->r_hi;
      }
    }
    int out = 0;
    for (int i0 = 0; i0 < cnt; i0 += 32) {
      const int i = i0 + lane;
      const bool live = i < cnt;
      const K k = live ? mine[i] : (K)0;
      const bool keep = live && (int)((k >> shift) & 0xff) == b_lo;
      const unsigned m = __ballot_sync(0xffffffffu, keep);
      if (keep) mine[out + __popc(m & ((1u << lane) - 1u))] = k;
      out += __popc(m);
      __syncwarp();
    }
    cnt = out;
    prefix |= (K)b_lo << shift;
    __syncthreads();
  }
  *out_lo = prefix;
  *out_hi = diverged ? khi : prefix;
}

// result of the order statistic in the reference's arithmetic
template <typename T> __device__ __forceinline__ float median_of(T lo, T hi) {
  // scipy.ndimage._measurements._select: integers are averaged in double
  return (float)(((double)lo + (double)hi) / 2.0);
}
template <> __device__ __forceinline__ float median_of<float>(float lo, float hi) { return (lo + hi) / 2.0f; }
template <> __device__ __forceinline__ float median_of<double>(double lo, double hi) { return (float)((lo + hi) / 2.0); }

template <typename T> __device__ __forceinline__ float percentile_of(T lo, T hi, double part) {
  // measurements.py:137: data[lo] + part * (data[hi] - data[lo]); the difference in the data dtype
  const T diff = (T)(hi - lo);
  return (float)((double)lo + part * (double)diff);
}

// the 0-based ranks lo <= hi among n values that the median / q-th percentile combines, and
// the percentile's weight of the upper one (scipy's median; measurements.percentile)
__device__ __forceinline__ void order_ranks(int stat, double q, int n, long long* lo, long long* hi, double* part) {
  *part = 0.0;
  if (stat == GM_STAT_MEDIAN) {
    *lo = (n - 1) / 2; *hi = n / 2;
  } else {
    const double frac = (double)(n - 1) * (q / 100.0);
    *lo = (long long)floor(frac);
    *hi = (long long)ceil(frac);
    *part = frac - floor(frac);
  }
}

// median / percentile of the n keys in `keys` in the reference's arithmetic (block-wide
// call; `keys` is consumed)
template <typename T>
__device__ float order_statistic(typename KeyOf<T>::type* keys, int n, int stat, double q, int* hist,
                                 SelectScratch<typename KeyOf<T>::type>* scratch) {
  typedef typename KeyOf<T>::type K;
  float result = __int_as_float(0x7fc00000);
  if (n > 0) {
    long long lo_rank, hi_rank;
    double part;
    order_ranks(stat, q, n, &lo_rank, &hi_rank, &part);
    K klo, khi;
    block_select2<K>(keys, n, lo_rank, hi_rank, &klo, &khi, hist, scratch);
    const T lo = KeyOf<T>::value(klo), hi = KeyOf<T>::value(khi);
    result = stat == GM_STAT_MEDIAN ? median_of<T>(lo, hi) : percentile_of<T>(lo, hi, part);
  }
  return result;
}

template <typename T>
__global__ void __launch_bounds__(SEL_THREADS, 3)
zonal_select_kernel(const PolyDev P, const T* __restrict__ raster, T nodata, int has_nodata,
                    const float* __restrict__ thresholds, int stat, double q,
                    const long long* __restrict__ area, const long long* __restrict__ big_offset,
                    typename KeyOf<T>::type* __restrict__ big_keys, int smem_capacity,
                    float* __restrict__ out, const int* __restrict__ work, int* __restrict__ too_big) {
  typedef typename KeyOf<T>::type K;
  extern __shared__ __align__(16) unsigned char sel_smem[];
  const int nw = SEL_THREADS / 32;
  int* cross = reinterpret_cast<int*>(sel_smem);
  const int warp = threadIdx.x >> 5;
  int* buf = cross + warp * P.cap;
  int* hbuf = cross + nw * P.cap + warp * 2 * PG_MAX_HSPANS;
  K* smem_keys = reinterpret_cast<K*>(sel_smem + ((size_t)(nw * P.cap + nw * 2 * PG_MAX_HSPANS) * sizeof(int) + 15) / 16 * 16);
  __shared__ int hist[256];
  __shared__ SelectScratch<K> select_scratch;
  __shared__ int cursor;
  const int n_listed = work[0];
  for (int item = blockIdx.x; item < n_listed; item += gridDim.x) {
    const int64_t p = work[2 + item];
    const long long a = area[p];
    if (a > smem_capacity && big_keys == nullptr) {   // optimistic launch without global key segments:
      if (threadIdx.x == 0) *too_big = 1;             // the host repeats the listed polygons with them
      continue;
    }
    K* keys = a <= smem_capacity ? smem_keys : big_keys + big_offset[p];
    if (threadIdx.x == 0) cursor = 0;
    __syncthreads();
    GatherVisitor<T> vis;
    vis.raster = raster; vis.width = P.width;
    vis.active = active_test(nodata, has_nodata, thresholds, p);
    vis.keys = keys; vis.cursor = &cursor; vis.capacity = a;
    scan_polygon(P, p, buf, hbuf, vis);
    __threadfence_block();
    __syncthreads();
    const int n = cursor;
    const float result = order_statistic<T>(keys, n, stat, q, hist, &select_scratch);
    if (threadIdx.x == 0) out[p] = result;
    __syncthreads();
  }
}

// 32-bit sortable keys of the dtypes the streaming select takes (float32 and integers up to 4 bytes)
template <typename T> struct Key32 {
  static __device__ __forceinline__ unsigned key(T v) {
    return std::is_signed<T>::value ? ((unsigned)(int)v ^ 0x80000000u) : (unsigned)v;
  }
  static __device__ __forceinline__ T value(unsigned k) {
    return std::is_signed<T>::value ? (T)(int)(k ^ 0x80000000u) : (T)k;
  }
};
template <> struct Key32<float> {
  static __device__ __forceinline__ unsigned key(float v) { return order_f32(v); }
  static __device__ __forceinline__ float value(unsigned k) { return unorder_f32(k); }
};

// ---- order statistics, one WARP per polygon (streaming select) -----------------------------------
// The usual polygon (<= ZW_MAXV vertices, <= ZW_BIG_ROWS rows, bounding box <= ZW_BIG_CELLS cells,
// rasters of up to 4 bytes per cell) is selected by ONE warp that streams it from the raster -- no
// block barrier, no shared key space, polygons fetched from an atomic counter like
// zonal_reduce_warp_kernel:
//   1. sample: every 16th row (lane = sample row, single-span rows only) is swept with scalar
//      loads, two rows in flight: range of the sampled keys, then a 256-bin histogram of the range
//      that is refined while the bins around the wanted rank still hold > 20 % of the sample.  The
//      bins that hold the sample ranks q * n_s -+ (3 sigma + 2) give a BRACKET [lo, hi] of keys;
//   2. main pass: the row walk of the reduce kernel (16-byte loads of whole aligned quads, edge cells
//      by one lane each).  Per cell, compared as VALUES (same order as the keys): count it, count it
//      as `below` when it is under the bracket, and when it lies in the bracket append it to the
//      lane's own column of a scratch table in global memory (a few dozen cells per lane, L2
//      resident) -- ten instructions per cell.  When the bracket spans < 256 distinct keys (byte
//      rasters, classes, constant areas) the cells go to an exact histogram instead;
//   3. the wanted ranks, now known from the exact count, are looked up among the bracket's keys:
//      256-bin histogram of the bracket, the bin of the rank, its <= 32 keys ranked by the lanes
//      (further levels while a bin holds more; at shift 0 a bin is one key).
// Small polygons (bounding box <= WS_DIRECT cells) skip the sample: every cell is "in the bracket".
// A polygon whose ranks fall outside the bracket (the sample misjudged the distribution) or whose
// bracket overflows a lane's column joins the deferred list for zonal_select_kernel, like the
// polygons this kernel does not take at all.  Results are bit-identical to the generic path: the
// same two keys are found, only by another route.
constexpr int WS_WARPS = 8;
constexpr int WS_MIN_BLOCKS = 4;
constexpr int WS_MAIN_BLOCKS = 3;        // the main kernel holds two batches of loads: 85 registers
constexpr int WS_CAP = 128;              // cells per lane in the scratch table ([slot][lane] per warp)
constexpr int WS_ROOM = 20;              // free slots a lane needs before a round of loads (<= 17 cells)
constexpr int WS_BINS = 1024;             // histogram bins per warp (dynamic shared memory)
constexpr int WS_BITS = 10;
constexpr int WS_DIRECT = 1536;          // bounding-box cells up to which every cell is kept
constexpr int WS_SAMPLE_STRIDE = 16;     // every 16th row is sampled
enum { WS_SAMPLE_RANGE = 0, WS_SAMPLE_HIST = 1, WS_MAIN_STASH = 2, WS_MAIN_HIST = 3 };

__device__ __forceinline__ void red_shared_inc(unsigned addr, bool p) {
  asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %1, 0;\n\t@q red.shared.add.u32 [%0], 1;\n\t}"
               :: "r"(addr), "r"((unsigned)p) : "memory");
}
__device__ __forceinline__ void store_if(unsigned* at, unsigned word, bool p) {
  asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %2, 0;\n\t@q st.global.u32 [%0], %1;\n\t}"
               :: "l"(at), "r"(word), "r"((unsigned)p) : "memory");
}

// bin of the warp's WS_BINS-entry table that holds the 0-based rank r, entries before it and
// entries in it; -1 when r is not below the table's total.  Warp-wide call.
__device__ __noinline__ int warp_find_bin(const int* hist, long long r, int* before, int* inside, int lane) {
  constexpr int PERL = WS_BINS / 32;
  const int4* mine4 = reinterpret_cast<const int4*>(hist) + (PERL / 4) * lane;
  int sum = 0;
#pragma unroll
  for (int j = 0; j < PERL / 4; ++j) { const int4 a = mine4[j]; sum += a.x + a.y + a.z + a.w; }
  int incl = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  const int excl = incl - sum;
  const bool mine = r >= excl && r < incl;
  const unsigned m = __ballot_sync(0xffffffffu, mine);
  if (m == 0) return -1;
  int bin = -1, e = 0, c = 0;
  if (mine) {
    int left = (int)(r - excl);
    e = excl;
    for (int j = 0; j < PERL; ++j) {
      const int h = hist[PERL * lane + j];
      if (left < h) { bin = PERL * lane + j; c = h; break; }
      left -= h; e += h;
    }
  }
  const int src = __ffs(m) - 1;
  *before = __shfl_sync(0xffffffffu, e, src);
  *inside = __shfl_sync(0xffffffffu, c, src);
  return __shfl_sync(0xffffffffu, bin, src);
}

// what a kept cell looks like in the scratch table: the raw bits of a float (the key is formed
// when the table is read), the key of an integer
template <typename T> struct StashWord {
  static __device__ __forceinline__ unsigned word(T v) { return Key32<T>::key(v); }
  static __device__ __forceinline__ unsigned key(unsigned w) { return w; }
};
template <> struct StashWord<float> {
  static __device__ __forceinline__ unsigned word(float v) { return __float_as_uint(v); }
  static __device__ __forceinline__ unsigned key(unsigned w) { return order_f32(__uint_as_float(w)); }
};

template <typename T>
struct WarpSelect {
  static constexpr int VEC = 4;
  typedef typename std::conditional<sizeof(T) == 4, uint4,
          typename std::conditional<sizeof(T) == 2, uint2, unsigned>::type>::type Quad;
  const T* raster; int width; T nodata; bool no_nodata;
  T vlo, vhi;               // the bracket as values: vlo <= v <= vhi
  unsigned lo, span;        // ... and as keys: key - lo <= span
  int shift;                // sample histogram: bin = (key - lo) >> shift
  unsigned hist_at;         // shared-memory address of this warp's 256 bins
  unsigned* column;         // this lane's column of the warp's scratch table (stride 32)
  int n_active, below, cnt; // per lane
  long long cells;
  unsigned kmin, kmax;
  float fmin_, fscale;      // float32 sample histogram: bin = (v - fmin_) * fscale (linear in the value)

  // the cell of the main pass when the bracket's cells are kept: count it, count it as below,
  // keep it -- nine instructions for float32 (predicated adds and store spelled out; the
  // compiler's own selection needs fifteen).  `fill` = the cell may be a filler that carries the
  // no-data value (lanes without a quad), which needs no test of its own.
  __device__ __forceinline__ void keep(T v, bool ok) {
    if constexpr (std::is_same<T, float>::value) {
      unsigned* at = column + (unsigned)cnt * 32u;
      asm volatile("{\n\t.reg .pred pa, pb, pi;\n\t"
                   "setp.ne.u32 pa, %7, 0;\n\t"
                   "setp.neu.and.f32 pa, %4, %5, pa;\n\t"   // active: a real cell that is not no data
                   "setp.lt.and.f32 pb, %4, %6, pa;\n\t"    // below the bracket
                   "setp.ge.and.f32 pi, %4, %6, pa;\n\t"
                   "setp.le.and.f32 pi, %4, %8, pi;\n\t"    // in the bracket
                   "@pa add.s32 %0, %0, 1;\n\t"
                   "@pb add.s32 %1, %1, 1;\n\t"
                   "@pi st.global.b32 [%3], %9;\n\t"
                   "@pi add.s32 %2, %2, 1;\n\t}"
                   : "+r"(n_active), "+r"(below), "+r"(cnt)
                   : "l"(at), "f"(v), "f"(no_nodata ? __int_as_float(0x7fc00000) : nodata), "f"(vlo),
                     "r"((unsigned)ok), "f"(vhi), "r"(__float_as_uint(v))
                   : "memory");
    } else {
      const bool active = ok & (no_nodata | (v != nodata));
      const bool in = active & (v >= vlo) & (v <= vhi);
      n_active += active ? 1 : 0;
      below += (active & (v < vlo)) ? 1 : 0;
      store_if(column + (unsigned)cnt * 32u, StashWord<T>::word(v), in);
      cnt += in ? 1 : 0;
    }
  }
  // any mode, chosen at run time (the sample sweeps and the rows the table cannot describe)
  __device__ __forceinline__ void take(int mode, T v, bool ok) {
    if (mode == WS_MAIN_STASH) { keep(v, ok); return; }
    const bool active = ok & (no_nodata | (v != nodata));
    const unsigned key = Key32<T>::key(v), rel = key - lo;
    if (mode == WS_SAMPLE_RANGE) {
      n_active += active ? 1 : 0;
      kmin = min(kmin, active ? key : 0xffffffffu);
      kmax = max(kmax, active ? key : 0u);
    } else {
      if (mode == WS_MAIN_HIST) n_active += active ? 1 : 0;
      below += (active & (key < lo)) ? 1 : 0;
      red_shared_inc(hist_at + ((rel >> shift) << 2), active & (rel <= span));
    }
  }
  // a lane's column is about to overflow: close the bracket (nothing is kept any more; the
  // polygon is deferred when the pass is over because cnt stays above the capacity)
  __device__ __forceinline__ void room() {
    if (__any_sync(0xffffffffu, cnt > WS_CAP - WS_ROOM)) {
      cnt = WS_CAP + 1; vlo = std::numeric_limits<T>::max(); vhi = std::numeric_limits<T>::lowest();
    }
  }
  // one batch of ZW_ROWS single-span rows of the row table (see WarpReduce) in the main pass:
  // whole aligned quads with one 16/8/4-byte load per lane and row, the edge cells (at most
  // VEC - 1 either side of a row) by lanes 8 b + c of row b.  The quad a lane takes is rotated
  // from row to row so that narrow polygons fill all columns evenly.  `issue` starts the loads,
  // `consume` takes the cells: the kernel issues two batches before it consumes the first.
  struct Batch { Quad qd[ZW_ROWS]; T edge; unsigned has; int longest; };
  __device__ __forceinline__ void issue(int y0, const int* tab, Batch& B) const {
    const int lane = threadIdx.x & 31;
    const T filler = no_nodata ? T(0) : nodata;
    Quad fillq;
    {
      T f[VEC];
#pragma unroll
      for (int j = 0; j < VEC; ++j) f[j] = filler;
      memcpy(&fillq, f, sizeof(Quad));
    }
    B.has = 0u; B.longest = 0;
#pragma unroll
    for (int b = 0; b < ZW_ROWS; ++b) {
      const int xh = tab[64 + b], xt = tab[96 + b];
      const int x = xh + VEC * ((lane + 7 * (y0 + b)) & 31);
      B.longest = max(B.longest, xt - xh);
      B.qd[b] = fillq;
      if (x < xt) {
        B.has |= 1u << b;
        B.qd[b] = __ldg(reinterpret_cast<const Quad*>(raster + (int64_t)(y0 + b) * width + x));
      }
    }
    // edge cells: lane = 8 * row + c, c < 3 in front of the quads, 3 <= c < 6 behind them
    const int eb = lane >> 3, ec = lane & 7;
    const bool head = ec < VEC - 1;
    const int ex = head ? tab[eb] + ec : tab[96 + eb] + ec - (VEC - 1);
    B.edge = filler;
    if (ec < 2 * (VEC - 1) && ex < (head ? min(tab[64 + eb], tab[32 + eb]) : tab[32 + eb])) {
      B.has |= 1u << 8;
      B.edge = __ldg(raster + (int64_t)(y0 + eb) * width + ex);
    }
  }
  template <bool EXACT> __device__ __forceinline__ void consume(int y0, const int* tab, const Batch& B) {
    const int lane = threadIdx.x & 31;
    if (!EXACT) room();
    // with a no-data value the fillers are inactive by themselves; without one they need `ok`
#pragma unroll
    for (int b = 0; b < ZW_ROWS; ++b) {
      T e[VEC];
      memcpy(e, &B.qd[b], sizeof(Quad));
      const bool ok = ((B.has >> b) & 1u) | !no_nodata;
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        if (EXACT) take(WS_MAIN_HIST, e[j], ok);
        else keep(e[j], ok);
      }
    }
    if (EXACT) take(WS_MAIN_HIST, B.edge, ((B.has >> 8) & 1u) | !no_nodata);
    else keep(B.edge, ((B.has >> 8) & 1u) | !no_nodata);
    if (B.longest > 32 * VEC) {   // rows of more than 32 quads: the rest
      const T filler = no_nodata ? T(0) : nodata;
      for (int k = 32 * VEC + VEC * lane; k - VEC * lane < B.longest; k += 32 * VEC) {
        if (!EXACT) room();
#pragma unroll 1
        for (int b = 0; b < ZW_ROWS; ++b) {
          const int x = tab[64 + b] + k;
          const bool ok = x < tab[96 + b];
          T e[VEC];
#pragma unroll
          for (int j = 0; j < VEC; ++j) e[j] = filler;
          if (ok) {
            const Quad qv = __ldg(reinterpret_cast<const Quad*>(raster + (int64_t)(y0 + b) * width + x));
            memcpy(e, &qv, sizeof(Quad));
          }
#pragma unroll
          for (int j = 0; j < VEC; ++j) take(EXACT ? WS_MAIN_HIST : WS_MAIN_STASH, e[j], ok);
        }
      }
    }
  }
};

// cells x0..x1 of row y, lane per cell, four loads in flight; any mode.  Not inlined: the rows
// the table cannot describe and the tails of very long sample rows are rare, and the kernel has
// to stay small enough for the instruction cache (32 warps per SM in different phases).
template <typename T>
__device__ __noinline__ void select_span(WarpSelect<T>& w, int mode, int y, int x0, int x1) {
  const T* row = w.raster + (int64_t)y * w.width;
  const int lane = threadIdx.x & 31;
  for (int x = x0 + lane; x - lane <= x1; x += 128) {
    if (mode == WS_MAIN_STASH) w.room();
    T v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) v[k] = x + 32 * k <= x1 ? __ldg(row + x + 32 * k) : T(0);
#pragma unroll
    for (int k = 0; k < 4; ++k) w.take(mode, v[k], x + 32 * k <= x1);
  }
}

// sample sweep: rows y0 + r * stride of the table (x0 in tab[r], end in tab[32 + r]), two rows
// and four cells per lane and row in flight.  RANGE: smallest / largest key and the number of
// active cells; HIST: bins of (key - lo) >> shift and the number of keys below lo.
template <typename T, int MODE>
__device__ __noinline__ void select_sample(WarpSelect<T>& w, int n_rows, const int* tab, int y0, int stride) {
  constexpr bool F = std::is_same<T, float>::value;   // float32: bins linear in the value, not the key
  const int lane = threadIdx.x & 31;
  const T nodata = w.nodata;
  const bool no_nodata = w.no_nodata;
  const unsigned lo = w.lo, span = w.span, hist_at = w.hist_at;
  const int shift = w.shift;
  const float f0 = w.fmin_, fs = w.fscale;
  int count = 0;
  unsigned kmin = 0xffffffffu, kmax = 0u;
  float vmin = INFINITY, vmax = -INFINITY;
  for (int r = 0; r < n_rows; r += 2) {
    T v[2][4];
    bool ok[2][4];
#pragma unroll
    for (int b = 0; b < 2; ++b) {
      const int rr = r + b < n_rows ? r + b : r;
      const int x0 = tab[rr], xe = r + b < n_rows ? tab[32 + rr] : 0;
      const T* row = w.raster + (int64_t)(y0 + rr * stride) * w.width + x0 + lane;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        ok[b][k] = x0 + lane + 32 * k < xe;
        v[b][k] = ok[b][k] ? __ldg(row + 32 * k) : T(0);
      }
    }
#pragma unroll
    for (int b = 0; b < 2; ++b)
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const bool active = ok[b][k] & (no_nodata | (v[b][k] != nodata));
        if constexpr (F) {
          const float x = (float)v[b][k];
          if (MODE == WS_SAMPLE_RANGE) {
            count += active ? 1 : 0;
            vmin = fminf(vmin, active ? x : INFINITY);      // (NaN cells leave the range alone)
            vmax = fmaxf(vmax, active ? x : -INFINITY);
          } else {
            const float rel = (x - f0) * fs;                  // NaN for NaN cells: neither below nor in a bin
            count += (active & (rel < 0.0f)) ? 1 : 0;
            const int bin = min((int)rel, WS_BINS - 1);
            red_shared_inc(hist_at + ((unsigned)bin << 2), active & (rel >= 0.0f) & (rel < (float)WS_BINS + 0.5f));
          }
        } else {
          const unsigned key = Key32<T>::key(v[b][k]);
          if (MODE == WS_SAMPLE_RANGE) {
            count += active ? 1 : 0;
            kmin = min(kmin, active ? key : 0xffffffffu);
            kmax = max(kmax, active ? key : 0u);
          } else {
            const unsigned rel = key - lo;
            count += (active & (key < lo)) ? 1 : 0;
            red_shared_inc(hist_at + ((rel >> shift) << 2), active & (rel <= span));
          }
        }
      }
  }
  if (MODE == WS_SAMPLE_RANGE) {
    w.n_active = count;
    if constexpr (F) { w.kmin = __float_as_uint(vmin); w.kmax = __float_as_uint(vmax); }
    else { w.kmin = kmin; w.kmax = kmax; }
  } else {
    w.below = count;
  }
  // (rows of more than 128 cells: their first 128 cells are the sample)
}

// visitor of the generic scanline for the rows the table cannot describe
template <typename T>
struct WarpSelectVisitor {
  WarpSelect<T>& w;
  int mode;
  __device__ __forceinline__ void span(int y, int x0, int x1) {
    if ((threadIdx.x & 31) == 0) w.cells += x1 - x0 + 1;
    select_span(w, mode, y, x0, x1);
  }
  __device__ __forceinline__ void hspan(int y, int x0, int x1, const int* buf, int n) {
    const T* row = w.raster + (int64_t)y * w.width;
    int extra = 0;
    for (int xb = x0; xb <= x1; xb += 32) {
      if (mode == WS_MAIN_STASH) w.room();
      const int x = xb + (threadIdx.x & 31);
      const bool ok = x <= x1 && !in_pairs(x, buf, n);
      w.take(mode, ok ? __ldg(row + x) : T(0), ok);
      extra += ok ? 1 : 0;
    }
    w.cells += extra;
  }
};

template <typename T>
__device__ __noinline__ void select_complex_row(const PolyDev& P, int64_t r0, int64_t r1, int y, int* buf,
                                                int* hbuf, WarpSelect<T>& w, int mode) {
  WarpSelectVisitor<T> vis{w, mode};
  generic_scanline(P, r0, r1, y, ZW_MAXV, buf, hbuf, vis);
}

// The select runs as THREE kernels, each a loop of warps over polygons (atomic counter) that
// executes ONE phase: with all phases in a single kernel the 32 warps of an SM sat in different
// parts of ~100 KB of code and 40-55 % of the issue slots were lost to instruction-cache misses
// (ncu r02c); split, every kernel's hot loop fits the instruction cache.
//   bracket kernel   sample -> state[p] = (lo, hi, what to do)
//   main kernel      the pass over all cells -> counts + the bracket's cells in the polygon's table
//                    (polygons with an exact histogram are finished here)
//   final kernel     ranks among the table's cells -> out[p]
// Polygons are processed in chunks of at most 131072 (GM_SELECT_CHUNK) so that the tables
// (WS_CAP x 32 words + 32 counts each, 2.2 GB per chunk) stay bounded; cfg4 is one chunk -- with
// four chunks of 32768 the tails of twelve launches cost 0.3 ms of 3.3.
enum { WS_SKIP = 0, WS_TABLE = 1, WS_EXACT = 2 };
struct SelectState { unsigned lo, hi; int what; int n_active; int below; int kept; };
constexpr int WS_TABLE_WORDS = WS_CAP * 32 + 32;     // cells + per-lane counts

#define WS_SHARED_TABLES                                                              \
  __shared__ double s_px[WS_WARPS][ZW_MAXV], s_py[WS_WARPS][ZW_MAXV];                 \
  __shared__ int s_prev[WS_WARPS][ZW_MAXV];                                           \
  __shared__ __align__(16) int s_cross[WS_WARPS][ZW_MAXC][32];                        \
  extern __shared__ __align__(16) int ws_hist[];        /* WS_WARPS x WS_BINS */      \
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;                         \
  double* px = s_px[warp];                                                            \
  double* py = s_py[warp];                                                            \
  int* prev = s_prev[warp];                                                           \
  int* hist = ws_hist + warp * WS_BINS;                                               \
  int (*cross)[32] = s_cross[warp];                                                   \
  const int* tab = &s_cross[warp][0][0];                                              \
  auto zero_hist = [&]() {                                                            \
    __syncwarp();                                                                     \
    _Pragma("unroll")                                                                 \
    for (int j = 0; j < WS_BINS / 32; ++j) hist[j * 32 + lane] = 0;                   \
    __syncwarp();                                                                     \
  };

template <typename T>
__global__ void __launch_bounds__(32 * WS_WARPS, WS_MIN_BLOCKS)
zonal_select_bracket_kernel(const PolyDev P, const T* __restrict__ raster, T nodata, int has_nodata,
                            int stat, double q, int64_t p_begin, int64_t p_end, int* __restrict__ counter,
                            SelectState* __restrict__ state, float* __restrict__ out,
                            long long* __restrict__ area, int* __restrict__ work) {
  // work[0]: length of the deferred list, work[2...]: the list
  WS_SHARED_TABLES
  const int maxx = P.width - 1;
  WarpSelect<T> w;
  w.raster = raster; w.width = P.width; w.nodata = nodata; w.no_nodata = !has_nodata;
  w.hist_at = (unsigned)__cvta_generic_to_shared(hist);
  w.column = nullptr;
  const double qf = stat == GM_STAT_MEDIAN ? 0.5 : q / 100.0;
  for (;;) {
    int64_t p = 0;
    if (lane == 0) p = p_begin + atomicAdd(counter, 1);
    p = __shfl_sync(0xffffffffu, p, 0);
    if (p >= p_end) break;
    const int64_t r0 = P.poly_offsets[p], r1 = P.poly_offsets[p + 1];
    const int miny = P.miny[p], maxy = P.maxy[p];
    int64_t v0 = 0, v1 = 0;
    if (r1 > r0) { v0 = P.ring_offsets[r0]; v1 = P.ring_offsets[r1]; }
    const int nv = (int)min((int64_t)(ZW_MAXV + 1), v1 - v0);
    const int nrows = maxy - miny + 1;
    if (nrows <= 0 || nv == 0) {     // no rows here (another stripe, outside the raster)
      if (lane == 0) { out[p] = __int_as_float(0x7fc00000); area[p] = 0; state[p].what = WS_SKIP; }
      continue;
    }
    bool defer = nv > ZW_MAXV || nv < 2 || nrows > ZW_BIG_ROWS;
    double boxw = 0.0;
    if (!defer) {
      boxw = fmax(stage_polygon(P, r0, r1, v0, nv, px, py, prev, lane), 0.0) + 1.0;
      defer = boxw * (double)nrows > (double)ZW_BIG_CELLS;
    }
    if (defer) {
      if (lane == 0) { work[2 + atomicAdd(work, 1)] = (int)p; state[p].what = WS_SKIP; }
      continue;
    }
    unsigned lo = 0u, hi = 0xffffffffu;
    if (sizeof(T) == 1) {
      hi = 255u;                       // byte rasters: an exact histogram of all keys, no sample
    } else if (boxw * (double)nrows > (double)WS_DIRECT) {
      const int stride = max(WS_SAMPLE_STRIDE, (nrows + 31) / 32);
      const int n_sr = (nrows + stride - 1) / stride;          // <= 32 sample rows, one per lane
      int sx0 = 0, sxe = 0;
      if (lane < n_sr) {
        const int y = miny + lane * stride;
        const int c = row_crossings_call(px, py, prev, nv, y, cross, lane);
        if (c == 2) {
          const int xa = cross[0][lane], xb = cross[1][lane];
          if (xa <= maxx && xb > 0) { sx0 = xa < 0 ? 0 : xa; sxe = xb > P.width ? P.width : xb; }
        }
      }
      __syncwarp();
      cross[0][lane] = sx0; cross[1][lane] = sxe;
      __syncwarp();
      // pass 0: range of the sampled keys; passes 1..: histograms of the bracket so far, until the
      // bins around the wanted ranks hold little more than the ranks' own margin
      int n_s = 0;
      long long ra = 0, rb = 0;
      bool open_lo = true, open_hi = true, usable = false;
      unsigned blo = 0u, bhi = 0xffffffffu;
      float vlo_s = 0.0f, vhi_s = 0.0f;      // float32: the bracket as values
      int sh = 0;
      for (int pass = 0; pass < 5; ++pass) {
        if (pass == 0) {
          select_sample<T, WS_SAMPLE_RANGE>(w, n_sr, tab, miny, stride);
          n_s = __reduce_add_sync(0xffffffffu, w.n_active);
          if constexpr (std::is_same<T, float>::value) {
            vlo_s = __uint_as_float(w.kmin); vhi_s = __uint_as_float(w.kmax);
            for (int o = 16; o > 0; o >>= 1) {
              vlo_s = fminf(vlo_s, __shfl_xor_sync(0xffffffffu, vlo_s, o));
              vhi_s = fmaxf(vhi_s, __shfl_xor_sync(0xffffffffu, vhi_s, o));
            }
          } else {
            blo = __reduce_min_sync(0xffffffffu, w.kmin);
            bhi = __reduce_max_sync(0xffffffffu, w.kmax);
          }
          if (n_s < 32) break;
          if (std::is_same<T, float>::value && !(vhi_s - vlo_s < INFINITY)) break;   // range not finite
          usable = true;
          const double fs = qf * (double)(n_s - 1);
          const double margin = 3.0 * sqrt(qf * (1.0 - qf) * (double)n_s) + 2.0;
          ra = (long long)floor(fs - margin); rb = (long long)ceil(fs + margin);
          open_lo = ra <= 0; open_hi = rb >= n_s - 1;
          ra = max(ra, 0LL); rb = min(rb, (long long)n_s - 1);
          continue;
        }
        zero_hist();
        float width = 0.0f;
        if constexpr (std::is_same<T, float>::value) {
          width = vhi_s - vlo_s;
          if (!(width > 0.0f)) break;                       // one value: the bracket is that value
          w.fmin_ = vlo_s; w.fscale = (float)WS_BINS / width;
        } else {
          const unsigned range = bhi - blo;
          sh = max(32 - __clz(range) - WS_BITS, 0);
          w.lo = blo; w.span = range; w.shift = sh;
        }
        select_sample<T, WS_SAMPLE_HIST>(w, n_sr, tab, miny, stride);
        const int below_s = __reduce_add_sync(0xffffffffu, w.below);
        __syncwarp();
        int ea = 0, ca = 0, eb = 0, cb = 0;
        const int ba = warp_find_bin(hist, ra - below_s, &ea, &ca, lane);
        const int bb = warp_find_bin(hist, rb - below_s, &eb, &cb, lane);
        if (ba < 0 || bb < 0) break;   // cannot happen (the ranks lie in the bracket); keep the bracket
        const long long wanted = rb - ra + 1, got = (long long)(eb + cb - ea);
        if constexpr (std::is_same<T, float>::value) {
          // one bin of slack either side covers the rounding of the bin arithmetic
          const float step = width / (float)WS_BINS;
          const float nlo = fmaxf(vlo_s, vlo_s + step * (float)(ba - 1));
          const float nhi = fminf(vhi_s, vlo_s + step * (float)(bb + 2));
          const bool narrower = nhi - nlo < 0.5f * width;
          vlo_s = nlo; vhi_s = nhi;
          if (!narrower || 3 * (got - wanted) <= wanted) break;
        } else {
          const unsigned long long top = (unsigned long long)blo + ((unsigned long long)(bb + 1) << sh) - 1ULL;
          const unsigned nhi = top < (unsigned long long)bhi ? (unsigned)top : bhi;
          blo = blo + ((unsigned)ba << sh);
          bhi = nhi;
          if (sh == 0 || 3 * (got - wanted) <= wanted) break;
        }
      }
      if constexpr (std::is_same<T, float>::value) {
        blo = order_f32(vlo_s); bhi = order_f32(vhi_s);
      }
      if (usable) {
        lo = open_lo ? 0u : blo;
        hi = open_hi ? 0xffffffffu : bhi;
      }
      __syncwarp();
    }
    // few distinct keys in the bracket: an exact histogram instead of the table
    if (lane == 0) {
      state[p].lo = lo; state[p].hi = hi;
      state[p].what = hi - lo < (unsigned)WS_BINS ? WS_EXACT : WS_TABLE;
    }
  }
}

template <typename T>
__global__ void __launch_bounds__(32 * WS_WARPS, WS_MAIN_BLOCKS)
zonal_select_main_kernel(const PolyDev P, const T* __restrict__ raster, T nodata, int has_nodata,
                         int mis, int edge_scalar, int stat, double q, int64_t p_begin, int64_t p_end,
                         int* __restrict__ counter, SelectState* __restrict__ state,
                         unsigned* __restrict__ tables, float* __restrict__ out,
                         long long* __restrict__ area, int* __restrict__ work) {
  WS_SHARED_TABLES
  __shared__ int s_buf[WS_WARPS][ZW_MAXV + 2 * PG_MAX_HSPANS];
  int* buf = s_buf[warp];
  int* hbuf = buf + ZW_MAXV;
  WarpSelect<T> w;
  w.raster = raster; w.width = P.width; w.nodata = nodata; w.no_nodata = !has_nodata;
  w.hist_at = (unsigned)__cvta_generic_to_shared(hist);
  for (;;) {
    int64_t p = 0;
    if (lane == 0) p = p_begin + atomicAdd(counter, 1);
    p = __shfl_sync(0xffffffffu, p, 0);
    if (p >= p_end) break;
    const int what = state[p].what;
    if (what == WS_SKIP) continue;
    const unsigned lo = state[p].lo, hi = state[p].hi;
    const int64_t r0 = P.poly_offsets[p], r1 = P.poly_offsets[p + 1];
    const int miny = P.miny[p], maxy = P.maxy[p];
    const int64_t v0 = P.ring_offsets[r0];
    const int nv = (int)(P.ring_offsets[r1] - v0);
    stage_polygon(P, r0, r1, v0, nv, px, py, prev, lane);
    const bool exact = what == WS_EXACT;
    const int main_mode = exact ? WS_MAIN_HIST : WS_MAIN_STASH;
    unsigned* table = tables + (size_t)(p - p_begin) * WS_TABLE_WORDS;
    w.column = table + lane;
    w.lo = lo; w.span = hi - lo; w.shift = 0;
    w.vlo = Key32<T>::value(lo); w.vhi = Key32<T>::value(hi);
    if (std::is_same<T, float>::value) {
      // keys beyond +-infinity are NaNs: as values they compare false with everything, so an open
      // end of the bracket is the infinity (NaN cells then count as "above", where they sort)
      if (lo < 0x007fffffu) w.vlo = (T)(-INFINITY);
      if (hi > 0xff800000u) w.vhi = (T)(INFINITY);
    }
    w.n_active = 0; w.below = 0; w.cnt = 0; w.cells = 0;
    if (exact) zero_hist();
    WarpSelectVisitor<T> scalar{w, main_mode};
    for (int base = miny; base <= maxy; base += 32) {
      const int y = base + lane;
      int cnt = 0;
      if (y <= maxy) cnt = row_crossings_call(px, py, prev, nv, y, cross, lane);
      unsigned single_mask;
      const unsigned complex_mask = row_table<WarpSelect<T>::VEC>(P, mis, edge_scalar, base, cnt, cross, w.cells,
                                                                   &single_mask, scalar);
      constexpr unsigned BM = (1u << ZW_ROWS) - 1u;
      if (sizeof(T) != 1 && exact) {
        // (rare: few distinct keys in a raster of wider cells) span by span with scalar loads
        for (int r = 0; r < 32; ++r)
          if (tab[r] < tab[32 + r]) select_span(w, WS_MAIN_HIST, base + r, tab[r], tab[32 + r] - 1);
      } else {
        // two batches of rows in flight: the loads of the second hide behind the cells of the first
        unsigned todo = 0u;
#pragma unroll
        for (int k = 0; k < 32 / ZW_ROWS; ++k) todo |= ((single_mask >> (k * ZW_ROWS)) & BM) ? 1u << k : 0u;
#pragma unroll 1
        while (todo) {
          const int rb = ZW_ROWS * (__ffs(todo) - 1);
          todo &= todo - 1;
          const int rb2 = todo ? ZW_ROWS * (__ffs(todo) - 1) : -1;
          todo &= todo - 1;
          typename WarpSelect<T>::Batch A, B;
          w.issue(base + rb, tab + rb, A);
          if (rb2 >= 0) w.issue(base + rb2, tab + rb2, B);
          w.template consume<sizeof(T) == 1>(base + rb, tab + rb, A);
          if (rb2 >= 0) w.template consume<sizeof(T) == 1>(base + rb2, tab + rb2, B);
        }
      }
      unsigned cm = complex_mask;
      while (cm) {
        const int r = __ffs(cm) - 1;
        cm &= cm - 1;
        select_complex_row(P, r0, r1, base + r, buf, hbuf, w, main_mode);
      }
      __syncwarp();
    }
    const bool overflow = __any_sync(0xffffffffu, w.cnt > WS_CAP);
    const int n = __reduce_add_sync(0xffffffffu, w.n_active);
    const int below = __reduce_add_sync(0xffffffffu, w.below);
    const int kept = __reduce_add_sync(0xffffffffu, w.cnt);
    long long cells = w.cells;
    for (int o = 16; o > 0; o >>= 1) cells += __shfl_xor_sync(0xffffffffu, cells, o);
    if (lane == 0) area[p] = cells;
    if (n == 0) {
      if (lane == 0) { out[p] = __int_as_float(0x7fc00000); state[p].what = WS_SKIP; }
      continue;
    }
    if (!exact) {
      // the final kernel takes it from here
      table[WS_CAP * 32 + lane] = (unsigned)w.cnt;
      if (lane == 0) { state[p].n_active = n; state[p].below = below; state[p].kept = overflow ? -1 : kept; }
      continue;
    }
    long long rank_lo, rank_hi;
    double part;
    order_ranks(stat, q, n, &rank_lo, &rank_hi, &part);
    const long long in_lo = rank_lo - below, in_hi = rank_hi - below;
    __syncwarp();
    int e0, c0, e1, c1;
    const int b_lo = in_lo >= 0 ? warp_find_bin(hist, in_lo, &e0, &c0, lane) : -1;
    const int b_hi = in_hi >= 0 ? warp_find_bin(hist, in_hi, &e1, &c1, lane) : -1;
    if (lane == 0) {
      state[p].what = WS_SKIP;
      if (b_lo >= 0 && b_hi >= 0) {
        const T vlo = Key32<T>::value(lo + (unsigned)b_lo), vhi = Key32<T>::value(lo + (unsigned)b_hi);
        out[p] = stat == GM_STAT_MEDIAN ? median_of<T>(vlo, vhi) : percentile_of<T>(vlo, vhi, part);
      } else {
        work[2 + atomicAdd(work, 1)] = (int)p;     // the ranks fell outside the bracket
      }
    }
  }
}

template <typename T>
__global__ void __launch_bounds__(32 * WS_WARPS, WS_MIN_BLOCKS)
zonal_select_final_kernel(int stat, double q, int64_t p_begin, int64_t p_end, int* __restrict__ counter,
                          const SelectState* __restrict__ state, const unsigned* __restrict__ tables,
                          float* __restrict__ out, int* __restrict__ work) {
  extern __shared__ __align__(16) int ws_hist[];        // WS_WARPS x WS_BINS
  __shared__ unsigned s_cand[WS_WARPS][32];
  __shared__ int s_ncand[WS_WARPS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int* hist = ws_hist + warp * WS_BINS;
  const unsigned hist_at = (unsigned)__cvta_generic_to_shared(hist);
  auto zero_hist = [&]() {
    __syncwarp();
#pragma unroll
    for (int j = 0; j < WS_BINS / 32; ++j) hist[j * 32 + lane] = 0;
    __syncwarp();
  };
  for (;;) {
    int64_t p = 0;
    if (lane == 0) p = p_begin + atomicAdd(counter, 1);
    p = __shfl_sync(0xffffffffu, p, 0);
    if (p >= p_end) break;
    if (state[p].what != WS_TABLE) continue;
    const int n = state[p].n_active, below = state[p].below, kept = state[p].kept;
    const unsigned lo = state[p].lo, hi = state[p].hi;
    const unsigned* column = tables + (size_t)(p - p_begin) * WS_TABLE_WORDS + lane;
    long long rank_lo, rank_hi;
    double part;
    order_ranks(stat, q, n, &rank_lo, &rank_hi, &part);
    long long in_lo = rank_lo - below, in_hi = rank_hi - below;
    unsigned klo = 0u, khi = 0u;
    bool found = false;
    if (kept >= 0 && in_lo >= 0 && in_hi < kept) {
      const int mine = (int)column[WS_CAP * 32];
      const int most = __reduce_max_sync(0xffffffffu, mine);
      // every lane walks `most` slots (its own beyond `mine` are skipped by predicate), eight
      // loads in flight; `sweep(f)` calls f(key, real) for each of the lane's kept cells
      auto sweep = [&](auto&& f) {
        for (int s = 0; s < most; s += 8) {
          unsigned wd[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) wd[j] = s + j < mine ? __ldcg(column + (s + j) * 32) : 0u;
#pragma unroll
          for (int j = 0; j < 8; ++j) f(StashWord<T>::key(wd[j]), s + j < mine);
        }
      };
      unsigned from = lo, range = hi - lo;
      for (;;) {
        const int sh = max(32 - __clz(range) - WS_BITS, 0);
        zero_hist();
        sweep([&](unsigned k, bool ok) {
          const unsigned rel = k - from;
          red_shared_inc(hist_at + ((rel >> sh) << 2), ok & (rel <= range));
        });
        __syncwarp();
        int e_lo = 0, c_lo = 0, e_hi = 0, c_hi = 0;
        const int b_lo = warp_find_bin(hist, in_lo, &e_lo, &c_lo, lane);
        const int b_hi = warp_find_bin(hist, in_hi, &e_hi, &c_hi, lane);
        if (b_lo < 0 || b_hi < 0) break;                 // (cannot happen: the ranks lie in the table)
        if (b_lo != b_hi) {
          // neighbouring ranks in different bins: the largest key of the one, the smallest of the other
          unsigned a = 0u, b = 0xffffffffu;
          sweep([&](unsigned k, bool ok) {
            const unsigned rel = k - from;
            const int d = (int)(rel >> sh);
            const bool in = ok & (rel <= range);
            a = max(a, (in & (d == b_lo)) ? k : 0u);
            b = min(b, (in & (d == b_hi)) ? k : 0xffffffffu);
          });
          klo = __reduce_max_sync(0xffffffffu, a);
          khi = __reduce_min_sync(0xffffffffu, b);
          found = true;
          break;
        }
        if (sh == 0) { klo = khi = from + (unsigned)b_lo; found = true; break; }
        if (c_lo <= 32) {
          // the bin's keys, one per lane, ranked against each other
          if (lane == 0) s_ncand[warp] = 0;
          __syncwarp();
          sweep([&](unsigned k, bool ok) {
            const unsigned rel = k - from;
            if (ok && rel <= range && (int)(rel >> sh) == b_lo) s_cand[warp][atomicAdd(&s_ncand[warp], 1) & 31] = k;
          });
          __syncwarp();
          const unsigned key = lane < c_lo ? s_cand[warp][lane] : 0xffffffffu;
          int rank = 0;
          for (int j = 0; j < c_lo; ++j) {
            const unsigned o = __shfl_sync(0xffffffffu, key, j);
            rank += (o < key) || (o == key && j < lane);
          }
          const unsigned m_lo = __ballot_sync(0xffffffffu, lane < c_lo && rank == (int)(in_lo - e_lo));
          const unsigned m_hi = __ballot_sync(0xffffffffu, lane < c_lo && rank == (int)(in_hi - e_lo));
          if (m_lo && m_hi) {
            klo = __shfl_sync(0xffffffffu, key, __ffs(m_lo) - 1);
            khi = __shfl_sync(0xffffffffu, key, __ffs(m_hi) - 1);
            found = true;
          }
          break;
        }
        from += (unsigned)b_lo << sh;
        range = (1u << sh) - 1u;
        in_lo -= e_lo; in_hi -= e_lo;
      }
    }
    if (lane == 0) {
      if (found) {
        const T vlo = Key32<T>::value(klo), vhi = Key32<T>::value(khi);
        out[p] = stat == GM_STAT_MEDIAN ? median_of<T>(vlo, vhi) : percentile_of<T>(vlo, vhi, part);
      } else {   // ranks outside the bracket, or more bracket cells than a column holds
        work[2 + atomicAdd(work, 1)] = (int)p;
      }
    }
  }
}

// ---- rasterise ---------------------------------------------------------------------------
// Tiles instead of atomics on the output: the raster is cut in tiles of RT_ROWS x RT_COLS cells,
// every polygon is listed with the tiles its bounding box touches (count, scan, fill), and ONE
// block per tile scan-converts its polygons into a tile of polygon indices in SHARED memory --
// atomicMax on shared memory, so that the LAST feature wins as in GDAL whatever order the warps
// work in -- and then writes the tile's burn values once, coalesced.  The output is written
// exactly once (its itemsize per cell), there is no index raster in HBM and no second pass.
constexpr int RT_ROWS = 16, RT_COLS = 256, RT_WARPS = 4;

// columns a polygon can touch (clamped to the raster; empty: lo > hi)
__global__ void poly_cols_kernel(const double* __restrict__ px, const int64_t* __restrict__ ring_offsets,
                                 const int64_t* __restrict__ poly_offsets, int64_t n_polygons, int width,
                                 int* __restrict__ minx, int* __restrict__ maxx) {
  const int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (p >= n_polygons) return;
  const int64_t v0 = ring_offsets[poly_offsets[p]], v1 = ring_offsets[poly_offsets[p + 1]];
  int lo = 1, hi = 0;
  if (v1 > v0) {
    double dmin = px[v0], dmax = px[v0];
    for (int64_t i = v0 + 1; i < v1; ++i) { dmin = fmin(dmin, px[i]); dmax = fmax(dmax, px[i]); }
    // crossings are floor(x + 0.5): one cell of slack either side covers every rounding
    lo = clamp_to_int(floor(dmin)) - 1;
    hi = clamp_to_int(floor(dmax)) + 1;
    if (lo < 0) lo = 0;
    if (hi >= width) hi = width - 1;
  }
  minx[p] = lo;
  maxx[p] = hi;
}

// pass 0: counts[tile] += 1 for every tile a polygon's box touches; pass 1: the polygon's id into
// the tile's list (cursor = running position, starts at the tile's offset)
__global__ void tile_bin_kernel(const int* __restrict__ miny, const int* __restrict__ maxy,
                                const int* __restrict__ minx, const int* __restrict__ maxx, int64_t n_polygons,
                                int tiles_x, int* __restrict__ counts_or_cursor, int* __restrict__ list) {
  const int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (p >= n_polygons) return;
  if (miny[p] > maxy[p] || minx[p] > maxx[p]) return;
  const int ty0 = miny[p] / RT_ROWS, ty1 = maxy[p] / RT_ROWS, tx0 = minx[p] / RT_COLS, tx1 = maxx[p] / RT_COLS;
  for (int ty = ty0; ty <= ty1; ++ty)
    for (int tx = tx0; tx <= tx1; ++tx) {
      const int at = atomicAdd(counts_or_cursor + (int64_t)ty * tiles_x + tx, 1);
      if (list) list[at] = (int)p;
    }
}

// exclusive scan of n ints in place by ONE block (n = number of tiles, a few hundred thousand);
// total[0] receives the sum
__global__ void __launch_bounds__(1024) tile_scan_kernel(int* __restrict__ data, int64_t n, int* __restrict__ total) {
  __shared__ int warp_sums[32];
  __shared__ int carry;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) carry = 0;
  __syncthreads();
  for (int64_t base = 0; base < n; base += 1024) {
    const int64_t i = base + tid;
    const int v = i < n ? data[i] : 0;
    int incl = v;
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    if (lane == 31) warp_sums[warp] = incl;
    __syncthreads();
    if (warp == 0) {
      int w = warp_sums[lane];
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, w, o);
        if (lane >= o) w += t;
      }
      warp_sums[lane] = w;
    }
    __syncthreads();
    const int before = carry + (warp > 0 ? warp_sums[warp - 1] : 0);
    if (i < n) data[i] = before + incl - v;
    __syncthreads();
    if (tid == 1023) carry = before + incl;
    __syncthreads();
  }
  if (tid == 0) *total = carry;
}

struct TileVisitor {
  int* tile; int x_lo, x_hi, y_lo; int label;       // tile = RT_ROWS x RT_COLS indices, columns x_lo..x_hi
  __device__ __forceinline__ void span(int y, int x0, int x1) {
    x0 = x0 < x_lo ? x_lo : x0;
    x1 = x1 > x_hi ? x_hi : x1;
    int* row = tile + (y - y_lo) * RT_COLS - x_lo;
    for (int x = x0 + (threadIdx.x & 31); x <= x1; x += 32) atomicMax(row + x, label);
  }
  __device__ __forceinline__ void hspan(int y, int x0, int x1, const int*, int) { span(y, x0, x1); }
};

template <typename T>
__global__ void __launch_bounds__(32 * RT_WARPS)
rasterize_tile_kernel(const PolyDev P, const int* __restrict__ tile_offsets, const int* __restrict__ tile_list,
                      int tiles_x, const T* __restrict__ burn, T nodata, T* __restrict__ dst) {
  extern __shared__ __align__(16) int rt_smem[];
  int* tile = rt_smem;                                        // RT_ROWS x RT_COLS polygon indices
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int* buf = tile + RT_ROWS * RT_COLS + warp * P.cap;         // crossings of the generic scanline
  int* hbuf = tile + RT_ROWS * RT_COLS + RT_WARPS * P.cap + warp * 2 * PG_MAX_HSPANS;
  __shared__ double s_px[RT_WARPS][ZW_MAXV], s_py[RT_WARPS][ZW_MAXV];
  __shared__ int s_prev[RT_WARPS][ZW_MAXV];
  __shared__ __align__(16) int s_cross[RT_WARPS][ZW_MAXC][32];
  const int tx = blockIdx.x % tiles_x, ty = blockIdx.x / tiles_x;
  const int x_lo = tx * RT_COLS, y_lo = ty * RT_ROWS;
  const int x_hi = min(x_lo + RT_COLS, P.width) - 1, y_hi = min(y_lo + RT_ROWS, P.height) - 1;
  for (int i = threadIdx.x; i < RT_ROWS * RT_COLS; i += blockDim.x) tile[i] = -1;
  __syncthreads();
  const int first = tile_offsets[blockIdx.x], last = tile_offsets[blockIdx.x + 1];
  for (int item = first + warp; item < last; item += RT_WARPS) {
    const int64_t p = tile_list[item];
    const int64_t r0 = P.poly_offsets[p], r1 = P.poly_offsets[p + 1];
    if (r1 <= r0) continue;
    const int64_t v0 = P.ring_offsets[r0], v1 = P.ring_offsets[r1];
    const int nv = (int)min((int64_t)(ZW_MAXV + 1), v1 - v0);
    const int ya = max(P.miny[p], y_lo), yb = min(P.maxy[p], y_hi);
    if (ya > yb) continue;
    TileVisitor vis{tile, x_lo, x_hi, y_lo, (int)p};
    if (nv == 1) {                 // point feature (GDALdllImagePoint): the cell that contains it
      const int x = clamp_to_int(floor(P.px[v0]));
      if (x >= x_lo && x <= x_hi) vis.span(ya, x, x);
      continue;
    }
    if (nv > ZW_MAXV) {            // many vertices: the whole warp works on one row at a time
      for (int y = ya; y <= yb; ++y) generic_scanline(P, r0, r1, y, P.cap, buf, hbuf, vis);
      continue;
    }
    stage_polygon(P, r0, r1, v0, nv, s_px[warp], s_py[warp], s_prev[warp], lane);
    for (int base = ya; base <= yb; base += 32) {
      const int y = base + lane;
      int cnt = 0;
      if (y <= yb) cnt = row_crossings_call(s_px[warp], s_py[warp], s_prev[warp], nv, y, s_cross[warp], lane);
      __syncwarp();
      const int rows_here = min(32, yb - base + 1);
      for (int r = 0; r < rows_here; ++r) {
        const int c = __shfl_sync(0xffffffffu, cnt, r);
        if (c < 0) { generic_scanline(P, r0, r1, base + r, P.cap, buf, hbuf, vis); continue; }
        for (int i = 0; i + 1 < c; i += 2) {
          const int xa = s_cross[warp][i][r], xb = s_cross[warp][i + 1][r] - 1;
          if (xa <= x_hi && xb >= x_lo) vis.span(base + r, xa, xb);
        }
      }
      __syncwarp();
    }
  }
  __syncthreads();
  // the tile leaves once: burn value of the winning polygon, `nodata` where there is none
  for (int i = threadIdx.x; i < RT_ROWS * RT_COLS; i += blockDim.x) {
    const int y = y_lo + i / RT_COLS, x = x_lo + i % RT_COLS;
    if (y <= y_hi && x <= x_hi) {
      const int l = tile[i];
      dst[(int64_t)y * P.width + x] = l < 0 ? nodata : burn[l];
    }
  }
}

// ---- multi-GPU order statistics: raw values out, segments in ---------------------------------
// Append the ACTIVE cell values under polygon p at values[offsets[p] ...] (any order).
template <typename T>
struct ValueVisitor {
  const T* raster; int width; ActiveTest<T> active;
  T* out; int* cursor; long long capacity;
  __device__ __forceinline__ void put(bool ok, T v) {
    const unsigned m = __ballot_sync(0xffffffffu, ok);
    if (m == 0) return;
    const int lane = threadIdx.x & 31;
    int base = 0;
    if (lane == 0) base = atomicAdd(cursor, __popc(m));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (ok) {
      const long long pos = base + __popc(m & ((1u << lane) - 1u));
      if (pos < capacity) out[pos] = v;
    }
  }
  __device__ __forceinline__ void span(int y, int x0, int x1) {
    const T* row = raster + (int64_t)y * width;
    const int lane = threadIdx.x & 31;
    for (int xb = x0; xb <= x1; xb += 32) {
      const int x = xb + lane;
      T v = T(0);
      bool ok = false;
      if (x <= x1) { v = __ldg(row + x); ok = active(v); }
      put(ok, v);
    }
  }
  __device__ __forceinline__ void hspan(int y, int x0, int x1, const int* buf, int n) {
    const T* row = raster + (int64_t)y * width;
    const int lane = threadIdx.x & 31;
    for (int xb = x0; xb <= x1; xb += 32) {
      const int x = xb + lane;
      T v = T(0);
      bool ok = false;
      if (x <= x1 && !in_pairs(x, buf, n)) { v = __ldg(row + x); ok = active(v); }
      put(ok, v);
    }
  }
};

template <typename T>
__global__ void __launch_bounds__(PG_THREADS)
zonal_values_kernel(const PolyDev P, const T* __restrict__ raster, T nodata, int has_nodata,
                    const float* __restrict__ thresholds, const long long* __restrict__ offsets,
                    T* __restrict__ values) {
  extern __shared__ int pg_smem[];
  __shared__ int cursor;
  const int warp = threadIdx.x >> 5;
  int* buf = pg_smem + warp * P.cap;
  int* hbuf = pg_smem + PG_WARPS * P.cap + warp * 2 * PG_MAX_HSPANS;
  for (int64_t p = blockIdx.x; p < P.n_polygons; p += gridDim.x) {
    if (threadIdx.x == 0) cursor = 0;
    __syncthreads();
    ValueVisitor<T> vis;
    vis.raster = raster; vis.width = P.width;
    vis.active = active_test(nodata, has_nodata, thresholds, p);
    vis.out = values + offsets[p]; vis.cursor = &cursor; vis.capacity = offsets[p + 1] - offsets[p];
    scan_polygon(P, p, buf, hbuf, vis);
    __syncthreads();
  }
}

// One block per segment: values -> sortable keys (in place in `keys`), then select.
template <typename T>
__global__ void __launch_bounds__(SEL_THREADS)
segment_select_kernel(const T* __restrict__ values, const long long* __restrict__ offsets, int64_t n_seg,
                      typename KeyOf<T>::type* __restrict__ keys, int stat, double q,
                      float* __restrict__ out) {
  typedef typename KeyOf<T>::type K;
  __shared__ int hist[256];
  __shared__ SelectScratch<K> select_scratch;
  for (int64_t seg = blockIdx.x; seg < n_seg; seg += gridDim.x) {
    const long long a = offsets[seg], b = offsets[seg + 1];
    K* k = keys + a;
    for (long long i = threadIdx.x; i < b - a; i += blockDim.x) k[i] = KeyOf<T>::key(values[a + i]);
    __syncthreads();
    const float result = order_statistic<T>(k, (int)(b - a), stat, q, hist, &select_scratch);
    if (threadIdx.x == 0) out[seg] = result;
    __syncthreads();
  }
}

// ---- host side ---------------------------------------------------------------------------------
// Polygon soup kept in HBM between calls (gm_polygons_upload): the CSR arrays and the
// largest vertex count, so that a request only runs the two small preparation kernels.
// What prepare_polygons derives from a soup for ONE raster grid (pixel-space vertices, row
// ranges, the active list): a resident soup keeps the last few, so that a repeated request --
// the same stripe of the same grid, step after step -- launches no preparation kernel at all.
struct PreparedPolygons {
  double geo[6];
  int height = 0, width = 0;
  int64_t row_begin = 0, row_end = 0;
  void *px = nullptr, *py = nullptr, *miny = nullptr, *maxy = nullptr, *active = nullptr, *n_active = nullptr;
  cudaEvent_t ready = nullptr;
  ~PreparedPolygons() {
    // (plain cudaFree waits for the device: kernels of other streams may still read these)
    void* all[] = {px, py, miny, maxy, active, n_active};
    for (void* p : all) if (p) cudaFree(p);
    if (ready) cudaEventDestroy(ready);
  }
};

struct ResidentPolygons {
  void *xy = nullptr, *rings = nullptr, *polys = nullptr;
  int64_t n_polygons = 0, n_rings = 0, n_vertices = 0, max_vertices = 1;
  int* error = nullptr;       // crossing-overflow flag of calls whose check is deferred
  std::mutex lock;
  std::vector<std::shared_ptr<PreparedPolygons>> prepared;   // most recent last, <= 4
  // the grid of the last call that found nothing prepared: an entry is only built (with plain,
  // device-synchronising allocations) when the SAME grid comes again -- a sweep of ever new
  // request windows over one soup keeps the stream-ordered per-call path
  struct Seen { double geo[6]; int height, width; int64_t rows[2]; };
  std::vector<Seen> seen;     // the last 8 such grids
};

struct PolyUpload {
  void *xy = nullptr, *px = nullptr, *py = nullptr, *rings = nullptr, *polys = nullptr;
  void *miny = nullptr, *maxy = nullptr, *error = nullptr, *active = nullptr, *n_active = nullptr;
  bool borrowed = false;   // xy / rings / polys belong to a ResidentPolygons
  bool deferred_error = false;                 // `error` is the resident soup's flag
  std::shared_ptr<PreparedPolygons> shared;    // px ... n_active belong to it
  PolyDev dev;
  cudaStream_t s;
  void release() {
    if (!shared) {
      void* own[] = {px, py, miny, maxy, active, n_active};
      for (void* p : own) if (p) cudaFreeAsync(p, s);
    }
    shared.reset();
    if (error && !deferred_error) cudaFreeAsync(error, s);
    if (!borrowed) {
      void* csr[] = {xy, rings, polys};
      for (void* p : csr) if (p) cudaFreeAsync(p, s);
    }
  }
};

static int64_t largest_polygon(const GmPolygons* polys) {
  int64_t max_vertices = 1;
  for (int64_t p = 0; p < polys->n_polygons; ++p) {
    const int64_t a = polys->ring_offsets[polys->poly_offsets[p]];
    const int64_t b = polys->ring_offsets[polys->poly_offsets[p + 1]];
    if (b - a > max_vertices) max_vertices = b - a;
  }
  return max_vertices;
}

static int prepare_polygons(const GmPolygons* polys, const double* geo, int height, int width,
                            int64_t row_begin, int64_t row_end, PolyUpload& u, cudaStream_t s,
                            bool stripe_call = false, bool cache = false) {
  // stripe_call (gm_zonal_partials_device): build the list of polygons with rows in this window
  // and leave the overflow flag of a resident soup to the finalisation; stripe_call or cache:
  // keep the prepared arrays with a resident soup
  u.s = s;
  if (!polys || !geo) return fail("polygons: null argument");
  if (geo[2] != 0.0 || geo[4] != 0.0 || geo[1] == 0.0 || geo[5] == 0.0)
    return fail("polygons: rotated or degenerate geotransform");
  const int64_t nv = polys->n_vertices, nr = polys->n_rings, np_ = polys->n_polygons;
  ResidentPolygons* resident = static_cast<ResidentPolygons*>(const_cast<void*>(polys->resident));
  if (resident && (resident->n_polygons != np_ || resident->n_rings != nr || resident->n_vertices != nv))
    return fail("polygons: resident handle does not match the descriptor");
  const int64_t max_vertices = resident ? resident->max_vertices : largest_polygon(polys);
  int cap = 32;
  while (cap < max_vertices && cap < PG_MAX_CROSSINGS) cap <<= 1;
  u.dev.n_polygons = np_; u.dev.height = height; u.dev.width = width; u.dev.cap = cap;
  u.dev.active = nullptr; u.dev.n_active = nullptr;
  if (resident) {
    u.borrowed = true;
    u.xy = resident->xy; u.rings = resident->rings; u.polys = resident->polys;
  } else {
    if (upload(&u.xy, polys->xy, sizeof(double) * 2 * nv, s)) return 1;
    if (upload(&u.rings, polys->ring_offsets, sizeof(int64_t) * (nr + 1), s)) return 1;
    if (upload(&u.polys, polys->poly_offsets, sizeof(int64_t) * (np_ + 1), s)) return 1;
  }
  u.dev.ring_offsets = (const int64_t*)u.rings; u.dev.poly_offsets = (const int64_t*)u.polys;
  const bool keep = (stripe_call || cache) && resident != nullptr;
  if (keep && stripe_call && resident->error) {
    u.error = resident->error; u.deferred_error = true;
  } else {
    GM_CUDA(cudaMallocAsync(&u.error, sizeof(int), s));
    GM_CUDA(cudaMemsetAsync(u.error, 0, sizeof(int), s));
  }
  u.dev.error = (int*)u.error;
  auto adopt = [&](const PreparedPolygons& q) {
    u.px = q.px; u.py = q.py; u.miny = q.miny; u.maxy = q.maxy; u.active = q.active; u.n_active = q.n_active;
  };
  if (keep) {
    std::lock_guard<std::mutex> guard(resident->lock);
    for (size_t i = 0; i < resident->prepared.size(); ++i) {
      std::shared_ptr<PreparedPolygons> q = resident->prepared[i];
      if (memcmp(q->geo, geo, sizeof(q->geo)) == 0 && q->height == height && q->width == width &&
          q->row_begin == row_begin && q->row_end == row_end && (!stripe_call || q->active)) {
        resident->prepared.erase(resident->prepared.begin() + (long)i);
        resident->prepared.push_back(q);
        GM_CUDA(cudaStreamWaitEvent(s, q->ready, 0));
        u.shared = q;
        adopt(*q);
        break;
      }
    }
  }
  if (!u.shared) {
    bool build = false;     // keep what this call prepares?
    if (keep) {
      std::lock_guard<std::mutex> guard(resident->lock);
      ResidentPolygons::Seen now;
      memcpy(now.geo, geo, sizeof(now.geo));
      now.height = height; now.width = width; now.rows[0] = row_begin; now.rows[1] = row_end;
      for (size_t i = 0; i < resident->seen.size() && !build; ++i) {
        const ResidentPolygons::Seen& o = resident->seen[i];
        build = memcmp(o.geo, now.geo, sizeof(now.geo)) == 0 && o.height == height && o.width == width &&
                o.rows[0] == row_begin && o.rows[1] == row_end;
      }
      if (!build) {
        if (resident->seen.size() >= 8) resident->seen.erase(resident->seen.begin());
        resident->seen.push_back(now);
      }
    }
    // (plain cudaMalloc for arrays that outlive the call: stream-ordered frees of another
    //  stream's pool blocks are not wanted here)
    auto alloc = [&](void** ptr, size_t bytes) -> cudaError_t {
      return build ? cudaMalloc(ptr, bytes) : cudaMallocAsync(ptr, bytes, s);
    };
    std::shared_ptr<PreparedPolygons> q;
    if (build) q = std::make_shared<PreparedPolygons>();
    void *px = nullptr, *py = nullptr, *miny = nullptr, *maxy = nullptr, *active = nullptr, *n_active = nullptr;
    cudaError_t e = alloc(&px, sizeof(double) * (nv > 0 ? nv : 1));
    if (e == cudaSuccess) e = alloc(&py, sizeof(double) * (nv > 0 ? nv : 1));
    if (e == cudaSuccess) e = alloc(&miny, sizeof(int) * (np_ > 0 ? np_ : 1));
    if (e == cudaSuccess) e = alloc(&maxy, sizeof(int) * (np_ > 0 ? np_ : 1));
    if (e == cudaSuccess && stripe_call) e = alloc(&active, sizeof(int) * (np_ > 0 ? np_ : 1));
    if (e == cudaSuccess && stripe_call) e = alloc(&n_active, sizeof(int));
    if (q) { q->px = px; q->py = py; q->miny = miny; q->maxy = maxy; q->active = active; q->n_active = n_active; }
    else { u.px = px; u.py = py; u.miny = miny; u.maxy = maxy; u.active = active; u.n_active = n_active; }
    if (e != cudaSuccess) return fail(std::string("polygons: ") + cudaGetErrorString(e));
    const double inv0 = -geo[0] / geo[1], inv1 = 1.0 / geo[1];
    const double inv3 = -geo[3] / geo[5], inv5 = 1.0 / geo[5];
    if (nv > 0) {
      poly_transform_kernel<<<(unsigned)((nv + 255) / 256), 256, 0, s>>>(
          (const double*)u.xy, (double*)px, (double*)py, nv, inv0, inv1, inv3, inv5);
      GM_LAUNCH_CHECK();
    }
    if (np_ > 0) {
      poly_rows_kernel<<<(unsigned)((np_ + 255) / 256), 256, 0, s>>>(
          (const double*)py, (const int64_t*)u.rings, (const int64_t*)u.polys, np_, height,
          (int)row_begin, (int)row_end, (int*)miny, (int*)maxy);
      GM_LAUNCH_CHECK();
    }
    if (stripe_call) {
      GM_CUDA(cudaMemsetAsync(n_active, 0, sizeof(int), s));
      if (np_ > 0) {
        poly_active_kernel<<<(unsigned)((np_ + 255) / 256), 256, 0, s>>>(
            (const int*)miny, (const int*)maxy, (const int64_t*)u.rings, (const int64_t*)u.polys, np_,
            (int*)active, (int*)n_active);
        GM_LAUNCH_CHECK();
      }
    }
    if (q) {
      memcpy(q->geo, geo, sizeof(q->geo));
      q->height = height; q->width = width; q->row_begin = row_begin; q->row_end = row_end;
      GM_CUDA(cudaEventCreateWithFlags(&q->ready, cudaEventDisableTiming));
      GM_CUDA(cudaEventRecord(q->ready, s));
      std::lock_guard<std::mutex> guard(resident->lock);
      if (resident->prepared.size() >= 4) resident->prepared.erase(resident->prepared.begin());
      resident->prepared.push_back(q);
      u.shared = q;
      adopt(*q);
    }
  }
  u.dev.px = (const double*)u.px; u.dev.py = (const double*)u.py;
  u.dev.miny = (const int*)u.miny; u.dev.maxy = (const int*)u.maxy;
  if (stripe_call) { u.dev.active = (const int*)u.active; u.dev.n_active = (const int*)u.n_active; }
  return 0;
}

static size_t scan_smem(int cap, int warps) {
  return (size_t)(warps * cap + warps * 2 * PG_MAX_HSPANS) * sizeof(int);
}

static int check_overflow(PolyUpload& u, cudaStream_t s) {
  if (u.deferred_error) return 0;     // gm_zonal_finalize_device reads the soup's flag
  int flag = 0;
  GM_CUDA(cudaMemcpyAsync(&flag, u.error, sizeof(int), cudaMemcpyDeviceToHost, s));
  GM_CUDA(cudaStreamSynchronize(s));
  if (flag) return fail("polygons: more than 4096 edge crossings (or 8 horizontal edges) on one scanline");
  return 0;
}

static unsigned poly_grid(int64_t n) {
  const int64_t cap = (int64_t)sm_count() * 32;
  return (unsigned)(n < cap ? (n > 0 ? n : 1) : cap);
}

// Where a raster of H x W cells stands against the grid of VEC-cell loads of the batched row
// walk: *mis = offset of its first cell from that grid; *edge_scalar = a load on its first or last
// row could reach outside the array (or the cells are not aligned to their own size), so those
// rows are read with scalar loads.
template <typename T>
static void raster_alignment(const void* raster, int vec, int H, int W, int* mis, int* edge_scalar) {
  *mis = (int)(((uintptr_t)raster / sizeof(T)) & (uintptr_t)(vec - 1));
  *edge_scalar = ((uintptr_t)raster % sizeof(T)) != 0 || *mis != 0 || (((int64_t)H * W + *mis) % vec) != 0;
}

// Partials and covered cells of every polygon: zonal_reduce_warp_kernel takes the usual polygons
// (`need`: the accumulators it keeps), zonal_reduce_kernel the ones it deferred to `work`, on a
// grid of `deferred_grid` blocks.
template <typename T>
static cudaError_t launch_reduce(const PolyUpload& u, const Staged& raster, T nd, int has_nodata,
                                 const float* thresholds, int need, unsigned deferred_grid, size_t smem_scan,
                                 GmZonalPartial* partial, long long* cells, int* work, cudaStream_t s) {
  const int64_t np_ = u.dev.n_polygons;
  int mis, edge_scalar;
  raster_alignment<T>(raster.dev, WarpReduce<T, ZW_ALL>::VEC, u.dev.height, u.dev.width, &mis, &edge_scalar);
  int64_t wblocks = (np_ + ZW_WARPS - 1) / ZW_WARPS;
  if (wblocks > (int64_t)sm_count() * ZW_MIN_BLOCKS) wblocks = (int64_t)sm_count() * ZW_MIN_BLOCKS;
  auto* warp_kernel = need == ZW_SUM ? &zonal_reduce_warp_kernel<T, ZW_SUM>
                    : need == ZW_MIN ? &zonal_reduce_warp_kernel<T, ZW_MIN>
                    : need == ZW_MAX ? &zonal_reduce_warp_kernel<T, ZW_MAX>
                    : &zonal_reduce_warp_kernel<T, ZW_ALL>;
  warp_kernel<<<(unsigned)wblocks, 32 * ZW_WARPS, 0, s>>>(u.dev, (const T*)raster.dev, nd, has_nodata, thresholds,
                                                           mis, edge_scalar, partial, cells, work);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  count_launch();
  zonal_reduce_kernel<T><<<deferred_grid, PG_THREADS, smem_scan, s>>>(
      u.dev, (const T*)raster.dev, nd, has_nodata, thresholds, partial, cells, work);
  e = cudaGetLastError();
  if (e == cudaSuccess) count_launch();
  return e;
}

// on a CUDA error: free what the calling function allocated so far (its `cleanup`) and fail
#define GM_TRY(expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) { cleanup(); return fail(std::string(#expr) + ": " + cudaGetErrorString(_e)); } } while (0)

template <typename T>
static int run_rasterize(PolyUpload& u, const void* burn, const void* nodata, Staged& out,
                         int64_t n_pixels, cudaStream_t s) {
  const int64_t np_ = u.dev.n_polygons;
  const int H = u.dev.height, W = u.dev.width;
  const int tiles_x = (W + RT_COLS - 1) / RT_COLS, tiles_y = (H + RT_ROWS - 1) / RT_ROWS;
  const int64_t n_tiles = (int64_t)tiles_x * tiles_y;
  T nd;
  memcpy(&nd, nodata, sizeof(T));
  void *dburn = nullptr, *dminx = nullptr, *dmaxx = nullptr, *doffsets = nullptr, *dcursor = nullptr;
  void *dlist = nullptr, *dtotal = nullptr;
  auto cleanup = [&]() {
    void* all[] = {dburn, dminx, dmaxx, doffsets, dcursor, dlist, dtotal};
    for (void* p : all) if (p) cudaFreeAsync(p, s);
  };
  if (upload(&dburn, burn, sizeof(T) * (size_t)(np_ > 0 ? np_ : 1), s)) { cleanup(); return 1; }
  GM_TRY(cudaMallocAsync(&doffsets, sizeof(int) * (size_t)(n_tiles + 1), s));
  GM_TRY(cudaMemsetAsync(doffsets, 0, sizeof(int) * (size_t)(n_tiles + 1), s));
  int total = 0;
  if (np_ > 0) {
    // polygons -> tiles: count, scan, fill
    GM_TRY(cudaMallocAsync(&dminx, sizeof(int) * np_, s));
    GM_TRY(cudaMallocAsync(&dmaxx, sizeof(int) * np_, s));
    GM_TRY(cudaMallocAsync(&dcursor, sizeof(int) * (size_t)(n_tiles + 1), s));
    GM_TRY(cudaMallocAsync(&dtotal, sizeof(int), s));
    const unsigned pb = (unsigned)((np_ + 255) / 256);
    poly_cols_kernel<<<pb, 256, 0, s>>>(u.dev.px, u.dev.ring_offsets, u.dev.poly_offsets, np_, W,
                                        (int*)dminx, (int*)dmaxx);
    tile_bin_kernel<<<pb, 256, 0, s>>>(u.dev.miny, u.dev.maxy, (const int*)dminx, (const int*)dmaxx, np_,
                                       tiles_x, (int*)doffsets, nullptr);
    tile_scan_kernel<<<1, 1024, 0, s>>>((int*)doffsets, n_tiles + 1, (int*)dtotal);
    GM_TRY(cudaGetLastError());
    count_launch(3);
    GM_TRY(cudaMemcpyAsync(&total, dtotal, sizeof(int), cudaMemcpyDeviceToHost, s));
    GM_TRY(cudaMemcpyAsync(dcursor, doffsets, sizeof(int) * (size_t)(n_tiles + 1), cudaMemcpyDeviceToDevice, s));
    GM_TRY(cudaStreamSynchronize(s));
    GM_TRY(cudaMallocAsync(&dlist, sizeof(int) * (size_t)(total > 0 ? total : 1), s));
    tile_bin_kernel<<<pb, 256, 0, s>>>(u.dev.miny, u.dev.maxy, (const int*)dminx, (const int*)dmaxx, np_,
                                       tiles_x, (int*)dcursor, (int*)dlist);
    GM_TRY(cudaGetLastError());
    count_launch();
  } else {
    GM_TRY(cudaMallocAsync(&dlist, sizeof(int), s));
  }
  const size_t smem = (size_t)RT_ROWS * RT_COLS * sizeof(int) + scan_smem(u.dev.cap, RT_WARPS);
  GM_TRY(cudaFuncSetAttribute(rasterize_tile_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  rasterize_tile_kernel<T><<<(unsigned)n_tiles, 32 * RT_WARPS, smem, s>>>(
      u.dev, (const int*)doffsets, (const int*)dlist, tiles_x, (const T*)dburn, nd, (T*)out.dev);
  GM_TRY(cudaGetLastError());
  count_launch();
  cleanup();
  (void)n_pixels;
  return 0;
}

template <typename T>
static int run_zonal(PolyUpload& u, const Staged& raster, const void* nodata, int has_nodata,
                     int stat, double q, const float* thresholds, float* out, int64_t* covered,
                     GmZonalPartial* partial, cudaStream_t s) {
  const int64_t np_ = u.dev.n_polygons;
  if (np_ == 0) return 0;
  T nd = T(0);
  if (has_nodata) memcpy(&nd, nodata, sizeof(T));
  void *darea = nullptr, *dthr = nullptr, *dpartial = nullptr, *dout = nullptr;
  void *doff = nullptr, *dtotal = nullptr, *dbig = nullptr, *scratch_work = nullptr, *scratch_list = nullptr;
  int rc = 0;
  auto cleanup = [&]() {
    void* all[] = {darea, dthr, dpartial, dout, doff, dtotal, dbig, scratch_work, scratch_list};
    for (void* p : all) if (p) cudaFreeAsync(p, s);
  };
  GM_TRY(cudaMallocAsync(&darea, sizeof(long long) * np_, s));
  if (thresholds && upload(&dthr, thresholds, sizeof(float) * np_, s)) { cleanup(); return 1; }
  const size_t smem_scan = scan_smem(u.dev.cap, PG_WARPS);
  if (smem_scan > 48 * 1024) {
    GM_TRY(cudaFuncSetAttribute(zonal_area_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_scan));
    GM_TRY(cudaFuncSetAttribute(zonal_reduce_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_scan));
  }
  const bool order_stat = stat == GM_STAT_MEDIAN || stat == GM_STAT_PERCENTILE;
  // covered cells per polygon on the host: straight into the caller's (page-locked) `covered`
  std::vector<long long> area_store;
  long long* area = reinterpret_cast<long long*>(covered);
  if (order_stat && !area) { area_store.resize(np_); area = area_store.data(); }
  // order statistics: the deferred list (work[0] entries from work[2]) of the polygons the
  // fast kernel does not take -- all of them when it does not apply
  void* dlist = nullptr;
  int n_listed = 0;
  std::vector<int> listed;
  bool area_done = false;
  bool selected = false;      // the listed polygons are done and `out` is on the host already
  if (order_stat) {
    GM_TRY(cudaMallocAsync(&dlist, sizeof(int) * (size_t)(np_ + 2), s));
    scratch_list = dlist;
    // the streaming select takes float32 and integers up to 4 bytes (32-bit sortable keys)
    const bool streaming = sizeof(T) <= 4 && !thresholds && out;
    if (streaming) {
      int mis, edge_scalar;
      raster_alignment<T>(raster.dev, WarpSelect<T>::VEC, u.dev.height, u.dev.width, &mis, &edge_scalar);
      // one warp per polygon, three kernels (bracket, main pass, final ranks) per chunk of
      // polygons; the bracket's cells of a chunk wait in per-polygon tables between the last two
      GM_TRY(cudaMallocAsync(&dout, sizeof(float) * np_, s));
      GM_TRY(cudaMemsetAsync(dlist, 0, 2 * sizeof(int), s));
      static const int64_t chunk_cap = getenv("GM_SELECT_CHUNK") ? atoll(getenv("GM_SELECT_CHUNK")) : 131072;
      const int64_t chunk = np_ < chunk_cap ? np_ : chunk_cap;
      const int64_t n_chunks = (np_ + chunk - 1) / chunk;
      void *dstate = nullptr, *dcounters = nullptr;
      GM_TRY(cudaMallocAsync(&dstate, sizeof(SelectState) * np_, s));
      GM_TRY(cudaMallocAsync(&dcounters, sizeof(int) * 3 * n_chunks, s));
      GM_TRY(cudaMemsetAsync(dcounters, 0, sizeof(int) * 3 * n_chunks, s));
      GM_TRY(cudaMallocAsync(&dbig, sizeof(unsigned) * (size_t)chunk * WS_TABLE_WORDS, s));
      if constexpr (sizeof(T) <= 4) {
        constexpr int ws_smem = WS_WARPS * WS_BINS * (int)sizeof(int);
        GM_TRY(cudaFuncSetAttribute(zonal_select_bracket_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, ws_smem));
        GM_TRY(cudaFuncSetAttribute(zonal_select_main_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, ws_smem));
        GM_TRY(cudaFuncSetAttribute(zonal_select_final_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, ws_smem));
        for (int64_t c = 0; c < n_chunks; ++c) {
          const int64_t p0 = c * chunk, p1 = p0 + chunk < np_ ? p0 + chunk : np_;
          int64_t wblocks = (p1 - p0 + WS_WARPS - 1) / WS_WARPS;
          if (wblocks > (int64_t)sm_count() * WS_MIN_BLOCKS) wblocks = (int64_t)sm_count() * WS_MIN_BLOCKS;
          int* counters = (int*)dcounters + 3 * c;
          zonal_select_bracket_kernel<T><<<(unsigned)wblocks, 32 * WS_WARPS, ws_smem, s>>>(
              u.dev, (const T*)raster.dev, nd, has_nodata, stat, q, p0, p1, counters, (SelectState*)dstate,
              (float*)dout, (long long*)darea, (int*)dlist);
          int64_t mblocks = (p1 - p0 + WS_WARPS - 1) / WS_WARPS;
          if (mblocks > (int64_t)sm_count() * WS_MAIN_BLOCKS) mblocks = (int64_t)sm_count() * WS_MAIN_BLOCKS;
          zonal_select_main_kernel<T><<<(unsigned)mblocks, 32 * WS_WARPS, ws_smem, s>>>(
              u.dev, (const T*)raster.dev, nd, has_nodata, mis, edge_scalar, stat, q, p0, p1, counters + 1,
              (SelectState*)dstate, (unsigned*)dbig, (float*)dout, (long long*)darea, (int*)dlist);
          zonal_select_final_kernel<T><<<(unsigned)wblocks, 32 * WS_WARPS, ws_smem, s>>>(
              stat, q, p0, p1, counters + 2, (const SelectState*)dstate, (const unsigned*)dbig, (float*)dout,
              (int*)dlist);
          count_launch(3);
        }
      }
      GM_TRY(cudaGetLastError());
      // the covered cells of the deferred polygons (the kernel reads the list's length on the
      // device), then ONE synchronisation for the list and all the counts
      zonal_area_kernel<<<poly_grid(np_ < 1024 ? np_ : 1024), PG_THREADS, smem_scan, s>>>(
          u.dev, (long long*)darea, (const int*)dlist);
      GM_TRY(cudaGetLastError());
      count_launch();
      // The deferred polygons are selected right away by the block-per-polygon kernel with their
      // keys in shared memory (the whole budget), its grid sized without knowing the list's
      // length: results, counts, the list and a "some polygon did not fit" flag come back under
      // ONE synchronisation.  Only when the flag is up does the host lay out global key segments
      // and repeat the listed polygons (below).
      {
        typedef typename KeyOf<T>::type K;
        const size_t shead = (scan_smem(u.dev.cap, SEL_THREADS / 32) + 15) / 16 * 16;
        const int capacity = (int)((200 * 1024 - shead) / sizeof(K));
        const size_t smem_sel = shead + (size_t)capacity * sizeof(K);
        GM_TRY(cudaFuncSetAttribute(zonal_select_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_sel));
        GM_TRY(cudaMallocAsync(&dtotal, sizeof(int), s));
        GM_TRY(cudaMemsetAsync(dtotal, 0, sizeof(int), s));
        zonal_select_kernel<T><<<poly_grid(np_ < 1024 ? np_ : 1024), SEL_THREADS, smem_sel, s>>>(
            u.dev, (const T*)raster.dev, nd, has_nodata, (const float*)dthr, stat, q,
            (const long long*)darea, nullptr, (K*)nullptr, capacity, (float*)dout, (const int*)dlist,
            (int*)dtotal);
        GM_TRY(cudaGetLastError());
        count_launch();
      }
      const int64_t head = np_ < 4096 ? np_ : 4096;
      std::vector<int> front(head + 2);
      int too_big = 0;
      GM_TRY(cudaMemcpyAsync(front.data(), dlist, sizeof(int) * (head + 2), cudaMemcpyDeviceToHost, s));
      GM_TRY(cudaMemcpyAsync(area, darea, sizeof(long long) * np_, cudaMemcpyDeviceToHost, s));
      GM_TRY(cudaMemcpyAsync(&too_big, dtotal, sizeof(int), cudaMemcpyDeviceToHost, s));
      GM_TRY(cudaMemcpyAsync(out, dout, sizeof(float) * np_, cudaMemcpyDeviceToHost, s));
      GM_TRY(cudaStreamSynchronize(s));
      area_done = true;
      selected = !too_big;
      cudaFreeAsync(dbig, s);
      cudaFreeAsync(dstate, s);
      cudaFreeAsync(dcounters, s);
      dbig = nullptr;
      n_listed = front[0];
      listed.assign(front.begin() + 2, front.begin() + 2 + (n_listed < head ? n_listed : head));
      if (getenv("GM_DEBUG_ZONAL")) fprintf(stderr, "gm_zonal_stats: %d of %lld polygons deferred to the generic select\n", n_listed, (long long)np_);
      if (n_listed > head) {
        listed.resize(n_listed);
        GM_TRY(cudaMemcpyAsync(listed.data(), (const int*)dlist + 2, sizeof(int) * n_listed, cudaMemcpyDeviceToHost, s));
        GM_TRY(cudaStreamSynchronize(s));
      }
    } else {
      n_listed = (int)np_;
      listed.resize(np_);
      std::vector<int> host(np_ + 2);
      host[0] = n_listed; host[1] = 0;
      for (int64_t p = 0; p < np_; ++p) { host[2 + p] = (int)p; listed[p] = (int)p; }
      GM_TRY(cudaMemcpyAsync(dlist, host.data(), sizeof(int) * (np_ + 2), cudaMemcpyHostToDevice, s));
      GM_TRY(cudaStreamSynchronize(s));
    }
    if (!area_done) {
      if (n_listed > 0) {
        // pixel centres inside the listed polygons (no raster access): `covered` and buffer sizes
        zonal_area_kernel<<<poly_grid(n_listed), PG_THREADS, smem_scan, s>>>(u.dev, (long long*)darea, (const int*)dlist);
        GM_TRY(cudaGetLastError());
        count_launch();
      }
      GM_TRY(cudaMemcpyAsync(area, darea, sizeof(long long) * np_, cudaMemcpyDeviceToHost, s));
      GM_TRY(cudaStreamSynchronize(s));
    }
  }

  if (!order_stat || partial) {
    // one pass: partials and the covered-cell counts together
    GM_TRY(cudaMallocAsync(&dpartial, sizeof(GmZonalPartial) * np_, s));
    // warps take the usual polygons one each; the rest goes through the block-per-polygon kernel
    void* dwork = nullptr;
    GM_TRY(cudaMallocAsync(&dwork, sizeof(int) * (size_t)(np_ + 2), s));
    scratch_work = dwork;
    GM_TRY(cudaMemsetAsync(dwork, 0, 2 * sizeof(int), s));
    const int need = partial ? ZW_ALL : stat == GM_STAT_MIN ? ZW_MIN : stat == GM_STAT_MAX ? ZW_MAX : ZW_SUM;
    GM_TRY(launch_reduce<T>(u, raster, nd, has_nodata, (const float*)dthr, need, poly_grid(np_), smem_scan,
                            (GmZonalPartial*)dpartial, (long long*)darea, (int*)dwork, s));
    if (!order_stat && covered) {
      static_assert(sizeof(long long) == sizeof(int64_t), "covered is int64");
      GM_TRY(cudaMemcpyAsync(covered, darea, sizeof(long long) * np_, cudaMemcpyDeviceToHost, s));
    }
    if (partial)
      GM_TRY(cudaMemcpyAsync(partial, dpartial, sizeof(GmZonalPartial) * np_, cudaMemcpyDeviceToHost, s));
    if (out && !order_stat) {
      GM_TRY(cudaMallocAsync(&dout, sizeof(float) * np_, s));
      zonal_finalize_kernel<<<(unsigned)((np_ + 255) / 256), 256, 0, s>>>(
          (const GmZonalPartial*)dpartial, stat, (float*)dout, np_);
      GM_TRY(cudaGetLastError());
      count_launch();
      GM_TRY(cudaMemcpyAsync(out, dout, sizeof(float) * np_, cudaMemcpyDeviceToHost, s));
    }
  }
  if (order_stat && out && !selected) {
    typedef typename KeyOf<T>::type K;
    if (!dout) GM_TRY(cudaMallocAsync(&dout, sizeof(float) * np_, s));
    if (n_listed > 0) {
      long long max_area = 0;
      for (int p : listed) max_area = area[p] > max_area ? area[p] : max_area;
      const size_t head = (scan_smem(u.dev.cap, SEL_THREADS / 32) + 15) / 16 * 16;
      const size_t budget = 200 * 1024 - head;
      long long capacity = (long long)(budget / sizeof(K));
      if (max_area < capacity) capacity = max_area > 0 ? max_area : 1;
      const size_t smem_sel = head + (size_t)capacity * sizeof(K);
      GM_TRY(cudaFuncSetAttribute(zonal_select_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_sel));
      // global key segments for the polygons that do not fit shared memory
      // (only polygons that exceed the shared-memory capacity read their offset: none -> no table)
      long long total = 0;
      for (int p : listed)
        if (area[p] > capacity) total += area[p];
      if (total > 0) {
        std::vector<long long> offsets(np_, 0);
        total = 0;
        for (int p : listed)
          if (area[p] > capacity) { offsets[p] = total; total += area[p]; }
        if (upload(&doff, offsets.data(), sizeof(long long) * np_, s)) { cleanup(); return 1; }
        GM_TRY(cudaStreamSynchronize(s));     // `offsets` is pageable and leaves scope here
      }
      GM_TRY(cudaMallocAsync(&dbig, sizeof(K) * (size_t)(total > 0 ? total : 1), s));
      zonal_select_kernel<T><<<poly_grid(n_listed), SEL_THREADS, smem_sel, s>>>(
          u.dev, (const T*)raster.dev, nd, has_nodata, (const float*)dthr, stat, q,
          (const long long*)darea, (const long long*)doff, (K*)dbig, (int)capacity, (float*)dout,
          (const int*)dlist, nullptr);
      GM_TRY(cudaGetLastError());
      count_launch();
    }
    GM_TRY(cudaMemcpyAsync(out, dout, sizeof(float) * np_, cudaMemcpyDeviceToHost, s));
  }
  GM_TRY(cudaStreamSynchronize(s));
  cleanup();
  return rc;
}

template <typename T>
static int run_zonal_values(PolyUpload& u, const Staged& raster, const void* nodata, int has_nodata,
                            const float* thresholds, const int64_t* counts, void* values_host,
                            cudaStream_t s) {
  const int64_t np_ = u.dev.n_polygons;
  std::vector<long long> offsets(np_ + 1, 0);
  for (int64_t p = 0; p < np_; ++p) offsets[p + 1] = offsets[p] + counts[p];
  const long long total = offsets[np_];
  if (np_ == 0 || total == 0) return 0;
  T nd = T(0);
  if (has_nodata) memcpy(&nd, nodata, sizeof(T));
  void *doff = nullptr, *dthr = nullptr, *dval = nullptr;
  int rc = upload(&doff, offsets.data(), sizeof(long long) * (np_ + 1), s);
  if (!rc && thresholds) rc = upload(&dthr, thresholds, sizeof(float) * np_, s);
  cudaError_t e = cudaSuccess;
  if (!rc) e = cudaMallocAsync(&dval, sizeof(T) * (size_t)total, s);
  if (!rc && e == cudaSuccess) {
    const size_t smem = scan_smem(u.dev.cap, PG_WARPS);
    if (smem > 48 * 1024)
      e = cudaFuncSetAttribute(zonal_values_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) {
      zonal_values_kernel<T><<<poly_grid(np_), PG_THREADS, smem, s>>>(
          u.dev, (const T*)raster.dev, nd, has_nodata, (const float*)dthr, (const long long*)doff, (T*)dval);
      e = cudaGetLastError();
      if (e == cudaSuccess) count_launch();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(values_host, dval, sizeof(T) * (size_t)total, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  }
  if (doff) cudaFreeAsync(doff, s);
  if (dthr) cudaFreeAsync(dthr, s);
  if (dval) cudaFreeAsync(dval, s);
  if (!rc && e != cudaSuccess) rc = fail(std::string("gm_zonal_values: ") + cudaGetErrorString(e));
  return rc;
}

template <typename T>
static int run_segment_select(const void* values, const int64_t* offsets, int64_t n_seg, int stat,
                              double q, float* out, cudaStream_t s) {
  typedef typename KeyOf<T>::type K;
  const int64_t total = offsets[n_seg];
  if (n_seg == 0) return 0;
  void *dval = nullptr, *doff = nullptr, *dkeys = nullptr, *dout = nullptr;
  int rc = upload(&dval, values, sizeof(T) * (size_t)total, s);
  if (!rc) rc = upload(&doff, offsets, sizeof(int64_t) * (n_seg + 1), s);
  cudaError_t e = cudaSuccess;
  if (!rc) e = cudaMallocAsync(&dkeys, sizeof(K) * (size_t)(total > 0 ? total : 1), s);
  if (!rc && e == cudaSuccess) e = cudaMallocAsync(&dout, sizeof(float) * n_seg, s);
  if (!rc && e == cudaSuccess) {
    segment_select_kernel<T><<<poly_grid(n_seg), SEL_THREADS, 0, s>>>(
        (const T*)dval, (const long long*)doff, n_seg, (K*)dkeys, stat, q, (float*)dout);
    e = cudaGetLastError();
    if (e == cudaSuccess) count_launch();
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, dout, sizeof(float) * n_seg, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  }
  void* all[] = {dval, doff, dkeys, dout};
  for (void* p : all) if (p) cudaFreeAsync(p, s);
  if (!rc && e != cudaSuccess) rc = fail(std::string("gm_segment_order_stat: ") + cudaGetErrorString(e));
  return rc;
}

// ---- multi-GPU reduce: partials that stay in HBM between the stripe pass and the all-reduce ----
// sums[3N] = (count, covered cells, sum) as float64 (counts are exact below 2^53) for ONE
// sum all-reduce, extremes[2N] = (min, -max) for ONE min all-reduce.
__global__ void zonal_pack_kernel(const GmZonalPartial* __restrict__ partial, const long long* __restrict__ cells,
                                  int64_t n, double* __restrict__ sums, double* __restrict__ extremes) {
  const int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (p >= n) return;
  const GmZonalPartial r = partial[p];
  sums[p] = (double)r.count; sums[n + p] = (double)cells[p]; sums[2 * n + p] = r.sum;
  extremes[p] = r.count > 0 ? r.vmin : DBL_MAX; extremes[n + p] = r.count > 0 ? -r.vmax : DBL_MAX;
}

__global__ void zonal_unpack_kernel(const double* __restrict__ sums, const double* __restrict__ extremes, int64_t n,
                                    int stat, float* __restrict__ out, long long* __restrict__ covered) {
  const int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (p >= n) return;
  const double count = sums[p];
  float v = __int_as_float(0x7fc00000);
  if (count > 0.0) {
    switch (stat) {
      case GM_STAT_COUNT: v = (float)count; break;
      case GM_STAT_SUM: v = (float)sums[2 * n + p]; break;
      case GM_STAT_MEAN: v = (float)(sums[2 * n + p] / count); break;
      case GM_STAT_MIN: v = (float)extremes[p]; break;
      case GM_STAT_MAX: v = (float)(-extremes[n + p]); break;
      default: break;
    }
  }
  out[p] = v;
  covered[p] = (long long)sums[n + p];
}

template <typename T>
static int run_zonal_partials_device(PolyUpload& u, const Staged& raster, const void* nodata, int has_nodata,
                                     const float* thresholds, double* sums, double* extremes, int stat,
                                     cudaStream_t s) {
  const int64_t np_ = u.dev.n_polygons;
  if (np_ == 0) return 0;
  T nd = T(0);
  if (has_nodata) memcpy(&nd, nodata, sizeof(T));
  void *darea = nullptr, *dthr = nullptr, *dpartial = nullptr, *dwork = nullptr;
  auto cleanup = [&]() {
    void* all[] = {darea, dthr, dpartial, dwork};
    for (void* p : all) if (p) cudaFreeAsync(p, s);
  };
  GM_TRY(cudaMallocAsync(&darea, sizeof(long long) * np_, s));
  GM_TRY(cudaMallocAsync(&dpartial, sizeof(GmZonalPartial) * np_, s));
  GM_TRY(cudaMallocAsync(&dwork, sizeof(int) * (size_t)(np_ + 2), s));
  GM_TRY(cudaMemsetAsync(dwork, 0, 2 * sizeof(int), s));
  // polygons without rows in this stripe are never visited: count 0 (zonal_pack_kernel turns
  // that into the neutral extremes)
  GM_TRY(cudaMemsetAsync(dpartial, 0, sizeof(GmZonalPartial) * np_, s));
  GM_TRY(cudaMemsetAsync(darea, 0, sizeof(long long) * np_, s));
  if (thresholds && upload(&dthr, thresholds, sizeof(float) * np_, s)) { cleanup(); return 1; }
  const size_t smem_scan = scan_smem(u.dev.cap, PG_WARPS);
  if (smem_scan > 48 * 1024)
    GM_TRY(cudaFuncSetAttribute(zonal_reduce_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_scan));
  // only what the statistic needs (a stripe call for the mean runs the sum-only kernel)
  const int need = stat == GM_STAT_MIN ? ZW_MIN : stat == GM_STAT_MAX ? ZW_MAX
                 : (stat == GM_STAT_SUM || stat == GM_STAT_MEAN || stat == GM_STAT_COUNT) ? ZW_SUM : ZW_ALL;
  GM_TRY(launch_reduce<T>(u, raster, nd, has_nodata, (const float*)dthr, need, poly_grid(np_ < 1024 ? np_ : 1024),
                          smem_scan, (GmZonalPartial*)dpartial, (long long*)darea, (int*)dwork, s));
  zonal_pack_kernel<<<(unsigned)((np_ + 255) / 256), 256, 0, s>>>(
      (const GmZonalPartial*)dpartial, (const long long*)darea, np_, sums, extremes);
  GM_TRY(cudaGetLastError());
  count_launch();
#undef GM_TRY
  cleanup();
  return 0;
}

}  // namespace gm

using namespace gm;

#define GM_RASTER_DISPATCH(dtype, CALL, WHAT)                                     \
  switch (dtype) {                                                                \
    case GM_U8: case GM_BOOL: { typedef uint8_t T; rc = CALL; break; }            \
    case GM_I8: { typedef int8_t T; rc = CALL; break; }                           \
    case GM_U16: { typedef uint16_t T; rc = CALL; break; }                        \
    case GM_I16: { typedef int16_t T; rc = CALL; break; }                         \
    case GM_U32: { typedef uint32_t T; rc = CALL; break; }                        \
    case GM_I32: { typedef int32_t T; rc = CALL; break; }                         \
    case GM_F32: { typedef float T; rc = CALL; break; }                           \
    case GM_F64: { typedef double T; rc = CALL; break; }                          \
    default: rc = fail(WHAT ": unsupported raster dtype");                        \
  }

extern "C" int gm_polygons_upload(const GmPolygons* polys, void** handle) {
  if (ensure_init()) return 1;
  if (!polys || !handle) return fail("gm_polygons_upload: null argument");
  cudaStream_t s = resolve_stream(nullptr);
  ResidentPolygons* r = new ResidentPolygons();
  r->n_polygons = polys->n_polygons; r->n_rings = polys->n_rings; r->n_vertices = polys->n_vertices;
  r->max_vertices = largest_polygon(polys);
  int rc = upload(&r->xy, polys->xy, sizeof(double) * 2 * r->n_vertices, s);
  if (!rc) rc = upload(&r->rings, polys->ring_offsets, sizeof(int64_t) * (r->n_rings + 1), s);
  if (!rc) rc = upload(&r->polys, polys->poly_offsets, sizeof(int64_t) * (r->n_polygons + 1), s);
  if (!rc && (cudaMalloc((void**)&r->error, sizeof(int)) != cudaSuccess ||
              cudaMemsetAsync(r->error, 0, sizeof(int), s) != cudaSuccess))
    rc = fail("gm_polygons_upload: no memory for the overflow flag");
  if (!rc && cudaStreamSynchronize(s) != cudaSuccess) rc = fail("gm_polygons_upload: copy failed");
  if (rc) {
    if (r->error) cudaFree(r->error);
    void* all[] = {r->xy, r->rings, r->polys};
    for (void* p : all) if (p) cudaFreeAsync(p, s);
    delete r;
    return 1;
  }
  *handle = r;
  return 0;
}

extern "C" int gm_polygons_free(void* handle) {
  if (!handle) return 0;
  ResidentPolygons* r = static_cast<ResidentPolygons*>(handle);
  cudaStream_t s = resolve_stream(nullptr);
  r->prepared.clear();
  if (r->error) cudaFree(r->error);
  void* all[] = {r->xy, r->rings, r->polys};
  for (void* p : all) if (p) cudaFreeAsync(p, s);
  delete r;
  return 0;
}

extern "C" int gm_zonal_values(const GmArray* raster, const void* nodata, int has_nodata,
                               const GmPolygons* polys, const double geo[6], const float* thresholds,
                               const int64_t* counts, void* values, void* stream) {
  if (ensure_init()) return 1;
  if (!raster || !polys || !counts || !values) return fail("gm_zonal_values: null argument");
  if (raster->shape[0] != 1) return fail("gm_zonal_values: one frame per call");
  cudaStream_t s = resolve_stream(stream);
  const int H = (int)raster->shape[1], W = (int)raster->shape[2];
  Staged in;
  PolyUpload u;
  int rc = in.open_input(*raster, s);
  if (!rc) rc = prepare_polygons(polys, geo, H, W, 0, H, u, s);
  if (!rc) {
    GM_RASTER_DISPATCH(raster->dtype, run_zonal_values<T>(u, in, nodata, has_nodata, thresholds, counts, values, s),
                       "gm_zonal_values")
  }
  if (!rc) rc = check_overflow(u, s);
  u.release();
  in.release();
  return rc;
}

extern "C" int gm_segment_order_stat(const void* values, int32_t dtype, const int64_t* offsets,
                                     int64_t n_segments, int stat, double q, float* out, void* stream) {
  if (ensure_init()) return 1;
  if (!offsets || !out || (n_segments > 0 && offsets[n_segments] > 0 && !values))
    return fail("gm_segment_order_stat: null argument");
  if (stat != GM_STAT_MEDIAN && stat != GM_STAT_PERCENTILE)
    return fail("gm_segment_order_stat: median or percentile expected");
  for (int64_t i = 0; i < n_segments; ++i)
    if (offsets[i + 1] - offsets[i] > 0x7fffffffLL) return fail("gm_segment_order_stat: segment too long");
  cudaStream_t s = resolve_stream(stream);
  int rc = 0;
  GM_RASTER_DISPATCH(dtype, run_segment_select<T>(values, offsets, n_segments, stat, q, out, s),
                     "gm_segment_order_stat")
  return rc;
}

extern "C" int gm_rasterize_polygons(const GmPolygons* polys, const double geo[6],
                                     const void* burn_values, const void* nodata, GmArray* dst,
                                     void* stream) {
  if (ensure_init()) return 1;
  if (!dst || !burn_values || !nodata) return fail("gm_rasterize_polygons: null argument");
  if (dst->shape[0] != 1) return fail("gm_rasterize_polygons: one band expected");
  cudaStream_t s = resolve_stream(stream);
  const int H = (int)dst->shape[1], W = (int)dst->shape[2];
  const int64_t n_pixels = (int64_t)H * W;
  Staged out;
  PolyUpload u;
  int rc = out.open_output(*dst, s);
  if (!rc && n_pixels > 0) {
    rc = prepare_polygons(polys, geo, H, W, 0, H, u, s);
    if (!rc) {
      switch (dst->dtype) {
        case GM_U8: case GM_BOOL: rc = run_rasterize<uint8_t>(u, burn_values, nodata, out, n_pixels, s); break;
        case GM_I32: rc = run_rasterize<int32_t>(u, burn_values, nodata, out, n_pixels, s); break;
        case GM_F64: rc = run_rasterize<double>(u, burn_values, nodata, out, n_pixels, s); break;
        case GM_F32: rc = run_rasterize<float>(u, burn_values, nodata, out, n_pixels, s); break;
        default: rc = fail("gm_rasterize_polygons: dtype must be uint8, int32, float32 or float64");
      }
    }
    if (!rc) rc = check_overflow(u, s);
    u.release();
  }
  if (!rc) rc = out.finish_output();
  const bool sync = out.owned;
  out.release();
  if (!rc && sync) GM_CUDA(cudaStreamSynchronize(s));
  return rc;
}

extern "C" int gm_zonal_stats(const GmArray* raster, const void* nodata, int has_nodata,
                              const GmPolygons* polys, const double geo[6], int stat, double q,
                              const float* thresholds, int64_t row_begin, int64_t row_end,
                              float* out, int64_t* covered, GmZonalPartial* partial, void* stream) {
  if (ensure_init()) return 1;
  if (!raster || !polys) return fail("gm_zonal_stats: null argument");
  if (raster->shape[0] != 1) return fail("gm_zonal_stats: one frame per call");
  if (stat < GM_STAT_SUM || stat > GM_STAT_PERCENTILE || stat == GM_STAT_STD || stat == GM_STAT_VAR)
    return fail("gm_zonal_stats: unsupported statistic");
  cudaStream_t s = resolve_stream(stream);
  const int H = (int)raster->shape[1], W = (int)raster->shape[2];
  if (row_begin < 0) row_begin = 0;
  if (row_end > H || row_end <= 0) row_end = H;
  Staged in;
  PolyUpload u;
  int rc = in.open_input(*raster, s);
  if (!rc) rc = prepare_polygons(polys, geo, H, W, row_begin, row_end, u, s, false, true);
  if (!rc) {
#define GM_Z(T) run_zonal<T>(u, in, nodata, has_nodata, stat, q, thresholds, out, covered, partial, s)
    switch (raster->dtype) {
      case GM_U8: case GM_BOOL: rc = GM_Z(uint8_t); break;
      case GM_I8: rc = GM_Z(int8_t); break;
      case GM_U16: rc = GM_Z(uint16_t); break;
      case GM_I16: rc = GM_Z(int16_t); break;
      case GM_U32: rc = GM_Z(uint32_t); break;
      case GM_I32: rc = GM_Z(int32_t); break;
      case GM_F32: rc = GM_Z(float); break;
      case GM_F64: rc = GM_Z(double); break;
      default: rc = fail("gm_zonal_stats: unsupported raster dtype");
    }
#undef GM_Z
  }
  if (!rc) rc = check_overflow(u, s);
  u.release();
  in.release();
  return rc;
}

extern "C" int gm_zonal_partials_device(const GmArray* raster, const void* nodata, int has_nodata,
                                        const GmPolygons* polys, const double geo[6],
                                        const float* thresholds, int64_t row_begin, int64_t row_end,
                                        double* sums, double* extremes, int stat, void* stream) {
  if (ensure_init()) return 1;
  if (!raster || !polys || !sums || !extremes) return fail("gm_zonal_partials_device: null argument");
  if (raster->shape[0] != 1) return fail("gm_zonal_partials_device: one frame per call");
  cudaStream_t s = resolve_stream(stream);
  const int H = (int)raster->shape[1], W = (int)raster->shape[2];
  if (row_begin < 0) row_begin = 0;
  if (row_end > H || row_end <= 0) row_end = H;
  Staged in;
  PolyUpload u;
  int rc = in.open_input(*raster, s);
  if (!rc) rc = prepare_polygons(polys, geo, H, W, row_begin, row_end, u, s, true);
  if (!rc) {
    GM_RASTER_DISPATCH(raster->dtype,
                       run_zonal_partials_device<T>(u, in, nodata, has_nodata, thresholds, sums, extremes, stat, s),
                       "gm_zonal_partials_device")
  }
  if (!rc) rc = check_overflow(u, s);
  u.release();
  in.release();
  return rc;
}

extern "C" int gm_zonal_finalize_device(const double* sums, const double* extremes, int64_t n_polygons,
                                        int stat, float* out, int64_t* covered, const GmPolygons* polys,
                                        void* stream) {
  if (ensure_init()) return 1;
  if (!sums || !extremes || !out || !covered) return fail("gm_zonal_finalize_device: null argument");
  if (n_polygons == 0) return 0;
  cudaStream_t s = resolve_stream(stream);
  // the stripe pass on a resident soup left its crossing-overflow flag on the device: it comes
  // back with the results, under the one synchronisation of this call
  ResidentPolygons* resident = polys ? static_cast<ResidentPolygons*>(const_cast<void*>(polys->resident)) : nullptr;
  int overflow = 0;
  void *dout = nullptr, *dcov = nullptr;
  GM_CUDA(cudaMallocAsync(&dout, sizeof(float) * n_polygons, s));
  GM_CUDA(cudaMallocAsync(&dcov, sizeof(long long) * n_polygons, s));
  zonal_unpack_kernel<<<(unsigned)((n_polygons + 255) / 256), 256, 0, s>>>(sums, extremes, n_polygons, stat,
                                                                          (float*)dout, (long long*)dcov);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) count_launch();
  if (e == cudaSuccess) e = cudaMemcpyAsync(out, dout, sizeof(float) * n_polygons, cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess) e = cudaMemcpyAsync(covered, dcov, sizeof(long long) * n_polygons, cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess && resident && resident->error)
    e = cudaMemcpyAsync(&overflow, resident->error, sizeof(int), cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  cudaFreeAsync(dout, s);
  cudaFreeAsync(dcov, s);
  if (e != cudaSuccess) return fail(std::string("gm_zonal_finalize_device: ") + cudaGetErrorString(e));
  if (overflow) {
    cudaMemsetAsync(resident->error, 0, sizeof(int), s);
    return fail("polygons: more than 4096 edge crossings (or 8 horizontal edges) on one scanline");
  }
  return 0;
}
