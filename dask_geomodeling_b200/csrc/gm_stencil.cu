// Spatial stencils of raster/spatial.py: HillShade, MovingMax, Dilate, Smooth.
// The source array carries the halo the reference block requested from its
// store (raster/spatial.py:27-108); every kernel reads (t, H+2m, W+2m) and
// writes the cropped (t, H, W).
#include "gm_common.cuh"
#include <cfloat>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <limits>
#include <algorithm>
#include <type_traits>
#include <cuda.h>          // CUtensorMap (types only: the encoder is fetched through the runtime)

namespace gm {


// ---- TMA tile staging ------------------------------------------------------------------------
// Stencil tiles with their halo are fetched by ONE cp.async.bulk.tensor (2-D tile mode) into
// shared memory and awaited on an mbarrier, instead of ~13 predicated loads per thread: the copy
// engine walks the rows, the threads only patch "no data" cells afterwards.  A tensor map needs
// a 16-byte aligned base and row pitch, so the TMA path is taken when the source window has
// such a pitch (the blocks ask their store for a window padded to it, see raster/spatial.py)
// and for tiles that lie wholly inside the window; everything else keeps the load path.
typedef CUresult (*TensorMapEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                         const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                         CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                         CUtensorMapFloatOOBfill);
static TensorMapEncodeTiled tensor_map_encoder() {
  static TensorMapEncodeTiled fn = []() -> TensorMapEncodeTiled {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      return nullptr;
    return reinterpret_cast<TensorMapEncodeTiled>(p);
  }();
  return fn;
}

// 2-D map over a (rows, cols) array of 4-byte cells with a row pitch of `pitch_cols` cells, box =
// (box_rows, box_cols).  Returns false when the array does not qualify (alignment) or the
// driver refuses; the caller then uses the load path.
static bool make_tile_map(CUtensorMap* map, const void* base, int64_t rows, int64_t cols, int64_t pitch_cols,
                          int box_rows, int box_cols, bool is_float) {
  if (getenv("GM_NO_TMA")) return false;
  TensorMapEncodeTiled encode = tensor_map_encoder();
  if (!encode || ((uintptr_t)base % 16) != 0 || (pitch_cols * 4) % 16 != 0 || (box_cols * 4) % 16 != 0 ||
      box_cols > 256 || box_rows > 256 || rows <= 0 || cols <= 0)
    return false;
  const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)pitch_cols * 4};
  const cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  const cuuint32_t elem[2] = {1, 1};
  return encode(map, is_float ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_INT32, 2,
                const_cast<void*>(base), dims, strides, box, elem, CU_TENSOR_MAP_INTERLEAVE_NONE,
                CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

__device__ __forceinline__ uint32_t st_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void st_mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(st_smem_u32(bar)), "r"(count));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void st_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(st_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void st_mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "ST_WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra ST_WAIT_DONE;\n"
      "bra ST_WAIT_LOOP;\n"
      "ST_WAIT_DONE:\n"
      "}\n" ::"r"(st_smem_u32(bar)), "r"(parity) : "memory");
}
// tile (x, y) of the map -> shared memory, completion counted on `bar`
__device__ __forceinline__ void st_tma_load_2d(void* smem_dst, const CUtensorMap* map, int x, int y, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
      ::"r"(st_smem_u32(smem_dst)), "l"(map), "r"(x), "r"(y), "r"(st_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void st_fence_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

template <typename T> static T read_scalar(const void* p) { T v; memcpy(&v, p, sizeof(T)); return v; }
static dim3 grid3(int W, int H, int bands, int bx, int by) {
  int gz = bands < 65535 ? bands : 65535;
  return dim3((W + bx - 1) / bx, (H + by - 1) / by, gz);
}

template <typename T> struct Lowest { static __host__ __device__ T value() { return std::numeric_limits<T>::lowest(); } };

// ---------------------------------------------------------------------------------
// HillShade (raster/spatial.py:353-417)
// ---------------------------------------------------------------------------------
// Horn gradient evaluated left to right in the array's dtype, divided by the
// resolution into float32, then the shading in float32 exactly in the order of
// the reference expression; the result is truncated to uint8.
template <typename T> struct HillArith;
// add2 / sub2: acc + 2 x and acc - 2 x.  Doubling is exact in binary floating point, so ONE fused
// multiply-add rounds exactly like the reference's separate product and sum.
template <> struct HillArith<float> {
  typedef float acc;
  static __device__ __forceinline__ float div(float v, double res) { return v / (float)res; }
  static __device__ __forceinline__ float mul(float v, double inv) { return v * (float)inv; }
  static __device__ __forceinline__ float add2(float acc_, float x) { return __fmaf_rn(2.0f, x, acc_); }
  static __device__ __forceinline__ float sub2(float acc_, float x) { return __fmaf_rn(-2.0f, x, acc_); }
};
template <> struct HillArith<double> {
  typedef double acc;
  static __device__ __forceinline__ float div(double v, double res) { return (float)(v / res); }
  static __device__ __forceinline__ float mul(double v, double inv) { return (float)(v * inv); }
  static __device__ __forceinline__ double add2(double acc_, double x) { return __fma_rn(2.0, x, acc_); }
  static __device__ __forceinline__ double sub2(double acc_, double x) { return __fma_rn(-2.0, x, acc_); }
};
template <typename T> struct HillArith {  // integer rasters: arithmetic wraps in T, division in double
  typedef T acc;
  static __device__ __forceinline__ float div(T v, double res) { return (float)((double)v / res); }
  static __device__ __forceinline__ float mul(T v, double inv) { return (float)((double)v * inv); }
  static __device__ __forceinline__ T add2(T acc_, T x) { return (T)(acc_ + (T)2 * x); }
  static __device__ __forceinline__ T sub2(T acc_, T x) { return (T)(acc_ - (T)2 * x); }
};

constexpr int HS_WARPS = 8;

template <typename A> __device__ __forceinline__ A shfl_down_any(A v, int d) {
  return __shfl_down_sync(0xffffffffu, v, d);
}
template <> __device__ __forceinline__ int8_t shfl_down_any<int8_t>(int8_t v, int d) { return (int8_t)__shfl_down_sync(0xffffffffu, (int)v, d); }
template <> __device__ __forceinline__ uint8_t shfl_down_any<uint8_t>(uint8_t v, int d) { return (uint8_t)__shfl_down_sync(0xffffffffu, (int)v, d); }
template <> __device__ __forceinline__ int16_t shfl_down_any<int16_t>(int16_t v, int d) { return (int16_t)__shfl_down_sync(0xffffffffu, (int)v, d); }
template <> __device__ __forceinline__ uint16_t shfl_down_any<uint16_t>(uint16_t v, int d) { return (uint16_t)__shfl_down_sync(0xffffffffu, (int)v, d); }
template <> __device__ __forceinline__ int64_t shfl_down_any<int64_t>(int64_t v, int d) { return (int64_t)__shfl_down_sync(0xffffffffu, (long long)v, d); }

// Four output columns per lane: the arithmetic per pixel is what it is (the reference's float32
// expression), but the work around it -- loads, shuffles, address steps, byte stores, loop
// control -- is shared by four pixels: a lane loads source columns 4m .. 4m+3 of a row, takes
// columns 4m+4, 4m+5 from its right-hand neighbour (two shuffles per row instead of two per
// pixel), and writes its four grey levels as ONE 32-bit store.  A warp covers 124 output
// columns per strip (lane 31 only feeds lane 30).  The Horn gradient and the two divisions
// are the reference's float32 expression; the shading uses the identity
//   sqrt(x^2+y^2) * sin(atan2(y, x) - az) = y*cos(az) - x*sin(az),
// fused multiply-adds and one hardware reciprocal square root (argument >= 1, 2^-22 relative
// error) -- a few ulp from the reference expression: SURVEY.md Appendix A-13 measured <= 1
// grey level on 4e-5 of the pixels for this form; the parity tests allow 1e-3.
constexpr int HQ_COLS = 124;   // output columns per warp
constexpr int HQ_ROWS = 64;
constexpr int HQ_AHEAD = 3;    // source rows fetched per batch (12 loads in flight per lane); a multiple of 3
static_assert(HQ_AHEAD % 3 == 0, "the ring of three row sets must close over a batch");

template <typename T, bool EXACT_INVERSE>
__global__ void __launch_bounds__(32 * HS_WARPS, 4)
hillshade_quad_kernel(const T* __restrict__ src, uint8_t* __restrict__ dst, T nodata, int has_nodata,
                      T fill, int bands, int H, int W, int SW, int quad_loads, double xres, double yres,
                      double inv_xres, double inv_yres, int dst_aligned,
                      float sin_alt, float cos_alt_zsf, float cos_az, float sin_az, float square_zsf) {
  // SW: columns of a source row (W + 2, or more when the window was padded to a 16-byte pitch);
  // quad_loads: 4-byte cells on that pitch -- a lane fetches its four columns with ONE 16-byte
  // load (they start at a multiple of four) instead of four loads 16 bytes apart
  typedef typename HillArith<T>::acc A;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t in_plane = (int64_t)(H + 2) * SW, out_plane = (int64_t)H * W;
  const int strips_x = (W + HQ_COLS - 1) / HQ_COLS;
  const int strips_y = (H + HQ_ROWS - 1) / HQ_ROWS;
  const int64_t strip = (int64_t)blockIdx.x * HS_WARPS + warp;
  if (strip >= (int64_t)bands * strips_y * strips_x) return;
  const int sx = (int)(strip % strips_x);
  const int sy = (int)((strip / strips_x) % strips_y);
  const int b = (int)(strip / ((int64_t)strips_x * strips_y));
  const int x0 = sx * HQ_COLS + 4 * lane, y0 = sy * HQ_ROWS;   // first output column of this lane
  const int rows = min(HQ_ROWS, H - y0);
  const int last_row = H + 1, last_col = SW - 1;
  const T* base = src + (int64_t)b * in_plane;
  // source columns of this lane, clamped into the array (clamped values only feed outputs
  // that are not written)
  int col[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) col[j] = min(x0 + j, last_col);
  auto clean = [&](T v) -> A { return (A)((has_nodata && v == nodata) ? fill : v); };
  const bool quad = sizeof(T) == 4 && quad_loads && x0 + 3 <= last_col;
  auto fetch = [&](int row, T (&v)[4]) {
    const T* p = base + (int64_t)min(row, last_row) * SW;
    if (sizeof(T) == 4 && quad) {
      const uint4 q = __ldg(reinterpret_cast<const uint4*>(p + x0));
      memcpy(&v[0], &q, 16);
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j) v[j] = __ldg(p + col[j]);
    }
  };
  auto load_row = [&](int row, A (&w)[6]) {
    T v[4];
    fetch(row, v);
#pragma unroll
    for (int j = 0; j < 4; ++j) w[j] = clean(v[j]);
    w[4] = shfl_down_any<A>(w[0], 1);
    w[5] = shfl_down_any<A>(w[1], 1);
  };
  // three live source rows in a ring of three register sets: a batch of HQ_AHEAD rows (a multiple
  // of 3) returns every set to its role, so no row is ever moved between registers
  A ring[3][6];
  load_row(y0, ring[0]);
  load_row(y0 + 1, ring[1]);
  const bool lane_writes = lane < 31 && x0 < W;
  const bool whole_quad = dst_aligned && x0 + 3 < W;
  uint8_t* o = dst + (int64_t)b * out_plane + (int64_t)y0 * W + x0;
  for (int r0 = 0; r0 < rows; r0 += HQ_AHEAD) {
    T next[HQ_AHEAD][4];
#pragma unroll
    for (int i = 0; i < HQ_AHEAD; ++i) fetch(y0 + r0 + i + 2, next[i]);
#pragma unroll
    for (int i = 0; i < HQ_AHEAD; ++i) {
      const int r = r0 + i;
      A (&a)[6] = ring[i % 3];
      A (&m)[6] = ring[(i + 1) % 3];
      A (&c)[6] = ring[(i + 2) % 3];
#pragma unroll
      for (int j = 0; j < 4; ++j) c[j] = clean(next[i][j]);
      c[4] = shfl_down_any<A>(c[0], 1);
      c[5] = shfl_down_any<A>(c[1], 1);
      unsigned packed = 0;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        // s0 s1 s2 = a[j..j+2] ; s3 . s5 = m[j], m[j+2] ; s6 s7 s8 = c[j..j+2]
        // gy = ((((s0 + 2 s1) + s2) - s6) - 2 s7) - s8 ; gx = ((((s0 + 2 s3) + s6) - s2) - 2 s5) - s8
        const A gy = HillArith<T>::sub2((HillArith<T>::add2(a[j], a[j + 1]) + a[j + 2]) - c[j], c[j + 1]) - c[j + 2];
        const A gx = HillArith<T>::sub2((HillArith<T>::add2(a[j], m[j]) + c[j]) - a[j + 2], m[j + 2]) - c[j + 2];
        float fy, fx;
        if (EXACT_INVERSE) {
          fy = HillArith<T>::mul((T)gy, inv_yres);
          fx = HillArith<T>::mul((T)gx, inv_xres);
        } else {
          fy = HillArith<T>::div((T)gy, yres);
          fx = HillArith<T>::div((T)gx, xres);
        }
        const float xx_plus_yy = __fmaf_rn(fx, fx, fy * fy);
        const float num = __fmaf_rn(-cos_alt_zsf, __fmaf_rn(fy, cos_az, -(fx * sin_az)), sin_alt);
        float inv_len;
        asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(inv_len) : "f"(__fmaf_rn(square_zsf, xx_plus_yy, 1.0f)));
        const float cang = num * inv_len;
        // np.where(cang <= 0, 0, 255 * cang).astype(uint8): the unsigned conversion truncates and
        // sends negative products (and NaN) to 0 by itself -- no compare / select
        const unsigned out = __float2uint_rz(255.0f * cang) & 0xffu;
        packed |= out << (8 * j);
      }
      if (lane_writes && r < rows) {
        uint8_t* q = o + (int64_t)r * W;
        if (whole_quad) {
          *reinterpret_cast<unsigned*>(q) = packed;
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (x0 + j < W) q[j] = (uint8_t)(packed >> (8 * j));
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------
// MovingMax (raster/spatial.py:192-213): circular footprint, chord per row
// ---------------------------------------------------------------------------------
// Tiled version for radii up to MM2_MAXR.  The disc is a stack of horizontal chords
// with only a few distinct half-widths (size 11: 2, 3, 4, 5), so per tile
//   1. the source tile + halo goes to shared memory (no data -> dtype minimum),
//   2. every tile row gets its running maximum over each distinct chord width
//      (one pass outwards from the centre, nested windows reuse the same loads),
//   3. an output pixel is the maximum of 2r+1 chord maxima, one per footprint row.
// 11 + K + 11 shared-memory accesses per pixel instead of the 97 taps of the disc.
constexpr int MM2_TX = 64, MM2_TY = 32, MM2_MAXR = 8, MM2_MAXK = MM2_MAXR + 1;
struct MMFootprint {
  int n_widths;
  int width[MM2_MAXK];            // distinct chord half-widths, ascending
  int level[2 * MM2_MAXR + 1];    // footprint row dy + r -> index into width[], -1: not in the disc
};

template <typename T>
__global__ void __launch_bounds__(256)
moving_max_tiled_kernel(const T* __restrict__ src, T* __restrict__ dst, T nodata, int has_nodata,
                        int bands, int H, int W, int r, const __grid_constant__ MMFootprint fp) {
  extern __shared__ __align__(16) unsigned char mm_smem[];
  const int tw = MM2_TX + 2 * r, th = MM2_TY + 2 * r;
  T* tile = reinterpret_cast<T*>(mm_smem);             // th x tw
  T* chord = tile + (size_t)th * tw;                   // n_widths x th x MM2_TX
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int SW = W + 2 * r, SH = H + 2 * r;
  const int64_t in_plane = (int64_t)SH * SW, out_plane = (int64_t)H * W;
  const int x0 = blockIdx.x * MM2_TX, y0 = blockIdx.y * MM2_TY;
  const T lowest = Lowest<T>::value();
  const int wmax = fp.width[fp.n_widths - 1];
  for (int b = blockIdx.z; b < bands; b += gridDim.z) {
    const T* plane = src + (int64_t)b * in_plane;
    __syncthreads();
    for (int ty = warp; ty < th; ty += 8) {
      const int gy = y0 + ty;
      for (int tx = lane; tx < tw; tx += 32) {
        const int gx = x0 + tx;
        T v = lowest;
        if (gy < SH && gx < SW) {
          v = __ldg(plane + (int64_t)gy * SW + gx);
          if (has_nodata && v == nodata) v = lowest;
        }
        tile[ty * tw + tx] = v;
      }
    }
    __syncthreads();
    for (int ty = warp; ty < th; ty += 8) {
      for (int tx = lane; tx < MM2_TX; tx += 32) {
        const T* c = tile + ty * tw + tx + r;
        T m = c[0];
        int k = 0;
        if (fp.width[0] == 0) { chord[(size_t)ty * MM2_TX + tx] = m; k = 1; }
        for (int d = 1; d <= wmax; ++d) {
          const T lo = c[-d], hi = c[d];
          m = lo > m ? lo : m;
          m = hi > m ? hi : m;
          if (d == fp.width[k]) { chord[((size_t)k * th + ty) * MM2_TX + tx] = m; ++k; }
        }
      }
    }
    __syncthreads();
    for (int ty = warp; ty < MM2_TY; ty += 8) {
      const int y = y0 + ty;
      if (y >= H) break;
      for (int tx = lane; tx < MM2_TX; tx += 32) {
        const int x = x0 + tx;
        if (x >= W) break;
        T best = lowest;
        for (int dy = 0; dy <= 2 * r; ++dy) {
          const int k = fp.level[dy];
          if (k < 0) continue;
          const T v = chord[((size_t)k * th + ty + dy) * MM2_TX + tx];
          best = v > best ? v : best;
        }
        // restore no data only where the centre was no data and nothing was found
        if (has_nodata && best == lowest &&
            __ldg(plane + (int64_t)(y + r) * SW + (x + r)) == nodata)
          best = nodata;
        dst[(int64_t)b * out_plane + (int64_t)y * W + x] = best;
      }
    }
  }
}


// max as one FMNMX / IMNMX.  For floats this differs from `v > m ? v : m` only when a NaN is
// present, which cannot happen here: sources turn NaN into no data (raster/sources.py:148)
// and every element-wise block replaces non-finite results by its fill value.
template <typename T> __device__ __forceinline__ T vmax(T a, T b) { return a > b ? a : b; }
template <> __device__ __forceinline__ float vmax<float>(float a, float b) { return fmaxf(a, b); }
template <> __device__ __forceinline__ double vmax<double>(double a, double b) { return fmax(a, b); }

// Compile-time footprint for the usual odd sizes: the three phases of the tiled kernel
// fully unrolled (no footprint look-ups, no branches): 11 + 11 shared loads, 4 shared stores
// and 21 max per pixel at size 11.
template <int SIZE> struct Disc {
  static constexpr int R = SIZE / 2;
  // chord half-width of footprint row dy: largest dx with dx^2 + dy^2 < (SIZE/2)^2, -1 if none
  static constexpr int half_width(int dy) {
    int w = -1;
    for (int dx = 0; dx <= R; ++dx)
      if (4 * (dx * dx + dy * dy) < SIZE * SIZE) w = dx;
    return w;
  }
  static constexpr bool used(int d) {
    for (int dy = -R; dy <= R; ++dy)
      if (half_width(dy) == d) return true;
    return false;
  }
  static constexpr int plane_of(int d) {   // index of width d among the used widths
    int k = 0;
    for (int e = 0; e < d; ++e) k += used(e) ? 1 : 0;
    return k;
  }
  static constexpr int n_planes() { return plane_of(R + 1); }
  static constexpr int wmax() { return half_width(0); }
};

template <typename T, int SIZE, int D>
__device__ __forceinline__ void chord_steps(const T* c, T& m, T* chord_px, int plane_stride) {
  if constexpr (D <= Disc<SIZE>::wmax()) {
    if constexpr (D > 0) {
      m = vmax<T>(m, vmax<T>(c[-D], c[D]));
    }
    if constexpr (Disc<SIZE>::used(D)) chord_px[Disc<SIZE>::plane_of(D) * plane_stride] = m;
    chord_steps<T, SIZE, D + 1>(c, m, chord_px, plane_stride);
  }
}

template <typename T, int SIZE, int DY>
__device__ __forceinline__ void disc_rows(const T* chord_px, int plane_stride, T& best) {
  constexpr int R = Disc<SIZE>::R;
  if constexpr (DY <= R) {
    constexpr int w = Disc<SIZE>::half_width(DY);
    if constexpr (w >= 0) {
      best = vmax<T>(best, chord_px[Disc<SIZE>::plane_of(w) * plane_stride + (DY + R) * MM2_TX]);
    }
    disc_rows<T, SIZE, DY + 1>(chord_px, plane_stride, best);
  }
}

template <typename T, int SIZE>
__global__ void __launch_bounds__(256)
moving_max_fixed_kernel(const T* __restrict__ src, T* __restrict__ dst, T nodata, int has_nodata,
                        int bands, int H, int W) {
  extern __shared__ __align__(16) unsigned char mm_smem[];
  constexpr int R = Disc<SIZE>::R;
  constexpr int TW = MM2_TX + 2 * R, TH = MM2_TY + 2 * R;
  constexpr int PLANE = TH * MM2_TX;
  T* tile = reinterpret_cast<T*>(mm_smem);             // TH x TW
  T* chord = tile + TH * TW;                           // n_planes x TH x MM2_TX
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int SW = W + 2 * R, SH = H + 2 * R;
  const int64_t in_plane = (int64_t)SH * SW, out_plane = (int64_t)H * W;
  const int x0 = blockIdx.x * MM2_TX, y0 = blockIdx.y * MM2_TY;
  const T lowest = Lowest<T>::value();
  for (int b = blockIdx.z; b < bands; b += gridDim.z) {
    const T* plane = src + (int64_t)b * in_plane;
    __syncthreads();
    // unconditional (clamped) loads, two tile rows per round: six requests in flight
    // per thread before the first value is tested
    constexpr int NJ = (TW + 31) / 32;
    for (int ty = warp; ty < TH; ty += 16) {
      T raw[2][NJ];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int gy = min(y0 + ty + 8 * h, SH - 1);
#pragma unroll
        for (int j = 0; j < NJ; ++j)
          raw[h][j] = __ldg(plane + (int64_t)gy * SW + min(x0 + lane + 32 * j, SW - 1));
      }
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int row = ty + 8 * h;
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
          const int tx = lane + 32 * j;
          const bool inside = y0 + row < SH && x0 + tx < SW;
          const T v = (!inside || (has_nodata && raw[h][j] == nodata)) ? lowest : raw[h][j];
          if (tx < TW && row < TH) tile[row * TW + tx] = v;
        }
      }
    }
    __syncthreads();
    for (int ty = warp; ty < TH; ty += 8) {
#pragma unroll
      for (int j = 0; j < MM2_TX / 32; ++j) {
        const int tx = lane + 32 * j;
        const T* c = tile + ty * TW + tx + R;
        T m = c[0];
        chord_steps<T, SIZE, 0>(c, m, chord + ty * MM2_TX + tx, PLANE);
      }
    }
    __syncthreads();
    for (int ty = warp; ty < MM2_TY; ty += 8) {
      const int y = y0 + ty;
      if (y >= H) break;
#pragma unroll
      for (int j = 0; j < MM2_TX / 32; ++j) {
        const int tx = lane + 32 * j;
        const int x = x0 + tx;
        if (x < W) {
          T best = lowest;
          disc_rows<T, SIZE, -R>(chord + ty * MM2_TX + tx, PLANE, best);
          if (has_nodata && best == lowest &&
              __ldg(plane + (int64_t)(y + R) * SW + (x + R)) == nodata)
            best = nodata;
          dst[(int64_t)b * out_plane + (int64_t)y * W + x] = best;
        }
      }
    }
  }
}

template <typename T, int SIZE>
static int launch_moving_max_fixed(const Staged& in, Staged& out, T nd, int has_nodata, int bands,
                                   int H, int W, cudaStream_t s) {
  constexpr int R = Disc<SIZE>::R;
  const size_t smem = ((size_t)(MM2_TX + 2 * R) * (MM2_TY + 2 * R) +
                       (size_t)Disc<SIZE>::n_planes() * (MM2_TY + 2 * R) * MM2_TX) * sizeof(T);
  auto kernel = moving_max_fixed_kernel<T, SIZE>;
  if (smem > 48 * 1024)
    GM_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kernel<<<grid3(W, H, bands, MM2_TX, MM2_TY), 256, smem, s>>>((const T*)in.dev, (T*)out.dev, nd,
                                                               has_nodata, bands, H, W);
  GM_LAUNCH_CHECK();
  return 0;
}

// 16-byte groups of four 4-byte cells (conflict-free shared-memory accesses)
template <typename T> struct Quad { T v[4]; };
template <typename T> __device__ __forceinline__ T vmin4(const T (&v)[4]) {
  const T a = v[0] < v[1] ? v[0] : v[1], b = v[2] < v[3] ? v[2] : v[3];
  return a < b ? a : b;
}
template <typename T> __device__ __forceinline__ Quad<T> lds_quad(const T* p) {
  Quad<T> q;
  const uint4 u = *reinterpret_cast<const uint4*>(p);
  memcpy(&q, &u, 16);
  return q;
}
template <typename T> __device__ __forceinline__ void sts_quad(T* p, const Quad<T>& q) {
  uint4 u;
  memcpy(&u, &q, 16);
  *reinterpret_cast<uint4*>(p) = u;
}

// Register-blocked version for 4-byte rasters: ONE phase after the tile is staged.  A
// thread owns 4 adjacent columns x MMB_ROWS rows of outputs and walks the MMB_ROWS + 2R tile rows
// they depend on: per tile row it reads its 4 + 2R values once (NQ conflict-free LDS.128), grows
// the nested chord maxima of its four columns in registers and folds the chord that footprint row
// dy = (tile row - output row) asks for into each of the (up to 2R + 1) output rows in reach.
// No chord planes in shared memory: 4 NQ (MMB_ROWS + 2R) / MMB_ROWS bytes of shared-memory reads per
// pixel (36 at size 11) instead of 92, and one block barrier per tile instead of three.
constexpr int MMB_TX = 128, MMB_ROWS = 8, MMB_TY = 8 * MMB_ROWS;

template <typename T, int SIZE, int D>
__device__ __forceinline__ void chord_regs(const T* w, T (&m)[4], T (*c)[4]) {
  constexpr int R = Disc<SIZE>::R;
  if constexpr (D <= Disc<SIZE>::wmax()) {
    if constexpr (D > 0) {
#pragma unroll
      for (int i = 0; i < 4; ++i) m[i] = vmax<T>(m[i], vmax<T>(w[R + i - D], w[R + i + D]));
    }
    if constexpr (Disc<SIZE>::used(D)) {
#pragma unroll
      for (int i = 0; i < 4; ++i) c[Disc<SIZE>::plane_of(D)][i] = m[i];
    }
    chord_regs<T, SIZE, D + 1>(w, m, c);
  }
}

template <typename T> __device__ __forceinline__ T vmax3(T a, T b, T c) { return vmax<T>(a, vmax<T>(b, c)); }

// folds the chords of tile rows RW (c0) and RW + 1 (c1) into output row J: one 3-input maximum
// when both rows are in the footprint of that output row
template <typename T, int SIZE, int RW, int J>
__device__ __forceinline__ void fold_rows(T (*c0)[4], T (*c1)[4], T (*best)[4]) {
  constexpr int R = Disc<SIZE>::R;
  if constexpr (J < MMB_ROWS) {
    constexpr int dy0 = RW - J - R, dy1 = dy0 + 1;
    constexpr int hw0 = (dy0 >= -R && dy0 <= R) ? Disc<SIZE>::half_width(dy0 < 0 ? -dy0 : dy0) : -1;
    constexpr int hw1 = (dy1 >= -R && dy1 <= R && RW + 1 < MMB_ROWS + 2 * R) ? Disc<SIZE>::half_width(dy1 < 0 ? -dy1 : dy1) : -1;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if constexpr (hw0 >= 0 && hw1 >= 0)
        best[J][i] = vmax3<T>(best[J][i], c0[Disc<SIZE>::plane_of(hw0)][i], c1[Disc<SIZE>::plane_of(hw1)][i]);
      else if constexpr (hw0 >= 0)
        best[J][i] = vmax<T>(best[J][i], c0[Disc<SIZE>::plane_of(hw0)][i]);
      else if constexpr (hw1 >= 0)
        best[J][i] = vmax<T>(best[J][i], c1[Disc<SIZE>::plane_of(hw1)][i]);
    }
    fold_rows<T, SIZE, RW, J + 1>(c0, c1, best);
  }
}

template <typename T, int SIZE, int TW, int RW>
__device__ __forceinline__ void row_chords(const T* seg, T (*c)[4]) {
  constexpr int R = Disc<SIZE>::R;
  constexpr int NQ = (4 + 2 * R + 3) / 4;
  if constexpr (RW < MMB_ROWS + 2 * R) {
    T w[4 * NQ];
#pragma unroll
    for (int k = 0; k < NQ; ++k) {
      const Quad<T> q = lds_quad<T>(seg + RW * TW + 4 * k);
#pragma unroll
      for (int i = 0; i < 4; ++i) w[4 * k + i] = q.v[i];
    }
    T m[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) m[i] = w[R + i];
    chord_regs<T, SIZE, 0>(w, m, c);
  }
}

template <typename T, int SIZE, int TW, int RW>
__device__ __forceinline__ void walk_rows(const T* seg, T (*best)[4]) {
  constexpr int R = Disc<SIZE>::R;
  if constexpr (RW < MMB_ROWS + 2 * R) {
    T c0[Disc<SIZE>::n_planes()][4], c1[Disc<SIZE>::n_planes()][4];
    row_chords<T, SIZE, TW, RW>(seg, c0);
    row_chords<T, SIZE, TW, RW + 1>(seg, c1);
    fold_rows<T, SIZE, RW, 0>(c0, c1, best);
    walk_rows<T, SIZE, TW, RW + 2>(seg, best);
  }
}

// Tiles are walked by persistent blocks (two per SM), x fastest so that the blocks running at
// one time share their halos in L2.  Two tile buffers per block: the bulk tensor copy of tile
// k + 1 is issued before tile k is computed, so its latency hides behind the arithmetic.
template <typename T, int SIZE>
__global__ void __launch_bounds__(256, 2)
moving_max_block_kernel(const T* __restrict__ src, T* __restrict__ dst, T nodata, int has_nodata,
                        int bands, int H, int W, int SW, int dst_aligned, int use_tma,
                        const __grid_constant__ CUtensorMap tile_map) {
  static_assert(sizeof(T) == 4, "quads of four 4-byte cells");
  extern __shared__ __align__(128) unsigned char mm_smem[];
  __shared__ __align__(8) uint64_t tile_bar[2];
  constexpr int R = Disc<SIZE>::R;
  constexpr int NQ = (4 + 2 * R + 3) / 4;                // quads per segment window
  constexpr int TW = MMB_TX - 4 + 4 * NQ;                // tile row stride: every window in bounds
  constexpr int TH = MMB_TY + 2 * R;
  constexpr int TILE_BYTES = (TH * TW * (int)sizeof(T) + 127) / 128 * 128;
  // (the bulk tensor copy wants a 128-byte aligned destination: 128 spare bytes are allocated)
  unsigned char* base = mm_smem + ((128u - (st_smem_u32(mm_smem) & 127u)) & 127u);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int SH = H + 2 * R;                 // SW >= W + 2 R: the window may carry pitch padding
  const int64_t in_plane = (int64_t)SH * SW, out_plane = (int64_t)H * W;
  const int tiles_x = (W + MMB_TX - 1) / MMB_TX, tiles_y = (H + MMB_TY - 1) / MMB_TY;
  const int64_t n_tiles = (int64_t)tiles_x * tiles_y * bands;
  const T lowest = Lowest<T>::value();
  uint32_t phases = 0u;                     // bit i: parity to wait for on tile_bar[i]
  if (use_tma) {
    if (threadIdx.x == 0) {
      st_mbar_init(&tile_bar[0], 1);
      st_mbar_init(&tile_bar[1], 1);
    }
    __syncthreads();
  }
  // tile t -> (band, y0, x0); a tile takes the bulk copy when it lies wholly inside the window
  auto locate = [&](int64_t t, int& b, int& y0, int& x0) {
    const int64_t per_band = (int64_t)tiles_x * tiles_y;
    b = (int)(t / per_band);
    const int r = (int)(t - b * per_band);
    y0 = (r / tiles_x) * MMB_TY;
    x0 = (r % tiles_x) * MMB_TX;
    return use_tma && x0 + TW <= SW && y0 + TH <= SH;
  };
  auto prefetch = [&](int64_t t, int buf) {
    int b, y0, x0;
    if (t < n_tiles && locate(t, b, y0, x0) && threadIdx.x == 0) {
      st_mbar_expect_tx(&tile_bar[buf], (uint32_t)(TH * TW * sizeof(T)));
      st_tma_load_2d(base + buf * TILE_BYTES, &tile_map, x0, b * SH + y0, &tile_bar[buf]);
    }
  };
  prefetch(blockIdx.x, 0);
  int buf = 0;
  for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x, buf ^= 1) {
    int b, y0, x0;
    const bool bulk = locate(t, b, y0, x0);
    const T* plane = src + (int64_t)b * in_plane;
    T* tile = reinterpret_cast<T*>(base + buf * TILE_BYTES);    // TH x TW
    // every thread is done with the other buffer (tile t - gridDim.x): its next tile may land
    if (use_tma) st_fence_async();
    __syncthreads();
    prefetch(t + gridDim.x, buf ^ 1);
    if (bulk) {
      st_mbar_wait(&tile_bar[buf], (phases >> buf) & 1u);
      phases ^= 1u << buf;
      if (has_nodata) {     // "no data" -> lowest, in place, a quad at a time
        constexpr int QUADS = TH * TW / 4;
        for (int i = threadIdx.x; i < QUADS; i += 256) {
          Quad<T> q = lds_quad<T>(tile + 4 * i);
          bool hit = false;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const bool nd = q.v[j] == nodata;
            q.v[j] = nd ? lowest : q.v[j];
            hit |= nd;
          }
          if (hit) sts_quad<T>(tile + 4 * i, q);
        }
      }
    } else {
      // clamped loads, four tile rows in flight per warp
      constexpr int NJ = (TW + 31) / 32;
      for (int ty = warp; ty < TH; ty += 32) {
        T raw[4][NJ];
#pragma unroll
        for (int h = 0; h < 4; ++h) {
          const int gy = min(y0 + ty + 8 * h, SH - 1);
#pragma unroll
          for (int j = 0; j < NJ; ++j)
            raw[h][j] = __ldg(plane + (int64_t)gy * SW + min(x0 + lane + 32 * j, SW - 1));
        }
#pragma unroll
        for (int h = 0; h < 4; ++h) {
          const int row = ty + 8 * h;
#pragma unroll
          for (int j = 0; j < NJ; ++j) {
            const int tx = lane + 32 * j;
            const bool in = y0 + row < SH && x0 + tx < SW;
            const T v = (!in || (has_nodata && raw[h][j] == nodata)) ? lowest : raw[h][j];
            if (tx < TW && row < TH) tile[row * TW + tx] = v;
          }
        }
      }
    }
    if (has_nodata || !bulk) __syncthreads();
    const int ty0 = warp * MMB_ROWS, x = x0 + 4 * lane;
    if (y0 + ty0 >= H || x >= W) continue;
    T best[MMB_ROWS][4];
#pragma unroll
    for (int j = 0; j < MMB_ROWS; ++j)
#pragma unroll
      for (int i = 0; i < 4; ++i) best[j][i] = lowest;
    walk_rows<T, SIZE, TW, 0>(tile + ty0 * TW + 4 * lane, best);
#pragma unroll
    for (int j = 0; j < MMB_ROWS; ++j) {
      const int y = y0 + ty0 + j;
      if (y >= H) break;
      // restore no data only where the centre was no data and nothing was found (rare: one test
      // for the quad)
      if (has_nodata && vmin4(best[j]) == lowest) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
          if (best[j][i] == lowest && x + i < W &&
              __ldg(plane + (int64_t)(y + R) * SW + (x + i + R)) == nodata)
            best[j][i] = nodata;
      }
      T* o = dst + (int64_t)b * out_plane + (int64_t)y * W + x;
      if (dst_aligned && x + 3 < W) {
        Quad<T> q;
#pragma unroll
        for (int i = 0; i < 4; ++i) q.v[i] = best[j][i];
        uint4 u;
        memcpy(&u, &q, 16);
        __stcs(reinterpret_cast<uint4*>(o), u);
      } else {
#pragma unroll
        for (int i = 0; i < 4; ++i)
          if (x + i < W) o[i] = best[j][i];
      }
    }
  }
}

template <typename T, int SIZE>
static int launch_moving_max_block(const Staged& in, Staged& out, T nd, int has_nodata, int bands,
                                   int H, int W, int SW, cudaStream_t s) {
  constexpr int R = Disc<SIZE>::R;
  constexpr int NQ = (4 + 2 * R + 3) / 4;
  constexpr int TW = MMB_TX - 4 + 4 * NQ, TH = MMB_TY + 2 * R;
  constexpr size_t TILE_BYTES = ((size_t)TW * TH * sizeof(T) + 127) / 128 * 128;
  const size_t smem = 2 * TILE_BYTES + 128;
  auto kernel = moving_max_block_kernel<T, SIZE>;
  static int sms = 0;
  if (!sms) {
    int dev = 0;
    GM_CUDA(cudaGetDevice(&dev));
    GM_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  }
  GM_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int aligned = ((uintptr_t)out.dev % 16 == 0) && (W % 4 == 0);
  static_assert((TW * TH) % 4 == 0 && (TW * sizeof(T)) % 16 == 0, "tile rows are whole 16-byte groups");
  CUtensorMap map;
  memset(&map, 0, sizeof(map));
  const int SH = H + 2 * R;
  const int use_tma = make_tile_map(&map, in.dev, (int64_t)bands * SH, SW, SW, TH, TW, std::is_same<T, float>::value);
  const int64_t n_tiles = (int64_t)((W + MMB_TX - 1) / MMB_TX) * ((H + MMB_TY - 1) / MMB_TY) * bands;
  const int grid = (int)std::min<int64_t>(n_tiles, 2 * (int64_t)sms);
  kernel<<<grid, 256, smem, s>>>((const T*)in.dev, (T*)out.dev, nd, has_nodata, bands, H, W, SW, aligned,
                                 use_tma, map);
  GM_LAUNCH_CHECK();
  return 0;
}

// 0: launched, 1: error, -1: no compile-time footprint for this dtype / size
template <typename T>
static int try_moving_max_fixed(int size, const Staged& in, Staged& out, T nd, int has_nodata,
                                int bands, int H, int W, int SW, cudaStream_t s) {
  if constexpr (std::is_same<T, float>::value || std::is_same<T, double>::value ||
                std::is_same<T, int16_t>::value || std::is_same<T, uint8_t>::value ||
                std::is_same<T, int32_t>::value) {
    if constexpr (sizeof(T) == 4) {
      switch (size) {
#define GM_CASE(N) case N: return launch_moving_max_block<T, N>(in, out, nd, has_nodata, bands, H, W, SW, s);
        GM_CASE(3) GM_CASE(5) GM_CASE(7) GM_CASE(9) GM_CASE(11) GM_CASE(13) GM_CASE(15)
#undef GM_CASE
        default: break;
      }
    }
    if (SW != W + 2 * (size / 2)) return -1;   // only the quad kernel reads a padded pitch
    switch (size) {
#define GM_CASE(N) case N: return launch_moving_max_fixed<T, N>(in, out, nd, has_nodata, bands, H, W, s);
      GM_CASE(3) GM_CASE(5) GM_CASE(7) GM_CASE(9) GM_CASE(11) GM_CASE(13) GM_CASE(15)
#undef GM_CASE
      default: break;
    }
  }
  return -1;
}

// Radii above 8, 8-byte cells from radius 7, and radius <= 8 where the tiled kernel's tile does
// not fit; any dtype, no size cap: the disc as 2r + 1 chords, each chord an O(1) range-maximum query.
// A block owns MMC_TX output columns x MMC_GROUPS * MMC_ROWS output rows and streams the
// source rows they depend on from top to bottom.  Per source row
//   1. the segment of MMC_TX + 2r cells is staged as level 0 (no data -> dtype minimum); the
//      loads of the next row are issued before this row's levels are built,
//   2. level k of the range-maximum ("sparse") table holds at p the maximum of cells
//      [p, p + 2^k), built from level k - 1 with one barrier per level,
//   3. a chord [x - w, x + w] of footprint row dy is max(M_k[x - w], M_k[x + w - 2^k + 1]),
//      k = floor(log2(2w + 1)); the host table `chord` holds both offsets per dy, and every
//      thread folds into the output rows of its group in reach one 3-input maximum per column.
// A thread keeps the running maxima of MMC_ROWS rows x MMC_COLS columns in registers.
// Work per pixel: 2r + 1 chords of two shared loads each, plus the table build, about
// log2(2r + 1) operations per staged cell shared by the block's rows.  Shared memory:
// levels x (MMC_TX + 2r) cells; the limit that leaves is checked on the host.
constexpr int MMC_THREADS = 256, MMC_GROUPS = 4, MMC_GROUP = MMC_THREADS / MMC_GROUPS, MMC_COLS = 4;
constexpr int MMC_TX = MMC_GROUP * MMC_COLS;   // 256 output columns
constexpr int MMC_ROWS = 8;                    // output rows per group: MMC_GROUPS * 8 per block
constexpr int MMC_PREFETCH = 8;                // staged cells per thread held in registers

template <typename T, bool FULL>
__device__ __forceinline__ void mmc_fold(const T* levels, const int2* __restrict__ chord, int sg, int r,
                                         int u, T (&best)[MMC_ROWS][MMC_COLS]) {
#pragma unroll
  for (int j = 0; j < MMC_ROWS; ++j) {
    const int d = sg - j;     // footprint row dy + r of output row j
    if (FULL || (unsigned)d <= (unsigned)(2 * r)) {
      const int2 o = __ldg(chord + d);
      const T* a = levels + o.x + u;
      const T* b = levels + o.y + u;
#pragma unroll
      for (int c = 0; c < MMC_COLS; ++c) best[j][c] = vmax3<T>(best[j][c], a[c * MMC_GROUP], b[c * MMC_GROUP]);
    }
  }
}

template <typename T>
__global__ void __launch_bounds__(MMC_THREADS, 1)   // ~200 registers: 2 blocks per SM spill
moving_max_chord_kernel(const T* __restrict__ src, T* __restrict__ dst, T nodata, int has_nodata,
                        int bands, int H, int W, int r, int n_levels, int pitch,
                        const int2* __restrict__ chord) {
  extern __shared__ __align__(16) unsigned char mm_smem[];
  T* levels = reinterpret_cast<T*>(mm_smem);          // n_levels x pitch, then MMC_TX sentinel cells
  const int tid = threadIdx.x, g = tid / MMC_GROUP, u = tid % MMC_GROUP;
  const int SW = W + 2 * r, SH = H + 2 * r;
  const int64_t in_plane = (int64_t)SH * SW, out_plane = (int64_t)H * W;
  const int x0 = blockIdx.x * MMC_TX, y0 = blockIdx.y * (MMC_GROUPS * MMC_ROWS);
  const int seg = MMC_TX + 2 * r;
  const int n_src = min(MMC_GROUPS * MMC_ROWS, H - y0) + 2 * r;   // source rows the block's outputs need
  const T lowest = Lowest<T>::value();
  // footprint rows without a chord (even sizes) point at the sentinel cells
  for (int i = tid; i < MMC_TX; i += MMC_THREADS) levels[n_levels * pitch + i] = lowest;
  for (int b = blockIdx.z; b < bands; b += gridDim.z) {
    const T* plane = src + (int64_t)b * in_plane;
    T pf[MMC_PREFETCH];
    auto fetch = [&](int s) {       // unconditional loads on clamped addresses
      const T* row = plane + (int64_t)min(y0 + s, SH - 1) * SW;
#pragma unroll
      for (int m = 0; m < MMC_PREFETCH; ++m) pf[m] = __ldg(row + min(x0 + tid + m * MMC_THREADS, SW - 1));
    };
    auto clean = [&](T v, int s, int i) {
      return (y0 + s < SH && x0 + i < SW && !(has_nodata && v == nodata)) ? v : lowest;
    };
    auto stage = [&](int s) {       // level 0 of source row s
#pragma unroll
      for (int m = 0; m < MMC_PREFETCH; ++m) {
        const int i = tid + m * MMC_THREADS;
        if (i < seg) levels[i] = clean(pf[m], s, i);
      }
      const T* row = plane + (int64_t)min(y0 + s, SH - 1) * SW;
      for (int i = tid + MMC_PREFETCH * MMC_THREADS; i < seg; i += MMC_THREADS)
        levels[i] = clean(__ldg(row + min(x0 + i, SW - 1)), s, i);
    };
    T best[MMC_ROWS][MMC_COLS];
#pragma unroll
    for (int j = 0; j < MMC_ROWS; ++j)
#pragma unroll
      for (int c = 0; c < MMC_COLS; ++c) best[j][c] = lowest;
    fetch(0);
    stage(0);
    for (int s = 0; s < n_src; ++s) {
      __syncthreads();                                  // level 0 of row s is in place
      if (s + 1 < n_src) fetch(s + 1);
      for (int k = 1; k < n_levels; ++k) {
        const int half = 1 << (k - 1), n = seg - 2 * half + 1;
        T* lk = levels + k * pitch;
        const T* prev = lk - pitch;
        for (int p = tid; p < n; p += MMC_THREADS) lk[p] = vmax<T>(prev[p], prev[p + half]);
        __syncthreads();
      }
      // output rows g * MMC_ROWS + j of this group take footprint row s - g * MMC_ROWS - j - r
      const int sg = s - g * MMC_ROWS;
      if (sg >= 0 && sg - (MMC_ROWS - 1) <= 2 * r) {
        if (sg >= MMC_ROWS - 1 && sg <= 2 * r) mmc_fold<T, true>(levels, chord, sg, r, u, best);
        else mmc_fold<T, false>(levels, chord, sg, r, u, best);
      }
      __syncthreads();                                  // every thread is done with row s
      if (s + 1 < n_src) stage(s + 1);
    }
#pragma unroll
    for (int j = 0; j < MMC_ROWS; ++j) {
      const int y = y0 + g * MMC_ROWS + j;
      if (y >= H) break;
#pragma unroll
      for (int c = 0; c < MMC_COLS; ++c) {
        const int x = x0 + u + c * MMC_GROUP;
        if (x >= W) continue;
        T v = best[j][c];
        // restore no data only where the centre was no data and nothing was found
        if (has_nodata && v == lowest && __ldg(plane + (int64_t)(y + r) * SW + (x + r)) == nodata) v = nodata;
        dst[(int64_t)b * out_plane + (int64_t)y * W + x] = v;
      }
    }
  }
}

static int floor_log2(int v) { int k = 0; while ((2 << k) <= v) ++k; return k; }

// shared memory of moving_max_chord_kernel for the chord half-widths `hw` (levels x pitch cells,
// then the sentinel cells)
template <typename T>
static size_t chord_smem(int r, int max_hw, int* n_levels, int* pitch) {
  *n_levels = floor_log2(2 * max_hw + 1) + 1;
  const int vec = 16 / (int)sizeof(T);
  *pitch = (MMC_TX + 2 * r + vec - 1) / vec * vec;
  return ((size_t)*n_levels * *pitch + MMC_TX) * sizeof(T);
}

template <typename T>
static int launch_moving_max_chord(const Staged& in, Staged& out, T nd, int has_nodata, int bands, int H,
                                   int W, int size, const std::vector<int>& hw, cudaStream_t s) {
  const int r = size / 2;
  const int max_hw = *std::max_element(hw.begin(), hw.end());
  int n_levels = 0, pitch = 0;
  const size_t smem = chord_smem<T>(r, std::max(max_hw, 0), &n_levels, &pitch);
  int dev = 0, limit = 0;
  GM_CUDA(cudaGetDevice(&dev));
  GM_CUDA(cudaDeviceGetAttribute(&limit, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  if (smem > (size_t)limit) {
    int largest = size, lv, pt;
    while (largest > 1 && chord_smem<T>(largest / 2, largest / 2, &lv, &pt) > (size_t)limit) largest -= 2;
    return fail("gm_moving_max: size " + std::to_string(size) + " needs " + std::to_string(smem) +
                " bytes of shared memory per block for " + std::to_string(sizeof(T)) +
                "-byte cells, above the device's " + std::to_string(limit) + "; the largest size for this dtype is " +
                std::to_string(largest));
  }
  // per footprint row: offsets of the two level-k windows that cover its chord, relative to the
  // block's first output column
  std::vector<int2> chord(2 * r + 1);
  for (int d = 0; d <= 2 * r; ++d) {
    const int w = hw[d];
    if (w < 0) {
      chord[d] = make_int2(n_levels * pitch, n_levels * pitch);   // the sentinel cells
      continue;
    }
    const int k = floor_log2(2 * w + 1);
    chord[d] = make_int2(k * pitch + r - w, k * pitch + r + w - (1 << k) + 1);
  }
  void* dev_chord = nullptr;
  if (upload(&dev_chord, chord.data(), (int64_t)chord.size() * sizeof(int2), s)) return 1;
  auto kernel = moving_max_chord_kernel<T>;
  if (smem > 48 * 1024)
    GM_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kernel<<<grid3(W, H, bands, MMC_TX, MMC_GROUPS * MMC_ROWS), MMC_THREADS, smem, s>>>(
      (const T*)in.dev, (T*)out.dev, nd, has_nodata, bands, H, W, r, n_levels, pitch, (const int2*)dev_chord);
  cudaError_t e = cudaGetLastError();
  cudaFreeAsync(dev_chord, s);
  if (e != cudaSuccess) return fail(std::string("moving_max launch: ") + cudaGetErrorString(e));
  count_launch();
  return 0;
}

// ---------------------------------------------------------------------------------
// Dilate (raster/spatial.py:146-155): 6-connected 3-D cross, values in order
// ---------------------------------------------------------------------------------
constexpr int DILATE_MAX_VALUES = 64;
template <typename T> struct DilateValues { T v[DILATE_MAX_VALUES]; int n; };

// Every source cell is ranked ONCE (rank = 1 + index of the cell's value in
// `values`, 0 if it is not listed; later values win, so the output is the value of the
// largest rank in the 7-point cross) into a byte tile in shared memory -- single-byte
// rasters through a 256-entry table -- and an output cell then takes the maximum of five
// bytes (plus the two time neighbours, ranked on the fly when there is more than one band).
constexpr int DL_TX = 128, DL_TY = 16;

template <typename T>
__device__ __forceinline__ int dilate_rank(T v, const T* vals, int n, const unsigned char* lut) {
  if constexpr (sizeof(T) == 1) {
    return lut[(unsigned char)v];
  } else {
    for (int i = n - 1; i >= 0; --i)
      if (v == vals[i]) return i + 1;
    return 0;
  }
}

template <typename T>
__global__ void __launch_bounds__(256)
dilate_tiled_kernel(const T* __restrict__ src, T* __restrict__ dst, int bands, int H, int W,
                    const __grid_constant__ DilateValues<T> values) {
  constexpr int TW = DL_TX + 2, TH = DL_TY + 2;
  __shared__ unsigned char rank[TH][TW + 2];
  __shared__ unsigned char lut[256];
  __shared__ T vals[DILATE_MAX_VALUES];
  const int SW = W + 2, SH = H + 2;
  const int64_t in_plane = (int64_t)SH * SW, out_plane = (int64_t)H * W;
  const int tid = threadIdx.x;
  const int x0 = blockIdx.x * DL_TX, y0 = blockIdx.y * DL_TY;
  if (tid < values.n) vals[tid] = values.v[tid];
  if (sizeof(T) == 1) {
    int r = 0;
    for (int i = 0; i < values.n; ++i)
      if ((unsigned char)values.v[i] == (unsigned char)tid) r = i + 1;
    lut[tid] = (unsigned char)r;
  }
  for (int b = blockIdx.z; b < bands; b += gridDim.z) {
    const T* plane = src + (int64_t)b * in_plane;
    __syncthreads();
    for (int i = tid; i < TW * TH; i += 256) {
      const int ty = i / TW, tx = i - ty * TW;
      const int gy = min(y0 + ty, SH - 1), gx = min(x0 + tx, SW - 1);   // clamped: never used beyond the array
      rank[ty][tx] = (unsigned char)dilate_rank<T>(__ldg(plane + (int64_t)gy * SW + gx), vals, values.n, lut);
    }
    __syncthreads();
    for (int i = tid; i < DL_TX * DL_TY; i += 256) {
      const int ty = i / DL_TX, tx = i - ty * DL_TX;
      const int x = x0 + tx, y = y0 + ty;
      if (x >= W || y >= H) continue;
      int best = max(max(rank[ty + 1][tx], rank[ty + 1][tx + 2]), max(rank[ty][tx + 1], rank[ty + 2][tx + 1]));
      best = max(best, (int)rank[ty + 1][tx + 1]);
      const T* c = plane + (int64_t)(y + 1) * SW + (x + 1);
      if (b > 0) best = max(best, dilate_rank<T>(__ldg(c - in_plane), vals, values.n, lut));
      if (b + 1 < bands) best = max(best, dilate_rank<T>(__ldg(c + in_plane), vals, values.n, lut));
      dst[(int64_t)b * out_plane + (int64_t)y * W + x] = best > 0 ? vals[best - 1] : __ldg(c);
    }
  }
}

// Single-byte rasters (the usual class rasters): four cells per thread, packed in one word.
// Ranks and original bytes are staged as words (4-byte left pad, so that an output word and
// its upper / lower neighbours are aligned word loads; the left / right neighbours are two
// byte permutes of adjacent words), the 5-point maximum is four bytewise maxima, and a word
// whose cross holds no listed value is copied through.
constexpr int DP_TX = 256, DP_TY = 16;            // outputs per block
constexpr int DP_WORDS = DP_TX / 4 + 2;           // words per staged row (one pad word each side)

template <typename T>
__global__ void __launch_bounds__(256)
dilate_packed_kernel(const T* __restrict__ src, T* __restrict__ dst, int bands, int H, int W, int dst_aligned,
                     const __grid_constant__ DilateValues<T> values) {
  static_assert(sizeof(T) == 1, "bytes");
  __shared__ unsigned rank[DP_TY + 2][DP_WORDS];
  __shared__ unsigned orig[DP_TY][DP_TX / 4];
  __shared__ unsigned char lut[256];
  __shared__ unsigned char vals[DILATE_MAX_VALUES + 1];
  const unsigned char* s8 = reinterpret_cast<const unsigned char*>(src);
  unsigned char* d8 = reinterpret_cast<unsigned char*>(dst);
  const int SW = W + 2, SH = H + 2;
  const int64_t in_plane = (int64_t)SH * SW, out_plane = (int64_t)H * W;
  const int tid = threadIdx.x;
  const int x0 = blockIdx.x * DP_TX, y0 = blockIdx.y * DP_TY;
  {
    int r = 0;
    for (int i = 0; i < values.n; ++i)
      if ((unsigned char)values.v[i] == (unsigned char)tid) r = i + 1;
    lut[tid] = (unsigned char)r;
    if (tid <= values.n) vals[tid] = tid ? (unsigned char)values.v[tid - 1] : 0;
  }
  for (int b = blockIdx.z; b < bands; b += gridDim.z) {
    const unsigned char* plane = s8 + (int64_t)b * in_plane;
    __syncthreads();
    // staged byte j of a row <-> source column x0 - 3 + j (output column c sits at byte c + 4)
    for (int task = tid; task < (DP_TY + 2) * DP_WORDS; task += 256) {
      const int ty = task / DP_WORDS, wx = task - ty * DP_WORDS;
      const int gy = y0 + ty;
      unsigned ranks = 0, bytes = 0;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int gx = x0 - 3 + 4 * wx + k;
        if (gy < SH && gx >= 0 && gx < SW) {
          const unsigned v = plane[(int64_t)gy * SW + gx];
          ranks |= (unsigned)lut[v] << (8 * k);
          bytes |= v << (8 * k);
        }
      }
      rank[ty][wx] = ranks;
      if (ty >= 1 && ty <= DP_TY && wx >= 1 && wx <= DP_TX / 4) orig[ty - 1][wx - 1] = bytes;
    }
    __syncthreads();
    for (int task = tid; task < DP_TY * (DP_TX / 4); task += 256) {
      const int ty = task / (DP_TX / 4), wx = task - ty * (DP_TX / 4);
      const int y = y0 + ty, x = x0 + 4 * wx;
      if (y >= H || x >= W) continue;
      const unsigned c = rank[ty + 1][wx + 1];
      const unsigned left = __byte_perm(rank[ty + 1][wx], c, 0x6543);       // ranks of columns x-1 .. x+2
      const unsigned right = __byte_perm(c, rank[ty + 1][wx + 2], 0x4321);  // ranks of columns x+1 .. x+4
      unsigned best = __vmaxu4(__vmaxu4(c, rank[ty][wx + 1]), __vmaxu4(rank[ty + 2][wx + 1], __vmaxu4(left, right)));
      unsigned out = orig[ty][wx];
      if (bands > 1) {   // the time neighbours of the 3-D cross, ranked on the fly
        unsigned tn = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          if (x + k < W) {
            const int64_t at = (int64_t)(y + 1) * SW + (x + k + 1);
            unsigned r = 0;
            if (b > 0) r = lut[plane[at - in_plane]];
            if (b + 1 < bands) r = max(r, (unsigned)lut[plane[at + in_plane]]);
            tn |= r << (8 * k);
          }
        }
        best = __vmaxu4(best, tn);
      }
      if (best) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const unsigned r = (best >> (8 * k)) & 0xffu;
          if (r) out = (out & ~(0xffu << (8 * k))) | ((unsigned)vals[r] << (8 * k));
        }
      }
      unsigned char* o = d8 + (int64_t)b * out_plane + (int64_t)y * W + x;
      if (dst_aligned && x + 3 < W) {
        *reinterpret_cast<unsigned*>(o) = out;
      } else {
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (x + k < W) o[k] = (unsigned char)(out >> (8 * k));
      }
    }
  }
}

// ---------------------------------------------------------------------------------
// Smooth (raster/spatial.py:273-307): scipy.ndimage.gaussian_filter restated
// ---------------------------------------------------------------------------------
// NI_Correlate1D, symmetric branch: tmp = c*w[0] + sum_{k=l..1} (a[-k] + a[+k])*w[k]
// accumulated in double, stored in the array dtype after EACH pass (y, then x).
// mode="constant": taps outside the array read `fill`.
constexpr int SM_TX = 32, SM_TY = 16, SM_MAXL = 64;

template <typename T> __device__ __forceinline__ T from_double(double v) { return (T)v; }

struct SmoothWeights { double wy[SM_MAXL + 1]; double wx[SM_MAXL + 1]; };

template <typename T>
__global__ void __launch_bounds__(SM_TX * SM_TY)
smooth_kernel(const T* __restrict__ src, T* __restrict__ dst, T nodata, int has_nodata, T fill,
              int bands, int SH, int SW, int H, int W, int my, int mx, int ly, int lx,
              const __grid_constant__ SmoothWeights wts) {
  extern __shared__ __align__(16) unsigned char sm_smem[];
  const int tw = SM_TX + 2 * lx, th = SM_TY + 2 * ly;
  T* tile = reinterpret_cast<T*>(sm_smem);     // th x tw input (no data -> fill)
  T* mid = tile + (size_t)th * tw;             // SM_TY x tw result of the y pass
  const int tid = threadIdx.y * SM_TX + threadIdx.x;
  const int64_t in_plane = (int64_t)SH * SW, out_plane = (int64_t)H * W;
  const int x0 = blockIdx.x * SM_TX, y0 = blockIdx.y * SM_TY;  // output coordinates
  for (int b = blockIdx.z; b < bands; b += gridDim.z) {
    __syncthreads();
    for (int i = tid; i < tw * th; i += SM_TX * SM_TY) {
      const int ty = i / tw, tx = i - ty * tw;
      const int gy = y0 + my - ly + ty, gx = x0 + mx - lx + tx;  // source coordinates
      T v = fill;
      if (gy >= 0 && gy < SH && gx >= 0 && gx < SW) {
        v = __ldg(src + (int64_t)b * in_plane + (int64_t)gy * SW + gx);
        if (has_nodata && v == nodata) v = fill;
      }
      tile[i] = v;
    }
    __syncthreads();
    // y pass for every column of the tile (including the x halo)
    for (int i = tid; i < SM_TY * tw; i += SM_TX * SM_TY) {
      const int ty = i / tw, tx = i - ty * tw;
      const T* c = tile + (ty + ly) * tw + tx;
      // rows of the haloed tile that lie outside the source array are `fill`
      // already; rows outside the y-filtered range cannot be requested
      double tmp = (double)c[0] * wts.wy[0];
      for (int k = ly; k >= 1; --k) tmp += ((double)c[-k * tw] + (double)c[k * tw]) * wts.wy[k];
      T r = ly > 0 ? from_double<T>(tmp) : c[0];
      // columns outside the source are padding for the x pass: constant `fill`
      const int gx = x0 + mx - lx + tx;
      if (gx < 0 || gx >= SW) r = fill;
      mid[i] = r;
    }
    __syncthreads();
    const int x = x0 + threadIdx.x, y = y0 + threadIdx.y;
    if (x < W && y < H) {
      const T* c = mid + threadIdx.y * tw + threadIdx.x + lx;
      T out;
      if (lx > 0) {
        double tmp = (double)c[0] * wts.wx[0];
        for (int k = lx; k >= 1; --k) tmp += ((double)c[-k] + (double)c[k]) * wts.wx[k];
        out = from_double<T>(tmp);
      } else {
        out = c[0];
      }
      dst[(int64_t)b * out_plane + (int64_t)y * W + x] = out;
    }
  }
}


__device__ __forceinline__ double smooth_fma(double a, double b, double c) { return fma(a, b, c); }
__device__ __forceinline__ float smooth_fma(float a, float b, float c) { return fmaf(a, b, c); }

static std::atomic<int> g_smooth_mode{-1};
static int smooth_mode() {
  int m = g_smooth_mode.load();
  if (m < 0) {
    const char* env = getenv("GM_SMOOTH");
    m = GM_SMOOTH_FMA;
    if (env && !strcmp(env, "exact")) m = GM_SMOOTH_EXACT;
    else if (env && !strcmp(env, "float32")) m = GM_SMOOTH_FLOAT32;
    g_smooth_mode.store(m);
  }
  return m;
}

// Fast path for ly == lx == L <= SMF_MAXL (every "exact"-mode request: size_px <= 6 gives
// L = int(4 * size_px / 3 + 0.5) <= 8).  Same arithmetic as smooth_kernel -- double
// accumulation in SciPy's tap order, array-dtype rounding after each pass -- organised so
// that the FP64 pipe, not shared memory, is the limit:
//   * the tile is converted to double ONCE when it is staged (conversions are slow-path
//     instructions; the generic kernel converts every tap);
//   * a thread produces 8 consecutive outputs of a column (y pass) or a row (x pass) from a
//     register window of 8 + 2L values: (8 + 2L) / 8 shared loads per output instead of
//     2L + 1;
//   * tile width incl. halo is 128 columns and 32 + 2L rows, so both passes are whole rounds
//     of the 256 threads; rows are padded to 129 doubles so that the x pass (lane = row) is
//     bank-conflict free; results leave through a staged, coalesced copy.
// Bound: 22 FP64 operations per pass per pixel (1 + 3L at L = 7) on a 64-lane FP64 pipe.
constexpr int SMF_TW = 128, SMF_TY = 32, SMF_RUN = 8, SMF_PITCH = SMF_TW + 1, SMF_MAXL = 8;

// ARITH: how a pass accumulates its 2 L + 1 taps
//   GM_SMOOTH_EXACT    double, multiply and add rounded separately: SciPy's correlate1d bit for bit
//   GM_SMOOTH_FMA      double, fused multiply-add: one rounding fewer per tap pair (the result can
//                      differ from SciPy's by the last bit of the ARRAY dtype where a double sum
//                      sits within 1e-16 of a rounding boundary); 1 + 2 L instead of 1 + 3 L FP64
//                      operations per output
//   GM_SMOOTH_FLOAT32  float32 rasters only: float accumulation with FFMA -- off the FP64 pipe
//                      altogether; error <= (2 L + 1) * 2^-24 relative, inside the stated 1e-6
template <typename T, int L, int ARITH>
__global__ void __launch_bounds__(256)
smooth_fast_kernel(const T* __restrict__ src, T* __restrict__ dst, T nodata, int has_nodata, T fill,
                   int bands, int SH, int SW, int H, int W, int my, int mx,
                   const __grid_constant__ SmoothWeights wts) {
  extern __shared__ __align__(16) unsigned char sm_smem[];
  constexpr int TX = SMF_TW - 2 * L;          // output columns per tile
  constexpr int TH = SMF_TY + 2 * L;          // staged rows
  constexpr int WIN = SMF_RUN + 2 * L;
  // Both tiles hold the ARRAY dtype (what SciPy stores between the passes); values are
  // widened to double when a thread fills its register window.  For float32 this halves the
  // shared memory of a double tile: 40 KB per CTA, four CTAs per SM.
  T* tile = reinterpret_cast<T*>(sm_smem);                 // TH x SMF_PITCH (source, no data -> fill)
  T* mid = tile + (size_t)TH * SMF_PITCH;                  // SMF_TY x SMF_PITCH (+ slack) after the y pass
  T* stage = tile;                                         // SMF_TY x TX results (reuses the tile)
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t in_plane = (int64_t)SH * SW, out_plane = (int64_t)H * W;
  const int x0 = blockIdx.x * TX, y0 = blockIdx.y * SMF_TY;  // output coordinates of the tile
  for (int b = blockIdx.z; b < bands; b += gridDim.z) {
    const T* plane = src + (int64_t)b * in_plane;
    __syncthreads();
    // source tile.  Tiles whose staged window lies inside the array (all but the outermost
    // ring of tiles) need no clamping and no inside test: straight rows, pointer steps
    const int wy0 = y0 + my - L, wx0 = x0 + mx - L;          // window origin in the source
    if (wy0 >= 0 && wx0 >= 0 && wy0 + TH <= SH && wx0 + SMF_TW <= SW) {
      const T* p = plane + (int64_t)(wy0 + warp) * SW + wx0 + lane;
      constexpr int ROUNDS = (TH + 7) / 8;
#pragma unroll 2
      for (int k = 0; k < ROUNDS; ++k) {
        const int row = warp + 8 * k;
        T raw[SMF_TW / 32];
        if (row < TH) {
#pragma unroll
          for (int j = 0; j < SMF_TW / 32; ++j) raw[j] = __ldg(p + 32 * j);
#pragma unroll
          for (int j = 0; j < SMF_TW / 32; ++j)
            tile[row * SMF_PITCH + lane + 32 * j] = (has_nodata && raw[j] == nodata) ? fill : raw[j];
        }
        p += (int64_t)8 * SW;
      }
    } else {
      // unconditional (clamped) loads, two tile rows = eight requests per thread per round
      for (int ty = warp; ty < TH; ty += 16) {
        T raw[2][SMF_TW / 32];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int gy = min(max(y0 + my - L + ty + 8 * h, 0), SH - 1);
#pragma unroll
          for (int j = 0; j < SMF_TW / 32; ++j)
            raw[h][j] = __ldg(plane + (int64_t)gy * SW + min(max(x0 + mx - L + lane + 32 * j, 0), SW - 1));
        }
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int row = ty + 8 * h;
          const int gy = y0 + my - L + row;
#pragma unroll
          for (int j = 0; j < SMF_TW / 32; ++j) {
            const int tx = lane + 32 * j;
            const int gx = x0 + mx - L + tx;
            const bool inside = gy >= 0 && gy < SH && gx >= 0 && gx < SW;
            const T v = (!inside || (has_nodata && raw[h][j] == nodata)) ? fill : raw[h][j];
            if (row < TH) tile[row * SMF_PITCH + tx] = v;
          }
        }
      }
    }
    __syncthreads();
    // y pass: task = (run of 8 rows, column); 4 x 128 tasks = two rounds of 256 threads
#pragma unroll 1
    for (int task = tid; task < (SMF_TY / SMF_RUN) * SMF_TW; task += 256) {
      const int tx = task & (SMF_TW - 1), run = task >> 7;
      const T* c = tile + (run * SMF_RUN) * SMF_PITCH + tx;
      typedef typename std::conditional<ARITH == GM_SMOOTH_FLOAT32, float, double>::type A;
      A win[WIN], wk[L + 1];
#pragma unroll
      for (int i = 0; i < WIN; ++i) win[i] = (A)c[i * SMF_PITCH];
#pragma unroll
      for (int k = 0; k <= L; ++k) wk[k] = (A)wts.wy[k];
      const int gx = x0 + mx - L + tx;
      const bool pad = gx < 0 || gx >= SW;   // columns outside the source: constant padding
#pragma unroll
      for (int o = 0; o < SMF_RUN; ++o) {
        A tmp = win[o + L] * wk[0];
#pragma unroll
        for (int k = L; k >= 1; --k) {
          if (ARITH == GM_SMOOTH_EXACT) tmp += (win[o + L - k] + win[o + L + k]) * wk[k];
          else tmp = smooth_fma(win[o + L - k] + win[o + L + k], wk[k], tmp);
        }
        const T r = from_double<T>(tmp);
        mid[(run * SMF_RUN + o) * SMF_PITCH + tx] = pad ? fill : r;
      }
    }
    __syncthreads();
    // x pass: lane = row, each warp takes runs of 8 output columns
#pragma unroll 1
    for (int run = warp; run * SMF_RUN < TX; run += 8) {
      const T* c = mid + lane * SMF_PITCH + run * SMF_RUN;
      typedef typename std::conditional<ARITH == GM_SMOOTH_FLOAT32, float, double>::type A;
      A win[WIN], wk[L + 1];
#pragma unroll
      for (int i = 0; i < WIN; ++i) win[i] = (A)c[i];  // may run into the next row / the slack: only feeds outputs >= TX
#pragma unroll
      for (int k = 0; k <= L; ++k) wk[k] = (A)wts.wx[k];
#pragma unroll
      for (int o = 0; o < SMF_RUN; ++o) {
        A tmp = win[o + L] * wk[0];
#pragma unroll
        for (int k = L; k >= 1; --k) {
          if (ARITH == GM_SMOOTH_EXACT) tmp += (win[o + L - k] + win[o + L + k]) * wk[k];
          else tmp = smooth_fma(win[o + L - k] + win[o + L + k], wk[k], tmp);
        }
        if (run * SMF_RUN + o < TX) stage[lane * TX + run * SMF_RUN + o] = from_double<T>(tmp);
      }
    }
    __syncthreads();
    if (x0 + TX <= W && y0 + SMF_TY <= H) {   // the tile's outputs lie inside the array
      T* o = dst + (int64_t)b * out_plane + (int64_t)(y0 + warp) * W + x0 + lane;
#pragma unroll
      for (int k = 0; k < SMF_TY / 8; ++k) {
        const T* st = stage + (warp + 8 * k) * TX + lane;
#pragma unroll
        for (int j = 0; j < (TX + 31) / 32; ++j)
          if (lane + 32 * j < TX) o[32 * j] = st[32 * j];
        o += (int64_t)8 * W;
      }
    } else {
      for (int ty = warp; ty < SMF_TY; ty += 8) {
        const int y = y0 + ty;
        if (y >= H) break;
        for (int tx = lane; tx < TX; tx += 32) {
          const int x = x0 + tx;
          if (x < W) dst[(int64_t)b * out_plane + (int64_t)y * W + x] = stage[ty * TX + tx];
        }
      }
    }
  }
}
template <typename T, int L, int ARITH>
static int launch_smooth_fast_as(const Staged& in, T* target, T nd, int has_nodata, T fill, int bands,
                                 int SH, int SW, int H, int W, int my, int mx, const SmoothWeights& wts,
                                 cudaStream_t s) {
  constexpr int TX = SMF_TW - 2 * L;
  const size_t smem = (((size_t)(SMF_TY + 2 * L) + SMF_TY) * SMF_PITCH + 2 * SMF_MAXL) * sizeof(T);
  auto kernel = smooth_fast_kernel<T, L, ARITH>;
  if (smem > 48 * 1024)
    GM_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kernel<<<grid3(W, H, bands, TX, SMF_TY), 256, smem, s>>>((const T*)in.dev, target, nd, has_nodata, fill,
                                                           bands, SH, SW, H, W, my, mx, wts);
  GM_LAUNCH_CHECK();
  return 0;
}

template <typename T, int L>
static int launch_smooth_fast(const Staged& in, T* target, T nd, int has_nodata, T fill, int bands,
                              int SH, int SW, int H, int W, int my, int mx, const SmoothWeights& wts,
                              cudaStream_t s) {
  const int mode = smooth_mode();
  if constexpr (std::is_same<T, float>::value) {
    if (mode == GM_SMOOTH_FLOAT32)
      return launch_smooth_fast_as<T, L, GM_SMOOTH_FLOAT32>(in, target, nd, has_nodata, fill, bands, SH, SW, H, W, my, mx, wts, s);
  }
  if (mode == GM_SMOOTH_EXACT)
    return launch_smooth_fast_as<T, L, GM_SMOOTH_EXACT>(in, target, nd, has_nodata, fill, bands, SH, SW, H, W, my, mx, wts, s);
  return launch_smooth_fast_as<T, L, GM_SMOOTH_FMA>(in, target, nd, has_nodata, fill, bands, SH, SW, H, W, my, mx, wts, s);
}

// 0: launched, 1: error, -1: no fast path for this dtype / radius
template <typename T>
static int try_smooth_fast(int L, const Staged& in, T* target, T nd, int has_nodata, T fill, int bands,
                           int SH, int SW, int H, int W, int my, int mx, const SmoothWeights& wts,
                           cudaStream_t s) {
  if constexpr (std::is_same<T, float>::value || std::is_same<T, double>::value ||
                std::is_same<T, int16_t>::value || std::is_same<T, uint8_t>::value ||
                std::is_same<T, int32_t>::value) {
    switch (L) {
#define GM_CASE(N) case N: return launch_smooth_fast<T, N>(in, target, nd, has_nodata, fill, bands, SH, SW, H, W, my, mx, wts, s);
      GM_CASE(1) GM_CASE(2) GM_CASE(3) GM_CASE(4) GM_CASE(5) GM_CASE(6) GM_CASE(7) GM_CASE(8)
#undef GM_CASE
      default: break;
    }
  }
  return -1;
}

// zoom-back of Smooth's "zoom" mode: ndimage.affine_transform(order=0,
// matrix=diag(1, zy, zx), offset=(0, oy, ox)) -> out[i, j] = in[floor(oy + i*zy + .5), ...]
template <typename T>
__global__ void zoom_nn_kernel(const T* __restrict__ src, T* __restrict__ dst, int bands, int H,
                               int W, double zy, double zx, double oy, double ox) {
  const int64_t plane = (int64_t)H * W, total = plane * bands;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int b = (int)(idx / plane);
    const int64_t r = idx - (int64_t)b * plane;
    const int i = (int)(r / W), j = (int)(r - (int64_t)i * W);
    const double cy = oy + (double)i * zy, cx = ox + (double)j * zx;
    T v = (T)0;  // cval
    if (cy >= 0.0 && cy <= (double)(H - 1) && cx >= 0.0 && cx <= (double)(W - 1)) {
      const int sy = (int)floor(cy + 0.5), sx = (int)floor(cx + 0.5);
      v = src[(int64_t)b * plane + (int64_t)sy * W + sx];
    }
    dst[idx] = v;
  }
}

// ---- host side ---------------------------------------------------------------------
template <typename T> static T cast_fill(double fill) { return (T)fill; }


template <typename T>
static int run_hillshade(const Staged& in, Staged& out, const void* nodata, int has_nodata,
                         double fill, int bands, int H, int W, int SW, double xres, double yres,
                         double alt_deg, double az_deg, cudaStream_t s) {
  const double alt = alt_deg * (M_PI / 180.0), az = az_deg * (M_PI / 180.0);
  // math.radians(x) = x * (pi / 180) in CPython
  const double zsf = 1.0 / 8.0;
  // a power-of-two resolution (in float32 for float rasters) has an exact reciprocal
  auto pow2 = [](double v) { int e; return v > 0 && std::frexp(v, &e) == 0.5 && e > -100 && e < 100; };
  const bool is_f32 = std::is_same<T, float>::value;
  const int exact = pow2(is_f32 ? (double)(float)xres : xres) && pow2(is_f32 ? (double)(float)yres : yres);
  const int qx = (W + HQ_COLS - 1) / HQ_COLS, qy = (H + HQ_ROWS - 1) / HQ_ROWS;
  const int64_t qstrips = (int64_t)bands * qx * qy;
  const unsigned qblocks = (unsigned)((qstrips + HS_WARPS - 1) / HS_WARPS);
  const int aligned = ((uintptr_t)out.dev % 4 == 0) && (W % 4 == 0);
  const int quad_loads = sizeof(T) == 4 && SW % 4 == 0 && (uintptr_t)in.dev % 16 == 0;
#define GM_HQ(EXACT)                                                                                \
  hillshade_quad_kernel<T, EXACT><<<qblocks, 32 * HS_WARPS, 0, s>>>(                                \
      (const T*)in.dev, (uint8_t*)out.dev, has_nodata ? read_scalar<T>(nodata) : T(0), has_nodata,   \
      cast_fill<T>(fill), bands, H, W, SW, quad_loads, xres, yres, 1.0 / xres, 1.0 / yres, aligned,  \
      (float)sin(alt), (float)(cos(alt) * zsf), (float)cos(az), (float)sin(az), (float)(zsf * zsf))
  if (exact) GM_HQ(true); else GM_HQ(false);
#undef GM_HQ
  GM_LAUNCH_CHECK();
  return 0;
}

template <typename T>
static int run_moving_max(const Staged& in, Staged& out, const void* nodata, int has_nodata,
                          int bands, int H, int W, int SW, int size, cudaStream_t s) {
  const int r = size / 2;
  // chord half-widths of the disc x^2 + y^2 < (size/2)^2 (utils.py:536-547)
  std::vector<int> hw(2 * r + 1);
  const double rad2 = (size / 2.0) * (size / 2.0);
  for (int dy = -r; dy <= r; ++dy) {
    int w = -1;
    for (int dx = 0; dx <= r; ++dx)
      if ((double)(dx * dx + dy * dy) < rad2) w = dx;
    hw[dy + r] = w;  // -1: the row is not part of the footprint
  }
  {
    const int fixed = try_moving_max_fixed<T>(size, in, out, has_nodata ? read_scalar<T>(nodata) : T(0),
                                              has_nodata, bands, H, W, SW, s);
    if (fixed >= 0) return fixed;
  }
  if (SW != W + 2 * r)
    return fail("gm_moving_max: a source wider than the output plus its halo (pitch padding) is only "
                "supported for 4-byte rasters and odd sizes 3..15");
  // The tiled kernel up to radius 8, except 8-byte cells at radius 7 and 8, where the chord
  // kernel is faster (16384^2 on a B200, profiles/r07_moving_max_sizes.json: int64 size 15 14.2
  // against 17.2 ms, float64 size 17 17.5 against 18.9; every 1-, 2- and 4-byte case and int64
  // up to size 11 run 1.6-4x faster tiled).  GM_MOVING_MAX_KERNEL=tiled or =chord overrides the
  // choice up to radius 8, so that tools/moving_max_bench.py can time the two against each other.
  const char* kernel_env = getenv("GM_MOVING_MAX_KERNEL");
  const bool tiled = kernel_env ? strcmp(kernel_env, "tiled") == 0 : !(sizeof(T) == 8 && r >= 7);
  if (r >= 1 && r <= MM2_MAXR && tiled) {
    MMFootprint fp;
    memset(&fp, 0, sizeof(fp));
    for (int i = 0; i < 2 * MM2_MAXR + 1; ++i) fp.level[i] = -1;
    std::vector<int> distinct;
    for (int w : hw) if (w >= 0) distinct.push_back(w);
    std::sort(distinct.begin(), distinct.end());
    distinct.erase(std::unique(distinct.begin(), distinct.end()), distinct.end());
    fp.n_widths = (int)distinct.size();
    for (int k = 0; k < fp.n_widths; ++k) fp.width[k] = distinct[k];
    for (int dy = 0; dy <= 2 * r; ++dy)
      if (hw[dy] >= 0)
        fp.level[dy] = (int)(std::find(distinct.begin(), distinct.end(), hw[dy]) - distinct.begin());
    const size_t tile_smem = ((size_t)(MM2_TX + 2 * r) * (MM2_TY + 2 * r) +
                              (size_t)fp.n_widths * (MM2_TY + 2 * r) * MM2_TX) * sizeof(T);
    if (tile_smem <= 200 * 1024) {
      auto tiled = moving_max_tiled_kernel<T>;
      if (tile_smem > 48 * 1024)
        GM_CUDA(cudaFuncSetAttribute(tiled, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tile_smem));
      tiled<<<grid3(W, H, bands, MM2_TX, MM2_TY), 256, tile_smem, s>>>(
          (const T*)in.dev, (T*)out.dev, has_nodata ? read_scalar<T>(nodata) : T(0), has_nodata,
          bands, H, W, r, fp);
      GM_LAUNCH_CHECK();
      return 0;
    }
  }
  return launch_moving_max_chord<T>(in, out, has_nodata ? read_scalar<T>(nodata) : T(0), has_nodata, bands, H,
                                    W, size, hw, s);
}

template <typename T>
static int run_dilate(const Staged& in, Staged& out, const void* values, int n_values, int bands,
                      int H, int W, cudaStream_t s) {
  if (n_values > DILATE_MAX_VALUES) return fail("gm_dilate: more than 64 values");
  DilateValues<T> dv;
  memset(&dv, 0, sizeof(dv));
  dv.n = n_values;
  memcpy(dv.v, values, sizeof(T) * n_values);
  if constexpr (sizeof(T) == 1) {
    const int aligned = ((uintptr_t)out.dev % 4 == 0) && (W % 4 == 0);
    dilate_packed_kernel<T><<<grid3(W, H, bands, DP_TX, DP_TY), 256, 0, s>>>(
        (const T*)in.dev, (T*)out.dev, bands, H, W, aligned, dv);
    GM_LAUNCH_CHECK();
    return 0;
  }
  dilate_tiled_kernel<T><<<grid3(W, H, bands, DL_TX, DL_TY), 256, 0, s>>>(
      (const T*)in.dev, (T*)out.dev, bands, H, W, dv);
  GM_LAUNCH_CHECK();
  return 0;
}

template <typename T>
static int run_smooth(const Staged& in, Staged& out, const void* nodata, int has_nodata,
                      double fill, const double* wy, int ly, const double* wx, int lx, int bands,
                      int SH, int SW, int H, int W, int my, int mx, int zoom, double zy, double zx,
                      double oy, double ox, cudaStream_t s) {
  if (ly > SM_MAXL || lx > SM_MAXL) return fail("gm_smooth: kernel radius above 64 taps");
  SmoothWeights wts;
  memset(&wts, 0, sizeof(wts));
  // scipy passes weights[::-1]; index k here is the distance from the centre
  for (int k = 0; k <= ly; ++k) wts.wy[k] = wy[ly + k];
  for (int k = 0; k <= lx; ++k) wts.wx[k] = wx[lx + k];
  const size_t smem = ((size_t)(SM_TX + 2 * lx) * (SM_TY + 2 * ly) +
                       (size_t)SM_TY * (SM_TX + 2 * lx)) * sizeof(T);
  auto kernel = smooth_kernel<T>;
  if (smem > 48 * 1024)
    GM_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  T* target = (T*)out.dev;
  void* tmp = nullptr;
  if (zoom) {
    GM_CUDA(cudaMallocAsync(&tmp, (size_t)bands * H * W * sizeof(T), s));
    target = (T*)tmp;
  }
  int fast = -1;
  if (ly == lx && ly >= 1 && ly <= SMF_MAXL)
    fast = try_smooth_fast<T>(ly, in, target, has_nodata ? read_scalar<T>(nodata) : T(0), has_nodata,
                              cast_fill<T>(fill), bands, SH, SW, H, W, my, mx, wts, s);
  if (fast == 1) {
    if (tmp) cudaFreeAsync(tmp, s);
    return 1;
  }
  if (fast == -1)
    kernel<<<grid3(W, H, bands, SM_TX, SM_TY), dim3(SM_TX, SM_TY), smem, s>>>(
        (const T*)in.dev, target, has_nodata ? read_scalar<T>(nodata) : T(0), has_nodata,
        cast_fill<T>(fill), bands, SH, SW, H, W, my, mx, ly, lx, wts);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    if (tmp) cudaFreeAsync(tmp, s);
    return fail(std::string("smooth launch: ") + cudaGetErrorString(e));
  }
  if (fast == -1) count_launch();
  if (zoom) {
    const int64_t total = (int64_t)bands * H * W;
    int64_t blocks = (total + 255) / 256;
    const int64_t cap = (int64_t)sm_count() * 16;
    if (blocks > cap) blocks = cap;
    zoom_nn_kernel<T><<<(unsigned)blocks, 256, 0, s>>>((const T*)tmp, (T*)out.dev, bands, H, W, zy,
                                                        zx, oy, ox);
    e = cudaGetLastError();
    cudaFreeAsync(tmp, s);
    if (e != cudaSuccess) return fail(std::string("zoom launch: ") + cudaGetErrorString(e));
    count_launch();
  }
  return 0;
}

// open both arrays, run `body`, download and release
template <typename F>
static int with_staged(const GmArray* src, GmArray* dst, void* stream, F body) {
  if (ensure_init()) return 1;
  if (!src || !dst) return fail("null array");
  cudaStream_t s = resolve_stream(stream);
  Staged in, out;
  int rc = in.open_input(*src, s);
  if (!rc) rc = out.open_output(*dst, s);
  if (!rc && array_count(*dst) > 0) rc = body(in, out, s);
  if (!rc) rc = out.finish_output();
  const bool sync = out.owned;
  in.release();
  out.release();
  if (!rc && sync) GM_CUDA(cudaStreamSynchronize(s));
  return rc;
}

#define GM_DISPATCH_NUMERIC(dtype, CALL)                                       \
  switch (dtype) {                                                             \
    case GM_U8: case GM_BOOL: { typedef uint8_t T; return CALL; }              \
    case GM_I8:  { typedef int8_t T; return CALL; }                            \
    case GM_U16: { typedef uint16_t T; return CALL; }                          \
    case GM_I16: { typedef int16_t T; return CALL; }                           \
    case GM_U32: { typedef uint32_t T; return CALL; }                          \
    case GM_I32: { typedef int32_t T; return CALL; }                           \
    case GM_I64: { typedef int64_t T; return CALL; }                           \
    case GM_F32: { typedef float T; return CALL; }                             \
    case GM_F64: { typedef double T; return CALL; }                            \
    default: return fail("unsupported dtype");                                 \
  }

}  // namespace gm

using namespace gm;

extern "C" int gm_hillshade(const GmArray* src, GmArray* dst, const void* nodata, int has_nodata,
                            double fill, double xres, double yres, double altitude_deg,
                            double azimuth_deg, void* stream) {
  return with_staged(src, dst, stream, [&](Staged& in, Staged& out, cudaStream_t s) -> int {
    const int bands = (int)dst->shape[0], H = (int)dst->shape[1], W = (int)dst->shape[2];
    if (dst->dtype != GM_U8) return fail("gm_hillshade: output must be uint8");
    // columns beyond W + 2 are pitch padding (ignored): with a 16-byte row pitch a lane reads its
    // four source columns with one load
    if (src->shape[0] != bands || src->shape[1] != H + 2 || src->shape[2] < W + 2)
      return fail("gm_hillshade: source must carry a 1 pixel halo");
    GM_DISPATCH_NUMERIC(src->dtype, run_hillshade<T>(in, out, nodata, has_nodata, fill, bands, H, W,
                                                     (int)src->shape[2], xres, yres, altitude_deg,
                                                     azimuth_deg, s));
  });
}

extern "C" int gm_moving_max(const GmArray* src, GmArray* dst, const void* nodata, int has_nodata,
                             int size, void* stream) {
  return with_staged(src, dst, stream, [&](Staged& in, Staged& out, cudaStream_t s) -> int {
    const int bands = (int)dst->shape[0], H = (int)dst->shape[1], W = (int)dst->shape[2];
    const int r = size / 2;
    if (src->dtype != dst->dtype) return fail("gm_moving_max: dtype mismatch");
    // columns beyond W + 2 r are pitch padding (ignored): they make the row pitch a multiple of
    // 16 bytes so that tiles can be fetched by TMA
    if (src->shape[0] != bands || src->shape[1] != H + 2 * r || src->shape[2] < W + 2 * r)
      return fail("gm_moving_max: source must carry a size//2 pixel halo");
    const int SW = (int)src->shape[2];
    GM_DISPATCH_NUMERIC(src->dtype, run_moving_max<T>(in, out, nodata, has_nodata, bands, H, W, SW, size, s));
  });
}

extern "C" int gm_dilate(const GmArray* src, GmArray* dst, const void* values, int n_values,
                         void* stream) {
  return with_staged(src, dst, stream, [&](Staged& in, Staged& out, cudaStream_t s) -> int {
    const int bands = (int)dst->shape[0], H = (int)dst->shape[1], W = (int)dst->shape[2];
    if (src->dtype != dst->dtype) return fail("gm_dilate: dtype mismatch");
    if (src->shape[0] != bands || src->shape[1] != H + 2 || src->shape[2] != W + 2)
      return fail("gm_dilate: source must carry a 1 pixel halo");
    GM_DISPATCH_NUMERIC(src->dtype, run_dilate<T>(in, out, values, n_values, bands, H, W, s));
  });
}

extern "C" int gm_set_smooth_mode(int mode) {
  if (mode < GM_SMOOTH_EXACT || mode > GM_SMOOTH_FLOAT32) return fail("gm_set_smooth_mode: bad mode");
  g_smooth_mode.store(mode);
  return 0;
}
extern "C" int gm_get_smooth_mode(void) { return smooth_mode(); }

extern "C" int gm_smooth(const GmArray* src, GmArray* dst, const void* nodata, int has_nodata,
                         double fill, const double* wy, int ly, const double* wx, int lx, int my,
                         int mx, int zoom, double zy, double zx, double oy, double ox, void* stream) {
  return with_staged(src, dst, stream, [&](Staged& in, Staged& out, cudaStream_t s) -> int {
    const int bands = (int)dst->shape[0], H = (int)dst->shape[1], W = (int)dst->shape[2];
    const int SH = (int)src->shape[1], SW = (int)src->shape[2];
    if (src->dtype != dst->dtype) return fail("gm_smooth: dtype mismatch");
    if (src->shape[0] != bands || SH != H + 2 * my || SW != W + 2 * mx)
      return fail("gm_smooth: source shape must be the output shape plus the margins");
    if (zoom && (my != 0 || mx != 0)) return fail("gm_smooth: zoom mode takes no margins");
    GM_DISPATCH_NUMERIC(src->dtype, run_smooth<T>(in, out, nodata, has_nodata, fill, wy, ly, wx, lx,
                                                  bands, SH, SW, H, W, my, mx, zoom, zy, zx, oy, ox, s));
  });
}
