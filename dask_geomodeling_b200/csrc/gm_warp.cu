// Nearest-neighbour warp across WGS 84 projections (replaces gdal.ReprojectImage in the
// reference's raster/sources.py:119-149 for EPSG:4326, EPSG:3857 and the UTM zones).
//
// Two kernels, chosen by the CRS pair:
//   - EPSG:4326 <-> EPSG:3857 is separable: the source column depends only on the target column
//     and the source row only on the target row.  One small kernel computes both index vectors,
//     the gather reads them (HBM-bound like resample_nn_kernel);
//   - pairs with a UTM zone evaluate the transverse Mercator series per cell in fp64, once per
//     cell for all bands.
#include "gm_common.cuh"
#include "gm_crs.cuh"

namespace gm {

constexpr int32_t kOutside = -1;   // no source cell: no data
constexpr int32_t kMiss = -2;      // a source cell outside the uploaded window

struct WarpArgs {
  int dst_kind, dst_zone, src_kind, src_zone;
  double dp, da, dq, dd;           // request geotransform (no rotation)
  double sp, sa, sq, sd;           // whole-source geotransform
  int64_t src_h, src_w, row0, col0;
};

// source (row, col) of the target centre (x, y) given in the request CRS, as floor()ed doubles
__device__ __forceinline__ void source_cell(const WarpArgs& w, double x, double y, double& fr,
                                            double& fc) {
  crs::to_degrees(x, y, w.dst_kind, w.dst_zone);
  crs::from_degrees(x, y, w.src_kind, w.src_zone);
  // GDAL's nearest-neighbour fudge, as window_geometry() in raster/sources.py
  fc = floor((x - w.sp) / w.sa + 1e-10);
  fr = floor((y - w.sq) / w.sd + 1e-10);
}

// kOutside / kMiss / index inside the window, for one axis
__device__ __forceinline__ int32_t classify(double f, int64_t n_src, int64_t origin, int64_t n_win) {
  if (!(f >= 0.0 && f < (double)n_src)) return kOutside;   // also NaN
  const int64_t k = (int64_t)f - origin;
  return (k >= 0 && k < n_win) ? (int32_t)k : kMiss;
}

// separable pairs: cols[j] for j < dw, then rows[i]; the other coordinate is held at 0 (valid in
// both CRSs), which the separable transforms do not read
__global__ void warp_axes_kernel(WarpArgs w, int dw, int dh, int64_t win_h, int64_t win_w,
                                 int32_t* __restrict__ cols, int32_t* __restrict__ rows) {
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < dw + dh; t += gridDim.x * blockDim.x) {
    double fr, fc;
    if (t < dw) {
      source_cell(w, w.dp + (t + 0.5) * w.da, 0.0, fr, fc);
      cols[t] = classify(fc, w.src_w, w.col0, win_w);
    } else {
      const int i = t - dw;
      source_cell(w, 0.0, w.dq + (i + 0.5) * w.dd, fr, fc);
      rows[i] = classify(fr, w.src_h, w.row0, win_h);
    }
  }
}

template <typename T>
__global__ void warp_gather_kernel(const T* __restrict__ src, T* __restrict__ dst, T nodata, int bands,
                                   int sh, int sw, int dh, int dw, const int32_t* __restrict__ cols,
                                   const int32_t* __restrict__ rows, unsigned long long* misses) {
  const int64_t plane = (int64_t)dh * dw;
  unsigned long long missed = 0;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < plane;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int i = (int)(idx / dw), j = (int)(idx - (int64_t)i * dw);
    const int32_t r = __ldg(rows + i), c = __ldg(cols + j);
    const bool inside = r >= 0 && c >= 0;
    missed += (!inside && r != kOutside && c != kOutside);
    const int64_t at = (int64_t)r * sw + c;
    for (int b = 0; b < bands; ++b) {
      T v = nodata;
      if (inside) {
        v = src[(int64_t)b * sh * sw + at];
        if (!is_finite(v)) v = nodata;
      }
      dst[(int64_t)b * plane + idx] = v;
    }
  }
  if (missed && misses) atomicAdd(misses, missed);
}

// pairs with a UTM zone: the full transform per cell
template <typename T>
__global__ void warp_cells_kernel(const T* __restrict__ src, T* __restrict__ dst, T nodata, int bands,
                                  int sh, int sw, int dh, int dw, WarpArgs w,
                                  unsigned long long* misses) {
  const int64_t plane = (int64_t)dh * dw;
  unsigned long long missed = 0;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < plane;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int i = (int)(idx / dw), j = (int)(idx - (int64_t)i * dw);
    double fr, fc;
    source_cell(w, w.dp + (j + 0.5) * w.da, w.dq + (i + 0.5) * w.dd, fr, fc);
    const int32_t r = classify(fr, w.src_h, w.row0, sh), c = classify(fc, w.src_w, w.col0, sw);
    const bool inside = r >= 0 && c >= 0;
    missed += (!inside && r != kOutside && c != kOutside);
    const int64_t at = (int64_t)r * sw + c;
    for (int b = 0; b < bands; ++b) {
      T v = nodata;
      if (inside) {
        v = src[(int64_t)b * sh * sw + at];
        if (!is_finite(v)) v = nodata;
      }
      dst[(int64_t)b * plane + idx] = v;
    }
  }
  if (missed && misses) atomicAdd(misses, missed);
}

template <typename T>
static int launch_warp(const GmArray* src, GmArray* dst, const void* nodata, const WarpArgs& w,
                       unsigned long long* misses, cudaStream_t s) {
  T nd;
  memcpy(&nd, nodata, sizeof(T));
  const int bands = (int)dst->shape[0], dh = (int)dst->shape[1], dw = (int)dst->shape[2];
  const int sh = (int)src->shape[1], sw = (int)src->shape[2];
  const int64_t plane = (int64_t)dh * dw;
  int64_t blocks = (plane + 255) / 256;
  const int64_t cap = (int64_t)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  if (crs::is_separable(w.src_kind, w.dst_kind)) {
    int32_t* axes = nullptr;
    GM_CUDA(cudaMallocAsync((void**)&axes, sizeof(int32_t) * ((int64_t)dw + dh), s));
    warp_axes_kernel<<<(unsigned)((dw + dh + 255) / 256), 256, 0, s>>>(w, dw, dh, sh, sw, axes,
                                                                       axes + dw);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) {
      count_launch();
      warp_gather_kernel<T><<<(unsigned)blocks, 256, 0, s>>>(
          (const T*)src->data, (T*)dst->data, nd, bands, sh, sw, dh, dw, axes, axes + dw, misses);
      e = cudaGetLastError();
    }
    cudaFreeAsync(axes, s);
    if (e != cudaSuccess) return fail(std::string("gm_warp_nn launch: ") + cudaGetErrorString(e));
    count_launch();
    return 0;
  }
  warp_cells_kernel<T><<<(unsigned)blocks, 256, 0, s>>>(
      (const T*)src->data, (T*)dst->data, nd, bands, sh, sw, dh, dw, w, misses);
  GM_LAUNCH_CHECK();
  return 0;
}

static int dispatch_warp(const GmArray* src, GmArray* dst, const void* nodata, const WarpArgs& w,
                         unsigned long long* misses, cudaStream_t s) {
  switch (src->dtype) {
    case GM_F32: return launch_warp<float>(src, dst, nodata, w, misses, s);
    case GM_F64: return launch_warp<double>(src, dst, nodata, w, misses, s);
    default: break;
  }
  switch (dtype_size(src->dtype)) {
    case 1: return launch_warp<uint8_t>(src, dst, nodata, w, misses, s);
    case 2: return launch_warp<uint16_t>(src, dst, nodata, w, misses, s);
    case 4: return launch_warp<uint32_t>(src, dst, nodata, w, misses, s);
    case 8: return launch_warp<uint64_t>(src, dst, nodata, w, misses, s);
  }
  return fail("gm_warp_nn: unsupported dtype");
}

}  // namespace gm

using namespace gm;

static bool valid_crs(int32_t kind, int32_t zone) {
  if (kind == GM_CRS_UTM) return zone != 0 && zone >= -60 && zone <= 60;
  return (kind == GM_CRS_GEOGRAPHIC || kind == GM_CRS_MERCATOR) && zone == 0;
}

extern "C" int gm_warp_nn(const GmArray* src, GmArray* dst, const void* nodata, const GmWarp* warp,
                          int64_t* misses, void* stream) {
  if (ensure_init()) return 1;
  if (!src || !dst || !nodata || !warp) return fail("gm_warp_nn: null argument");
  if (src->dtype != dst->dtype) return fail("gm_warp_nn: dtype mismatch");
  if (src->space != GM_DEVICE || dst->space != GM_DEVICE)
    return fail("gm_warp_nn: operands must be device resident");
  if (src->shape[0] != dst->shape[0]) return fail("gm_warp_nn: band count mismatch");
  if (!valid_crs(warp->src_kind, warp->src_zone) || !valid_crs(warp->dst_kind, warp->dst_zone))
    return fail("gm_warp_nn: unsupported CRS");
  if (warp->dst_geo[2] != 0.0 || warp->dst_geo[4] != 0.0 || warp->src_geo[2] != 0.0 ||
      warp->src_geo[4] != 0.0)
    return fail("gm_warp_nn: rotated geotransforms are not supported");
  if (dst->shape[1] > INT32_MAX || dst->shape[2] > INT32_MAX || src->shape[1] > INT32_MAX ||
      src->shape[2] > INT32_MAX)
    return fail("gm_warp_nn: raster side exceeds 2^31 - 1");
  if (misses) *misses = 0;
  if (array_count(*dst) == 0) return 0;
  cudaStream_t s = resolve_stream(stream);
  WarpArgs w;
  w.dst_kind = warp->dst_kind; w.dst_zone = warp->dst_zone;
  w.src_kind = warp->src_kind; w.src_zone = warp->src_zone;
  w.dp = warp->dst_geo[0]; w.da = warp->dst_geo[1]; w.dq = warp->dst_geo[3]; w.dd = warp->dst_geo[5];
  w.sp = warp->src_geo[0]; w.sa = warp->src_geo[1]; w.sq = warp->src_geo[3]; w.sd = warp->src_geo[5];
  w.src_h = warp->src_height; w.src_w = warp->src_width;
  w.row0 = warp->win_row0; w.col0 = warp->win_col0;
  if (!misses) return dispatch_warp(src, dst, nodata, w, nullptr, s);

  unsigned long long* counter = nullptr;
  GM_CUDA(cudaMallocAsync((void**)&counter, sizeof(*counter), s));
  int rc = 0;
  cudaError_t e = cudaMemsetAsync(counter, 0, sizeof(*counter), s);
  if (e != cudaSuccess) rc = fail(std::string("gm_warp_nn: ") + cudaGetErrorString(e));
  if (rc == 0) rc = dispatch_warp(src, dst, nodata, w, counter, s);
  unsigned long long host = 0;
  if (rc == 0) {
    e = cudaMemcpyAsync(&host, counter, sizeof(host), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) rc = fail(std::string("gm_warp_nn: ") + cudaGetErrorString(e));
  }
  cudaFreeAsync(counter, s);
  if (rc == 0) *misses = (int64_t)host;
  return rc;
}
