// Input adaptor kernels: constant fill and nearest-neighbour resample/crop/pad
// (replaces the GDAL warp in the reference's raster/sources.py:119-149).
#include "gm_common.cuh"

namespace gm {

template <typename T>
__global__ void fill_kernel(T* __restrict__ dst, T value, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x)
    dst[i] = value;
}


// out[b, i, j] = src[b, floor(row0 + i*row_step), floor(col0 + j*col_step)], or
// nodata outside the source window; non-finite floats become nodata
// (raster/sources.py:146-148).
template <typename T>
__global__ void resample_nn_kernel(const T* __restrict__ src, T* __restrict__ dst, T nodata,
                                   int bands, int sh, int sw, int dh, int dw,
                                   double col0, double col_step, double row0, double row_step) {
  const int64_t plane = (int64_t)dh * dw;
  const int64_t total = plane * bands;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int b = (int)(idx / plane);
    const int64_t r = idx - (int64_t)b * plane;
    const int i = (int)(r / dw), j = (int)(r - (int64_t)i * dw);
    const double fr = floor(row0 + i * row_step), fc = floor(col0 + j * col_step);
    T v = nodata;
    if (fr >= 0.0 && fr < (double)sh && fc >= 0.0 && fc < (double)sw) {
      v = src[((int64_t)b * sh + (int64_t)fr) * sw + (int64_t)fc];
      if (!is_finite(v)) v = nodata;
    }
    dst[idx] = v;
  }
}

template <typename T>
static int launch_resample(const GmArray* src, GmArray* dst, const void* nodata, double col0,
                           double col_step, double row0, double row_step, cudaStream_t s) {
  const int64_t total = array_count(*dst);
  if (total == 0) return 0;
  T nd;
  memcpy(&nd, nodata, sizeof(T));
  int64_t blocks = (total + 255) / 256;
  const int64_t cap = (int64_t)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  resample_nn_kernel<T><<<(unsigned)blocks, 256, 0, s>>>(
      (const T*)src->data, (T*)dst->data, nd, (int)dst->shape[0], (int)src->shape[1],
      (int)src->shape[2], (int)dst->shape[1], (int)dst->shape[2], col0, col_step, row0, row_step);
  GM_LAUNCH_CHECK();
  return 0;
}

}  // namespace gm

using namespace gm;

extern "C" int gm_fill(void* dst, int32_t dtype, const void* value, int64_t count, void* stream) {
  if (ensure_init()) return 1;
  if (count <= 0) return 0;
  cudaStream_t s = resolve_stream(stream);
  int64_t blocks = (count + 255) / 256;
  const int64_t cap = (int64_t)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  switch (dtype_size(dtype)) {
    case 1: { uint8_t v; memcpy(&v, value, 1); fill_kernel<<<(unsigned)blocks, 256, 0, s>>>((uint8_t*)dst, v, count); break; }
    case 2: { uint16_t v; memcpy(&v, value, 2); fill_kernel<<<(unsigned)blocks, 256, 0, s>>>((uint16_t*)dst, v, count); break; }
    case 4: { uint32_t v; memcpy(&v, value, 4); fill_kernel<<<(unsigned)blocks, 256, 0, s>>>((uint32_t*)dst, v, count); break; }
    case 8: { uint64_t v; memcpy(&v, value, 8); fill_kernel<<<(unsigned)blocks, 256, 0, s>>>((uint64_t*)dst, v, count); break; }
    default: return fail("gm_fill: unsupported dtype");
  }
  GM_LAUNCH_CHECK();
  return 0;
}

extern "C" int gm_resample_nn(const GmArray* src, GmArray* dst, const void* nodata, double col0,
                              double col_step, double row0, double row_step, void* stream) {
  if (ensure_init()) return 1;
  if (!src || !dst || !nodata) return fail("gm_resample_nn: null argument");
  if (src->dtype != dst->dtype) return fail("gm_resample_nn: dtype mismatch");
  if (src->space != GM_DEVICE || dst->space != GM_DEVICE)
    return fail("gm_resample_nn: operands must be device resident");
  if (src->shape[0] != dst->shape[0]) return fail("gm_resample_nn: band count mismatch");
  cudaStream_t s = resolve_stream(stream);
  switch (src->dtype) {
    case GM_F32: return launch_resample<float>(src, dst, nodata, col0, col_step, row0, row_step, s);
    case GM_F64: return launch_resample<double>(src, dst, nodata, col0, col_step, row0, row_step, s);
    default: break;
  }
  switch (dtype_size(src->dtype)) {
    case 1: return launch_resample<uint8_t>(src, dst, nodata, col0, col_step, row0, row_step, s);
    case 2: return launch_resample<uint16_t>(src, dst, nodata, col0, col_step, row0, row_step, s);
    case 4: return launch_resample<uint32_t>(src, dst, nodata, col0, col_step, row0, row_step, s);
    case 8: return launch_resample<uint64_t>(src, dst, nodata, col0, col_step, row0, row_step, s);
  }
  return fail("gm_resample_nn: unsupported dtype");
}
