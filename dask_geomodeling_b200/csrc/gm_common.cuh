// Shared internals of libgeokernels.so (not part of the ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <vector>
#include <atomic>
#include <cstdio>
#include <cstring>
#include "../../include/geokernels.h"

namespace gm {

void set_error(const std::string& msg);
int  fail(const std::string& msg);               // sets the error, returns 1
cudaStream_t resolve_stream(void* stream);       // NULL -> library stream
int  ensure_init();
int  sm_count();
void count_launch(int n = 1);

#define GM_CUDA(expr)                                                          \
  do {                                                                         \
    cudaError_t _e = (expr);                                                   \
    if (_e != cudaSuccess) {                                                   \
      return gm::fail(std::string(#expr) + ": " + cudaGetErrorString(_e));     \
    }                                                                          \
  } while (0)

#define GM_LAUNCH_CHECK()                                                      \
  do {                                                                         \
    cudaError_t _e = cudaGetLastError();                                       \
    if (_e != cudaSuccess) {                                                   \
      return gm::fail(std::string("kernel launch: ") + cudaGetErrorString(_e));\
    }                                                                          \
    gm::count_launch();                                                        \
  } while (0)

__host__ __device__ inline int dtype_size(int dt) {
  switch (dt) {
    case GM_BOOL: case GM_U8: case GM_I8: return 1;
    case GM_U16: case GM_I16: return 2;
    case GM_U32: case GM_I32: case GM_F32: return 4;
    case GM_I64: case GM_F64: return 8;
  }
  return 0;
}

// non-finite float source values become no data in the resample / warp gathers
template <typename T> __device__ __forceinline__ bool is_finite(T v) { return true; }
template <> __device__ __forceinline__ bool is_finite<float>(float v) { return isfinite(v); }
template <> __device__ __forceinline__ bool is_finite<double>(double v) { return isfinite(v); }

inline int64_t array_count(const GmArray& a) { return a.shape[0] * a.shape[1] * a.shape[2]; }
inline int64_t array_bytes(const GmArray& a) { return array_count(a) * dtype_size(a.dtype); }

// Device view of an array that may live on the host: uploads on construction
// (inputs) and/or downloads on finish() (outputs).  All work is stream-ordered.
struct Staged {
  void* dev = nullptr;
  void* host = nullptr;
  int64_t bytes = 0;
  bool owned = false;
  cudaStream_t stream = nullptr;
  int open_input(const GmArray& a, cudaStream_t s);
  int open_output(const GmArray& a, cudaStream_t s);
  int finish_output();      // async D2H if staged
  void release();           // free staging buffer
};

// Small host table -> device copy helper (stream ordered).
int upload(void** dev, const void* host, int64_t bytes, cudaStream_t s);

}  // namespace gm
