// Ceiling probe of the cfg2 chain (Reclassify, Clip, Step, IsData on int16 + float32 -> bool):
// the byte pattern of the specialised kernel gm_jit.cu generates for it, with trivial work per pixel.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o chain_ceiling tools/chain_ceiling.cu
//   ./chain_ceiling [edge = 16384] [blocks per SM = 0] [launches = 1000]
// (tools/chain_ceiling.py compiles and runs it.)  Same access pattern as gm_fused on cfg2: 256
// threads, a thread owns groups of V = 4 pixels (8 B of int16, 16 B of float32, 4 B out), loads
// U = 4 groups before it evaluates any, ld.global.cs / st.global.cs, one block per chunk of 256 U
// groups.  `blocks per SM` > 0 caps the grid at SMs x that many blocks, which then stride over the
// chunks (what gm_fused does for programs with tables in shared memory).  Per pixel it computes
// out = (a != 32767) & (b != FLT_MAX).  The time of one launch, over `launches` launches after a
// warm-up, is what the chain could take under this access pattern if evaluating it cost nothing.
#include <cuda_runtime.h>
#include <cfloat>
#include <cstdint>
#include <cstdio>
#include <cstdlib>

#define CHECK(x)                                                                          \
  do {                                                                                    \
    cudaError_t e_ = (x);                                                                 \
    if (e_ != cudaSuccess) {                                                              \
      fprintf(stderr, "%s:%d %s: %s\n", __FILE__, __LINE__, #x, cudaGetErrorString(e_)); \
      return 1;                                                                           \
    }                                                                                     \
  } while (0)

constexpr int V = 4, U = 4, T = 256;

__device__ __forceinline__ uint32_t flag(uint32_t a16, uint32_t b) {
  return ((a16 & 0xffffu) != 0x7fffu) & (__uint_as_float(b) != FLT_MAX);
}
__device__ __forceinline__ uint32_t flags(uint2 a, uint4 b) {
  return flag(a.x, b.x) | flag(a.x >> 16, b.y) << 8 | flag(a.y, b.z) << 16 | flag(a.y >> 16, b.w) << 24;
}

__global__ void __launch_bounds__(T) chain_ceiling(const int16_t* __restrict__ a, const float* __restrict__ b,
                                                   uint8_t* __restrict__ out, long long n) {
  const long long groups = n / V, chunk = (long long)T * U, n_chunks = groups / chunk;
  const uint2* a2 = reinterpret_cast<const uint2*>(a);
  const uint4* b4 = reinterpret_cast<const uint4*>(b);
  uint32_t* o4 = reinterpret_cast<uint32_t*>(out);
  for (long long c = blockIdx.x; c < n_chunks; c += gridDim.x) {
    const long long g0 = c * chunk + threadIdx.x;
    uint2 x[U];
    uint4 y[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      x[u] = __ldcs(a2 + g0 + u * T);
      y[u] = __ldcs(b4 + g0 + u * T);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) __stcs(o4 + g0 + u * T, flags(x[u], y[u]));
  }
  for (long long px = n_chunks * chunk * V + (long long)blockIdx.x * T + threadIdx.x; px < n;
       px += (long long)gridDim.x * T)
    out[px] = (uint8_t)flag((uint16_t)a[px], __float_as_uint(b[px]));
}

__global__ void fill(int16_t* a, float* b, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const uint32_t h = (uint32_t)(i * 2654435761u);
    a[i] = (h % 13 == 0) ? (int16_t)32767 : (int16_t)(h % 49);
    b[i] = (h % 11 == 0) ? FLT_MAX : (float)(h % 100);
  }
}

int main(int argc, char** argv) {
  const long long edge = argc > 1 ? atoll(argv[1]) : 16384;
  const int per_sm = argc > 2 ? atoi(argv[2]) : 0;
  const int launches = argc > 3 ? atoi(argv[3]) : 1000;
  const long long n = edge * edge;
  cudaDeviceProp prop;
  CHECK(cudaGetDeviceProperties(&prop, 0));
  int16_t* a;
  float* b;
  uint8_t* out;
  CHECK(cudaMalloc(&a, n * sizeof(int16_t)));
  CHECK(cudaMalloc(&b, n * sizeof(float)));
  CHECK(cudaMalloc(&out, n));
  fill<<<prop.multiProcessorCount * 8, 256>>>(a, b, n);
  CHECK(cudaGetLastError());
  const long long per_block = (long long)T * U * V;
  long long grid = (n + per_block - 1) / per_block;
  if (per_sm > 0 && grid > (long long)prop.multiProcessorCount * per_sm) grid = (long long)prop.multiProcessorCount * per_sm;
  if (grid < 1) grid = 1;
  for (int i = 0; i < 20; ++i) chain_ceiling<<<(unsigned)grid, T>>>(a, b, out, n);
  CHECK(cudaDeviceSynchronize());
  cudaEvent_t t0, t1;
  CHECK(cudaEventCreate(&t0));
  CHECK(cudaEventCreate(&t1));
  CHECK(cudaEventRecord(t0));
  for (int i = 0; i < launches; ++i) chain_ceiling<<<(unsigned)grid, T>>>(a, b, out, n);
  CHECK(cudaEventRecord(t1));
  CHECK(cudaEventSynchronize(t1));
  CHECK(cudaGetLastError());
  float ms = 0;
  CHECK(cudaEventElapsedTime(&ms, t0, t1));
  ms /= launches;

  // check a sample of the output against the rule on the host
  const long long m = n < (1 << 20) ? n : (1 << 20);
  int16_t* ha = (int16_t*)malloc(m * sizeof(int16_t));
  float* hb = (float*)malloc(m * sizeof(float));
  uint8_t* ho = (uint8_t*)malloc(m);
  CHECK(cudaMemcpy(ha, a + (n - m), m * sizeof(int16_t), cudaMemcpyDeviceToHost));
  CHECK(cudaMemcpy(hb, b + (n - m), m * sizeof(float), cudaMemcpyDeviceToHost));
  CHECK(cudaMemcpy(ho, out + (n - m), m, cudaMemcpyDeviceToHost));
  long long bad = 0;
  for (long long i = 0; i < m; ++i) bad += ho[i] != (uint8_t)(ha[i] != 32767 && hb[i] != FLT_MAX);

  const double bytes = 7.0 * (double)n;
  printf("{\"device\": \"%s\", \"sms\": %d, \"edge\": %lld, \"blocks_per_sm\": %d, \"grid\": %lld, "
         "\"launches\": %d, \"ms_per_launch\": %.4f, \"tb_per_s\": %.3f, \"gpx_per_s\": %.1f, "
         "\"mismatches\": %lld}\n",
         prop.name, prop.multiProcessorCount, edge, per_sm, grid, launches, ms, bytes / (ms * 1e-3) / 1e12,
         (double)n / (ms * 1e-3) / 1e9, bad);
  CHECK(cudaFree(a));
  CHECK(cudaFree(b));
  CHECK(cudaFree(out));
  return bad ? 2 : 0;
}
