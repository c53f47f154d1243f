// Ceiling probe of the cfg2 chain (Reclassify, Clip, Step, IsData on int16 + float32 -> bool):
// the byte pattern of the specialised kernel gm_jit.cu generates for it, with trivial work per pixel.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o chain_ceiling tools/chain_ceiling.cu
//   ./chain_ceiling [edge = 16384] [blocks per SM = 0] [launches = 1000] [skeleton = 0] [W = 0] [K = 1]
// (tools/chain_ceiling.py compiles and runs it.)  Same access pattern as gm_fused on cfg2: 256
// threads, a thread owns groups of V = 4 pixels (8 B of int16, 16 B of float32, 4 B out), loads
// U = 4 groups before it evaluates any, ld.global.cs / st.global.cs, one block per K chunks of
// 256 U groups.  `blocks per SM` > 0 caps the grid at SMs x that many blocks, which then stride over
// the chunks (what gm_fused does for programs with tables in shared memory).  Per pixel it computes
// out = (a != 32767) & (b != FLT_MAX), plus W dependent multiply-adds that do not change it (the
// work dial: 0, 8, 16 or 24).  The time of one launch, over `launches` launches after a warm-up, is
// what the chain could take under this access pattern and skeleton if evaluating it cost W
// instructions per pixel.
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

// `W` extra dependent integer multiply-adds per pixel, seeded from both inputs; `zero` (0 at run time)
// folds the result into the flag, so the compiler must compute it and the output does not change.
template <int W>
__device__ __forceinline__ uint32_t flag(uint32_t a16, uint32_t b, uint32_t zero) {
  uint32_t f = ((a16 & 0xffffu) != 0x7fffu) & (__uint_as_float(b) != FLT_MAX);
  if constexpr (W > 0) {
    uint32_t h = a16 ^ b;
#pragma unroll
    for (int w = 0; w < W; ++w) h = h * 0x9E3779B1u + 0x7F4A7C15u;
    f ^= h & zero;
  }
  return f;
}
template <int W>
__device__ __forceinline__ uint32_t flags(uint2 a, uint4 b, uint32_t zero) {
  return flag<W>(a.x, b.x, zero) | flag<W>(a.x >> 16, b.y, zero) << 8 | flag<W>(a.y, b.z, zero) << 16 |
         flag<W>(a.y >> 16, b.w, zero) << 24;
}

// Kernel skeletons:
//   SINGLE     one chunk per block, loads placed by the compiler (what gm_fused did until r04);
//   PINNED     one chunk per block, a block barrier after the 2 U loads (a load cannot sink below it);
//   PIPELINED  K consecutive chunks per block in two register sets: the loads of chunk c + 1 are
//              issued before chunk c is evaluated (the prologue loads the first chunk).
enum Skeleton { SINGLE = 0, PINNED = 1, PIPELINED = 2 };

__device__ __forceinline__ void load_chunk(uint2 (&x)[U], uint4 (&y)[U], const uint2* a2, const uint4* b4, long long g0) {
#pragma unroll
  for (int u = 0; u < U; ++u) {
    x[u] = __ldcs(a2 + g0 + u * T);
    y[u] = __ldcs(b4 + g0 + u * T);
  }
}
template <int W>
__device__ __forceinline__ void eval_chunk(const uint2 (&x)[U], const uint4 (&y)[U], uint32_t* o4, long long g0,
                                           uint32_t zero) {
#pragma unroll
  for (int u = 0; u < U; ++u) __stcs(o4 + g0 + u * T, flags<W>(x[u], y[u], zero));
}

template <int MODE, int W>
__global__ void __launch_bounds__(T) chain_ceiling(const int16_t* __restrict__ a, const float* __restrict__ b,
                                                   uint8_t* __restrict__ out, long long n, int K, uint32_t zero) {
  const long long groups = n / V, chunk = (long long)T * U, n_chunks = groups / chunk;
  const uint2* a2 = reinterpret_cast<const uint2*>(a);
  const uint4* b4 = reinterpret_cast<const uint4*>(b);
  uint32_t* o4 = reinterpret_cast<uint32_t*>(out);
  if (MODE == PIPELINED) {
    for (long long c0 = (long long)blockIdx.x * K; c0 < n_chunks; c0 += (long long)gridDim.x * K) {
      const long long c1 = c0 + K < n_chunks ? c0 + K : n_chunks;
      uint2 x0[U], x1[U];
      uint4 y0[U], y1[U];
      load_chunk(x0, y0, a2, b4, c0 * chunk + threadIdx.x);
      for (long long c = c0; c < c1; c += 2) {
        if (c + 1 < c1) load_chunk(x1, y1, a2, b4, (c + 1) * chunk + threadIdx.x);
        eval_chunk<W>(x0, y0, o4, c * chunk + threadIdx.x, zero);
        if (c + 1 == c1) break;
        if (c + 2 < c1) load_chunk(x0, y0, a2, b4, (c + 2) * chunk + threadIdx.x);
        eval_chunk<W>(x1, y1, o4, (c + 1) * chunk + threadIdx.x, zero);
      }
    }
  } else {
    for (long long c = blockIdx.x; c < n_chunks; c += gridDim.x) {
      const long long g0 = c * chunk + threadIdx.x;
      uint2 x[U];
      uint4 y[U];
      load_chunk(x, y, a2, b4, g0);
      if (MODE == PINNED) __syncthreads();
      eval_chunk<W>(x, y, o4, g0, zero);
    }
  }
  for (long long px = n_chunks * chunk * V + (long long)blockIdx.x * T + threadIdx.x; px < n;
       px += (long long)gridDim.x * T)
    out[px] = (uint8_t)flag<W>((uint16_t)a[px], __float_as_uint(b[px]), zero);
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
  const int skeleton = argc > 4 ? atoi(argv[4]) : SINGLE;
  const int work = argc > 5 ? atoi(argv[5]) : 0;
  const int K = skeleton == PIPELINED && argc > 6 ? atoi(argv[6]) : 1;
  typedef void (*Kernel)(const int16_t*, const float*, uint8_t*, long long, int, uint32_t);
  const Kernel kernels[3][4] = {
      {chain_ceiling<SINGLE, 0>, chain_ceiling<SINGLE, 8>, chain_ceiling<SINGLE, 16>, chain_ceiling<SINGLE, 24>},
      {chain_ceiling<PINNED, 0>, chain_ceiling<PINNED, 8>, chain_ceiling<PINNED, 16>, chain_ceiling<PINNED, 24>},
      {chain_ceiling<PIPELINED, 0>, chain_ceiling<PIPELINED, 8>, chain_ceiling<PIPELINED, 16>,
       chain_ceiling<PIPELINED, 24>}};
  if (skeleton < 0 || skeleton > 2 || work % 8 || work < 0 || work > 24 || K < 1) {
    fprintf(stderr, "skeleton 0..2, W in {0, 8, 16, 24}, K >= 1\n");
    return 1;
  }
  const Kernel kernel = kernels[skeleton][work / 8];
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
  const long long per_block = (long long)T * U * V * K;
  long long grid = (n + per_block - 1) / per_block;
  if (per_sm > 0 && grid > (long long)prop.multiProcessorCount * per_sm) grid = (long long)prop.multiProcessorCount * per_sm;
  if (grid < 1) grid = 1;
  for (int i = 0; i < 20; ++i) kernel<<<(unsigned)grid, T>>>(a, b, out, n, K, 0u);
  CHECK(cudaDeviceSynchronize());
  cudaEvent_t t0, t1;
  CHECK(cudaEventCreate(&t0));
  CHECK(cudaEventCreate(&t1));
  CHECK(cudaEventRecord(t0));
  for (int i = 0; i < launches; ++i) kernel<<<(unsigned)grid, T>>>(a, b, out, n, K, 0u);
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
  printf("{\"device\": \"%s\", \"sms\": %d, \"edge\": %lld, \"skeleton\": \"%s\", \"W\": %d, \"K\": %d, "
         "\"blocks_per_sm\": %d, \"grid\": %lld, "
         "\"launches\": %d, \"ms_per_launch\": %.4f, \"tb_per_s\": %.3f, \"gpx_per_s\": %.1f, "
         "\"mismatches\": %lld}\n",
         prop.name, prop.multiProcessorCount, edge, (const char*[]){"single", "pinned", "pipelined"}[skeleton], work, K,
         per_sm, grid, launches, ms, bytes / (ms * 1e-3) / 1e12,
         (double)n / (ms * 1e-3) / 1e9, bad);
  CHECK(cudaFree(a));
  CHECK(cudaFree(b));
  CHECK(cudaFree(out));
  return bad ? 2 : 0;
}
