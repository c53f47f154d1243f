// Fused element-wise evaluator: one HBM pass per program.
//
// Persistent CTAs walk tiles of TILE = 256 * V pixels.  For every tile
//   - one elected thread streams the tile of every input raster from HBM into
//     shared memory with TMA bulk copies (cp.async.bulk + mbarrier complete_tx),
//     double buffered so that the next tile is in flight while this one is
//     being evaluated;
//   - all threads interpret the program once for their V pixels: the instruction
//     stream sits in the kernel parameter (constant) bank and is decoded
//     warp-uniformly, the accumulator lives in registers, the machine registers
//     and the staged inputs are read straight from shared memory (consecutive
//     lanes touch consecutive words: conflict free);
//   - results are staged in shared memory and leave with TMA bulk stores.
// Two machines are instantiated: 32-bit slots (classes I32/F32, V = 16) and 64-bit
// slots (all four classes, V = 8).
//
// What each instruction does to a pixel is defined once, in gm_eval_ops.cuh, which the
// specialised kernels (gm_jit.cu) share; this file owns the staging, the operand addressing and the
// dispatch of classes and opcodes.
#include "gm_common.cuh"
#include "gm_jit.h"
#include <type_traits>

// The transcendentals and the integer power are kept out of line: rare, large, and they would
// otherwise dictate the register allocation of the whole interpreter.
#define GM_OUTLINE __device__ __noinline__
#include "gm_eval_ops.cuh"

namespace gm {

constexpr int THREADS = 256;
constexpr int NSTAGE = 2;

struct DevTable {
  const int64_t* keys;   // sorted keys (int64 or float64 bits)
  const uint64_t* vals;  // 8-byte values
  const uint8_t* hit;    // per entry: 1 mapped, 2 mapped onto the fill value
  int64_t base;
  int32_t n;
  int32_t kind;
};

struct EvalParams {
  int32_t n_instr;
  int32_t n_inputs;
  int32_t n_outputs;
  int32_t n_tables;
  int32_t tables_in_smem;
  int32_t n_regs;
  int64_t n;
  const void* in[GM_MAX_INPUTS];
  void* out[GM_MAX_OUTPUTS];
  int32_t in_dtype[GM_MAX_INPUTS];
  int32_t out_dtype[GM_MAX_OUTPUTS];
  int32_t in_off[GM_MAX_INPUTS];    // byte offset of the input inside one input stage
  int32_t out_off[GM_MAX_OUTPUTS];  // byte offset of the output inside one output stage
  int32_t in_stage_bytes, out_stage_bytes;
  int32_t regs_off, tables_off, bar_off;  // byte offsets in dynamic shared memory
  int32_t pad;
  DevTable tab[GM_MAX_TABLES];
  GmInstr instr[GM_MAX_INSTR];
};

template <int W> struct SlotOf;
template <> struct SlotOf<4> { typedef uint32_t type; };
template <> struct SlotOf<8> { typedef uint64_t type; };

// ---- mbarrier / TMA bulk copy wrappers (PTX) -----------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra WAIT_DONE;\n"
      "bra WAIT_LOOP;\n"
      "WAIT_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(smem_dst)),
      "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void bulk_store(void* gdst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst),
               "r"(smem_u32(smem_src)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- class / dtype dispatch, hoisted out of the per-pixel loops ---------------------------
// Every multi-way decision (storage dtype, value class) is taken ONCE per instruction
// and selects a fully specialised, branch-free loop over the V pixels of the thread.
template <int W, typename F>
__device__ __forceinline__ void with_class(int cls, F&& f) {
  if (cls == GM_C_I32) f(int32_t(0));
  else if (cls == GM_C_F32) f(float(0));
  else if constexpr (W == 8) {
    if (cls == GM_C_I64) f(int64_t(0)); else f(double(0));
  }
}

// acc[i] = f(acc[i], i) for the V pixels of the thread
template <int V, typename S, typename F> __device__ __forceinline__ void each(S (&acc)[V], F&& f) {
#pragma unroll
  for (int i = 0; i < V; ++i) acc[i] = f(acc[i], i);
}

// operand b of pixel i: a slot in shared memory (register file or a staged input that already is a
// slot of the right class)
template <typename S> __device__ __forceinline__ uint64_t b_at(const S* __restrict__ bp, int i) {
  return (uint64_t)bp[i * THREADS + threadIdx.x];
}

// x[i] (class `from`) -> class `to`; the sentinel k becomes NaN when asked (float targets)
template <int W, int V, typename S>
__device__ __forceinline__ void convert_all(S (&x)[V], int from, int to, bool nanify, uint64_t k) {
  if (from == to) return;
  with_class<W>(from, [&](auto ft) {
    typedef decltype(ft) From;
    with_class<W>(to, [&](auto tt) {
      typedef decltype(tt) To;
      if constexpr (!std::is_same<From, To>::value) each(x, [&](S v, int) { return cvt<From, To>(v, nanify, k); });
    });
  });
}

// staged input (storage type ST) -> slots of the input's natural class
template <typename ST, int V, typename S>
__device__ __forceinline__ void read_loop(const unsigned char* base, S (&x)[V]) {
  const ST* p = reinterpret_cast<const ST*>(base) + threadIdx.x;
#pragma unroll
  for (int i = 0; i < V; ++i) {
    const ST v = p[i * THREADS];
    if constexpr (std::is_same<ST, float>::value) x[i] = (S)__float_as_uint(v);
    else if constexpr (std::is_same<ST, double>::value) x[i] = (S)__double_as_longlong(v);
    else if constexpr (std::is_signed<ST>::value && sizeof(ST) < 8) x[i] = (S)(uint32_t)(int32_t)v;
    else x[i] = (S)v;
  }
}

template <int W, int V, typename S>
__device__ __forceinline__ void read_input(const unsigned char* base, int dtype, S (&x)[V]) {
  switch (dtype) {
    case GM_BOOL: case GM_U8: read_loop<uint8_t, V, S>(base, x); break;
    case GM_I8: read_loop<int8_t, V, S>(base, x); break;
    case GM_U16: read_loop<uint16_t, V, S>(base, x); break;
    case GM_I16: read_loop<int16_t, V, S>(base, x); break;
    case GM_I32: case GM_F32: case GM_U32: read_loop<uint32_t, V, S>(base, x); break;
    default:
      if constexpr (W == 8) read_loop<uint64_t, V, S>(base, x);
      break;
  }
}

template <typename ST, int V, typename S>
__device__ __forceinline__ void write_loop(unsigned char* base, const S (&x)[V]) {
  ST* p = reinterpret_cast<ST*>(base) + threadIdx.x;
#pragma unroll
  for (int i = 0; i < V; ++i) p[i * THREADS] = (ST)x[i];
}

template <int W, int V, typename S>
__device__ __forceinline__ void write_output(unsigned char* base, int dtype, const S (&x)[V]) {
  switch (dtype) {
    case GM_BOOL: case GM_U8: case GM_I8: write_loop<uint8_t, V, S>(base, x); break;
    case GM_U16: case GM_I16: write_loop<uint16_t, V, S>(base, x); break;
    case GM_I32: case GM_F32: case GM_U32: write_loop<uint32_t, V, S>(base, x); break;
    default:
      if constexpr (W == 8) write_loop<uint64_t, V, S>(base, x);
      break;
  }
}

// ---- typed instructions ------------------------------------------------------------------------
// Binary arithmetic / comparison: acc and b both hold class T; b is the immediate k0 (IMM) or a
// slot in shared memory (`bp`).
template <int OP, typename T, bool IMM, int V, typename S>
__device__ __forceinline__ void binary_loop(const GmInstr& in, S (&acc)[V], const S* __restrict__ bp) {
  const bool fa = in.flags & GM_F_ND_A, fb = (in.flags & GM_F_ND_B) && !IMM;
  const uint64_t k0 = in.k[0], k1 = in.k[1], k2 = in.k[2], k3 = in.k[3];
  each(acc, [&](S a, int i) {
    const uint64_t b = IMM ? k0 : b_at(bp, i);
    if constexpr (OP >= GM_OP_EQ) return compare<OP, T>(a, b, fa, fb, k1, k2, k3);
    else return math<OP, T>(a, b, fa, fb, k1, k2, k3);
  });
}

template <typename T, bool IMM, int V, typename S>
__device__ __forceinline__ void exec_binary(const GmInstr& in, S (&acc)[V], const S* __restrict__ bp) {
  switch (in.op) {
    case GM_OP_ADD:  binary_loop<GM_OP_ADD, T, IMM>(in, acc, bp); break;
    case GM_OP_SUB:  binary_loop<GM_OP_SUB, T, IMM>(in, acc, bp); break;
    case GM_OP_RSUB: binary_loop<GM_OP_RSUB, T, IMM>(in, acc, bp); break;
    case GM_OP_MUL:  binary_loop<GM_OP_MUL, T, IMM>(in, acc, bp); break;
    case GM_OP_DIV:  binary_loop<GM_OP_DIV, T, IMM>(in, acc, bp); break;
    case GM_OP_RDIV: binary_loop<GM_OP_RDIV, T, IMM>(in, acc, bp); break;
    case GM_OP_POW:  binary_loop<GM_OP_POW, T, IMM>(in, acc, bp); break;
    case GM_OP_RPOW: binary_loop<GM_OP_RPOW, T, IMM>(in, acc, bp); break;
    case GM_OP_EQ: binary_loop<GM_OP_EQ, T, IMM>(in, acc, bp); break;
    case GM_OP_NE: binary_loop<GM_OP_NE, T, IMM>(in, acc, bp); break;
    case GM_OP_GT: binary_loop<GM_OP_GT, T, IMM>(in, acc, bp); break;
    case GM_OP_GE: binary_loop<GM_OP_GE, T, IMM>(in, acc, bp); break;
    case GM_OP_LT: binary_loop<GM_OP_LT, T, IMM>(in, acc, bp); break;
    case GM_OP_LE: binary_loop<GM_OP_LE, T, IMM>(in, acc, bp); break;
    default: break;
  }
}

// Unary instructions that look at acc (class A) in the compare class T.
template <typename T, typename A, int V, typename S>
__device__ __forceinline__ void exec_unary(const GmInstr& in, S (&acc)[V], const DevTable* __restrict__ tabs) {
  const bool fa = in.flags & GM_F_ND_A;
  const uint64_t k0 = in.k[0], k1 = in.k[1], k2 = in.k[2], k3 = in.k[3], k4 = in.k[4], k5 = in.k[5];
  switch (in.op) {
    case GM_OP_EXP: case GM_OP_LOG: case GM_OP_LOG10:
      if constexpr (IsFloat<T>::value && std::is_same<T, A>::value) {
        if (in.op == GM_OP_EXP) each(acc, [&](S a, int) { return transcend<GM_OP_EXP, T>(a, fa, k1, k3); });
        else if (in.op == GM_OP_LOG) each(acc, [&](S a, int) { return transcend<GM_OP_LOG, T>(a, fa, k1, k3); });
        else each(acc, [&](S a, int) { return transcend<GM_OP_LOG10, T>(a, fa, k1, k3); });
      }
      break;
    case GM_OP_MASK: {
      const bool has = in.flags & GM_F_ND_T, cl = in.flags & GM_F_CLOSE, fin = in.flags & GM_F_ND_FINITE;
      each(acc, [&](S a, int) { return mask<T, A>(a, has, cl, fin, k0, k1, k3, k4); });
      break;
    }
    case GM_OP_MASKBELOW:
      each(acc, [&](S a, int) { return mask_below<T, A>(a, k0, k5); });
      break;
    case GM_OP_STEP:
      each(acc, [&](S a, int) { return step<T, A>(a, fa, k0, k1, k2, k3, k4); });
      break;
    case GM_OP_CLASSIFY: {
      const DevTable& t = tabs[in.aux];
      const bool right = in.flags & GM_F_RIGHT;
      each(acc, [&](S a, int) { return classify<T, A>(a, fa, right, t.keys, t.n, k1, k3); });
      break;
    }
    default: break;
  }
}

template <typename A, bool DENSE, bool ND_ONLY, int V, typename S>
__device__ __forceinline__ void exec_reclass(const GmInstr& in, S (&acc)[V], const DevTable& t) {
  const bool select = in.flags & GM_F_SELECT, fa = in.flags & GM_F_ND_A, out_f64 = in.cls_out == GM_C_F64;
  const uint64_t k1 = in.k[1], k3 = in.k[3];
  each(acc, [&](S a, int) {
    return reclass<A, DENSE, ND_ONLY>(a, select, fa, out_f64, t.keys, t.vals, t.hit, t.n, t.base, k1, k3);
  });
}

template <typename A, int V, typename S>
__device__ __forceinline__ void dispatch_reclass(const GmInstr& in, S (&acc)[V], const DevTable& t) {
  const bool nd_only = in.flags & GM_F_ND_T;
  if (t.kind == GM_TABLE_DENSE) {
    if (nd_only) exec_reclass<A, true, true>(in, acc, t);
    else exec_reclass<A, true, false>(in, acc, t);
  } else {
    if (nd_only) exec_reclass<A, false, true>(in, acc, t);
    else exec_reclass<A, false, false>(in, acc, t);
  }
}

// ---- the kernel ---------------------------------------------------------------------------------
template <int W, int V>
__global__ void __launch_bounds__(THREADS, 3)
eval_kernel(const __grid_constant__ EvalParams p) {
  typedef typename SlotOf<W>::type S;
  constexpr int TILE = THREADS * V;
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ DevTable tabs[GM_MAX_TABLES];
  const int tid = threadIdx.x;
  auto in_stage_ptr = [&](int s) { return smem + (size_t)s * p.in_stage_bytes; };
  auto out_stage_ptr = [&](int s) {
    return smem + (size_t)NSTAGE * p.in_stage_bytes + (size_t)s * p.out_stage_bytes;
  };
  S* regs = reinterpret_cast<S*>(smem + p.regs_off);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + p.bar_off);

  // lookup tables -> shared memory; barriers
  if (tid == 0) {
    size_t off = p.tables_off;
    for (int t = 0; t < p.n_tables; ++t) {
      DevTable d = p.tab[t];
      if (p.tables_in_smem) {
        if (d.keys) { d.keys = reinterpret_cast<const int64_t*>(smem + off); off += (size_t)d.n * 8; }
        if (d.vals) { d.vals = reinterpret_cast<const uint64_t*>(smem + off); off += (size_t)d.n * 8; }
        if (d.hit)  { d.hit = smem + off; off += ((size_t)d.n + 15) / 16 * 16; }
      }
      tabs[t] = d;
    }
    for (int s = 0; s < NSTAGE; ++s) mbar_init(&bars[s], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (p.tables_in_smem) {
    for (int t = 0; t < p.n_tables; ++t) {
      const DevTable g = p.tab[t];
      const DevTable s = tabs[t];
      if (g.keys) for (int i = tid; i < g.n; i += THREADS) const_cast<int64_t*>(s.keys)[i] = g.keys[i];
      if (g.vals) for (int i = tid; i < g.n; i += THREADS) const_cast<uint64_t*>(s.vals)[i] = g.vals[i];
      if (g.hit)  for (int i = tid; i < g.n; i += THREADS) const_cast<uint8_t*>(s.hit)[i] = g.hit[i];
    }
    __syncthreads();
  }

  const int64_t n = p.n;
  const int64_t n_tiles = (n + TILE - 1) / TILE;
  const int64_t n_full = n / TILE;  // tiles that can travel as TMA bulk copies

  auto issue_loads = [&](int64_t tile, int stage) {
    // one thread: arm the barrier with the byte count, then one bulk copy per input
    uint32_t total = 0;
    for (int k = 0; k < p.n_inputs; ++k) total += (uint32_t)TILE * dtype_size(p.in_dtype[k]);
    mbar_expect_tx(&bars[stage], total);
    for (int k = 0; k < p.n_inputs; ++k) {
      const uint32_t bytes = (uint32_t)TILE * dtype_size(p.in_dtype[k]);
      bulk_load(in_stage_ptr(stage) + p.in_off[k],
                reinterpret_cast<const unsigned char*>(p.in[k]) + (size_t)tile * bytes, bytes, &bars[stage]);
    }
  };

  int64_t tile = blockIdx.x;
  if (tid == 0 && tile < n_full && p.n_inputs > 0) issue_loads(tile, 0);

  for (int it = 0; tile < n_tiles; tile += gridDim.x, ++it) {
    const int stage = it & 1;
    const bool full = tile < n_full;
    const int64_t next = tile + gridDim.x;
    if (tid == 0) {
      bulk_wait_read<1>();  // the output stage used two tiles ago has been drained
      if (next < n_full && p.n_inputs > 0) issue_loads(next, stage ^ 1);
    }
    const int64_t base = tile * TILE;
    if (full) {
      if (p.n_inputs > 0) mbar_wait(&bars[stage], (uint32_t)((it >> 1) & 1));
    } else {
      // ragged last tile: plain guarded copies into the stage
      for (int k = 0; k < p.n_inputs; ++k) {
        const int sz = dtype_size(p.in_dtype[k]);
        const unsigned char* g = reinterpret_cast<const unsigned char*>(p.in[k]) + (size_t)base * sz;
        unsigned char* d = in_stage_ptr(stage) + p.in_off[k];
        const int64_t valid = (n - base) * sz;
        for (int64_t i = tid; i < (int64_t)TILE * sz; i += THREADS) d[i] = i < valid ? g[i] : 0;
      }
      __syncthreads();
    }
    __syncthreads();  // also orders tid 0's wait_group before everyone's output writes

    S acc[V];
#pragma unroll
    for (int i = 0; i < V; ++i) acc[i] = 0;

    for (int pc = 0; pc < p.n_instr; ++pc) {
      const GmInstr& in = p.instr[pc];
      const int op = in.op;
      // operand b: pointer into shared memory (register file or a staged input that
      // already is a slot of the right class)
      const S* bp = nullptr;
      if (in.src_kind == GM_SRC_REG) bp = regs + (size_t)in.src * TILE;
      else if (in.src_kind == GM_SRC_INPUT) bp = reinterpret_cast<const S*>(in_stage_ptr(stage) + p.in_off[in.src]);

      switch (op) {
        case GM_OP_LOAD:
        case GM_OP_MATB: {
          // acc (LOAD) or reg[aux] (MATB) = convert(source); sentinel -> NaN when asked
          const bool nanify = (in.flags & GM_F_NAN) && (in.flags & GM_F_ND_B);
          if (op == GM_OP_LOAD) {
            if (in.src_kind == GM_SRC_INPUT)
              read_input<W, V, S>(in_stage_ptr(stage) + p.in_off[in.src], p.in_dtype[in.src], acc);
            else if (in.src_kind == GM_SRC_REG) {
#pragma unroll
              for (int i = 0; i < V; ++i) acc[i] = bp[i * THREADS + tid];
            } else {
#pragma unroll
              for (int i = 0; i < V; ++i) acc[i] = (S)in.k[0];
            }
            convert_all<W, V, S>(acc, in.cls_b, in.cls_out, nanify, in.k[2]);
          } else {
            S tmp[V];
            if (in.src_kind == GM_SRC_INPUT)
              read_input<W, V, S>(in_stage_ptr(stage) + p.in_off[in.src], p.in_dtype[in.src], tmp);
            else if (in.src_kind == GM_SRC_REG) {
#pragma unroll
              for (int i = 0; i < V; ++i) tmp[i] = bp[i * THREADS + tid];
            } else {
#pragma unroll
              for (int i = 0; i < V; ++i) tmp[i] = (S)in.k[0];
            }
            convert_all<W, V, S>(tmp, in.cls_b, in.cls_out, nanify, in.k[2]);
            S* rp = regs + (size_t)in.aux * TILE + tid;
#pragma unroll
            for (int i = 0; i < V; ++i) rp[i * THREADS] = tmp[i];
          }
          break;
        }
        case GM_OP_ST: {
          S* rp = regs + (size_t)in.aux * TILE + tid;
#pragma unroll
          for (int i = 0; i < V; ++i) rp[i * THREADS] = acc[i];
          break;
        }
        case GM_OP_OUT:
          write_output<W, V, S>(out_stage_ptr(stage) + p.out_off[in.aux], p.out_dtype[in.aux], acc);
          break;
        case GM_OP_CVT:
          convert_all<W, V, S>(acc, in.cls_a, in.cls_out, (in.flags & GM_F_NAN) && (in.flags & GM_F_ND_A),
                               in.k[1]);
          break;
        case GM_OP_ISDATA:
        case GM_OP_ISNODATA: {
          const bool fa = in.flags & GM_F_ND_A;
          const bool want_nodata = op == GM_OP_ISNODATA;
          const uint64_t k1 = in.k[1];
          with_class<W>(in.cls_a, [&](auto tag) {
            typedef decltype(tag) A;
            each(acc, [&](S a, int) { return is_data<A>(a, fa, want_nodata, k1); });
          });
          break;
        }
        case GM_OP_CLIP: {
          const uint64_t k1 = in.k[1], k2 = in.k[2];
          if (in.flags & GM_F_B_BOOL) {
            each(acc, [&](S a, int i) { return clip<int32_t, 1>(a, b_at(bp, i), k1, k2); });
          } else if (in.flags & GM_F_ND_B) {
            with_class<W>(in.cls_b, [&](auto tag) {
              typedef decltype(tag) B;
              each(acc, [&](S a, int i) { return clip<B, 2>(a, b_at(bp, i), k1, k2); });
            });
          }
          break;
        }
        case GM_OP_AND: case GM_OP_OR: case GM_OP_XOR: case GM_OP_NOT: {
          const bool imm = in.src_kind == GM_SRC_IMM;
          const uint64_t yimm = in.k[0] != 0;
          auto y = [&](int i) { return imm ? yimm : b_at(bp, i); };
          if (op == GM_OP_AND) each(acc, [&](S a, int i) { return logic<GM_OP_AND>(a, y(i)); });
          else if (op == GM_OP_OR) each(acc, [&](S a, int i) { return logic<GM_OP_OR>(a, y(i)); });
          else if (op == GM_OP_XOR) each(acc, [&](S a, int i) { return logic<GM_OP_XOR>(a, y(i)); });
          else each(acc, [&](S a, int) { return logic<GM_OP_NOT>(a, 0); });
          break;
        }
        case GM_OP_RECLASS:
          if (in.cls_a == GM_C_I32) dispatch_reclass<int32_t>(in, acc, tabs[in.aux]);
          else if constexpr (W == 8) dispatch_reclass<int64_t>(in, acc, tabs[in.aux]);
          break;
        case GM_OP_OVERLAY: {
          const bool has = in.flags & GM_F_ND_T, cl = in.flags & GM_F_CLOSE, fin = in.flags & GM_F_ND_FINITE;
          const int kind = (int)in.aux;
          const uint64_t k2 = in.k[2], k4 = in.k[4];
          with_class<W>(in.cls, [&](auto tag) {
            typedef decltype(tag) T;
            with_class<W>(in.cls_out, [&](auto otag) {
              typedef decltype(otag) To;
              each(acc, [&](S a, int i) {
                return overlay<T, To>(a, b_at(bp, i), has, cl, fin, kind, k2, k4);
              });
            });
          });
          break;
        }
        case GM_OP_EXP: case GM_OP_LOG: case GM_OP_LOG10:
        case GM_OP_MASK: case GM_OP_MASKBELOW: case GM_OP_STEP: case GM_OP_CLASSIFY:
          with_class<W>(in.cls, [&](auto tag) {
            typedef decltype(tag) T;
            with_class<W>(in.cls_a, [&](auto atag) {
              typedef decltype(atag) A;
              exec_unary<T, A>(in, acc, tabs);
            });
          });
          break;
        default: {  // binary arithmetic / comparison
          const bool imm = in.src_kind == GM_SRC_IMM;
          with_class<W>(in.cls, [&](auto tag) {
            typedef decltype(tag) T;
            if (imm) exec_binary<T, true>(in, acc, bp);
            else exec_binary<T, false>(in, acc, bp);
          });
          break;
        }
      }
    }

    // results leave through the async proxy: make the generic-proxy writes visible first
    fence_async_smem();
    __syncthreads();
    if (full) {
      if (tid == 0) {
        for (int k = 0; k < p.n_outputs; ++k) {
          const uint32_t bytes = (uint32_t)TILE * dtype_size(p.out_dtype[k]);
          bulk_store(reinterpret_cast<unsigned char*>(p.out[k]) + (size_t)tile * bytes,
                     out_stage_ptr(stage) + p.out_off[k], bytes);
        }
        bulk_commit();
      }
    } else {
      for (int k = 0; k < p.n_outputs; ++k) {
        const int sz = dtype_size(p.out_dtype[k]);
        unsigned char* g = reinterpret_cast<unsigned char*>(p.out[k]) + (size_t)base * sz;
        const unsigned char* s = out_stage_ptr(stage) + p.out_off[k];
        const int64_t valid = (n - base) * sz;
        for (int64_t i = tid; i < valid; i += THREADS) g[i] = s[i];
      }
    }
  }
  if (tid == 0) bulk_wait_read<0>();  // shared memory must outlive the last bulk stores
}

static bool wide(int cls) { return cls == GM_C_I64 || cls == GM_C_F64; }
static bool is_binary(int op) {
  return (op >= GM_OP_ADD && op <= GM_OP_RPOW) || (op >= GM_OP_EQ && op <= GM_OP_LE);
}
static int validate(const GmProgram* prog, const GmArray* inputs) {
  if (!prog) return fail("gm_eval_program: null program");
  if (prog->n_instr < 1 || prog->n_instr > GM_MAX_INSTR) return fail("gm_eval_program: bad instruction count");
  if (prog->n_inputs < 0 || prog->n_inputs > GM_MAX_INPUTS) return fail("gm_eval_program: too many inputs");
  if (prog->n_outputs < 1 || prog->n_outputs > GM_MAX_OUTPUTS) return fail("gm_eval_program: bad output count");
  if (prog->n_tables < 0 || prog->n_tables > GM_MAX_TABLES) return fail("gm_eval_program: too many tables");
  if (prog->word != 4 && prog->word != 8) return fail("gm_eval_program: word must be 4 or 8");
  for (int i = 0; i < prog->n_instr; ++i) {
    const GmInstr& in = prog->instr[i];
    if (in.op >= GM_OP_COUNT_) return fail("gm_eval_program: unknown opcode");
    if (in.src_kind == GM_SRC_REG && in.src >= GM_NREG) return fail("gm_eval_program: bad register");
    if (in.src_kind == GM_SRC_INPUT && in.src >= prog->n_inputs) return fail("gm_eval_program: bad input index");
    if ((in.op == GM_OP_ST || in.op == GM_OP_MATB) && in.aux >= GM_NREG) return fail("gm_eval_program: bad register");
    if (in.op == GM_OP_OUT && (int)in.aux >= prog->n_outputs) return fail("gm_eval_program: bad output index");
    if ((in.op == GM_OP_CLASSIFY || in.op == GM_OP_RECLASS) && (int)in.aux >= prog->n_tables)
      return fail("gm_eval_program: bad table index");
    if (in.cls > GM_C_F64 || in.cls_a > GM_C_F64 || in.cls_b > GM_C_F64 || in.cls_out > GM_C_F64)
      return fail("gm_eval_program: bad class");
    if (prog->word == 4) {
      if (wide(in.cls_a) || wide(in.cls_out) || wide(in.cls) ||
          (in.src_kind != GM_SRC_NONE && wide(in.cls_b)))
        return fail("gm_eval_program: 64-bit class in a 32-bit program");
    }
    const bool direct_b = in.src_kind == GM_SRC_INPUT && in.op != GM_OP_LOAD && in.op != GM_OP_MATB;
    if (direct_b) {
      // a staged input is only a valid b operand when its storage already is a slot
      const int dt = inputs[in.src].dtype;
      if (dtype_size(dt) != prog->word || natural_class(dt) != in.cls_b)
        return fail("gm_eval_program: input used as operand without conversion");
    }
    if (is_binary(in.op) && (in.cls_a != in.cls || (in.src_kind != GM_SRC_NONE && in.cls_b != in.cls)))
      return fail("gm_eval_program: arithmetic operands must already hold the compute class");
    if (in.op == GM_OP_OVERLAY && in.aux != GM_RED_REPLACE && in.aux != GM_RED_COUNT &&
        in.cls_out != GM_C_F32 && in.cls_out != GM_C_F64)
      return fail("gm_eval_program: overlay max / min / sum / product need a float accumulator");
  }
  return 0;
}

}  // namespace gm

using namespace gm;

template <int W, int V>
static int launch_eval(EvalParams& p, const GmProgram* prog, size_t table_bytes, cudaStream_t s) {
  const int tile = THREADS * V;
  // dynamic shared memory layout: [input stages][output stages][registers][tables][barriers]
  size_t off = 0;
  int in_stage = 0, out_stage = 0;
  for (int k = 0; k < prog->n_inputs; ++k) {
    p.in_off[k] = in_stage;
    in_stage += (tile * dtype_size(p.in_dtype[k]) + 127) / 128 * 128;
  }
  for (int k = 0; k < prog->n_outputs; ++k) {
    p.out_off[k] = out_stage;
    out_stage += (tile * dtype_size(p.out_dtype[k]) + 127) / 128 * 128;
  }
  p.in_stage_bytes = in_stage;
  p.out_stage_bytes = out_stage;
  off = (size_t)NSTAGE * in_stage + (size_t)NSTAGE * out_stage;
  p.regs_off = (int)off;
  off += (size_t)p.n_regs * tile * W;
  p.tables_off = (int)off;
  const size_t budget = 200 * 1024;
  p.tables_in_smem = (table_bytes > 0 && off + table_bytes + 64 <= budget) ? 1 : 0;
  if (p.tables_in_smem) off += (table_bytes + 15) / 16 * 16;
  p.bar_off = (int)off;
  off += 64;
  if (off > 227 * 1024) return -1;  // caller retries with a smaller tile
  auto kernel = eval_kernel<W, V>;
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)off);
  int per_sm = 1;
  if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, THREADS, off);
  if (e != cudaSuccess) return fail(std::string("eval launch setup: ") + cudaGetErrorString(e));
  if (per_sm < 1) per_sm = 1;
  const int64_t n_tiles = (p.n + tile - 1) / tile;
  int64_t grid = (int64_t)sm_count() * per_sm;
  if (grid > n_tiles) grid = n_tiles;
  kernel<<<(unsigned)grid, THREADS, off, s>>>(p);
  e = cudaGetLastError();
  if (e != cudaSuccess) return fail(std::string("eval kernel launch: ") + cudaGetErrorString(e));
  count_launch();
  return 0;
}

// Back-end selection: GM_EVAL_AUTO specialises (NVRTC) from kJitMinPixels pixels on and
// interprets below that, where a launch is latency-bound and a compile would not pay.
static std::atomic<int> g_eval_mode{-1};
static const int64_t kJitMinPixels = 1 << 18;

static int eval_mode() {
  int m = g_eval_mode.load(std::memory_order_relaxed);
  if (m >= 0) return m;
  const char* env = getenv("GM_EVAL");
  m = GM_EVAL_AUTO;
  if (env && !strcmp(env, "interp")) m = GM_EVAL_INTERPRET;
  else if (env && !strcmp(env, "jit")) m = GM_EVAL_SPECIALISE;
  g_eval_mode.store(m);
  return m;
}

extern "C" int gm_set_eval_mode(int mode) {
  if (mode < GM_EVAL_AUTO || mode > GM_EVAL_SPECIALISE) return fail("gm_set_eval_mode: bad mode");
  g_eval_mode.store(mode);
  return 0;
}
extern "C" int gm_get_eval_mode(void) { return eval_mode(); }

extern "C" int gm_eval_program(const GmProgram* prog, const GmArray* inputs, GmArray* outputs,
                               int64_t n_pixels, void* stream) {
  if (ensure_init()) return 1;
  if (validate(prog, inputs)) return 1;
  if (n_pixels < 0) return fail("gm_eval_program: negative pixel count");
  cudaStream_t s = resolve_stream(stream);
  const int mode = eval_mode();
  const bool specialise = mode == GM_EVAL_SPECIALISE || (mode == GM_EVAL_AUTO && n_pixels >= kJitMinPixels);
  const bool need_tables = !(specialise && jit_tables_baked(prog));

  EvalParams p;
  memset(&p, 0, sizeof(p));
  p.n_instr = prog->n_instr;
  p.n_inputs = prog->n_inputs;
  p.n_outputs = prog->n_outputs;
  p.n_tables = prog->n_tables;
  p.n = n_pixels;
  memcpy(p.instr, prog->instr, sizeof(GmInstr) * prog->n_instr);
  int n_regs = 0;
  for (int i = 0; i < prog->n_instr; ++i) {
    const GmInstr& in = prog->instr[i];
    if (in.src_kind == GM_SRC_REG && in.src + 1 > n_regs) n_regs = in.src + 1;
    if ((in.op == GM_OP_ST || in.op == GM_OP_MATB) && (int)in.aux + 1 > n_regs) n_regs = in.aux + 1;
  }
  p.n_regs = n_regs;

  Staged sin[GM_MAX_INPUTS], sout[GM_MAX_OUTPUTS];
  std::vector<void*> scratch;
  int rc = 0;
  auto cleanup = [&]() {
    for (int i = 0; i < prog->n_inputs; ++i) sin[i].release();
    for (int i = 0; i < prog->n_outputs; ++i) sout[i].release();
    for (void* d : scratch) cudaFreeAsync(d, s);
  };

  for (int i = 0; i < prog->n_inputs && !rc; ++i) {
    if (array_count(inputs[i]) != n_pixels) { rc = fail("gm_eval_program: input size mismatch"); break; }
    if (!dtype_size(inputs[i].dtype)) { rc = fail("gm_eval_program: bad input dtype"); break; }
    if (((uintptr_t)inputs[i].data & 15u) && inputs[i].space == GM_DEVICE) {
      rc = fail("gm_eval_program: device input not 16-byte aligned"); break;
    }
    rc = sin[i].open_input(inputs[i], s);
    p.in[i] = sin[i].dev;
    p.in_dtype[i] = inputs[i].dtype;
  }
  for (int i = 0; i < prog->n_outputs && !rc; ++i) {
    if (array_count(outputs[i]) != n_pixels) { rc = fail("gm_eval_program: output size mismatch"); break; }
    if (!dtype_size(outputs[i].dtype)) { rc = fail("gm_eval_program: bad output dtype"); break; }
    if (((uintptr_t)outputs[i].data & 15u) && outputs[i].space == GM_DEVICE) {
      rc = fail("gm_eval_program: device output not 16-byte aligned"); break;
    }
    rc = sout[i].open_output(outputs[i], s);
    p.out[i] = sout[i].dev;
    p.out_dtype[i] = outputs[i].dtype;
  }
  size_t table_bytes = 0;
  for (int t = 0; t < prog->n_tables && !rc && need_tables; ++t) {
    const GmTable& g = prog->tables[t];
    DevTable& d = p.tab[t];
    d.n = g.n; d.kind = g.kind; d.base = g.base;
    void* dev = nullptr;
    if (g.keys) {
      rc = upload(&dev, g.keys, (int64_t)g.n * 8, s); if (rc) break;
      scratch.push_back(dev); d.keys = (const int64_t*)dev; table_bytes += (size_t)g.n * 8;
    }
    if (g.vals) {
      rc = upload(&dev, g.vals, (int64_t)g.n * 8, s); if (rc) break;
      scratch.push_back(dev); d.vals = (const uint64_t*)dev; table_bytes += (size_t)g.n * 8;
    }
    if (g.hit) {
      rc = upload(&dev, g.hit, (int64_t)g.n, s); if (rc) break;
      scratch.push_back(dev); d.hit = (const uint8_t*)dev; table_bytes += ((size_t)g.n + 15) / 16 * 16;
    }
  }
  if (rc) { cleanup(); return 1; }

  if (n_pixels > 0 && specialise) {
    const void* tk[GM_MAX_TABLES] = {}; const void* tv[GM_MAX_TABLES] = {}; const void* th[GM_MAX_TABLES] = {};
    for (int t = 0; t < prog->n_tables; ++t) { tk[t] = p.tab[t].keys; tv[t] = p.tab[t].vals; th[t] = p.tab[t].hit; }
    if (jit_launch(prog, p.in, p.in_dtype, p.out, p.out_dtype, tk, tv, th, n_pixels, s)) { cleanup(); return 1; }
  } else if (n_pixels > 0) {
    // widest tile that fits shared memory: more pixels per thread = less decode per pixel
    if (prog->word == 4) {
      rc = launch_eval<4, 16>(p, prog, table_bytes, s);
      if (rc == -1) rc = launch_eval<4, 8>(p, prog, table_bytes, s);
      if (rc == -1) rc = launch_eval<4, 4>(p, prog, table_bytes, s);
    } else {
      rc = launch_eval<8, 8>(p, prog, table_bytes, s);
      if (rc == -1) rc = launch_eval<8, 4>(p, prog, table_bytes, s);
      if (rc == -1) rc = launch_eval<8, 2>(p, prog, table_bytes, s);
    }
    if (rc == -1) rc = fail("gm_eval_program: program does not fit shared memory");
    if (rc) { cleanup(); return 1; }
  }
  bool staged_out = false;
  for (int i = 0; i < prog->n_outputs; ++i) {
    if (sout[i].finish_output()) { cleanup(); return 1; }
    staged_out |= sout[i].owned;
  }
  cleanup();
  if (staged_out) GM_CUDA(cudaStreamSynchronize(s));
  return 0;
}
