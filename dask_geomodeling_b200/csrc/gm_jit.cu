// Specialising back end of the fused evaluator.
//
// gm_eval_program hands a validated GmProgram to jit_launch().  The program is
// translated ONCE into a straight-line CUDA kernel that calls, per instruction, the
// device function of gm_eval_ops.cuh that the interpreter runs too (classes become
// template arguments, flags and constants literals, small lookup tables __device__
// arrays; gm_jit_prelude.cuh adds the memory access of generated code), compiled
// for sm_100a with NVRTC (-fmad=false, IEEE division) and cached by a hash of the
// program.  The generated kernel keeps every pixel in registers:
//
//   * a thread owns groups of V = 16 / (widest element) consecutive pixels, so the
//     widest raster moves as 128-bit accesses and every warp access of every raster
//     is one fully used contiguous segment (no shared-memory staging needed);
//   * U groups per thread make a chunk (U*V = 16 pixels, 96 B per thread on cfg2), loaded before
//     it is evaluated, streaming cache hints on both sides; where two chunks of input fit the
//     register budget (kTwoSetWords), a block walks K consecutive chunks in two register sets and
//     issues the loads of chunk c + 1 before it evaluates chunk c;
//   * a small dense Reclassify table is two 32-bit literal words, other baked lookup tables
//     live in shared memory (see JitLayout).
//
// The interpreter in gm_eval.cu stays the zero-latency path for small rasters; the
// parity tests check the two against each other and against the oracle.
#include "gm_common.cuh"
#include "gm_jit.h"
#include <dlfcn.h>
#include <deque>
#include <memory>
#include <mutex>
#include <unordered_map>
#include <sys/stat.h>
#include <unistd.h>

namespace gm {

static const char* kPrelude =
#include "build/gm_jit_prelude.inc"
    ;

// ---- NVRTC through dlopen (the library must load on machines without it) --------------
typedef struct _nvrtcProgram* nvrtcProgram;
struct Nvrtc {
  void* handle = nullptr;
  int (*CreateProgram)(nvrtcProgram*, const char*, const char*, int, const char* const*, const char* const*);
  int (*CompileProgram)(nvrtcProgram, int, const char* const*);
  int (*GetCUBINSize)(nvrtcProgram, size_t*);
  int (*GetCUBIN)(nvrtcProgram, char*);
  int (*GetProgramLogSize)(nvrtcProgram, size_t*);
  int (*GetProgramLog)(nvrtcProgram, char*);
  int (*DestroyProgram)(nvrtcProgram*);
  const char* (*GetErrorString)(int);
};

static Nvrtc g_nvrtc;
static std::mutex g_jit_mutex;

static int load_nvrtc() {
  if (g_nvrtc.handle) return 0;
  const char* env = getenv("GM_NVRTC_PATH");
  const char* candidates[] = {env, "libnvrtc.so.12", "/usr/local/cuda/lib64/libnvrtc.so.12",
                              "libnvrtc.so"};
  void* h = nullptr;
  for (const char* c : candidates) {
    if (!c || !*c) continue;
    h = dlopen(c, RTLD_NOW | RTLD_LOCAL);
    if (h) break;
  }
  if (!h) return fail("NVRTC (libnvrtc.so.12) not found: set GM_NVRTC_PATH or GM_EVAL=interp");
#define GM_SYM(name)                                                                   \
  *(void**)(&g_nvrtc.name) = dlsym(h, "nvrtc" #name);                                  \
  if (!g_nvrtc.name) return fail("libnvrtc lacks nvrtc" #name)
  GM_SYM(CreateProgram); GM_SYM(CompileProgram); GM_SYM(GetCUBINSize); GM_SYM(GetCUBIN);
  GM_SYM(GetProgramLogSize); GM_SYM(GetProgramLog); GM_SYM(DestroyProgram); GM_SYM(GetErrorString);
#undef GM_SYM
  g_nvrtc.handle = h;
  return 0;
}

// ---- source generation ----------------------------------------------------------------------
static const char* class_type(int cls) {
  switch (cls) {
    case GM_C_I32: return "int32_t";
    case GM_C_F32: return "float";
    case GM_C_I64: return "int64_t";
    default: return "double";
  }
}
static bool class_is_float(int cls) { return cls == GM_C_F32 || cls == GM_C_F64; }
static bool class_fits(int cls, int word) { return word == 8 || cls == GM_C_I32 || cls == GM_C_F32; }

static const char* storage_type(int dt) {
  switch (dt) {
    case GM_BOOL: case GM_U8: return "uint8_t";
    case GM_I8: return "int8_t";
    case GM_U16: return "uint16_t";
    case GM_I16: return "int16_t";
    case GM_I64: case GM_F64: return "uint64_t";
    default: return "uint32_t";
  }
}

static std::string hex(uint64_t v) {
  char buf[32];
  snprintf(buf, sizeof(buf), "0x%llxULL", (unsigned long long)v);
  return buf;
}
static std::string num(long long v) { return std::to_string(v); }
static const char* tf(bool b) { return b ? "true" : "false"; }
static std::string lit(int v) { return "Lit<" + num(v) + ">()"; }   // Lit of the prelude

// Where each lookup table lives.  A baked table's contents are part of the module (and of the
// cache key): a dense ND_ONLY Reclassify table of at most 64 entries as two 32-bit literal words
// (`bits`, reclass_bits), any other baked table in shared memory (`in_smem`).  A table that is not
// baked is read from global memory through the pointers of the parameter block.
struct JitLayout {
  int V, U;        // pixels per group, groups per thread and chunk
  bool two_sets;   // the hot loop prefetches the next chunk into a second register set (see generate)
  bool baked[GM_MAX_TABLES];
  bool in_smem[GM_MAX_TABLES];
  bool bits[GM_MAX_TABLES];
};

// The two-set hot loop holds two chunks of input in registers: 2 * U * (32-bit words of one group of
// every input).  It is used while that stays within kTwoSetWords and the program has no tables in
// shared memory; cfg2 (int16 + float32: 48 words) then compiles to 64 registers without spills, so
// 4 blocks of 256 stay resident per SM.  Wider programs (cfg1, two float32 inputs: 64 words, 45 -> 77
// registers and 13.8 -> 21.8 instructions per pixel unbaked; four float32 inputs: 80 -> 154
// registers; eight float64 inputs spill) keep the single-set loop.
static const int kTwoSetWords = 48;
// Chunks per block of the two-set loop, at most: on one B200 at 1000 W (cfg2 chain, bench.py --legs
// chain, before the warp barrier of the loads was added) 1, 2, 4 and 8 took 0.336, 0.318, 0.291 and
// 0.297 ms per step, the single-set loop with one chunk per block 0.309 ms.  Fewer on small rasters,
// so that the grid still fills the resident blocks of every SM (see jit_launch).
static const int kMaxChunksPerBlock = 4;
static const int kBakeLimit = 2048;  // table entries baked into the module / held in smem
static const int kBitsLimit = 64;    // entries of a table held as two 32-bit words

// Every use of table t is an ND_ONLY Reclassify of an I32 key, the table is dense, and its key range
// lies inside int32 (the 32-bit range test of reclass_bits).
static bool bits_table(const GmProgram* prog, int t) {
  const GmTable& g = prog->tables[t];
  if (g.kind != GM_TABLE_DENSE || !g.hit || g.n < 1 || g.n > kBitsLimit || g.base < INT32_MIN ||
      g.base + g.n - 1 > INT32_MAX)
    return false;
  for (int pc = 0; pc < prog->n_instr; ++pc) {
    const GmInstr& in = prog->instr[pc];
    if ((in.op == GM_OP_RECLASS || in.op == GM_OP_CLASSIFY) && in.aux == t &&
        (in.op != GM_OP_RECLASS || !(in.flags & GM_F_ND_T) || in.cls_a != GM_C_I32))
      return false;
  }
  return true;
}

static JitLayout plan_layout(const GmProgram* prog, const int* in_dtype, const int* out_dtype) {
  JitLayout L;
  int widest = 1;
  for (int i = 0; i < prog->n_inputs; ++i) widest = std::max(widest, dtype_size(in_dtype[i]));
  for (int i = 0; i < prog->n_outputs; ++i) widest = std::max(widest, dtype_size(out_dtype[i]));
  L.V = 16 / widest;
  L.U = std::max(2, 16 / L.V);
  int total = 0;
  for (int t = 0; t < prog->n_tables; ++t) total += prog->tables[t].n;
  bool smem_tables = false;
  for (int t = 0; t < GM_MAX_TABLES; ++t) {
    L.baked[t] = t < prog->n_tables && total <= kBakeLimit;
    L.bits[t] = L.baked[t] && bits_table(prog, t);
    L.in_smem[t] = L.baked[t] && !L.bits[t];
    smem_tables = smem_tables || L.in_smem[t];
  }
  int words = 0;   // 32-bit words of one group of every input
  for (int i = 0; i < prog->n_inputs; ++i) words += std::max(1, L.V * dtype_size(in_dtype[i]) / 4);
  L.two_sets = !smem_tables && 2 * L.U * words <= kTwoSetWords;
  return L;
}

// Constant k[i] of instruction pc.  The constants (sentinels, thresholds, fill values, scalar
// operands) are NOT baked into the source: they travel in the kernel's parameter block
// (p.k[pc][i], read through the constant bank like a literal would be), so that the compiled
// kernel -- and its cache key -- depend on the structure of the program only.  Changing a
// scalar of a view (a slider on Multiply(x, k), another threshold) reuses the kernel.
//
// A program that keeps being launched with the SAME constants on a large raster is compiled a
// second time with the constants as literals (`bake`): the compiler then folds them (about 8 %
// fewer instructions on the cfg2 chain).  See jit_launch.
static thread_local const GmProgram* t_bake = nullptr;   // non-null while generating a baked kernel
static std::string kref(int pc, int i) {
  if (t_bake) return hex(t_bake->instr[pc].k[i]);
  return "p.k[" + num(pc) + "][" + num(i) + "]";
}

// operand b of instruction `in` as an expression of type uint64_t
static std::string operand_b(const GmInstr& in, int pc) {
  if (in.src_kind == GM_SRC_REG) return "(uint64_t)r" + num(in.src);
  if (in.src_kind == GM_SRC_INPUT) return "(uint64_t)i" + num(in.src);
  if (in.src_kind == GM_SRC_IMM) return kref(pc, 0);
  return "0ULL";
}

static std::string convert_expr(const std::string& x, int from, int to, bool nanify, const std::string& k, int word) {
  if (from == to || !class_fits(from, word) || !class_fits(to, word)) return x;
  return std::string("cvt<") + class_type(from) + ", " + class_type(to) + ">(" + x + ", " + tf(nanify) + ", " +
         k + ")";
}

static std::string table_args(const GmProgram* prog, int t) {
  const GmTable& g = prog->tables[t];
  std::string s;
  s += g.keys ? "t" + num(t) + "k" : std::string("(const int64_t*)0");
  s += ", ";
  s += g.vals ? "t" + num(t) + "v" : std::string("(const uint64_t*)0");
  s += ", ";
  s += g.hit ? "t" + num(t) + "h" : std::string("(const uint8_t*)0");
  return s;
}

// IsData / IsNoData at pc + 1 over the result of a Step at pc, folded into the Step (the IsNd arm
// functor of the prelude).  The Step has no other consumer: the IsData directly follows it and
// replaces the accumulator.  Only in a baked kernel, where the compares of constant arms become
// literals: with the constants in the parameter block the fold costs instructions (cfg2: 21.6 ->
// 25.3 per pixel in tools/jit_sass.py).  Only Step: the same fold over Clip measured more
// instructions, and Clip / Mask / MaskBelow have at most one constant arm to gain.
static const GmInstr* folded_is_data(const GmProgram* prog, int pc) {
  const GmInstr& in = prog->instr[pc];
  if (!t_bake || pc + 1 >= prog->n_instr) return nullptr;
  const GmInstr& nd = prog->instr[pc + 1];
  const bool producer = in.op == GM_OP_STEP;
  const bool is_data = nd.op == GM_OP_ISDATA || nd.op == GM_OP_ISNODATA;
  return producer && is_data && (nd.flags & GM_F_ND_A) && class_fits(nd.cls_a, prog->word) ? &nd : nullptr;
}

// `fold`: the IsData / IsNoData that folded_is_data found for this instruction, or null
static std::string emit_instruction(const GmProgram* prog, const GmInstr& in, const JitLayout& L,
                                    const GmInstr* fold) {
  const int word = prog->word;
  const int pc = (int)(&in - prog->instr);
  const bool fa = in.flags & GM_F_ND_A, fb = in.flags & GM_F_ND_B;
  const std::string b = operand_b(in, pc);
  const std::string arm = fold ? std::string(", IsNd<") + class_type(fold->cls_a) + ">{" + kref(pc + 1, 1) + "}" : "";
  std::string s, call;   // call: a Step, which takes the arm functor
  switch (in.op) {
    case GM_OP_LOAD:
    case GM_OP_MATB: {
      std::string src = in.src_kind == GM_SRC_REG     ? "r" + num(in.src)
                        : in.src_kind == GM_SRC_INPUT ? "i" + num(in.src)
                                                      : "(S)" + kref(pc, 0);
      const bool nanify = (in.flags & GM_F_NAN) && fb;
      const std::string v = convert_expr(src, in.cls_b, in.cls_out, nanify, kref(pc, 2), word);
      s = (in.op == GM_OP_LOAD ? std::string("acc") : "r" + num(in.aux)) + " = " + v + ";";
      break;
    }
    case GM_OP_ST: s = "r" + num(in.aux) + " = acc;"; break;
    case GM_OP_OUT: s = "o" + num(in.aux) + " = acc;"; break;
    case GM_OP_CVT:
      s = "acc = " + convert_expr("acc", in.cls_a, in.cls_out, (in.flags & GM_F_NAN) && fa, kref(pc, 1), word) + ";";
      break;
    case GM_OP_ISDATA:
    case GM_OP_ISNODATA:
      if (class_fits(in.cls_a, word))
        s = std::string("acc = is_data<") + class_type(in.cls_a) + ">(acc, " + tf(fa) + ", " +
            tf(in.op == GM_OP_ISNODATA) + ", " + kref(pc, 1) + ");";
      break;
    case GM_OP_CLIP: {
      int mode = (in.flags & GM_F_B_BOOL) ? 1 : (fb ? 2 : 0);
      if (mode == 2 && !class_fits(in.cls_b, word)) mode = 0;
      s = std::string("acc = clip<") + class_type(mode == 2 ? in.cls_b : GM_C_I32) + ", " + num(mode) +
          ">(acc, " + b + ", " + kref(pc, 1) + ", " + kref(pc, 2) + ");";
      break;
    }
    case GM_OP_AND: case GM_OP_OR: case GM_OP_XOR: case GM_OP_NOT: {
      std::string y = b;
      if (in.op == GM_OP_NOT) y = "0ULL";
      else if (in.src_kind == GM_SRC_IMM) y = "(uint64_t)(" + kref(pc, 0) + " != 0)";
      s = "acc = logic<" + num(in.op) + ">(acc, " + y + ");";
      break;
    }
    case GM_OP_RECLASS: {
      const GmTable& g = prog->tables[in.aux];
      const char* A = in.cls_a == GM_C_I32 ? "int32_t" : "int64_t";
      if (in.cls_a != GM_C_I32 && word != 8) break;
      if (L.bits[in.aux]) {
        const unsigned lut = ((in.flags & GM_F_SELECT) ? 0u : 1u) | 2u;   // as in reclass
        uint32_t w[2] = {0, 0};
        for (int i = 0; i < g.n; ++i) w[i / 32] |= ((lut >> g.hit[i]) & 1u) << (i % 32);
        s = std::string("acc = reclass_bits(acc, ") + tf(in.flags & GM_F_SELECT) + ", " + tf(fa) + ", " +
            num(w[0]) + "u, " + num(w[1]) + "u, " + num(g.n) + "u, " + num(g.base) + ", " + kref(pc, 1) + ");";
        break;
      }
      s = std::string("acc = reclass<") + A + ", " + tf(g.kind == GM_TABLE_DENSE) + ", " +
          tf(in.flags & GM_F_ND_T) + ">(acc, " + tf(in.flags & GM_F_SELECT) + ", " + tf(fa) + ", " +
          tf(in.cls_out == GM_C_F64) + ", " + table_args(prog, in.aux) + ", " + num(g.n) + ", " +
          num(g.base) + "LL, " + kref(pc, 1) + ", " + kref(pc, 3) + ");";
      break;
    }
    case GM_OP_OVERLAY:
      if (class_fits(in.cls, word) && class_fits(in.cls_out, word))
        s = std::string("acc = overlay<") + class_type(in.cls) + ", " + class_type(in.cls_out) + ">(acc, " + b +
            ", " + lit((in.flags & GM_F_ND_T) != 0) + ", " + lit((in.flags & GM_F_CLOSE) != 0) + ", " +
            lit((in.flags & GM_F_ND_FINITE) != 0) + ", " + lit((int)in.aux) + ", " + kref(pc, 2) + ", " + kref(pc, 4) + ");";
      break;
    case GM_OP_EXP: case GM_OP_LOG: case GM_OP_LOG10:
      if (class_fits(in.cls, word) && class_is_float(in.cls) && in.cls == in.cls_a)
        s = "acc = transcend<" + num(in.op) + ", " + class_type(in.cls) + ">(acc, " + tf(fa) + ", " +
            kref(pc, 1) + ", " + kref(pc, 3) + ");";
      break;
    case GM_OP_MASK:
      if (class_fits(in.cls, word) && class_fits(in.cls_a, word))
        s = std::string("acc = mask<") + class_type(in.cls) + ", " + class_type(in.cls_a) + ">(acc, " +
            lit((in.flags & GM_F_ND_T) != 0) + ", " + lit((in.flags & GM_F_CLOSE) != 0) + ", " + lit((in.flags & GM_F_ND_FINITE) != 0) +
            ", " + kref(pc, 0) + ", " + kref(pc, 1) + ", " + kref(pc, 3) + ", " + kref(pc, 4) + ");";
      break;
    case GM_OP_MASKBELOW:
      if (class_fits(in.cls, word) && class_fits(in.cls_a, word))
        s = std::string("acc = mask_below<") + class_type(in.cls) + ", " + class_type(in.cls_a) + ">(acc, " +
            kref(pc, 0) + ", " + kref(pc, 5) + ");";
      break;
    case GM_OP_STEP:
      if (class_fits(in.cls, word) && class_fits(in.cls_a, word))
        call = std::string("step<") + class_type(in.cls) + ", " + class_type(in.cls_a) + ">(acc, " + tf(fa) +
               ", " + kref(pc, 0) + ", " + kref(pc, 1) + ", " + kref(pc, 2) + ", " + kref(pc, 3) + ", " +
               kref(pc, 4) + arm + ")";
      break;
    case GM_OP_CLASSIFY:
      if (class_fits(in.cls, word) && class_fits(in.cls_a, word))
        s = std::string("acc = classify<") + class_type(in.cls) + ", " + class_type(in.cls_a) + ">(acc, " +
            tf(fa) + ", " + tf(in.flags & GM_F_RIGHT) + ", t" + num(in.aux) + "k, " + num(prog->tables[in.aux].n) +
            ", " + kref(pc, 1) + ", " + kref(pc, 3) + ");";
      break;
    default: {  // binary arithmetic / comparison
      if (!class_fits(in.cls, word)) break;
      const bool imm = in.src_kind == GM_SRC_IMM;
      const bool is_cmp = in.op >= GM_OP_EQ && in.op <= GM_OP_LE;
      s = std::string("acc = ") + (is_cmp ? "compare<" : "math<") + num(in.op) + ", " + class_type(in.cls) +
          ">(acc, " + b + ", " + tf(fa) + ", " + tf(fb && !imm) + ", " + kref(pc, 1) + ", " + kref(pc, 2) +
          ", " + kref(pc, 3) + ");";
      break;
    }
  }
  if (!call.empty())
    s = fold ? "acc = data_flag<S>(" + call + ", " + tf(fold->op == GM_OP_ISNODATA) + ");"
             : "acc = " + call + ";";
  return s;
}

static void emit_table_data(std::string& src, const GmProgram* prog, const JitLayout& L) {
  for (int t = 0; t < prog->n_tables; ++t) {
    if (!L.in_smem[t]) continue;
    const GmTable& g = prog->tables[t];
    const std::string id = num(t);
    if (g.keys) {
      src += "__device__ const int64_t g_t" + id + "k[" + num(std::max(g.n, 1)) + "] = {";
      for (int i = 0; i < g.n; ++i) src += "(int64_t)" + hex(((const uint64_t*)g.keys)[i]) + ",";
      src += "};\n";
    }
    if (g.vals) {
      src += "__device__ const uint64_t g_t" + id + "v[" + num(std::max(g.n, 1)) + "] = {";
      for (int i = 0; i < g.n; ++i) src += hex(((const uint64_t*)g.vals)[i]) + ",";
      src += "};\n";
    }
    if (g.hit) {
      src += "__device__ const uint8_t g_t" + id + "h[" + num(std::max(g.n, 1)) + "] = {";
      for (int i = 0; i < g.n; ++i) src += num(g.hit[i]) + ",";
      src += "};\n";
    }
  }
}

static std::string generate(const GmProgram* prog, const int* in_dtype, const int* out_dtype,
                            const JitLayout& L) {
  const int V = L.V, U = L.U;
  std::string src;
  src.reserve(1 << 16);
  src += "#define GM_WORD " + num(prog->word) + "\n";
  src += kPrelude;
  src += "\nstruct Params { const void* in[" + num(GM_MAX_INPUTS) + "]; void* out[" + num(GM_MAX_OUTPUTS) +
         "]; long long n; long long chunks_per_block; const int64_t* tk[" + num(GM_MAX_TABLES) + "]; const uint64_t* tv[" +
         num(GM_MAX_TABLES) + "]; const uint8_t* th[" + num(GM_MAX_TABLES) + "]; unsigned long long k[" +
         num(GM_MAX_INSTR) + "][6]; };\n";
  emit_table_data(src, prog, L);

  // Tables in shared memory are file-scope __shared__ arrays (compile-time addresses); the others
  // travel as global pointers through pixel() and group(); bits tables are literals of reclass_bits.
  std::string tab_params, tab_args;
  for (int t = 0; t < prog->n_tables; ++t) {
    const GmTable& g = prog->tables[t];
    const std::string id = num(t), n = num(std::max(g.n, 1));
    if (L.bits[t]) continue;
    if (L.in_smem[t]) {
      if (g.keys) src += "__shared__ int64_t t" + id + "k[" + n + "];\n";
      if (g.vals) src += "__shared__ uint64_t t" + id + "v[" + n + "];\n";
      if (g.hit) src += "__shared__ uint8_t t" + id + "h[" + n + "];\n";
    } else {
      tab_params += ", const int64_t* __restrict__ t" + id + "k, const uint64_t* __restrict__ t" + id +
                    "v, const uint8_t* __restrict__ t" + id + "h";
      tab_args += ", t" + id + "k, t" + id + "v, t" + id + "h";
    }
  }

  // ---- one pixel ---------------------------------------------------------------------
  src += "GM_DEV void pixel(const Params& p";
  bool first = false;
  for (int i = 0; i < prog->n_inputs; ++i) { src += std::string(first ? "" : ", ") + "S i" + num(i); first = false; }
  for (int i = 0; i < prog->n_outputs; ++i) { src += std::string(first ? "" : ", ") + "S& o" + num(i); first = false; }
  src += tab_params + ") {\n  S acc = 0, r0 = 0, r1 = 0, r2 = 0, r3 = 0;\n";
  for (int pc = 0; pc < prog->n_instr; ++pc) {
    const GmInstr* fold = folded_is_data(prog, pc);
    const std::string line = emit_instruction(prog, prog->instr[pc], L, fold);
    if (!line.empty()) src += "  " + line + "\n";
    if (fold && !line.empty()) ++pc;
  }
  src += "  (void)r0; (void)r1; (void)r2; (void)r3;\n}\n";

  // ---- one group of V pixels held in 32-bit words ---------------------------------------
  auto words = [&](int dt) { return std::max(1, V * dtype_size(dt) / 4); };
  src += "GM_DEV void group(const Params& p";
  first = false;
  for (int i = 0; i < prog->n_inputs; ++i) { src += std::string(first ? "" : ", ") + "const uint32_t* a" + num(i); first = false; }
  for (int i = 0; i < prog->n_outputs; ++i) { src += std::string(first ? "" : ", ") + "uint32_t* w" + num(i); first = false; }
  src += tab_params + ") {\n";
  // 1-byte outputs are packed four pixels to a word (pack_bytes), the others stored per pixel
  auto packed = [&](int i) { return dtype_size(out_dtype[i]) == 1 && V % 4 == 0; };
  for (int j = 0; j < V; ++j) {
    src += "  ";
    for (int i = 0; i < prog->n_outputs; ++i) src += "S o" + num(i) + "_" + num(j) + "; ";
    src += "pixel(p";
    first = false;
    for (int i = 0; i < prog->n_inputs; ++i) {
      src += std::string(first ? "" : ", ") + "element<" + storage_type(in_dtype[i]) + ", " + num(j) + ">(a" + num(i) + ")";
      first = false;
    }
    for (int i = 0; i < prog->n_outputs; ++i) { src += std::string(first ? "" : ", ") + "o" + num(i) + "_" + num(j); first = false; }
    src += tab_args + ");";
    for (int i = 0; i < prog->n_outputs; ++i) {
      const std::string o = "o" + num(i) + "_" + num(j), w = "w" + num(i);
      if (!packed(i))
        src += " set_element<" + num(dtype_size(out_dtype[i])) + ", " + num(j) + ">(" + w + ", " + o + ");";
      else if (j % 4 == 3)
        src += " " + w + "[" + num(j / 4) + "] = pack_bytes(o" + num(i) + "_" + num(j - 3) + ", o" + num(i) + "_" +
               num(j - 2) + ", o" + num(i) + "_" + num(j - 1) + ", " + o + ");";
    }
    src += "\n";
  }
  src += "}\n";

  // ---- the kernel -------------------------------------------------------------------------
  src += "extern \"C\" __global__ void __launch_bounds__(256) gm_fused(const __grid_constant__ Params p) {\n";
  src += "  const int tid = threadIdx.x;\n";
  for (int t = 0; t < prog->n_tables; ++t) {
    const GmTable& g = prog->tables[t];
    const std::string id = num(t);
    if (L.bits[t]) continue;
    if (L.in_smem[t]) {
      src += "  for (int i = tid; i < " + num(g.n) + "; i += 256) {";
      if (g.keys) src += " t" + id + "k[i] = g_t" + id + "k[i];";
      if (g.vals) src += " t" + id + "v[i] = g_t" + id + "v[i];";
      if (g.hit) src += " t" + id + "h[i] = g_t" + id + "h[i];";
      src += " }\n";
    } else {
      src += "  const int64_t* t" + id + "k = p.tk[" + id + "]; const uint64_t* t" + id + "v = p.tv[" + id +
             "]; const uint8_t* t" + id + "h = p.th[" + id + "];\n";
    }
  }
  if (prog->n_tables) src += "  __syncthreads();\n";
  for (int i = 0; i < prog->n_inputs; ++i)
    src += "  const unsigned char* __restrict__ in" + num(i) + " = (const unsigned char*)p.in[" + num(i) + "];\n";
  for (int i = 0; i < prog->n_outputs; ++i)
    src += "  unsigned char* __restrict__ out" + num(i) + " = (unsigned char*)p.out[" + num(i) + "];\n";
  src += "  const long long groups = p.n / " + num(V) + ";\n";
  src += "  const long long chunk = 256LL * " + num(U) + ";\n";
  src += "  const long long n_chunks = groups / chunk;\n";
  // full chunks: U groups per thread.  The loads of a chunk are emitted before its evaluation; `set`
  // selects a register set of the two-set loop (-1: the single set), `g0` is the chunk's first group
  // of this thread.
  auto load_set = [&](int set, const std::string& g0, bool fence) {
    const std::string idx = set < 0 ? "" : "[" + num(set) + "]";
    std::string t = "      #pragma unroll\n      for (int u = 0; u < " + num(U) + "; ++u) {\n";
    for (int i = 0; i < prog->n_inputs; ++i) {
      const int bytes = V * dtype_size(in_dtype[i]);
      t += "        load_group<" + num(bytes) + ">(a" + num(i) + idx + "[u], in" + num(i) + " + (" + g0 +
           " + u * 256LL) * " + num(bytes) + ");\n";
    }
    return t + (fence ? "        __syncwarp();\n" : "") + "      }\n";
  };
  auto eval_set = [&](int set, const std::string& g0) {
    const std::string idx = set < 0 ? "" : "[" + num(set) + "]";
    std::string t = "      #pragma unroll\n      for (int u = 0; u < " + num(U) + "; ++u) {\n";
    for (int i = 0; i < prog->n_outputs; ++i) t += "        uint32_t w" + num(i) + "[" + num(words(out_dtype[i])) + "];\n";
    t += "        group(p";
    bool first = false;
    for (int i = 0; i < prog->n_inputs; ++i) { t += std::string(first ? "" : ", ") + "a" + num(i) + idx + "[u]"; first = false; }
    for (int i = 0; i < prog->n_outputs; ++i) { t += std::string(first ? "" : ", ") + "w" + num(i); first = false; }
    t += tab_args + ");\n";
    for (int i = 0; i < prog->n_outputs; ++i) {
      const int bytes = V * dtype_size(out_dtype[i]);
      t += "        store_group<" + num(bytes) + ">(out" + num(i) + " + (" + g0 + " + u * 256LL) * " + num(bytes) +
           ", w" + num(i) + ");\n";
    }
    return t + "      }\n";
  };
  if (L.two_sets) {
    // p.chunks_per_block consecutive chunks per block in two register sets: the loads of chunk c + 1
    // are issued before chunk c is evaluated.  The warp barrier after each group's loads keeps ptxas
    // from sinking them into the evaluation (tools/jit_sass.py: without it the unbaked cfg2 kernel
    // issues them after ~140 of ~350 instructions; one barrier after all of them is not enough).
    src += "  const long long K = p.chunks_per_block;\n";
    src += "  for (long long c0 = (long long)blockIdx.x * K; c0 < n_chunks; c0 += (long long)gridDim.x * K) {\n";
    src += "    const long long c1 = c0 + K < n_chunks ? c0 + K : n_chunks;\n";
    for (int i = 0; i < prog->n_inputs; ++i)
      src += "    uint32_t a" + num(i) + "[2][" + num(U) + "][" + num(words(in_dtype[i])) + "];\n";
    src += load_set(0, "c0 * chunk + tid", true);
    src += "    for (long long c = c0; c < c1; c += 2) {\n";
    src += "      if (c + 1 < c1) {\n" + load_set(1, "(c + 1) * chunk + tid", true) + "      }\n";
    src += eval_set(0, "c * chunk + tid");
    src += "      if (c + 1 == c1) break;\n";
    src += "      if (c + 2 < c1) {\n" + load_set(0, "(c + 2) * chunk + tid", true) + "      }\n";
    src += eval_set(1, "(c + 1) * chunk + tid");
    src += "    }\n  }\n";
  } else {
    // one chunk at a time, all its loads first (ptxas may still sink some of them)
    src += "  for (long long c = blockIdx.x; c < n_chunks; c += gridDim.x) {\n";
    src += "    const long long g0 = c * chunk + tid;\n";
    for (int i = 0; i < prog->n_inputs; ++i)
      src += "    uint32_t a" + num(i) + "[" + num(U) + "][" + num(words(in_dtype[i])) + "];\n";
    src += load_set(-1, "g0", false) + eval_set(-1, "g0");
    src += "  }\n";
  }
  // remaining whole groups: one per thread
  src += "  for (long long g = n_chunks * chunk + (long long)blockIdx.x * 256 + tid; g < groups; g += (long long)gridDim.x * 256) {\n";
  for (int i = 0; i < prog->n_inputs; ++i) {
    const int bytes = V * dtype_size(in_dtype[i]);
    src += "    uint32_t a" + num(i) + "[" + num(words(in_dtype[i])) + "]; load_group<" + num(bytes) + ">(a" + num(i) +
           ", in" + num(i) + " + g * " + num(bytes) + ");\n";
  }
  for (int i = 0; i < prog->n_outputs; ++i)
    src += "    uint32_t w" + num(i) + "[" + num(words(out_dtype[i])) + "];\n";
  src += "    group(p";
  first = false;
  for (int i = 0; i < prog->n_inputs; ++i) { src += std::string(first ? "" : ", ") + "a" + num(i); first = false; }
  for (int i = 0; i < prog->n_outputs; ++i) { src += std::string(first ? "" : ", ") + "w" + num(i); first = false; }
  src += tab_args + ");\n";
  for (int i = 0; i < prog->n_outputs; ++i) {
    const int bytes = V * dtype_size(out_dtype[i]);
    src += "    store_group<" + num(bytes) + ">(out" + num(i) + " + g * " + num(bytes) + ", w" + num(i) + ");\n";
  }
  src += "  }\n";
  // ragged tail: fewer than V pixels, one thread each
  src += "  if (blockIdx.x == 0) {\n    const long long px = groups * " + num(V) + " + tid;\n    if (px < p.n) {\n";
  for (int i = 0; i < prog->n_outputs; ++i) src += "      S o" + num(i) + ";\n";
  src += "      pixel(p";
  first = false;
  for (int i = 0; i < prog->n_inputs; ++i) {
    const std::string st = storage_type(in_dtype[i]);
    src += std::string(first ? "" : ", ") + "slot_of<" + st + ">(((const " + st + "*)in" + num(i) + ")[px])";
    first = false;
  }
  for (int i = 0; i < prog->n_outputs; ++i) { src += std::string(first ? "" : ", ") + "o" + num(i); first = false; }
  src += tab_args + ");\n";
  for (int i = 0; i < prog->n_outputs; ++i) {
    const char* ot = dtype_size(out_dtype[i]) == 1 ? "uint8_t" : dtype_size(out_dtype[i]) == 2 ? "uint16_t"
                     : dtype_size(out_dtype[i]) == 4 ? "uint32_t" : "uint64_t";
    src += std::string("      ((") + ot + "*)out" + num(i) + ")[px] = (" + ot + ")o" + num(i) + ";\n";
  }
  src += "    }\n  }\n}\n";
  return src;
}

// ---- cache ------------------------------------------------------------------------------------
struct JitKernel {
  std::string key;
  cudaLibrary_t library = nullptr;
  cudaKernel_t kernel = nullptr;
  JitLayout layout;
  int blocks_per_sm = 8;
  ~JitKernel() { if (library) cudaLibraryUnload(library); }
};

// Kernels in memory: at most kMaxKernels, the oldest is unloaded first (a launch in flight keeps
// its kernel alive through the shared pointer).  Compiled cubins are also kept on disk
// (GM_JIT_CACHE=<dir>, default ~/.cache/dask_geomodeling_b200/jit, "off" disables), keyed by a
// hash of the generated source, so that a new process does not pay the NVRTC compile again.
static const size_t kMaxKernels = 256;
static std::unordered_map<std::string, std::shared_ptr<JitKernel>> g_kernels;
static std::deque<std::string> g_kernel_order;
static std::unordered_map<std::string, std::string> g_last_constants;   // structure key -> constants of its last launch
static const int64_t kBakeFromPixels = 1 << 22;
static std::atomic<int64_t> g_disk_hits{0};
static std::atomic<int64_t> g_compiles{0};
static std::string g_last_source;

static std::string program_key(const GmProgram* prog, const int* in_dtype, const int* out_dtype,
                               const JitLayout& L) {
  std::string key;
  auto put = [&](const void* p, size_t n) { key.append((const char*)p, n); };
  put(&prog->word, 4); put(&prog->n_instr, 4); put(&prog->n_inputs, 4); put(&prog->n_outputs, 4);
  put(&prog->n_tables, 4);
  for (int pc = 0; pc < prog->n_instr; ++pc) {     // the structure of an instruction, not its constants
    GmInstr shape = prog->instr[pc];
    memset(shape.k, 0, sizeof(shape.k));
    put(&shape, sizeof(GmInstr));
  }
  put(in_dtype, sizeof(int) * prog->n_inputs);
  put(out_dtype, sizeof(int) * prog->n_outputs);
  for (int t = 0; t < prog->n_tables; ++t) {
    const GmTable& g = prog->tables[t];
    const char has[4] = {(char)(g.keys != nullptr), (char)(g.vals != nullptr), (char)(g.hit != nullptr),
                         (char)L.baked[t]};
    put(&g.n, 4); put(&g.kind, 4); put(&g.base, 8); put(has, 4);
    if (L.baked[t]) {
      if (g.keys) put(g.keys, (size_t)g.n * 8);
      if (g.vals) put(g.vals, (size_t)g.n * 8);
      if (g.hit) put(g.hit, (size_t)g.n);
    }
  }
  return key;
}

// source -> sm_100a cubin.  GM_JIT_DUMP=<prefix> writes <prefix>.cu / <prefix>.cubin of
// the last compile (for cuobjdump -sass / ncu source correlation).
static int nvrtc_compile(const std::string& source, std::vector<char>& cubin) {
  if (load_nvrtc()) return 1;
  nvrtcProgram np = nullptr;
  int rc = g_nvrtc.CreateProgram(&np, source.c_str(), "gm_fused.cu", 0, nullptr, nullptr);
  if (rc) return fail(std::string("nvrtcCreateProgram: ") + g_nvrtc.GetErrorString(rc));
  const char* opts[] = {"--gpu-architecture=sm_100a", "-std=c++17", "-fmad=false", "-prec-div=true",
                        "-prec-sqrt=true", "-ftz=false", "-lineinfo", "-default-device"};
  rc = g_nvrtc.CompileProgram(np, (int)(sizeof(opts) / sizeof(opts[0])), opts);
  if (rc) {
    size_t n = 0;
    g_nvrtc.GetProgramLogSize(np, &n);
    std::string log(n, '\0');
    if (n) g_nvrtc.GetProgramLog(np, &log[0]);
    g_nvrtc.DestroyProgram(&np);
    return fail(std::string("NVRTC failed (") + g_nvrtc.GetErrorString(rc) + "):\n" + log);
  }
  size_t size = 0;
  g_nvrtc.GetCUBINSize(np, &size);
  cubin.resize(size);
  g_nvrtc.GetCUBIN(np, cubin.data());
  g_nvrtc.DestroyProgram(&np);
  if (const char* prefix = getenv("GM_JIT_DUMP")) {
    if (FILE* f = fopen((std::string(prefix) + ".cu").c_str(), "w")) { fwrite(source.data(), 1, source.size(), f); fclose(f); }
    if (FILE* f = fopen((std::string(prefix) + ".cubin").c_str(), "wb")) { fwrite(cubin.data(), 1, cubin.size(), f); fclose(f); }
  }
  return 0;
}

static std::string cache_dir() {
  const char* env = getenv("GM_JIT_CACHE");
  if (env && (!strcmp(env, "off") || !strcmp(env, "0"))) return "";
  if (env && *env) return env;
  const char* xdg = getenv("XDG_CACHE_HOME");
  const char* home = getenv("HOME");
  if (xdg && *xdg) return std::string(xdg) + "/dask_geomodeling_b200/jit";
  if (home && *home) return std::string(home) + "/.cache/dask_geomodeling_b200/jit";
  return "";
}

static std::string source_hash(const std::string& source) {
  // two independent 64-bit FNV-1a style hashes of the whole source (prelude included: a new
  // library version never picks up an old cubin)
  uint64_t a = 1469598103934665603ULL, b = 0x9E3779B97F4A7C15ULL;
  for (unsigned char c : source) {
    a = (a ^ c) * 1099511628211ULL;
    b = (b + c) * 0xD6E8FEB86659FD93ULL;
    b ^= b >> 29;
  }
  char buf[40];
  snprintf(buf, sizeof(buf), "%016llx%016llx", (unsigned long long)a, (unsigned long long)b);
  return buf;
}

static void make_dirs(const std::string& path) {
  for (size_t i = 1; i <= path.size(); ++i)
    if (i == path.size() || path[i] == '/') mkdir(path.substr(0, i).c_str(), 0755);
}

static bool read_cached_cubin(const std::string& path, std::vector<char>& cubin) {
  FILE* f = fopen(path.c_str(), "rb");
  if (!f) return false;
  fseek(f, 0, SEEK_END);
  const long n = ftell(f);
  fseek(f, 0, SEEK_SET);
  bool ok = n > 0;
  if (ok) {
    cubin.resize((size_t)n);
    ok = fread(cubin.data(), 1, (size_t)n, f) == (size_t)n;
  }
  fclose(f);
  return ok;
}

static void write_cached_cubin(const std::string& dir, const std::string& path, const std::vector<char>& cubin) {
  make_dirs(dir);
  const std::string tmp = path + ".tmp" + std::to_string((long long)getpid());
  FILE* f = fopen(tmp.c_str(), "wb");
  if (!f) return;
  const bool ok = fwrite(cubin.data(), 1, cubin.size(), f) == cubin.size();
  fclose(f);
  if (!ok || rename(tmp.c_str(), path.c_str()) != 0) remove(tmp.c_str());
}

static int compile_kernel(const std::string& source, JitKernel* k) {
  std::vector<char> cubin;
  const std::string dir = cache_dir();
  const std::string path = dir.empty() ? "" : dir + "/" + source_hash(source) + ".cubin";
  if (!path.empty() && read_cached_cubin(path, cubin)) {
    g_disk_hits.fetch_add(1);
  } else {
    cubin.clear();
    if (nvrtc_compile(source, cubin)) return 1;
    g_compiles.fetch_add(1);
    if (!path.empty()) write_cached_cubin(dir, path, cubin);
  }
  cudaError_t e = cudaLibraryLoadData(&k->library, cubin.data(), nullptr, nullptr, 0, nullptr, nullptr, 0);
  if (e != cudaSuccess) return fail(std::string("cudaLibraryLoadData: ") + cudaGetErrorString(e));
  e = cudaLibraryGetKernel(&k->kernel, k->library, "gm_fused");
  if (e != cudaSuccess) return fail(std::string("cudaLibraryGetKernel: ") + cudaGetErrorString(e));
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, (const void*)k->kernel, 256, 0) == cudaSuccess &&
      per_sm > 0)
    k->blocks_per_sm = per_sm;
  else
    cudaGetLastError();
  return 0;
}

struct JitParams {
  const void* in[GM_MAX_INPUTS];
  void* out[GM_MAX_OUTPUTS];
  long long n;
  long long chunks_per_block;   // of the two-set loop; 1 otherwise
  const int64_t* tk[GM_MAX_TABLES];
  const uint64_t* tv[GM_MAX_TABLES];
  const uint8_t* th[GM_MAX_TABLES];
  unsigned long long k[GM_MAX_INSTR][6];
};

int jit_tables_baked(const GmProgram* prog) {
  int total = 0;
  for (int t = 0; t < prog->n_tables; ++t) total += prog->tables[t].n;
  return total <= kBakeLimit;
}

int jit_launch(const GmProgram* prog, const void* const* in, const int* in_dtype, void* const* out,
               const int* out_dtype, const void* const* tkeys, const void* const* tvals,
               const void* const* thit, int64_t n, cudaStream_t s) {
  const JitLayout L = plan_layout(prog, in_dtype, out_dtype);
  const std::string key = program_key(prog, in_dtype, out_dtype, L);
  // the constants of this launch (they select the baked variant, if there is one)
  std::string constants;
  for (int pc = 0; pc < prog->n_instr; ++pc) constants.append((const char*)prog->instr[pc].k, sizeof(prog->instr[pc].k));
  const std::string baked_key = key + '#' + constants;
  std::shared_ptr<JitKernel> k;
  {
    std::lock_guard<std::mutex> lock(g_jit_mutex);
    auto build = [&](const std::string& as, bool bake) -> std::shared_ptr<JitKernel> {
      t_bake = bake ? prog : nullptr;
      std::string source = generate(prog, in_dtype, out_dtype, L);
      t_bake = nullptr;
      std::shared_ptr<JitKernel> fresh = std::make_shared<JitKernel>();
      fresh->key = as;
      fresh->layout = L;
      g_last_source = source;
      if (compile_kernel(source, fresh.get())) return nullptr;
      if (g_kernels.size() >= kMaxKernels && !g_kernel_order.empty()) {
        g_kernels.erase(g_kernel_order.front());     // unloaded when its last launch has returned
        g_kernel_order.pop_front();
      }
      g_kernels[as] = fresh;
      g_kernel_order.push_back(as);
      return fresh;
    };
    auto baked = g_kernels.find(baked_key);
    if (baked != g_kernels.end()) {
      k = baked->second;
    } else {
      auto it = g_kernels.find(key);
      k = it != g_kernels.end() ? it->second : build(key, false);
      if (!k) return 1;
      // the same constants again on a large raster: from now on the literal-specialised kernel
      std::string& last = g_last_constants[key];
      if (n >= kBakeFromPixels && last == constants && !getenv("GM_JIT_NO_BAKE")) {
        std::shared_ptr<JitKernel> special = build(baked_key, true);
        if (special) k = special;
      }
      last = constants;
    }
  }
  JitParams p;
  memset(&p, 0, sizeof(p));
  for (int i = 0; i < prog->n_inputs; ++i) p.in[i] = in[i];
  for (int i = 0; i < prog->n_outputs; ++i) p.out[i] = out[i];
  p.n = n;
  for (int pc = 0; pc < prog->n_instr; ++pc)
    for (int i = 0; i < 6; ++i) p.k[pc][i] = prog->instr[pc].k[i];
  for (int t = 0; t < prog->n_tables; ++t) {
    p.tk[t] = (const int64_t*)tkeys[t];
    p.tv[t] = (const uint64_t*)tvals[t];
    p.th[t] = (const uint8_t*)thit[t];
  }
  // One block per chunk of 256 * U groups, or per K chunks in the two-set loop.  A grid of resident
  // blocks that strides over the chunks streams slower (tools/chain_ceiling.cu on one B200: 0.29-0.30 ms
  // against 0.263 ms for the cfg2 pattern), so the grid is capped at the resident blocks only when every
  // block first copies its lookup tables into shared memory (those programs keep the single-set loop).
  // K shrinks on small rasters, so that the grid still fills every SM's resident blocks.
  const int64_t resident = (int64_t)sm_count() * k->blocks_per_sm;
  const int64_t chunk_px = 256LL * L.U * L.V;
  p.chunks_per_block = 1;
  if (L.two_sets)
    p.chunks_per_block = std::max<int64_t>(1, std::min<int64_t>(kMaxChunksPerBlock, n / chunk_px / resident));
  const int64_t per_block = chunk_px * p.chunks_per_block;
  int64_t grid = (n + per_block - 1) / per_block;
  bool smem_tables = false;
  for (int t = 0; t < prog->n_tables; ++t) smem_tables = smem_tables || L.in_smem[t];
  if (smem_tables && grid > resident) grid = resident;
  if (grid > INT32_MAX) grid = INT32_MAX;
  if (grid < 1) grid = 1;
  void* args[] = {&p};
  cudaError_t e = cudaLaunchKernel((const void*)k->kernel, dim3((unsigned)grid), dim3(256), args, 0, s);
  if (e != cudaSuccess) return fail(std::string("specialised kernel launch: ") + cudaGetErrorString(e));
  count_launch();
  return 0;
}

int64_t jit_compile_count() { return g_compiles.load(); }

}  // namespace gm

using namespace gm;

// Test / inspection hooks: the CUDA source generated for `prog`, with its constants as kernel
// parameters or baked (no GPU needed).
static int jit_source(const GmProgram* prog, const int32_t* in_dtype, const int32_t* out_dtype, bool bake,
                      char* buffer, int64_t capacity, int64_t* length) {
  if (!prog || !length) return fail("gm_jit_source: null argument");
  if (prog->n_instr < 1 || prog->n_instr > GM_MAX_INSTR || prog->n_inputs > GM_MAX_INPUTS ||
      prog->n_outputs > GM_MAX_OUTPUTS || prog->n_tables > GM_MAX_TABLES)
    return fail("gm_jit_source: bad program");
  const JitLayout L = plan_layout(prog, in_dtype, out_dtype);
  t_bake = bake ? prog : nullptr;
  const std::string source = generate(prog, in_dtype, out_dtype, L);
  t_bake = nullptr;
  *length = (int64_t)source.size();
  if (buffer && capacity > 0) {
    const size_t n = std::min((size_t)capacity - 1, source.size());
    memcpy(buffer, source.data(), n);
    buffer[n] = 0;
  }
  return 0;
}

extern "C" int gm_jit_source(const GmProgram* prog, const int32_t* in_dtype, const int32_t* out_dtype,
                             char* buffer, int64_t capacity, int64_t* length) {
  return jit_source(prog, in_dtype, out_dtype, false, buffer, capacity, length);
}

extern "C" int gm_jit_baked_source(const GmProgram* prog, const int32_t* in_dtype, const int32_t* out_dtype,
                                   char* buffer, int64_t capacity, int64_t* length) {
  return jit_source(prog, in_dtype, out_dtype, true, buffer, capacity, length);
}

// Compile `prog` with NVRTC without loading it (works without a GPU): used by the CPU
// test-suite to prove that every generated kernel is valid sm_100a code.
extern "C" int gm_jit_check(const GmProgram* prog, const int32_t* in_dtype, const int32_t* out_dtype,
                            int64_t* cubin_bytes) {
  if (!prog) return fail("gm_jit_check: null program");
  const JitLayout L = plan_layout(prog, in_dtype, out_dtype);
  const std::string source = generate(prog, in_dtype, out_dtype, L);
  std::vector<char> cubin;
  std::lock_guard<std::mutex> lock(g_jit_mutex);
  if (nvrtc_compile(source, cubin)) return 1;
  if (cubin_bytes) *cubin_bytes = (int64_t)cubin.size();
  return 0;
}

extern "C" int64_t gm_jit_compile_count(void) { return jit_compile_count(); }
