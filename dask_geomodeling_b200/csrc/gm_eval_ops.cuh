// Per-pixel semantics of the fused evaluator's bytecode: the only definition of what each
// instruction does to one slot.  Both back ends compile this text:
//   - the interpreter (gm_eval.cu, nvcc) with 32- and 64-bit slots, class and opcode dispatch
//     hoisted out of its loops over the pixels of a thread;
//   - the specialised kernels (gm_jit.cu, NVRTC): build.py splices this file into
//     gm_jit_prelude.cuh, and the generator calls these functions with literal flags.
//
// The slot type S (uint32_t or uint64_t) is deduced from the accumulator.  Value classes and the
// opcode are template parameters; per-instruction flags are plain arguments, which the interpreter
// tests warp-uniformly at run time and the generator passes as literals (the compiler folds them).
// Mask and Overlay take theirs as deduced types instead: bool / int from the interpreter, Lit<v>
// (gm_jit_prelude.cuh) from generated code.  A function is optimised before it is inlined, and
// there a plain literal argument came too late to fold their branches back to the code of one
// flag combination.  Constants arrive as raw bits (GmInstr::k).
//
// The includer provides int32_t & co. and GM_OUTLINE, the qualifiers of the large, rarely used
// helpers (pow, exp, log, integer power): the interpreter keeps them out of line, the specialised
// kernel inlines them.  No standard-library header is used: NVRTC compiles this without any.
//
// Reference: raster/elemwise.py:235-299, :551-638, :726-757, raster/misc.py:98-123, :208-222,
// :245-251, :309-328, :387-399, :482-515, raster/reduction.py:38-119.
#ifndef GM_EVAL_OPS_CUH
#define GM_EVAL_OPS_CUH
#include "../../include/gm_bytecode.h"

#define GM_DEV __device__ __forceinline__

template <typename T> struct IsFloat { static constexpr bool value = false; };
template <> struct IsFloat<float> { static constexpr bool value = true; };
template <> struct IsFloat<double> { static constexpr bool value = true; };

// ---- raw slot bits <-> typed value ------------------------------------------
template <typename T> struct Raw;
template <> struct Raw<int32_t> {
  static GM_DEV int32_t get(uint64_t b) { return (int32_t)(uint32_t)b; }
  static GM_DEV uint64_t put(int32_t v) { return (uint64_t)(uint32_t)v; }
};
template <> struct Raw<float> {
  static GM_DEV float get(uint64_t b) { return __uint_as_float((uint32_t)b); }
  static GM_DEV uint64_t put(float v) { return (uint64_t)__float_as_uint(v); }
};
template <> struct Raw<int64_t> {
  static GM_DEV int64_t get(uint64_t b) { return (int64_t)b; }
  static GM_DEV uint64_t put(int64_t v) { return (uint64_t)v; }
};
template <> struct Raw<double> {
  static GM_DEV double get(uint64_t b) { return __longlong_as_double((long long)b); }
  static GM_DEV uint64_t put(double v) { return (uint64_t)__double_as_longlong(v); }
};

template <typename T> GM_DEV T quiet_nan() { return T(0); }
template <> GM_DEV float quiet_nan<float>() { return __int_as_float(0x7fc00000); }
template <> GM_DEV double quiet_nan<double>() { return __longlong_as_double(0x7ff8000000000000LL); }

// ---- arithmetic (wrap-around integers, IEEE floats) ---------------------------------
GM_DEV int32_t w_add(int32_t a, int32_t b) { return (int32_t)((uint32_t)a + (uint32_t)b); }
GM_DEV int64_t w_add(int64_t a, int64_t b) { return (int64_t)((uint64_t)a + (uint64_t)b); }
GM_DEV float w_add(float a, float b) { return a + b; }
GM_DEV double w_add(double a, double b) { return a + b; }
GM_DEV int32_t w_sub(int32_t a, int32_t b) { return (int32_t)((uint32_t)a - (uint32_t)b); }
GM_DEV int64_t w_sub(int64_t a, int64_t b) { return (int64_t)((uint64_t)a - (uint64_t)b); }
GM_DEV float w_sub(float a, float b) { return a - b; }
GM_DEV double w_sub(double a, double b) { return a - b; }
GM_DEV int32_t w_mul(int32_t a, int32_t b) { return (int32_t)((uint32_t)a * (uint32_t)b); }
GM_DEV int64_t w_mul(int64_t a, int64_t b) { return (int64_t)((uint64_t)a * (uint64_t)b); }
GM_DEV float w_mul(float a, float b) { return a * b; }
GM_DEV double w_mul(double a, double b) { return a * b; }

template <typename T> GM_DEV T w_div(T a, T b) {
  if constexpr (IsFloat<T>::value) return a / b; else return b == 0 ? T(0) : a / b;
}
// numpy integer power: square-and-multiply with wrap-around.  A negative
// exponent raises in numpy; here it yields 0 (documented limitation).
template <typename T> GM_OUTLINE T int_pow(T base, T e) {
  if (e < 0) return 0;
  T r = 1;
  while (e) {
    if (e & 1) r = w_mul(r, base);
    e >>= 1;
    if (e) base = w_mul(base, base);
  }
  return r;
}
GM_OUTLINE float t_pow(float a, float b) { return powf(a, b); }
GM_OUTLINE double t_pow(double a, double b) { return pow(a, b); }
GM_OUTLINE float t_exp(float a) { return expf(a); }
GM_OUTLINE double t_exp(double a) { return exp(a); }
GM_OUTLINE float t_log(float a) { return logf(a); }
GM_OUTLINE double t_log(double a) { return log(a); }
GM_OUTLINE float t_log10(float a) { return log10f(a); }
GM_OUTLINE double t_log10(double a) { return log10(a); }
template <typename T> GM_DEV T w_pow(T a, T b) {
  if constexpr (IsFloat<T>::value) return t_pow(a, b); else return int_pow<T>(a, b);
}
template <typename T> GM_DEV bool finite_(T v) {
  if constexpr (IsFloat<T>::value) return isfinite(v); else return true;
}
template <typename T> GM_DEV T abs_(T v) {
  if constexpr (IsFloat<T>::value) return fabs(v); else return v < 0 ? -v : v;
}
// np.isclose(x, y): less_equal(abs(x - y), tol) & isfinite(y) | (x == y)
template <typename T> GM_DEV bool close_(T x, T y, T tol, bool y_finite) {
  return ((abs_(w_sub(x, y)) <= tol) && y_finite) || (x == y);
}

// ---- instructions ---------------------------------------------------------------------------
// LOAD / MATB / CVT: numpy astype From -> To; the sentinel k becomes NaN when asked (float targets)
template <typename From, typename To, typename S> GM_DEV S cvt(S x, bool nanify, uint64_t k) {
  const From v = Raw<From>::get(x);
  To r = (To)v;
  if constexpr (IsFloat<To>::value) r = (nanify && v == Raw<From>::get(k)) ? quiet_nan<To>() : r;
  return (S)Raw<To>::put(r);
}

// binary arithmetic in class T: invalid operands (sentinels k1 of a, k2 of b) or a non-finite
// result -> fill k3
template <int OP, typename T, typename S>
GM_DEV S math(S a, uint64_t b, bool fa, bool fb, uint64_t k1, uint64_t k2, uint64_t k3) {
  const T x = Raw<T>::get(a), y = Raw<T>::get(b);
  T r;
  if constexpr (OP == GM_OP_ADD) r = w_add(x, y);
  else if constexpr (OP == GM_OP_SUB) r = w_sub(x, y);
  else if constexpr (OP == GM_OP_RSUB) r = w_sub(y, x);
  else if constexpr (OP == GM_OP_MUL) r = w_mul(x, y);
  else if constexpr (OP == GM_OP_DIV) r = w_div(x, y);
  else if constexpr (OP == GM_OP_RDIV) r = w_div(y, x);
  else if constexpr (OP == GM_OP_POW) r = w_pow(x, y);
  else r = w_pow(y, x);
  const bool bad = !finite_(r) || (fa && x == Raw<T>::get(k1)) || (fb && y == Raw<T>::get(k2));
  return (S)Raw<T>::put(bad ? Raw<T>::get(k3) : r);
}

// comparison in class T: a boolean, or the fill k3 (slot bits) for invalid operands
template <int OP, typename T, typename S>
GM_DEV S compare(S a, uint64_t b, bool fa, bool fb, uint64_t k1, uint64_t k2, uint64_t k3) {
  const T x = Raw<T>::get(a), y = Raw<T>::get(b);
  bool r;
  if constexpr (OP == GM_OP_EQ) r = x == y;
  else if constexpr (OP == GM_OP_NE) r = x != y;
  else if constexpr (OP == GM_OP_GT) r = x > y;
  else if constexpr (OP == GM_OP_GE) r = x >= y;
  else if constexpr (OP == GM_OP_LT) r = x < y;
  else r = x <= y;
  const bool bad = (fa && x == Raw<T>::get(k1)) || (fb && y == Raw<T>::get(k2));
  return bad ? (S)k3 : (S)(r ? 1u : 0u);
}

// EXP / LOG / LOG10 in the float class T
template <int OP, typename T, typename S> GM_DEV S transcend(S a, bool fa, uint64_t k1, uint64_t k3) {
  const T x = Raw<T>::get(a);
  T r;
  if constexpr (OP == GM_OP_EXP) r = t_exp(x);
  else if constexpr (OP == GM_OP_LOG) r = t_log(x);
  else r = t_log10(x);
  const bool bad = !finite_(r) || (fa && x == Raw<T>::get(k1));
  return (S)Raw<T>::put(bad ? Raw<T>::get(k3) : r);
}

template <typename S> GM_DEV S data_flag(bool is_nd, bool want_nodata) {
  return (S)((is_nd == want_nodata) ? 1u : 0u);
}

// ISDATA (want_nodata false) / ISNODATA of a in class A, sentinel k1
template <typename A, typename S> GM_DEV S is_data(S a, bool fa, bool want_nodata, uint64_t k1) {
  return data_flag<S>(fa && Raw<A>::get(a) == Raw<A>::get(k1), want_nodata);
}

template <int OP, typename S> GM_DEV S logic(S a, uint64_t b) {
  const bool x = (uint32_t)a != 0u, y = (uint32_t)b != 0u;
  bool r;
  if constexpr (OP == GM_OP_AND) r = x && y;
  else if constexpr (OP == GM_OP_OR) r = x || y;
  else if constexpr (OP == GM_OP_XOR) r = x != y;
  else r = !x;
  return (S)(r ? 1u : 0u);
}

// Clip: masked cells become the sentinel k1.  MODE 0 = no mask information, 1 = b is a boolean
// mask, 2 = b holds class B with sentinel k2
template <typename B, int MODE, typename S> GM_DEV S clip(S a, uint64_t b, uint64_t k1, uint64_t k2) {
  if constexpr (MODE == 1) return ((uint32_t)b == 0u) ? (S)k1 : a;
  else if constexpr (MODE == 2) return (Raw<B>::get(b) == Raw<B>::get(k2)) ? (S)k1 : a;
  else return a;
}

// Mask (raster/misc.py:208-222): data -> value k0, no data -> fill k3; the sentinel test (class T,
// k1) is np.isclose with tolerance k4 when `cl`
template <typename T, typename A, typename S, typename Has, typename Cl, typename Fin>
GM_DEV S mask(S a, Has has, Cl cl, Fin fin, uint64_t k0, uint64_t k1, uint64_t k3, uint64_t k4) {
  const T x = (T)Raw<A>::get(a);
  const bool nod = has && (cl ? close_(x, Raw<T>::get(k1), Raw<T>::get(k4), fin) : x == Raw<T>::get(k1));
  return nod ? (S)k3 : (S)k0;
}

// MaskBelow (raster/misc.py:249-250): threshold k0 in class T, sentinel k5 as slot bits
template <typename T, typename A, typename S> GM_DEV S mask_below(S a, uint64_t k0, uint64_t k5) {
  return ((T)Raw<A>::get(a) < Raw<T>::get(k0)) ? (S)k5 : a;
}

// What Step makes of each arm of its select: `Id` keeps the value (see IsNd in the prelude).
template <typename S> struct Id {
  GM_DEV S operator()(uint64_t v) const { return (S)v; }
};

// Step (raster/misc.py:316-326): location k0 in class T, sentinel k1 in class A, left / at / right
// k2 / k3 / k4 as slot bits
template <typename T, typename A, typename S, typename F = Id<S>>
GM_DEV auto step(S a, bool fa, uint64_t k0, uint64_t k1, uint64_t k2, uint64_t k3, uint64_t k4, F f = F()) {
  const A raw = Raw<A>::get(a);
  const T x = (T)raw, loc = Raw<T>::get(k0);
  auto r = f(a);
  r = x < loc ? f(k2) : r;
  r = x == loc ? f(k3) : r;
  r = x > loc ? f(k4) : r;
  r = (fa && raw == Raw<A>::get(k1)) ? f(a) : r;
  return r;
}

// Classify: np.digitize(values, bins, right) (raster/misc.py:396), bins ascending; no data -> k3
template <typename T, typename A, typename S>
GM_DEV S classify(S a, bool fa, bool right, const int64_t* keys, int n, uint64_t k1, uint64_t k3) {
  const A raw = Raw<A>::get(a);
  const T x = (T)raw;
  int lo = 0, hi = n;
  if (x != x) lo = n;  // NaN sorts last
  else
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      const T e = Raw<T>::get((uint64_t)keys[mid]);
      const bool go = right ? (e < x) : (e <= x);
      if (go) lo = mid + 1; else hi = mid;
    }
  return (fa && raw == Raw<A>::get(k1)) ? (S)k3 : (S)(uint32_t)lo;
}

// Overlay, the FillNoData step (raster/elemwise.py:752-755): acc = isdata(b) ? astype(b) : acc.
// The sentinel test (np.isclose with tolerance k4 when `cl`) runs in class T = class of b, To is
// the class of acc.  With a GmReduce kind the step reduces instead (reduce_rasters):
// acc = isdata(b) ? red(acc, astype(b)) : acc, with max / min / sum / product in a float class To
// where NaN marks "no value yet" (NaN cells of b are skipped as the np.nan* functions do), or
// count (acc + 1 in any class).  Validation rejects max / min / sum / product over other classes.
template <typename T, typename To, typename S, typename Has, typename Cl, typename Fin, typename Kind>
GM_DEV S overlay(S a, uint64_t b, Has has, Cl cl, Fin fin, Kind kind, uint64_t k2, uint64_t k4) {
  const T y = Raw<T>::get(b);
  const bool nod = has && (cl ? close_(y, Raw<T>::get(k2), Raw<T>::get(k4), fin) : y == Raw<T>::get(k2));
  To next = (To)y;
  if (kind == GM_RED_COUNT) {
    next = (To)(Raw<To>::get(a) + (To)1);
  } else if (kind != GM_RED_REPLACE) {
    if constexpr (IsFloat<To>::value) {
      const To old = Raw<To>::get(a);
      if (next != next) next = old;
      else if (old == old) {
        if (kind == GM_RED_MAX) next = next > old ? next : old;
        else if (kind == GM_RED_MIN) next = next < old ? next : old;
        else if (kind == GM_RED_SUM) next = old + next;
        else next = old * next;
      }
    }
  }
  return nod ? a : (S)Raw<To>::put(next);
}

// Reclassify (raster/misc.py:505-514): mapped -> target, else fill k3 (select) or astype(values).
// With ND_ONLY only the "result has data" boolean is produced (enough when the result merely masks
// another raster), which keeps the whole program in 32-bit slots.  The source sentinel (k1, fa)
// maps onto the fill.  A full result needs 64-bit slots: with 32-bit ones a is returned.
template <typename A, bool DENSE, bool ND_ONLY, typename S>
GM_DEV S reclass(S a, bool select, bool fa, bool out_f64, const int64_t* keys, const uint64_t* vals,
                 const uint8_t* hit, int n, int64_t base, uint64_t k1, uint64_t k3) {
  const int64_t key = (int64_t)Raw<A>::get(a);
  int found = 0;  // 0 miss, 1 mapped, 2 mapped onto the fill value
  uint64_t val = k3;
  if constexpr (DENSE) {
    const uint64_t idx = (uint64_t)(key - base);
    if (idx < (uint64_t)n) {
      found = hit[idx];
      if constexpr (!ND_ONLY) val = found ? vals[idx] : val;
    }
  } else {
    int lo = 0, hi = n;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (keys[mid] < key) lo = mid + 1; else hi = mid;
    }
    if (lo < n && keys[lo] == key) {
      found = hit ? hit[lo] : 1;
      if constexpr (!ND_ONLY) val = vals[lo];
    }
  }
  found = (fa && key == (int64_t)k1) ? 2 : found;
  if constexpr (ND_ONLY) {
    const unsigned lut = (select ? 0u : 1u) | 2u;  // result for [miss, mapped, mapped onto the fill]
    return (S)((lut >> found) & 1u);
  } else if constexpr (sizeof(S) == 8) {
    // unmapped cells keep astype(values): class A -> the (64-bit) target class
    const S keep = out_f64 ? (S)Raw<double>::put((double)Raw<A>::get(a)) : (S)Raw<int64_t>::put((int64_t)Raw<A>::get(a));
    return found ? (S)val : (select ? (S)k3 : keep);
  } else {
    return a;
  }
}

#endif  // GM_EVAL_OPS_CUH
