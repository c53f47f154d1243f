// Device-side building blocks of the specialised evaluator kernels.
//
// This file is NOT compiled by nvcc: build.py embeds it as a string in
// libgeokernels.so and gm_jit.cu prepends it to every kernel it generates from a
// GmProgram, which NVRTC then compiles for sm_100a (-fmad=false, IEEE div/sqrt).
// One function per bytecode instruction, operating on ONE pixel held in registers;
// every flag and class of the instruction is a template parameter and every
// constant a literal, so the generated kernel contains only the arithmetic of the
// fused blocks.  The semantics are those of the interpreter in gm_eval.cu (same
// reference citations: raster/elemwise.py:235-299, :551-638, :726-757 and
// raster/misc.py:98-123, :208-222, :245-251, :309-328, :387-399, :482-515).
//
// GM_WORD (4 or 8) is defined by the generator before this text.

typedef signed char int8_t;
typedef unsigned char uint8_t;
typedef short int16_t;
typedef unsigned short uint16_t;
typedef int int32_t;
typedef unsigned int uint32_t;
typedef long long int64_t;
typedef unsigned long long uint64_t;

#if GM_WORD == 8
typedef uint64_t S;
#else
typedef uint32_t S;
#endif

#define GM_DEV __device__ __forceinline__

template <typename A, typename B> struct Same { static constexpr bool value = false; };
template <typename A> struct Same<A, A> { static constexpr bool value = true; };
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

// ---- storage element -> slot of the input's natural class -------------------------
template <typename ST> GM_DEV S slot_of(ST v) { return (S)v; }
template <> GM_DEV S slot_of<int8_t>(int8_t v) { return (S)(uint32_t)(int32_t)v; }
template <> GM_DEV S slot_of<int16_t>(int16_t v) { return (S)(uint32_t)(int32_t)v; }
template <> GM_DEV S slot_of<int32_t>(int32_t v) { return (S)(uint32_t)v; }

// element J of a group of elements of type ST held in consecutive 32-bit words
template <typename ST, int J> GM_DEV S element(const uint32_t* w) {
  if constexpr (sizeof(ST) == 8) {
    return (S)((uint64_t)w[2 * J] | ((uint64_t)w[2 * J + 1] << 32));
  } else if constexpr (sizeof(ST) == 4) {
    return slot_of<ST>((ST)w[J]);
  } else if constexpr (sizeof(ST) == 2) {
    return slot_of<ST>((ST)(uint16_t)(w[J / 2] >> (16 * (J % 2))));
  } else {
    return slot_of<ST>((ST)(uint8_t)(w[J / 4] >> (8 * (J % 4))));
  }
}

// four 1-byte elements (truncating) as one 32-bit word, in one expression: the compiler merges the
// bytes with 3-input LOP3s (fewer instructions on cfg2 than set_element per byte or byte permutes)
GM_DEV uint32_t pack_bytes(S s0, S s1, S s2, S s3) {
  return ((uint32_t)s0 & 0xffu) | ((uint32_t)s1 & 0xffu) << 8 | ((uint32_t)s2 & 0xffu) << 16 |
         ((uint32_t)s3 & 0xffu) << 24;
}

// store slot `s` as element J (SZ bytes, truncating) of a group held in 32-bit words
template <int SZ, int J> GM_DEV void set_element(uint32_t* w, S s) {
  if constexpr (SZ == 8) {
    w[2 * J] = (uint32_t)(uint64_t)s;
    w[2 * J + 1] = (uint32_t)((uint64_t)s >> 32);
  } else if constexpr (SZ == 4) {
    w[J] = (uint32_t)s;
  } else if constexpr (SZ == 2) {
    if constexpr (J % 2 == 0) w[J / 2] = (uint32_t)s & 0xffffu;
    else w[J / 2] |= ((uint32_t)s & 0xffffu) << 16;
  } else {
    if constexpr (J % 4 == 0) w[J / 4] = (uint32_t)s & 0xffu;
    else w[J / 4] |= ((uint32_t)s & 0xffu) << (8 * (J % 4));
  }
}

// streaming loads / stores of 2, 4, 8 or 16 bytes (each byte is touched once)
template <int BYTES> GM_DEV void load_group(uint32_t* w, const void* p) {
  if constexpr (BYTES == 16) {
    const uint4 v = __ldcs(reinterpret_cast<const uint4*>(p));
    w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
  } else if constexpr (BYTES == 8) {
    const uint2 v = __ldcs(reinterpret_cast<const uint2*>(p));
    w[0] = v.x; w[1] = v.y;
  } else if constexpr (BYTES == 4) {
    w[0] = __ldcs(reinterpret_cast<const unsigned int*>(p));
  } else if constexpr (BYTES == 2) {
    w[0] = __ldcs(reinterpret_cast<const unsigned short*>(p));
  } else {
    w[0] = __ldcs(reinterpret_cast<const unsigned char*>(p));
  }
}
template <int BYTES> GM_DEV void store_group(void* p, const uint32_t* w) {
  if constexpr (BYTES == 16) {
    __stcs(reinterpret_cast<uint4*>(p), make_uint4(w[0], w[1], w[2], w[3]));
  } else if constexpr (BYTES == 8) {
    __stcs(reinterpret_cast<uint2*>(p), make_uint2(w[0], w[1]));
  } else if constexpr (BYTES == 4) {
    __stcs(reinterpret_cast<unsigned int*>(p), w[0]);
  } else if constexpr (BYTES == 2) {
    __stcs(reinterpret_cast<unsigned short*>(p), (unsigned short)w[0]);
  } else {
    __stcs(reinterpret_cast<unsigned char*>(p), (unsigned char)w[0]);
  }
}

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
template <typename T> GM_DEV T int_pow(T base, T e) {
  if (e < 0) return 0;
  T r = 1;
  while (e) {
    if (e & 1) r = w_mul(r, base);
    e >>= 1;
    if (e) base = w_mul(base, base);
  }
  return r;
}
GM_DEV float t_pow(float a, float b) { return powf(a, b); }
GM_DEV double t_pow(double a, double b) { return pow(a, b); }
GM_DEV float t_exp(float a) { return expf(a); }
GM_DEV double t_exp(double a) { return exp(a); }
GM_DEV float t_log(float a) { return logf(a); }
GM_DEV double t_log(double a) { return log(a); }
GM_DEV float t_log10(float a) { return log10f(a); }
GM_DEV double t_log10(double a) { return log10(a); }
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
enum {
  OP_LOAD = 0, OP_ST, OP_OUT, OP_CVT, OP_ADD, OP_SUB, OP_RSUB, OP_MUL, OP_DIV, OP_RDIV,
  OP_POW, OP_RPOW, OP_EXP, OP_LOG, OP_LOG10, OP_EQ, OP_NE, OP_GT, OP_GE, OP_LT, OP_LE,
  OP_AND, OP_OR, OP_XOR, OP_NOT, OP_ISDATA, OP_ISNODATA, OP_OVERLAY, OP_CLIP, OP_MASK,
  OP_MASKBELOW, OP_STEP, OP_CLASSIFY, OP_RECLASS, OP_MATB
};

// numpy astype From -> To; the sentinel becomes NaN when asked (float targets)
template <typename From, typename To, bool NANIFY> GM_DEV S cvt(S x, uint64_t k) {
  const From v = Raw<From>::get(x);
  To r = (To)v;
  if constexpr (IsFloat<To>::value && NANIFY) r = (v == Raw<From>::get(k)) ? quiet_nan<To>() : r;
  return (S)Raw<To>::put(r);
}

// binary arithmetic: invalid operands or a non-finite result -> fill
template <int OP, typename T, bool FA, bool FB>
GM_DEV S math(S a, uint64_t b, uint64_t k1, uint64_t k2, uint64_t k3) {
  const T x = Raw<T>::get(a), y = Raw<T>::get(b);
  T r;
  if constexpr (OP == OP_ADD) r = w_add(x, y);
  else if constexpr (OP == OP_SUB) r = w_sub(x, y);
  else if constexpr (OP == OP_RSUB) r = w_sub(y, x);
  else if constexpr (OP == OP_MUL) r = w_mul(x, y);
  else if constexpr (OP == OP_DIV) r = w_div(x, y);
  else if constexpr (OP == OP_RDIV) r = w_div(y, x);
  else if constexpr (OP == OP_POW) r = w_pow(x, y);
  else r = w_pow(y, x);
  bool bad = !finite_(r);
  if constexpr (FA) bad = bad || (x == Raw<T>::get(k1));
  if constexpr (FB) bad = bad || (y == Raw<T>::get(k2));
  return (S)Raw<T>::put(bad ? Raw<T>::get(k3) : r);
}

template <int OP, typename T, bool FA, bool FB>
GM_DEV S compare(S a, uint64_t b, uint64_t k1, uint64_t k2, uint64_t k3) {
  const T x = Raw<T>::get(a), y = Raw<T>::get(b);
  bool r;
  if constexpr (OP == OP_EQ) r = x == y;
  else if constexpr (OP == OP_NE) r = x != y;
  else if constexpr (OP == OP_GT) r = x > y;
  else if constexpr (OP == OP_GE) r = x >= y;
  else if constexpr (OP == OP_LT) r = x < y;
  else r = x <= y;
  bool bad = false;
  if constexpr (FA) bad = bad || (x == Raw<T>::get(k1));
  if constexpr (FB) bad = bad || (y == Raw<T>::get(k2));
  return bad ? (S)k3 : (S)(r ? 1u : 0u);
}

template <int OP, typename T, bool FA> GM_DEV S transcend(S a, uint64_t k1, uint64_t k3) {
  const T x = Raw<T>::get(a);
  const T r = OP == OP_EXP ? t_exp(x) : OP == OP_LOG ? t_log(x) : t_log10(x);
  bool bad = !finite_(r);
  if constexpr (FA) bad = bad || (x == Raw<T>::get(k1));
  return (S)Raw<T>::put(bad ? Raw<T>::get(k3) : r);
}

template <bool WANT_NODATA> GM_DEV S data_flag(bool is_nd) { return (S)((is_nd == WANT_NODATA) ? 1u : 0u); }

template <typename A, bool FA, bool WANT_NODATA> GM_DEV S is_data(S a, uint64_t k1) {
  bool is_nd = false;
  if constexpr (FA) is_nd = Raw<A>::get(a) == Raw<A>::get(k1);
  return data_flag<WANT_NODATA>(is_nd);
}

// What Step makes of each arm of its select.  `Id` keeps the value; `IsNd` is an IsData / IsNoData
// over Step's result folded into it (baked kernels only): it compares every arm with the no-data
// value instead of the selected one -- the same result, but the compare of a constant arm is a
// compare of two literals, which the compiler folds.
struct Id {
  GM_DEV S operator()(uint64_t v) const { return (S)v; }
};
template <typename C> struct IsNd {
  uint64_t nd;
  GM_DEV bool operator()(uint64_t v) const { return Raw<C>::get(v) == Raw<C>::get(nd); }
};

template <int OP> GM_DEV S logic(S a, uint64_t b) {
  const bool x = (uint32_t)a != 0u, y = (uint32_t)b != 0u;
  bool r;
  if constexpr (OP == OP_AND) r = x && y;
  else if constexpr (OP == OP_OR) r = x || y;
  else if constexpr (OP == OP_XOR) r = x != y;
  else r = !x;
  return (S)(r ? 1u : 0u);
}

// Clip: MODE 0 = no mask information, 1 = boolean mask, 2 = sentinel of class B
template <typename B, int MODE> GM_DEV S clip(S a, uint64_t b, uint64_t k1, uint64_t k2) {
  if constexpr (MODE == 1) return ((uint32_t)b == 0u) ? (S)k1 : a;
  else if constexpr (MODE == 2) return (Raw<B>::get(b) == Raw<B>::get(k2)) ? (S)k1 : a;
  else return a;
}

template <typename T, typename A, bool HAS, bool CL, bool FIN>
GM_DEV S mask(S a, uint64_t k0, uint64_t k1, uint64_t k3, uint64_t k4) {
  const T x = (T)Raw<A>::get(a);
  bool nod = false;
  if constexpr (HAS) {
    if constexpr (CL) nod = close_(x, Raw<T>::get(k1), Raw<T>::get(k4), FIN);
    else nod = x == Raw<T>::get(k1);
  }
  return nod ? (S)k3 : (S)k0;
}

template <typename T, typename A> GM_DEV S mask_below(S a, uint64_t k0, uint64_t k5) {
  return ((T)Raw<A>::get(a) < Raw<T>::get(k0)) ? (S)k5 : a;
}

template <typename T, typename A, bool FA, typename F = Id>
GM_DEV auto step(S a, uint64_t k0, uint64_t k1, uint64_t k2, uint64_t k3, uint64_t k4, F f = F()) {
  const A raw = Raw<A>::get(a);
  const T x = (T)raw, loc = Raw<T>::get(k0);
  auto r = f(a);
  r = x < loc ? f(k2) : r;
  r = x == loc ? f(k3) : r;
  r = x > loc ? f(k4) : r;
  if constexpr (FA) r = (raw == Raw<A>::get(k1)) ? f(a) : r;
  return r;
}

// np.digitize(values, bins, right), bins ascending
template <typename T, typename A, bool FA, bool RIGHT>
GM_DEV S classify(S a, const int64_t* keys, int n, uint64_t k1, uint64_t k3) {
  const A raw = Raw<A>::get(a);
  const T x = (T)raw;
  int lo = 0, hi = n;
  if (x != x) lo = n;  // NaN sorts last
  else
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      const T e = Raw<T>::get((uint64_t)keys[mid]);
      const bool go = RIGHT ? (e < x) : (e <= x);
      if (go) lo = mid + 1; else hi = mid;
    }
  if constexpr (FA) return (raw == Raw<A>::get(k1)) ? (S)k3 : (S)(uint32_t)lo;
  return (S)(uint32_t)lo;
}

// FillNoData step: acc = isdata(b) ? astype(b) : acc; KIND != 0: the reducing forms of
// reduce_rasters (1 max, 2 min, 3 sum, 4 product over a float class with NaN = no value yet,
// 5 count)
template <typename T, typename To, bool HAS, bool CL, bool FIN, int KIND>
GM_DEV S overlay(S a, uint64_t b, uint64_t k2, uint64_t k4) {
  const T y = Raw<T>::get(b);
  bool nod = false;
  if constexpr (HAS) {
    if constexpr (CL) nod = close_(y, Raw<T>::get(k2), Raw<T>::get(k4), FIN);
    else nod = y == Raw<T>::get(k2);
  }
  To next = (To)y;
  if constexpr (KIND == 5) {
    next = (To)(Raw<To>::get(a) + (To)1);
  } else if constexpr (KIND != 0) {
    const To old = Raw<To>::get(a);
    if (next != next) next = old;
    else if (old == old) {
      if constexpr (KIND == 1) next = next > old ? next : old;
      else if constexpr (KIND == 2) next = next < old ? next : old;
      else if constexpr (KIND == 3) next = old + next;
      else next = old * next;
    }
  }
  return nod ? a : (S)Raw<To>::put(next);
}

// Reclassify.  found: 0 miss, 1 mapped, 2 mapped onto the fill value
template <typename A, bool DENSE, bool ND_ONLY, bool SELECT, bool FA, bool OUT_F64>
GM_DEV S reclass(S a, const int64_t* keys, const uint64_t* vals, const uint8_t* hit, int n,
                 int64_t base, uint64_t k1, uint64_t k3) {
  const int64_t key = (int64_t)Raw<A>::get(a);
  int found = 0;
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
  if constexpr (FA) found = (key == (int64_t)k1) ? 2 : found;
  if constexpr (ND_ONLY) {
    const unsigned lut = (SELECT ? 0u : 1u) | 2u;
    return (S)((lut >> found) & 1u);
  } else {
#if GM_WORD == 8
    S keep;
    if constexpr (OUT_F64) keep = (S)Raw<double>::put((double)Raw<A>::get(a));
    else keep = (S)Raw<int64_t>::put((int64_t)Raw<A>::get(a));
    return found ? (S)val : (SELECT ? (S)k3 : keep);
#else
    return a;
#endif
  }
}

// Reclassify, ND_ONLY, through a dense table of at most 64 entries of an I32 key, held as the two
// 32-bit words lo:hi.  Their bit i is the result for key base + i, (lut >> hit[i]) & 1 with the lut
// of reclass (the generator folds it in); a key outside the table is found = 0, the sentinel
// found = 2.  [base, base + n) lies inside int32, so one unsigned compare of the 32-bit difference
// is the range test of reclass.
template <bool SELECT, bool FA>
GM_DEV S reclass_bits(S a, uint32_t lo, uint32_t hi, uint32_t n, int32_t base, uint64_t k1) {
  const unsigned lut = (SELECT ? 0u : 1u) | 2u;
  const int32_t key = Raw<int32_t>::get(a);
  const uint32_t idx = (uint32_t)key - (uint32_t)base;
  const uint32_t w = idx < 32u ? lo : hi;
  unsigned r = idx < n ? (w >> (idx & 31u)) & 1u : lut & 1u;
  // key == k1 as int64: a sentinel outside int32 never matches (uniform, or folded when baked)
  if constexpr (FA) r = (key == (int32_t)k1 && (int64_t)k1 == (int64_t)(int32_t)k1) ? (lut >> 2) & 1u : r;
  return (S)r;
}
