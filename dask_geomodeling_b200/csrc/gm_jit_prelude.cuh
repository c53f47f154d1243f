// Device-side building blocks of the specialised evaluator kernels.
//
// This file is NOT compiled by nvcc: build.py embeds it as a string in libgeokernels.so, with
// gm_eval_ops.cuh and gm_bytecode.h spliced in where they are included, and gm_jit.cu prepends it
// to every kernel it generates from a GmProgram, which NVRTC then compiles for sm_100a
// (-fmad=false, IEEE div/sqrt).  What each instruction does to a pixel is defined in
// gm_eval_ops.cuh, shared with the interpreter; the generator calls those functions with every
// class and flag of the instruction as a template argument or literal and every constant a
// literal, so the generated kernel contains only the arithmetic of the fused blocks.  This file
// adds what only generated code needs: moving pixels between memory and slots, and the register
// bit tables of Reclassify.
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

#define GM_OUTLINE __device__ __forceinline__
#include "gm_eval_ops.cuh"

// a flag or kind as a compile-time constant, for the functions that deduce its type (Mask, Overlay)
template <int V> struct Lit {
  constexpr operator int() const { return V; }
};

#if GM_WORD == 8
typedef uint64_t S;
#else
typedef uint32_t S;
#endif

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

// An IsData / IsNoData over Step's result folded into the Step (baked kernels only): used as Step's
// arm functor, it compares every arm with the no-data value instead of the selected one -- the same
// result, but the compare of a constant arm is a compare of two literals, which the compiler folds.
template <typename C> struct IsNd {
  uint64_t nd;
  GM_DEV bool operator()(uint64_t v) const { return Raw<C>::get(v) == Raw<C>::get(nd); }
};

// Reclassify, ND_ONLY, through a dense table of at most 64 entries of an I32 key, held as the two
// 32-bit words lo:hi.  Their bit i is the result for key base + i, (lut >> hit[i]) & 1 with the lut
// of reclass (the generator folds it in); a key outside the table is found = 0, the sentinel
// found = 2.  [base, base + n) lies inside int32, so one unsigned compare of the 32-bit difference
// is the range test of reclass.
GM_DEV S reclass_bits(S a, bool select, bool fa, uint32_t lo, uint32_t hi, uint32_t n, int32_t base, uint64_t k1) {
  const unsigned lut = (select ? 0u : 1u) | 2u;
  const int32_t key = Raw<int32_t>::get(a);
  const uint32_t idx = (uint32_t)key - (uint32_t)base;
  const uint32_t w = idx < 32u ? lo : hi;
  unsigned r = idx < n ? (w >> (idx & 31u)) & 1u : lut & 1u;
  // key == k1 as int64: a sentinel outside int32 never matches (uniform, or folded when baked)
  if (fa) r = (key == (int32_t)k1 && (int64_t)k1 == (int64_t)(int32_t)k1) ? (lut >> 2) & 1u : r;
  return (S)r;
}
