/*
 * gm_bytecode.h -- the instruction set of the fused element-wise evaluator (GmProgram in
 * geokernels.h): value classes, opcodes, reduction kinds, operand sources, flags and table kinds.
 *
 * It depends on nothing, so that the device code NVRTC compiles for the specialised kernels can
 * take these definitions as they are (build.py splices this file into that text).
 */
#ifndef GM_BYTECODE_H
#define GM_BYTECODE_H

/* ---- value classes the evaluator computes in ----------------------------- */
enum GmClass { GM_C_I32 = 0, GM_C_I64 = 1, GM_C_F32 = 2, GM_C_F64 = 3 };

/* One accumulator + GM_NREG registers per pixel; every instruction is
 * acc = op(acc, b) where b is a register, an input pixel or an immediate.
 * Arithmetic and comparison instructions are homogeneous: acc and b already
 * hold class `cls` (the compiler inserts CVT / MATB conversions); b may come
 * straight from an input only when the input's storage is a slot of that class.
 * Sentinel ("no data") semantics are evaluated exactly as the reference does
 * between blocks: raster/elemwise.py:235-299 (math/compare/logic),
 * :551-638 (Invert/IsData/IsNoData), :726-757 (FillNoData);
 * raster/misc.py:98-123 (Clip) :208-222 (Mask) :245-251 (MaskBelow)
 * :309-328 (Step) :387-399 (Classify) :482-515 (Reclassify).
 */
enum GmOp {
  GM_OP_LOAD = 0,   /* acc = convert(b: cls_b -> cls_out)                   */
  GM_OP_ST,         /* reg[aux] = acc                                       */
  GM_OP_OUT,        /* out[aux][pixel] = acc                                */
  GM_OP_CVT,        /* acc: cls_a -> cls_out (numpy astype)                 */
  GM_OP_ADD, GM_OP_SUB, GM_OP_RSUB, GM_OP_MUL, GM_OP_DIV, GM_OP_RDIV,
  GM_OP_POW, GM_OP_RPOW,
  GM_OP_EXP, GM_OP_LOG, GM_OP_LOG10,
  GM_OP_EQ, GM_OP_NE, GM_OP_GT, GM_OP_GE, GM_OP_LT, GM_OP_LE,
  GM_OP_AND, GM_OP_OR, GM_OP_XOR, GM_OP_NOT,
  GM_OP_ISDATA, GM_OP_ISNODATA,
  GM_OP_OVERLAY,    /* FillNoData step: acc = isdata(b) ? b : acc; with aux = a
                       GmReduce kind the step reduces instead (reduce_rasters,
                       raster/reduction.py:38-119): acc = isdata(b) ? red(acc, b) : acc */
  GM_OP_CLIP,       /* acc = masked(b) ? k1 : acc                           */
  GM_OP_MASK,       /* acc = isnodata(acc) ? k3 : k0                        */
  GM_OP_MASKBELOW,  /* acc = acc < k0 ? k1 : acc                            */
  GM_OP_STEP,       /* left/at/right around k0                              */
  GM_OP_CLASSIFY,   /* np.digitize against table aux                        */
  GM_OP_RECLASS,    /* sorted/dense table lookup, table aux                 */
  GM_OP_MATB,       /* reg[aux] = convert(b: cls_b -> cls_out), acc untouched */
  GM_OP_COUNT_
};

/* reduction kinds of GM_OP_OVERLAY (aux): max / min / sum / product keep acc in a float class
 * where NaN means "no value yet" and skip NaN cells like np.nanmax etc.; count adds one        */
enum GmReduce { GM_RED_REPLACE = 0, GM_RED_MAX = 1, GM_RED_MIN = 2, GM_RED_SUM = 3, GM_RED_PRODUCT = 4,
                GM_RED_COUNT = 5 };

enum GmSrcKind { GM_SRC_NONE = 0, GM_SRC_REG = 1, GM_SRC_INPUT = 2, GM_SRC_IMM = 3 };

enum GmFlags {
  GM_F_ND_A      = 1,   /* k1 holds the sentinel of acc (class cls_a)       */
  GM_F_ND_B      = 2,   /* k2 holds the sentinel of b   (class cls_b)       */
  GM_F_CLOSE     = 4,   /* float sentinel test is np.isclose, k4 = tol      */
  GM_F_ND_FINITE = 8,   /* isfinite(sentinel) (term of np.isclose)          */
  GM_F_B_BOOL    = 16,  /* Clip: b is a boolean mask                        */
  GM_F_RIGHT     = 32,  /* Classify: right=True                             */
  GM_F_SELECT    = 64,  /* Reclassify: select=True                          */
  GM_F_ND_T      = 128, /* Mask/Overlay: sentinel given in class `cls` (k1/k2);
                           Reclassify: produce only the is-data boolean     */
  GM_F_NAN       = 32   /* LOAD/MATB/CVT to a float class: the sentinel (k2 for
                           b, k1 for acc) converts to NaN, so that the typed
                           op that follows needs no sentinel test of its own */
};

enum GmTableKind { GM_TABLE_SORTED = 0, GM_TABLE_DENSE = 1 };

#endif /* GM_BYTECODE_H */
