"""Compiler from element-wise block expressions to evaluator bytecode.

An expression is a DAG of ``Node`` objects over ``Leaf`` inputs (rasters that
are already materialised) and python/numpy scalars.  ``evaluate`` infers the
NumPy result dtypes and no data sentinels exactly as the reference blocks do
(raster/elemwise.py:134-152, :235-299; raster/misc.py; SURVEY.md Appendix B),
lowers the DAG to the accumulator machine of include/geokernels.h and runs it
in ONE CUDA launch through ``gm_eval_program``.
"""
import ctypes

import numpy as np

from .. import _native
from ..utils import get_dtype_max, get_uint_dtype, get_int_dtype

C_I32, C_I64, C_F32, C_F64 = 0, 1, 2, 3
_WIDE = (C_I64, C_F64)

# GmOp (order matters: it is the enum in include/gm_bytecode.h)
_OPS = [
    "LOAD", "ST", "OUT", "CVT", "ADD", "SUB", "RSUB", "MUL", "DIV", "RDIV", "POW", "RPOW",
    "EXP", "LOG", "LOG10", "EQ", "NE", "GT", "GE", "LT", "LE", "AND", "OR", "XOR", "NOT",
    "ISDATA", "ISNODATA", "OVERLAY", "CLIP", "MASK", "MASKBELOW", "STEP", "CLASSIFY", "RECLASS",
    "MATB",
]
OP = {name: i for i, name in enumerate(_OPS)}
SRC_NONE, SRC_REG, SRC_INPUT, SRC_IMM = 0, 1, 2, 3
F_ND_A, F_ND_B, F_CLOSE, F_ND_FINITE, F_B_BOOL, F_RIGHT, F_SELECT, F_ND_T = 1, 2, 4, 8, 16, 32, 64, 128
F_NAN = 32  # LOAD / MATB / CVT: sentinel -> NaN (shares the bit of F_RIGHT)

DENSE_TABLE_LIMIT = 4096
RED_KINDS = {"max": 1, "min": 2, "sum": 3, "product": 4, "count": 5}   # GmReduce


class FusionLimit(Exception):
    """The expression does not fit one program (registers, inputs, length)."""


class Leaf(object):
    def __init__(self, index):
        self.index = index


class Node(object):
    """``op`` applied to ``children`` (Leaf | Node | scalar) with literal ``params``."""

    def __init__(self, op, children, **params):
        self.op = op
        self.children = list(children)
        self.params = params


def dtype_class(dtype):
    dtype = np.dtype(dtype)
    if dtype == np.float32:
        return C_F32
    if dtype == np.float64:
        return C_F64
    if dtype in (np.dtype("u4"), np.dtype("i8")):
        return C_I64
    if dtype == bool or (dtype.kind in "iu" and dtype.itemsize <= 4):
        return C_I32
    raise TypeError("dtype '{}' is not supported by the CUDA raster path".format(dtype))


def _bits(value, cls):
    """Raw 64-bit pattern of ``value`` in class ``cls``."""
    if cls == C_I32:
        return int(value) & 0xFFFFFFFF
    if cls == C_I64:
        return int(value) & 0xFFFFFFFFFFFFFFFF
    with np.errstate(over="ignore"):
        if cls == C_F32:
            return int(np.array(value, dtype=np.float32).view(np.uint32))
        return int(np.array(value, dtype=np.float64).view(np.uint64))


def _is_scalar(x):
    return isinstance(x, (bool, int, float, np.generic))


def sentinel(dtype, nodata):
    """Value ``v`` such that ``values == nodata`` (NumPy semantics) is exactly
    ``values == v`` in ``dtype``; None when the comparison can never be true."""
    if nodata is None:
        return None
    dtype = np.dtype(dtype)
    try:
        if dtype == bool:
            return None
        if dtype.kind in "iu":
            if isinstance(nodata, (float, np.floating)) and not float(nodata).is_integer():
                return None
            v = int(nodata)
            info = np.iinfo(dtype)
            return v if info.min <= v <= info.max else None
        with np.errstate(over="ignore"):
            v = dtype.type(nodata)
        if np.isnan(v) or float(v) != float(nodata):
            return None
        return v
    except (TypeError, ValueError, OverflowError):
        return None


def _isclose_terms(dtype, nodata):
    """(compare dtype, y, tol, isfinite(y)) reproducing ``np.isclose(values, nodata)``
    term by term (numpy/_core/numeric.py isclose): ``abs(x - y) <= atol + rtol*abs(y)``."""
    y = nodata
    if isinstance(y, (bool, int)) and not isinstance(y, np.generic):
        y = float(y)
    elif isinstance(y, np.generic):
        y = np.asarray(y, dtype=np.result_type(y, 1.0))[()]
    probe = np.zeros(1, dtype=dtype)
    with np.errstate(all="ignore"):
        cmp_dtype = (probe - y).dtype
        rhs = 1e-8 + 1e-5 * abs(y)
        if isinstance(rhs, np.generic):
            cmp_dtype = np.result_type(cmp_dtype, rhs)
        tol = np.asarray(rhs).astype(cmp_dtype)[()]
        yy = np.asarray(y).astype(cmp_dtype)[()]
    return np.dtype(cmp_dtype), yy, tol, bool(np.isfinite(y))


def _cast_into(value, dtype):
    """What ``array[index] = value`` stores in an array of ``dtype``."""
    with np.errstate(all="ignore"):
        return np.asarray(value).astype(dtype)[()]


def _compare_dtype(dtypes_and_scalars):
    return np.result_type(*dtypes_and_scalars)


class _Typed(object):
    __slots__ = ("dtype", "nodata")

    def __init__(self, dtype, nodata):
        self.dtype = np.dtype(dtype)
        self.nodata = nodata

    @property
    def cls(self):
        return dtype_class(self.dtype)


_MATH = {"add": "ADD", "subtract": "SUB", "multiply": "MUL", "divide": "DIV", "power": "POW"}
_REVERSED = {"SUB": "RSUB", "DIV": "RDIV", "POW": "RPOW", "ADD": "ADD", "MUL": "MUL",
             "EQ": "EQ", "NE": "NE", "GT": "LT", "LT": "GT", "GE": "LE", "LE": "GE",
             "AND": "AND", "OR": "OR", "XOR": "XOR"}
_COMPARE = {"equal": "EQ", "not_equal": "NE", "greater": "GT", "greater_equal": "GE",
            "less": "LT", "less_equal": "LE"}
_LOGIC = {"logical_and": "AND", "logical_or": "OR", "logical_xor": "XOR"}
_UNARY_MATH = {"exp": "EXP", "log": "LOG", "log10": "LOG10"}


class _Compiler(object):
    """Lowers an expression DAG to the accumulator machine.

    ``word`` is the slot width the program is compiled for (4 or 8 bytes); a
    staged input can be used directly as the b operand of an instruction only
    when its storage already is a slot of the class the instruction computes in,
    otherwise it is first converted into a scratch register (MATB)."""

    def __init__(self, leaves, word=4):
        self.leaves = leaves  # list of _Typed for every input
        self.word = word
        self.instr = []
        self.tables = []      # dicts with numpy arrays (kept alive until launch)
        self.free_regs = list(range(_native.GM_NREG))
        self.uses = {}
        self.in_reg = {}      # id(node) -> (reg, _Typed)
        self.wide = False

    # -- helpers ---------------------------------------------------------------
    def emit(self, op, cls=C_I32, cls_a=C_I32, cls_b=C_I32, cls_out=C_I32, src=(SRC_NONE, 0),
             flags=0, aux=0, k=()):
        if len(self.instr) >= _native.GM_MAX_INSTR:
            raise FusionLimit("program too long")
        kk = [0] * 6
        for i, v in enumerate(k):
            kk[i] = v
        for c in (cls, cls_a, cls_out) + ((cls_b,) if src[0] != SRC_NONE else ()):
            if c in _WIDE:
                self.wide = True
        self.instr.append(dict(op=OP[op], cls=cls, cls_a=cls_a, cls_b=cls_b, cls_out=cls_out,
                               src_kind=src[0], src=src[1], flags=flags, aux=aux, k=kk))

    def count_uses(self, node):
        if not isinstance(node, Node):
            return
        self.uses[id(node)] = self.uses.get(id(node), 0) + 1
        if self.uses[id(node)] == 1:
            for c in node.children:
                self.count_uses(c)

    def alloc_reg(self):
        if not self.free_regs:
            raise FusionLimit("out of registers")
        return self.free_regs.pop(0)

    def free_reg(self, reg):
        self.free_regs.append(reg)
        self.free_regs.sort()

    def release(self, x):
        """Called once per consumed use of a node that lives in a register."""
        if isinstance(x, Node) and id(x) in self.in_reg:
            self.uses[id(x)] -= 1
            if self.uses[id(x)] <= 0:
                reg, _ = self.in_reg.pop(id(x))
                self.free_reg(reg)

    def is_complex(self, x):
        return isinstance(x, Node) and id(x) not in self.in_reg

    def to_acc(self, x):
        """Bring ``x`` into the accumulator in its own class.  Returns (typed, flags,
        k1): the sentinel test a consuming instruction has to do on acc."""
        if isinstance(x, Leaf):
            t = self.leaves[x.index]
            self.emit("LOAD", cls_b=t.cls, cls_out=t.cls, src=(SRC_INPUT, x.index))
        elif isinstance(x, Node):
            if id(x) in self.in_reg:
                reg, t = self.in_reg[id(x)]
                self.emit("LOAD", cls_b=t.cls, cls_out=t.cls, src=(SRC_REG, reg))
                self.release(x)
            else:
                t = self.node(x)
                if self.uses.get(id(x), 1) > 1:
                    reg = self.alloc_reg()
                    self.emit("ST", cls_a=t.cls, cls_out=t.cls, aux=reg)
                    self.in_reg[id(x)] = (reg, t)
                    self.release(x)
        else:
            raise TypeError("scalar cannot be the accumulator operand")
        s = sentinel(t.dtype, t.nodata)
        if s is None:
            return t, 0, 0
        return t, F_ND_A, _bits(s, t.cls)

    def acc_to_class(self, t, want):
        """Convert acc from the class of ``t`` to ``want``; returns the (flags, k1)
        sentinel test still to be done on the converted acc.  A sentinel entering a
        float class from another class becomes NaN (no test needed afterwards)."""
        s = sentinel(t.dtype, t.nodata)
        if t.cls == want:
            return (F_ND_A, _bits(s, want)) if s is not None else (0, 0)
        nanify = s is not None and want in (C_F32, C_F64)
        last = self.instr[-1] if self.instr else None
        if last is not None and last["op"] == OP["LOAD"] and last["src_kind"] in (SRC_INPUT, SRC_REG) \
                and last["cls_out"] == t.cls:
            # fold the conversion into the load that just produced acc
            last["cls_out"] = want
            if nanify:
                last["flags"] |= F_ND_B | F_NAN
                last["k"][2] = _bits(s, t.cls)
            if want in _WIDE:
                self.wide = True
        else:
            self.emit("CVT", cls_a=t.cls, cls_out=want, flags=(F_ND_A | F_NAN) if nanify else 0,
                      k=(0, _bits(s, t.cls) if nanify else 0))
        if s is not None and not nanify:
            return F_ND_A, _bits(s, want)   # injective integer widening
        return 0, 0

    def spill_to_reg(self, x):
        """Evaluate node ``x`` and park it in a register (if not there yet)."""
        if id(x) in self.in_reg:
            return
        t = self.node(x)
        reg = self.alloc_reg()
        self.emit("ST", cls_a=t.cls, cls_out=t.cls, aux=reg)
        self.in_reg[id(x)] = (reg, t)
        if self.uses.get(id(x), 1) <= 1:
            self.uses[id(x)] = 1

    def _direct(self, src, typed, want):
        """Can (src, typed) be read as a slot of class ``want`` without conversion?"""
        if typed.cls != want:
            return False
        if src[0] == SRC_REG:
            return True
        return typed.dtype.itemsize == self.word and typed.dtype != np.dtype("u4")

    def b_operand(self, x, want, nan_ok=True):
        """Make ``x`` available as operand b in class ``want``.  Returns
        (src, typed|None, k0, flags, k2, scratch register to free or None)."""
        if _is_scalar(x):
            return (SRC_IMM, 0), None, x, 0, 0, None
        if isinstance(x, Leaf):
            typed, src = self.leaves[x.index], (SRC_INPUT, x.index)
        else:
            reg, typed = self.in_reg[id(x)]
            src = (SRC_REG, reg)
        s = sentinel(typed.dtype, typed.nodata)
        if self._direct(src, typed, want):
            return src, typed, 0, (F_ND_B if s is not None else 0), (_bits(s, want) if s is not None else 0), None
        nanify = nan_ok and s is not None and want != typed.cls and want in (C_F32, C_F64)
        scratch = self.alloc_reg()
        self.emit("MATB", cls_b=typed.cls, cls_out=want, src=src, aux=scratch,
                  flags=(F_ND_B | F_NAN) if nanify else 0, k=(0, 0, _bits(s, typed.cls) if nanify else 0))
        flags, k2 = 0, 0
        if s is not None and not nanify:
            flags, k2 = F_ND_B, _bits(s, want)
        return (SRC_REG, scratch), typed, 0, flags, k2, scratch

    def order_operands(self, a, b):
        """Pick the accumulator operand; returns (a, b, swapped) with b no longer complex."""
        if _is_scalar(a) and _is_scalar(b):
            raise TypeError("at least one operand must be a raster")
        swapped = False
        if self.is_complex(a) and self.is_complex(b):
            self.spill_to_reg(b)
        elif self.is_complex(b) or _is_scalar(a):
            a, b, swapped = b, a, True
        return a, b, swapped

    def operand_type(self, x):
        if isinstance(x, Leaf):
            return self.leaves[x.index]
        if isinstance(x, Node) and id(x) in self.in_reg:
            return self.in_reg[id(x)][1]
        return None

    # -- per-op lowering -----------------------------------------------------------
    def node(self, n):
        handler = getattr(self, "op_" + n.op, None)
        if handler is None:
            if n.op in _MATH:
                return self.math(n)
            if n.op in _COMPARE:
                return self.compare(n)
            if n.op in _LOGIC:
                return self.logic(n)
            if n.op in _UNARY_MATH:
                return self.unary_math(n)
            raise NotImplementedError(n.op)
        return handler(n)

    def _binary(self, op, a, b, choose_class, out_cls, fill_bits, scalar_bits):
        """acc = op(a, b).  ``choose_class(ta, tb, scalar)`` picks the compute class
        once the accumulator operand has been evaluated (tb is None for a scalar b);
        ``fill_bits(T)`` / ``scalar_bits(v, T)`` encode the fill and an immediate."""
        a, b, swapped = self.order_operands(a, b)
        if swapped:
            op = _REVERSED[op]
        ta, _, _ = self.to_acc(a)
        tb = self.operand_type(b)
        T = choose_class(ta, tb, b if tb is None else None)
        fa, k1 = self.acc_to_class(ta, T)
        src, tb, k0, fb, k2, scratch = self.b_operand(b, T)
        if tb is None:
            k0 = scalar_bits(k0, T)
        self.emit(op, cls=T, cls_a=T, cls_b=T, cls_out=T if out_cls is None else out_cls, src=src,
                  flags=fa | fb, k=(k0, k1, k2, fill_bits(T)))
        if scratch is not None:
            self.free_reg(scratch)
        self.release(b)
        return T

    def math(self, n):
        dtype = np.dtype(n.params["dtype"])
        fill = n.params["fillvalue"]
        T = dtype_class(dtype)
        a, b = n.children
        if n.op == "power" and self._power_needs_mask(a, b, T):
            return self._masked_power(n, dtype, fill, T)

        def scalar_bits(v, cls):
            with np.errstate(all="ignore"):
                return _bits(np.asarray(v).astype(dtype)[()], cls)

        self._binary(_MATH[n.op], a, b, lambda ta, tb, sc: T, None, lambda cls: _bits(fill, cls),
                     scalar_bits)
        return _Typed(dtype, fill)

    def _needs_nan(self, x, T):
        t = self.operand_type(x)
        if t is None:
            return isinstance(x, Node)  # unknown until evaluated: be conservative
        return t.cls != T and sentinel(t.dtype, t.nodata) is not None

    def _power_needs_mask(self, a, b, T):
        # pow(NaN, 0) == pow(1, NaN) == 1: the sentinel -> NaN substitution used when an
        # operand changes class would leak through np.power
        if T not in (C_F32, C_F64):
            return False
        return any(not _is_scalar(x) and self._needs_nan(x, T) for x in (a, b))

    def _masked_power(self, n, dtype, fill, T):
        a, b = n.children
        if any(isinstance(x, Node) for x in (a, b)):
            raise FusionLimit("power with mixed operand classes is evaluated on its own")
        # validity mask of the raster operands, then the power on converted operands
        rasters = [x for x in (a, b) if isinstance(x, Leaf)]
        mask_reg = self.alloc_reg()
        for i, x in enumerate(rasters):
            t, fa, k1 = self.to_acc(x)
            self.emit("ISDATA", cls_a=t.cls, flags=fa, k=(0, k1))
            if i > 0:
                self.emit("AND", src=(SRC_REG, mask_reg))
            self.emit("ST", aux=mask_reg)

        def scalar_bits(v, cls):
            with np.errstate(all="ignore"):
                return _bits(np.asarray(v).astype(dtype)[()], cls)

        saved = [self.leaves[x.index] for x in rasters]
        try:
            for x in rasters:  # operands enter the power without sentinel handling
                self.leaves[x.index] = _Typed(saved[rasters.index(x)].dtype, None)
            self._binary(_MATH[n.op], a, b, lambda ta, tb, sc: T, None, lambda cls: _bits(fill, cls),
                         scalar_bits)
        finally:
            for x, t in zip(rasters, saved):
                self.leaves[x.index] = t
        self.emit("CLIP", cls_a=T, cls_b=C_I32, cls_out=T, src=(SRC_REG, mask_reg), flags=F_B_BOOL,
                  k=(0, _bits(fill, T)))
        self.free_reg(mask_reg)
        return _Typed(dtype, fill)

    def unary_math(self, n):
        dtype = np.dtype(n.params["dtype"])
        fill = n.params["fillvalue"]
        T = dtype_class(dtype)
        ta, _, _ = self.to_acc(n.children[0])
        fa, k1 = self.acc_to_class(ta, T)
        self.emit(_UNARY_MATH[n.op], cls=T, cls_a=T, cls_out=T, flags=fa, k=(0, k1, 0, _bits(fill, T)))
        return _Typed(dtype, fill)

    def compare(self, n):
        a, b = n.children

        def choose(ta, tb, scalar):
            # NumPy compares in the common type of both operands (python scalars are weak)
            T = dtype_class(_compare_dtype([ta.dtype, tb.dtype if tb is not None else scalar]))
            if T in (C_I32, C_I64):
                fits = scalar is None or -2 ** 31 <= int(scalar) < 2 ** 31
                narrow = ta.cls == C_I32 and (tb is None or tb.cls == C_I32)
                if T == C_I32 and not fits:
                    T = C_I64
                elif T == C_I64 and fits and narrow:
                    T = C_I32   # exact in 32 bits, keeps the program narrow
            return T

        fill = 1 if n.op == "not_equal" else 0
        self._binary(_COMPARE[n.op], a, b, choose, C_I32, lambda cls: fill,
                     lambda v, cls: _bits(int(v) if cls in (C_I32, C_I64) else v, cls))
        return _Typed(bool, None)

    def logic(self, n):
        a, b = n.children
        a, b, swapped = self.order_operands(a, b)
        self.to_acc(a)
        src, tb, k0, _, _, scratch = self.b_operand(b, C_I32)
        if tb is None:
            k0 = 1 if k0 else 0
        self.emit(_LOGIC[n.op], src=src, k=(k0,))
        if scratch is not None:
            self.free_reg(scratch)
        self.release(b)
        return _Typed(bool, None)

    def op_invert(self, n):
        self.to_acc(n.children[0])
        self.emit("NOT")
        return _Typed(bool, None)

    def _is_data(self, n, op):
        child = n.children[0]
        if isinstance(child, Node) and child.op == "reclassify" and self.uses.get(id(child), 1) <= 1:
            self.op_reclassify(child, nd_only=True)   # acc = "has data" boolean
            if op == "ISNODATA":
                self.emit("NOT")
            return _Typed(bool, None)
        t, fa, k1 = self.to_acc(child)
        self.emit(op, cls_a=t.cls, flags=fa, k=(0, k1))
        return _Typed(bool, None)

    def op_isdata(self, n):
        return self._is_data(n, "ISDATA")

    def op_isnodata(self, n):
        return self._is_data(n, "ISNODATA")

    def op_fillnodata(self, n):
        dtype = np.dtype(n.params["dtype"])
        fill = get_dtype_max(dtype)
        T = dtype_class(dtype)
        for c in n.children:
            if self.is_complex(c):
                self.spill_to_reg(c)
        self.emit("LOAD", cls_b=T, cls_out=T, src=(SRC_IMM, 0), k=(_bits(fill, T),))
        for c in n.children:
            tc = self.operand_type(c)
            flags, cmp_cls, k2, k4 = 0, tc.cls, 0, 0
            if tc.nodata is not None:
                if tc.dtype.kind == "f":
                    cmp_dtype, y, tol, fin = _isclose_terms(tc.dtype, tc.nodata)
                    cmp_cls = dtype_class(cmp_dtype)
                    flags = F_ND_T | F_CLOSE | (F_ND_FINITE if fin else 0)
                    k2, k4 = _bits(y, cmp_cls), _bits(tol, cmp_cls)
                else:
                    s = sentinel(tc.dtype, tc.nodata)
                    if s is not None:
                        flags, k2 = F_ND_T, _bits(s, cmp_cls)
            saved = None
            if isinstance(c, Leaf):  # the sentinel test happens inside OVERLAY, in cmp_cls
                saved, self.leaves[c.index] = self.leaves[c.index], _Typed(tc.dtype, None)
            try:
                src, _, _, _, _, scratch = self.b_operand(c, cmp_cls, nan_ok=False)
            finally:
                if saved is not None:
                    self.leaves[c.index] = saved
            self.emit("OVERLAY", cls=cmp_cls, cls_a=T, cls_b=cmp_cls, cls_out=T, src=src, flags=flags,
                      k=(0, 0, k2, 0, k4))
            if scratch is not None:
                self.free_reg(scratch)
            self.release(c)
        return _Typed(dtype, fill)

    def _overlay_operand(self, c):
        """Flags and constants of an OVERLAY step for child ``c`` (its has-data test is
        utils.get_index: np.isclose for floats, == otherwise): (typed, cmp class, flags, k2, k4)."""
        tc = self.operand_type(c)
        flags, cmp_cls, k2, k4 = 0, tc.cls, 0, 0
        if tc.nodata is not None:
            if tc.dtype.kind == "f":
                cmp_dtype, y, tol, fin = _isclose_terms(tc.dtype, tc.nodata)
                cmp_cls = dtype_class(cmp_dtype)
                flags = F_ND_T | F_CLOSE | (F_ND_FINITE if fin else 0)
                k2, k4 = _bits(y, cmp_cls), _bits(tol, cmp_cls)
            else:
                s = sentinel(tc.dtype, tc.nodata)
                if s is not None:
                    flags, k2 = F_ND_T, _bits(s, cmp_cls)
        return tc, cmp_cls, flags, k2, k4

    def op_reduce(self, n):
        """reduce_rasters (raster/reduction.py:38-119): 'last' / 'first' overlay the children,
        'count' counts those with data, 'max' / 'min' / 'sum' / 'product' reduce them in the
        float dtype NumPy's nan-functions would use (np.result_type(dtype, float16); a NaN
        accumulator means "no value yet") and cast the result back, all-'no data' cells -> fill."""
        p = n.params
        statistic = p["statistic"]
        dtype = np.dtype(p["dtype"])
        nodata = p["fillvalue"]
        T = dtype_class(dtype)
        children = list(n.children)
        if statistic == "first":
            children = children[::-1]
        for c in children:
            if self.is_complex(c):
                self.spill_to_reg(c)
        if statistic in ("last", "first"):
            kind, acc_dtype, init = 0, dtype, _cast_into(nodata, dtype)
        elif statistic == "count":
            kind, acc_dtype, init = RED_KINDS["count"], dtype, 0
        else:
            work = np.result_type(dtype, np.float16)
            if statistic in ("sum", "product") and work != dtype:
                raise NotImplementedError(
                    "reduce_rasters('{}') of {} rasters accumulates in {} on the CPU path; the CUDA path "
                    "reduces float32 / float64 rasters only".format(statistic, dtype, work))
            acc_dtype = np.dtype("f8") if work == np.float64 else np.dtype("f4")
            kind, init = RED_KINDS[statistic], float("nan")
        A = dtype_class(acc_dtype)
        self.emit("LOAD", cls_b=A, cls_out=A, src=(SRC_IMM, 0), k=(_bits(init, A),))
        for c in children:
            tc, cmp_cls, flags, k2, k4 = self._overlay_operand(c)
            saved = None
            if isinstance(c, Leaf):  # the sentinel test happens inside OVERLAY, in cmp_cls
                saved, self.leaves[c.index] = self.leaves[c.index], _Typed(tc.dtype, None)
            try:
                src, _, _, _, _, scratch = self.b_operand(c, cmp_cls, nan_ok=False)
            finally:
                if saved is not None:
                    self.leaves[c.index] = saved
            self.emit("OVERLAY", cls=cmp_cls, cls_a=A, cls_b=cmp_cls, cls_out=A, src=src, flags=flags,
                      aux=kind, k=(0, 0, k2, 0, k4))
            if scratch is not None:
                self.free_reg(scratch)
            self.release(c)
        if statistic in ("last", "first", "count"):
            return _Typed(dtype, nodata)
        # acc (float, NaN = every child was 'no data') -> out dtype, NaN cells -> fill
        fill = 0 if statistic == "sum" else nodata
        value_reg, mask_reg = self.alloc_reg(), self.alloc_reg()
        self.emit("ST", cls_a=A, cls_out=A, aux=value_reg)
        self.emit("EQ", cls=A, cls_a=A, cls_b=A, cls_out=C_I32, src=(SRC_REG, value_reg))   # NaN != NaN
        self.emit("ST", aux=mask_reg)
        self.emit("LOAD", cls_b=A, cls_out=A, src=(SRC_REG, value_reg))
        if A != T:
            self.emit("CVT", cls_a=A, cls_out=T)
        self.emit("CLIP", cls_a=T, cls_b=C_I32, cls_out=T, src=(SRC_REG, mask_reg), flags=F_B_BOOL,
                  k=(0, _bits(_cast_into(fill, dtype), T)))
        self.free_reg(value_reg)
        self.free_reg(mask_reg)
        return _Typed(dtype, nodata)

    def op_clip(self, n):
        store, mask = n.children
        mask_is_reclass = (isinstance(mask, Node) and mask.op == "reclassify"
                           and self.uses.get(id(mask), 1) <= 1 and id(mask) not in self.in_reg)
        if mask_is_reclass:
            self.op_reclassify(mask, nd_only=True)
            reg = self.alloc_reg()
            self.emit("ST", aux=reg)
            self.in_reg[id(mask)] = (reg, _Typed(bool, None))
            self.uses[id(mask)] = 1
        elif self.is_complex(mask):
            self.spill_to_reg(mask)
        ts, _, _ = self.to_acc(store)
        tm = self.operand_type(mask)
        saved = None
        if isinstance(mask, Leaf):  # CLIP tests the sentinel itself, in the mask's own class
            saved, self.leaves[mask.index] = self.leaves[mask.index], _Typed(tm.dtype, None)
        try:
            src, _, _, _, _, scratch = self.b_operand(mask, tm.cls, nan_ok=False)
        finally:
            if saved is not None:
                self.leaves[mask.index] = saved
        flags, k2 = 0, 0
        if tm.dtype == bool:
            flags = F_B_BOOL
        else:
            s = sentinel(tm.dtype, tm.nodata)
            if s is not None:
                flags, k2 = F_ND_B, _bits(s, tm.cls)
        nd = _cast_into(ts.nodata, ts.dtype) if ts.nodata is not None else 0
        self.emit("CLIP", cls_a=ts.cls, cls_b=tm.cls, cls_out=ts.cls, src=src, flags=flags,
                  k=(0, _bits(nd, ts.cls), k2))
        if scratch is not None:
            self.free_reg(scratch)
        self.release(mask)
        return _Typed(ts.dtype, ts.nodata)

    def op_mask(self, n):
        value = n.params["value"]
        if isinstance(value, float):
            out_dtype = np.dtype("float32")
        elif value >= 0:
            out_dtype = get_uint_dtype(value)
        else:
            out_dtype = get_int_dtype(value)
        fill = 1 if value == 0 else 0
        out_cls = dtype_class(out_dtype)
        ta, _, _ = self.to_acc(n.children[0])
        flags, cmp_cls, k1, k4 = 0, ta.cls, 0, 0
        if ta.nodata is not None:
            if ta.dtype.kind == "f":
                cmp_dtype, y, tol, fin = _isclose_terms(ta.dtype, ta.nodata)
                cmp_cls = dtype_class(cmp_dtype)
                flags = F_ND_T | F_CLOSE | (F_ND_FINITE if fin else 0)
                k1, k4 = _bits(y, cmp_cls), _bits(tol, cmp_cls)
            else:
                s = sentinel(ta.dtype, ta.nodata)
                if s is not None:
                    flags, k1 = F_ND_T, _bits(s, cmp_cls)
        self.emit("MASK", cls=cmp_cls, cls_a=ta.cls, cls_out=out_cls, flags=flags,
                  k=(_bits(_cast_into(value, out_dtype), out_cls), k1, 0,
                     _bits(_cast_into(fill, out_dtype), out_cls), k4))
        return _Typed(out_dtype, fill)

    def _scalar_compare_class(self, ta, value):
        T = dtype_class(_compare_dtype([ta.dtype, value]))
        if T == C_I32 and not (-2 ** 31 <= int(value) < 2 ** 31):
            T = C_I64
        return T

    def op_maskbelow(self, n):
        value = n.params["value"]
        ta, _, _ = self.to_acc(n.children[0])
        T = self._scalar_compare_class(ta, value)
        nd = _cast_into(ta.nodata, ta.dtype)
        self.emit("MASKBELOW", cls=T, cls_a=ta.cls, cls_out=ta.cls,
                  k=(_bits(value, T), 0, 0, 0, 0, _bits(nd, ta.cls)))
        return _Typed(ta.dtype, ta.nodata)

    def op_step(self, n):
        p = n.params
        ta, _, _ = self.to_acc(n.children[0])
        T = self._scalar_compare_class(ta, p["value"])
        s = sentinel(ta.dtype, ta.nodata)
        flags, k1 = (F_ND_A, _bits(s, ta.cls)) if s is not None else (0, 0)
        cast = lambda v: _bits(_cast_into(v, ta.dtype), ta.cls)  # noqa: E731
        self.emit("STEP", cls=T, cls_a=ta.cls, cls_out=ta.cls, flags=flags,
                  k=(_bits(p["value"], T), k1, cast(p["left"]), cast(p["at"]), cast(p["right"])))
        return _Typed(ta.dtype, ta.nodata)

    def op_classify(self, n):
        bins = np.asarray(n.params["bins"])
        out_dtype = get_uint_dtype(len(bins) + 2)
        fill = get_dtype_max(out_dtype)
        ta, _, _ = self.to_acc(n.children[0])
        small = ta.dtype == bool or (ta.dtype.kind in "iu" and ta.dtype.itemsize <= 2)
        if bins.dtype.kind in "iu" and ta.dtype.kind in "iub":
            fits = len(bins) == 0 or (bins.min() >= -2 ** 31 and bins.max() < 2 ** 31)
            T = C_I32 if (ta.cls == C_I32 and fits) else C_I64
            keys = bins.astype(np.int64)
            if T == C_I32:
                keys = keys.astype(np.int32).view(np.uint32).astype(np.uint64).view(np.int64)
        else:
            as32 = bins.astype(np.float32)
            exact32 = bool(np.all(as32.astype(np.float64) == bins.astype(np.float64)))
            if exact32 and (ta.dtype == np.float32 or small):
                T = C_F32   # identical ordering to the float64 comparison NumPy performs
                keys = as32.view(np.uint32).astype(np.uint64).view(np.int64)
            else:
                T = C_F64
                keys = bins.astype(np.float64).view(np.int64)
        table = dict(keys=np.ascontiguousarray(keys), vals=None, hit=None, base=0, n=len(bins), kind=0)
        self.tables.append(table)
        if len(self.tables) > _native.GM_MAX_TABLES:
            raise FusionLimit("too many tables")
        s = sentinel(ta.dtype, ta.nodata)
        flags, k1 = (F_ND_A, _bits(s, ta.cls)) if s is not None else (0, 0)
        if n.params["right"]:
            flags |= F_RIGHT
        self.emit("CLASSIFY", cls=T, cls_a=ta.cls, cls_out=C_I32, flags=flags, aux=len(self.tables) - 1,
                  k=(0, k1, 0, _bits(fill, C_I32)))
        return _Typed(out_dtype, fill)

    def op_reclassify(self, n, nd_only=False):
        p = n.params
        dtype = np.dtype(p["dtype"])
        fill = p["fillvalue"]
        pairs = p["data"]
        source = np.asarray([s for s, _ in pairs]).astype(np.int64)
        target = np.asarray([t for _, t in pairs]).astype(dtype)
        ta, _, _ = self.to_acc(n.children[0])
        # the source's own sentinel maps onto the fill unless the user mapped it
        # explicitly (raster/misc.py:495-497); it is tested by the instruction itself
        # so that a far-away sentinel does not blow up the dense table
        flags, k1 = 0, 0
        s = sentinel(ta.dtype, ta.nodata)
        if ta.nodata is not None and not np.any(source == ta.nodata) and s is not None:
            flags, k1 = F_ND_A, _bits(int(s), C_I64)
        order = np.argsort(source)
        source, target = source[order], target[order]
        T = dtype_class(dtype)
        with np.errstate(all="ignore"):
            is_fill = target == dtype.type(fill)
        hit = np.where(is_fill, 2, 1).astype(np.uint8)
        vals = target.view(np.uint64)
        span = int(source[-1] - source[0]) + 1 if len(source) else 0
        if 0 < span <= DENSE_TABLE_LIMIT:
            base = int(source[0])
            dense_vals = np.zeros(span, dtype=np.uint64)
            dense_hit = np.zeros(span, dtype=np.uint8)
            dense_vals[source - base] = vals
            dense_hit[source - base] = hit
            table = dict(keys=None, vals=None if nd_only else dense_vals, hit=dense_hit, base=base,
                         n=span, kind=1)
        else:
            table = dict(keys=np.ascontiguousarray(source), vals=np.ascontiguousarray(vals),
                         hit=np.ascontiguousarray(hit), base=0, n=len(source), kind=0)
        self.tables.append(table)
        if len(self.tables) > _native.GM_MAX_TABLES:
            raise FusionLimit("too many tables")
        flags |= (F_SELECT if p["select"] else 0) | (F_ND_T if nd_only else 0)
        out_cls = C_I32 if nd_only else T
        if not nd_only:
            self.wide = True
        self.emit("RECLASS", cls=C_I32 if nd_only else C_I64, cls_a=ta.cls, cls_out=out_cls, flags=flags,
                  aux=len(self.tables) - 1, k=(0, k1, 0, _bits(fill, T) if not nd_only else 0))
        return _Typed(bool, None) if nd_only else _Typed(dtype, fill)


_STORE_CODE = {}


def _build_program(compiler, n_inputs, n_outputs):
    prog = _native.GmProgram()
    prog.n_instr = len(compiler.instr)
    prog.n_inputs = n_inputs
    prog.n_outputs = n_outputs
    prog.word = 8 if compiler.wide else 4
    prog.n_tables = len(compiler.tables)
    for dst, src in zip(prog.instr, compiler.instr):
        for name in ("op", "cls", "cls_a", "cls_b", "cls_out", "src_kind", "src", "flags", "aux"):
            setattr(dst, name, src[name])
        for i in range(6):
            dst.k[i] = src["k"][i]
    for dst, t in zip(prog.tables, compiler.tables):
        dst.keys = t["keys"].ctypes.data if t["keys"] is not None else None
        dst.vals = t["vals"].ctypes.data if t["vals"] is not None else None
        dst.hit = t["hit"].ctypes.data if t["hit"] is not None else None
        dst.base, dst.n, dst.kind = t["base"], t["n"], t["kind"]
    return prog


def _compile(roots, leaf_types, word):
    comp = _Compiler([_Typed(d, nd) for d, nd in leaf_types], word)
    for r in roots:
        comp.count_uses(r)
    results = []
    for i, r in enumerate(roots):
        t, _, _ = comp.to_acc(r)
        results.append(t)
        comp.emit("OUT", cls_a=t.cls, cls_out=t.cls, aux=i)
    # inputs whose natural class is wide force the 64-bit machine
    if any(dtype_class(d) in _WIDE for d, _ in leaf_types):
        comp.wide = True
    return comp, results


def compile_expression(roots, leaf_types):
    """Lower ``roots`` (list of Node) to a GmProgram with one output per root.

    Returns (program, compiler, [result _Typed per root]).  The program is first
    compiled for 32-bit slots; if any class turns out to be 64-bit it is compiled
    again for 64-bit slots (operand directness depends on the slot width)."""
    if len(leaf_types) > _native.GM_MAX_INPUTS or len(roots) > _native.GM_MAX_OUTPUTS:
        raise FusionLimit("too many inputs/outputs")
    comp, results = _compile(roots, leaf_types, 4)
    if comp.wide:
        comp, results = _compile(roots, leaf_types, 8)
        comp.wide = True
    return _build_program(comp, len(leaf_types), len(roots)), comp, results


def run_program(prog, inputs, out_dtypes, shape, keep_on_device):
    """Launch ``prog`` over ``inputs`` (numpy or DeviceArray); returns the outputs."""
    lib = _native.lib()
    n = int(np.prod(shape, dtype=np.int64))
    in_desc = (_native.GmArray * max(len(inputs), 1))()
    staged = []
    any_device = keep_on_device or any(_native.is_device(a) for a in inputs)
    for i, a in enumerate(inputs):
        if not _native.is_device(a):
            a = np.ascontiguousarray(a)
            if any_device:
                a = _native.DeviceArray.from_host(a)
        staged.append(a)
        in_desc[i] = _native.as_gm_array(a, (1, 1, n))
    outputs = []
    out_desc = (_native.GmArray * len(out_dtypes))()
    for i, dt in enumerate(out_dtypes):
        out = _native.DeviceArray(shape, dt) if any_device else _native.pinned_empty(shape, dt)
        outputs.append(out)
        out_desc[i] = _native.as_gm_array(out, (1, 1, n))
    _native.check(lib.gm_eval_program(ctypes.byref(prog), in_desc, out_desc, n, _native.current_stream()))
    if any_device and not keep_on_device:
        outputs = [o.to_host() for o in outputs]
    return outputs


def evaluate(roots, leaves, keep_on_device=False, compiled=None):
    """Evaluate expression roots over ``leaves`` = [(values, no_data_value), ...].

    Returns [(values, dtype, no_data_value), ...] per root.  ``compiled`` = the result of an
    earlier ``compile_expression`` for the same roots and leaf types (see core/fusion.py).
    """
    shapes = [tuple(v.shape) for v, _ in leaves]
    shape = shapes[0]
    arrays = [v for v, _ in leaves]
    if any(s != shape for s in shapes):
        shape = np.broadcast_shapes(*shapes)
        arrays = [np.ascontiguousarray(np.broadcast_to(np.asarray(a), shape)) for a in arrays]
    if compiled is None:
        compiled = compile_expression(roots, [(v.dtype, nd) for v, nd in leaves])
    prog, comp, results = compiled
    outs = run_program(prog, arrays, [t.dtype for t in results], shape, keep_on_device)
    del comp  # tables stay alive until the (synchronous) upload inside the call is done
    return [(o, t.dtype, t.nodata) for o, t in zip(outs, results)]


class CompiledProgram(object):
    """A program compiled once and launched many times on device-resident
    arrays (what ``bench.py`` times; no host work besides the launch)."""

    def __init__(self, roots, leaf_types):
        self.program, self._compiler, self.results = compile_expression(roots, leaf_types)

    def launch(self, inputs, outputs):
        lib = _native.lib()
        n = inputs[0].size if inputs else outputs[0].size
        in_desc = (_native.GmArray * max(len(inputs), 1))()
        for i, a in enumerate(inputs):
            in_desc[i] = _native.as_gm_array(a, (1, 1, n))
        out_desc = (_native.GmArray * len(outputs))()
        for i, a in enumerate(outputs):
            out_desc[i] = _native.as_gm_array(a, (1, 1, n))
        _native.check(lib.gm_eval_program(ctypes.byref(self.program), in_desc, out_desc, n,
                                          _native.current_stream()))
