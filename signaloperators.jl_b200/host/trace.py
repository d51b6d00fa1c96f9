"""Tracing of `OperateOn` closures into expression DAGs the GPU sink can lower.

`OperateOn(fn, xs...)` (src/mapsignal.jl:131-145) applies an arbitrary function per sample.  The GPU sink
cannot run Python, so `fn` is called once, on the host, with `Sym` tracer values in place of samples: one per
argument, or one tuple of `Sym` per argument (one entry per channel) when `bychannel=False`.  What comes back is
a DAG over the arguments and Float64 constants, which host/lowering.py turns into a device program.

Supported: `+ - * / %`, unary `-` and `+`, `**`, `abs()`, `round(x)`, `math.floor/ceil/trunc`, the numpy ufuncs
of `UNARY` / `BINARY` below (`np.tanh(x)`, `np.maximum(x, 0)`, ...), and `np.clip(x, lo, hi)` with constant
bounds.  Anything that needs the VALUE of a sample on the host raises a `TraceError` naming the construct:
branching (`if x > 0`, `and`/`or`), comparisons, the builtin `min`/`max` (they compare), and conversions to a
Python number (`float(x)`, `math.sqrt(x)` and the other `math` functions).
"""
from __future__ import annotations

import numpy as np


class TraceError(TypeError):
    """The closure does something a traced sample cannot stand for."""


# numpy ufunc -> function name of the device (include/signalops.h SIGOPS_EFN_*), or an arithmetic operator
UNARY = {np.absolute: "abs", np.fabs: "abs", np.sign: "sign", np.floor: "floor", np.ceil: "ceil", np.trunc: "trunc",
         np.rint: "round", np.sqrt: "sqrt", np.exp: "exp", np.exp2: "exp2", np.expm1: "expm1",
         np.log: "log", np.log2: "log2", np.log10: "log10", np.log1p: "log1p", np.sin: "sin", np.cos: "cos",
         np.tan: "tan", np.tanh: "tanh", np.sinh: "sinh", np.cosh: "cosh", np.arctan: "atan", np.cbrt: "cbrt",
         np.negative: "neg", np.positive: "pos", np.square: "square", np.reciprocal: "reciprocal"}
BINARY = {np.add: "+", np.subtract: "-", np.multiply: "*", np.divide: "/", np.minimum: "min", np.maximum: "max",
          np.copysign: "copysign", np.fmod: "rem", np.remainder: "mod", np.power: "pow", np.hypot: "hypot"}


class Node:
    """One operation of the traced expression.  kind: "arg" (key = argument index, or (argument, channel)),
    "const" (value), or a function / operator name with its operands in `args`."""
    __slots__ = ("kind", "args", "value", "key")

    def __init__(self, kind, args=(), value=None, key=None):
        self.kind, self.args, self.value, self.key = kind, tuple(args), value, key

    def __repr__(self):
        if self.kind == "arg":
            return f"arg{self.key}"
        if self.kind == "const":
            return repr(self.value)
        return f"{self.kind}({', '.join(map(repr, self.args))})"


def _node(v, what):
    if isinstance(v, Sym):
        return v.node
    if isinstance(v, (bool, np.bool_)):
        raise TraceError(f"a boolean operand in {what}")
    if isinstance(v, (int, float, np.integer, np.floating)):
        return Node("const", value=float(v))
    raise TraceError(f"operand {v!r} of {what} is neither a traced sample nor a number")


def _sym(kind, *args, value=None):
    return Sym(Node(kind, [_node(a, kind) for a in args], value=value))


def _refuse(construct):
    def f(self, *a, **k):
        raise TraceError(f"{construct} on a traced sample: the GPU sink compiles the closure once for all samples, "
                         "so it cannot depend on a sample's value")
    return f


class Sym:
    """A traced sample.  Operations build the expression; anything that needs a concrete value raises."""
    __slots__ = ("node",)
    __array_priority__ = 1000

    def __init__(self, node):
        self.node = node

    # arithmetic
    def __add__(self, o): return _sym("+", self, o)
    def __radd__(self, o): return _sym("+", o, self)
    def __sub__(self, o): return _sym("-", self, o)
    def __rsub__(self, o): return _sym("-", o, self)
    def __mul__(self, o): return _sym("*", self, o)
    def __rmul__(self, o): return _sym("*", o, self)
    def __truediv__(self, o): return _sym("/", self, o)
    def __rtruediv__(self, o): return _sym("/", o, self)
    def __mod__(self, o): return _sym("mod", self, o)        # Python's float % is Julia's mod
    def __rmod__(self, o): return _sym("mod", o, self)
    def __neg__(self): return _sym("neg", self)
    def __pos__(self): return self
    def __abs__(self): return _sym("abs", self)
    def __floor__(self): return _sym("floor", self)
    def __ceil__(self): return _sym("ceil", self)
    def __trunc__(self): return _sym("trunc", self)

    def __round__(self, ndigits=None):
        if ndigits is not None:
            raise TraceError("round(x, ndigits) on a traced sample (only round(x) is supported)")
        return _sym("round", self)

    def __pow__(self, o):
        # an integer literal 2 is x*x (Julia's `literal_pow`); other exponents are pow
        if isinstance(o, (int, np.integer)) and not isinstance(o, bool) and o == 2:
            return _sym("*", self, self)
        return _sym("pow", self, o)

    def __rpow__(self, o): return _sym("pow", o, self)

    def clip(self, lo=None, hi=None, out=None, **kw):
        """np.clip(x, lo, hi): Julia's clamp(x, lo, hi) with constant bounds."""
        if out is not None or kw:
            raise TraceError("np.clip with out= or other options on a traced sample")
        if isinstance(lo, Sym) or isinstance(hi, Sym):
            raise TraceError("np.clip with traced bounds (only constant bounds are supported)")
        lo = -np.inf if lo is None else float(lo)
        hi = np.inf if hi is None else float(hi)
        return Sym(Node("clamp", [self.node], value=(lo, hi)))

    def __array_ufunc__(self, ufunc, method, *inputs, **kw):
        if method != "__call__" or kw:
            raise TraceError(f"numpy ufunc {ufunc.__name__}.{method} with options on a traced sample")
        if ufunc in UNARY:
            name = UNARY[ufunc]
            (x,) = inputs
            if name == "pos":
                return x
            if name == "square":
                return _sym("*", x, x)
            if name == "reciprocal":
                return _sym("/", 1.0, x)
            return _sym(name, x)
        if ufunc in BINARY:
            a, b = inputs
            if BINARY[ufunc] == "pow" and not isinstance(b, Sym):
                return a.__pow__(b)
            return _sym(BINARY[ufunc], a, b)
        raise TraceError(f"numpy function {ufunc.__name__} is not supported on traced samples")

    # everything that needs a value
    __bool__ = _refuse("branching (`if`, `while`, `and`, `or`, a conditional expression)")
    __lt__ = __le__ = __gt__ = __ge__ = _refuse("a comparison (`<`, `>`, ... or the builtin min/max)")
    __eq__ = __ne__ = _refuse("a comparison (`==`, `!=`)")
    __float__ = __int__ = __index__ = __complex__ = _refuse(
        "a conversion to a Python number (float(), int(), math.sqrt and the other math functions)")
    __floordiv__ = __rfloordiv__ = _refuse("`//` (floor division)")
    __hash__ = object.__hash__

    def __repr__(self):
        return f"Sym({self.node!r})"


def _unpack(v, n_out, what):
    if n_out is None:
        if isinstance(v, (tuple, list)):
            raise TraceError(f"{what} returned {len(v)} values per sample")
        return _node(v, what)
    vs = tuple(v) if isinstance(v, (tuple, list)) else (v,)
    if len(vs) != n_out:
        raise TraceError(f"{what} returned {len(vs)} channels, expected {n_out}")
    return tuple(_node(e, what) for e in vs)


def same(a, b):
    """Whether two traced expressions are the same expression (constants compared bit for bit)."""
    return (a.kind == b.kind and a.key == b.key and repr(a.value) == repr(b.value) and len(a.args) == len(b.args)
            and all(same(p, q) for p, q in zip(a.args, b.args)))


def trace_generator(fn, nchannels):
    """Call the generator closure of `Signal(fn, ...)` on one tracer value standing for its argument (the phase or the
    time of a frame) and return one Node per channel.  Raises whatever `fn` raises on a tracer: a TraceError for what
    a traced sample cannot stand for, or any other error of a closure that needs a number."""
    name = getattr(fn, "__name__", repr(fn))
    return _unpack(fn(Sym(Node("arg", key=0))), nchannels, f"Signal({name})")


def trace(fn, nargs, channels=None):
    """Call `fn` on tracer values.  bychannel (channels is None): one Sym per argument, returns one Node.  Otherwise
    `channels[k]` channels of argument k arrive as a tuple of Sym, and a tuple of Nodes (one per output channel) is
    returned.  Raises TraceError when `fn` does something a traced sample cannot stand for."""
    name = getattr(fn, "__name__", repr(fn))
    if channels is None:
        args = [Sym(Node("arg", key=k)) for k in range(nargs)]
        return _unpack(fn(*args), None, f"OperateOn({name})")
    args = [tuple(Sym(Node("arg", key=(k, c))) for c in range(nc)) for k, nc in enumerate(channels)]
    v = fn(*args)
    return _unpack(v, len(v) if isinstance(v, (tuple, list)) else 1, f"OperateOn({name})")
