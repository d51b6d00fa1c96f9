"""Generator functions the device can evaluate (the `Functor` hook of
src/functions.jl:65-66,88): Julia closures cannot cross a C ABI, so the GPU sink
recognises an enumerated set, traces other closures into device programs
(host/trace.py, host/lowering.py) and materialises the rest on the host."""
from __future__ import annotations

import math

import numpy as np

from . import graph as G

FN_SIN, FN_COS, FN_SAW, FN_AFFINE_SIN, FN_AFFINE_COS, FN_IDENTITY = 1, 2, 3, 4, 5, 6


class Sawtooth(G.Functor):
    """README sound3: `ϕ -> ϕ/π - 1`"""

    def __call__(self, phi):
        return phi / math.pi - 1


class AffineSin(G.Functor):
    """README sound4: `ϕ -> 0.5sin(ϕ) + 0.5` generalised to a*sin(ϕ)+b"""

    def __init__(self, a=0.5, b=0.5):
        self.a, self.b = float(a), float(b)

    def __call__(self, phi):
        return self.a * math.sin(phi) + self.b


class AffineCos(G.Functor):
    def __init__(self, a=0.5, b=0.5):
        self.a, self.b = float(a), float(b)

    def __call__(self, phi):
        return self.a * math.cos(phi) + self.b


def is_sin(fn):
    """Stands in for dispatch on `typeof(sin)` (src/functions.jl:57-60)."""
    return fn is G.sin or fn is math.sin or fn is np.sin


def functor_code(fn):
    if is_sin(fn):
        return FN_SIN, 0.0, 0.0
    if fn is G.cos or fn is math.cos or fn is np.cos:
        return FN_COS, 0.0, 0.0
    if fn is G.identity:
        return FN_IDENTITY, 0.0, 0.0
    if isinstance(fn, Sawtooth):
        return FN_SAW, 0.0, 0.0
    if isinstance(fn, AffineSin):
        return FN_AFFINE_SIN, fn.a, fn.b
    if isinstance(fn, AffineCos):
        return FN_AFFINE_COS, fn.a, fn.b
    return None


def _const(nd, value=None):
    return nd.kind == "const" and (value is None or nd.value == value)


def _arg(nd):
    return nd.kind == "arg"


def _scaled(nd, fn):
    """`a*fn(arg)` or `fn(arg)*a` -> a; `fn(arg)` -> 1."""
    if nd.kind == fn and _arg(nd.args[0]):
        return 1.0
    if nd.kind == "*":
        p, q = nd.args
        if _const(p) and q.kind == fn and _arg(q.args[0]):
            return p.value
        if _const(q) and p.kind == fn and _arg(p.args[0]):
            return q.value
    return None


def generator_shape(nd):
    """(code, a, b) of the device generator a traced generator expression (host/trace.py) is exactly, or None.  Only
    rewrites that keep every bit are taken: `a*sin(arg) + b` evaluates as the device's `a*sin(x) + b` in any operand
    order of `+` and `*`, and `- b` as `+ (-b)`.  `sin(arg)` is AFFINE_SIN(1, 0), not FN_SIN, which is the `sinpi`
    form of the builtin `sin` only (src/functions.jl:57-60)."""
    if _arg(nd):
        return FN_IDENTITY, 0.0, 0.0
    if nd.kind == "-" and _const(nd.args[1], 1.0) and nd.args[0].kind == "/":
        p, q = nd.args[0].args
        if _arg(p) and _const(q, math.pi):
            return FN_SAW, 0.0, 0.0
    if nd.kind == "cos" and _arg(nd.args[0]):
        return FN_COS, 0.0, 0.0
    if nd.kind == "sin" and _arg(nd.args[0]):
        return FN_AFFINE_SIN, 1.0, 0.0
    if nd.kind in ("+", "-"):
        p, q = nd.args
        if nd.kind == "+" and _const(p):
            p, q = q, p
        if _const(q):
            b = q.value if nd.kind == "+" else -q.value
            for fn, code in (("sin", FN_AFFINE_SIN), ("cos", FN_AFFINE_COS)):
                a = _scaled(p, fn)
                if a is not None:
                    return code, a, b
    return None
