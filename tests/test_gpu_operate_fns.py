"""OperateOn with Base math functions and traced closures on the device (SIGOPS_OP_FN1 / FN2 / POPFN2), against the
CPU oracle, which calls the Python closure per sample.

Tolerances are BASELINE.json's (Float64 1e-9 of the RMS, Float32 1e-5); the exact functions (abs, sign, the roundings,
sqrt, clamp, min, max, copysign, rem, mod) must match bit for bit.  The `test_*` functions that take the `gpu` fixture
also run on the plan emulator (tests/test_operate_fns_emulated.py); the dispatch cases at the end need the device."""
import re

import numpy as np
import pytest

import oracle
from signalops import (Bandpass, Filt, GPUSink, Hz, Lowpass, Normpower, Operate, OperateOn, Signal, ToFramerate, Until, kHz, s,
                       sink, sink_batch)

pytestmark = pytest.mark.gpu

F64_TOL = 1e-9
F32_TOL = 1e-5


def rms(a):
    a = np.asarray(a, dtype=np.float64)
    return float(np.sqrt(np.mean(a ** 2))) if a.size else 0.0


def check(gpu, make, tol=F64_TOL, exact=False):
    want, fs = oracle.sink(make())
    got, fs2 = sink(make(), gpu)
    assert fs == fs2 and got.shape == want.shape and got.dtype == want.dtype
    if exact:
        assert np.array_equal(got, want, equal_nan=True)
    else:
        err = float(np.max(np.abs(got.astype(np.float64) - want.astype(np.float64)))) / max(rms(want), 1e-300)
        assert err <= tol, f"max err / rms = {err:g}"
    return got


def data(shape, dtype=np.float64, seed=7, kind="normal"):
    rng = np.random.default_rng(seed)
    if kind == "positive":
        x = rng.uniform(0.05, 4.0, shape)
    elif kind == "unit":
        x = rng.uniform(-0.95, 0.95, shape)
    else:
        x = 2.0 * rng.standard_normal(shape)
    if np.dtype(dtype).kind == "i":
        return np.round(8 * x).astype(dtype)
    return x.astype(dtype)


# (name, closure, input domain, exact)
UNARY = [
    ("abs", abs, "normal", True),
    ("sign", np.sign, "normal", True),
    ("floor", np.floor, "normal", True),
    ("ceil", np.ceil, "normal", True),
    ("trunc", np.trunc, "normal", True),
    ("round", np.rint, "normal", True),
    ("sqrt", np.sqrt, "positive", True),
    ("clamp", lambda v: np.clip(v, -1.0, 1.0), "normal", True),
    ("exp", np.exp, "normal", False),
    ("exp2", np.exp2, "normal", False),
    ("expm1", np.expm1, "normal", False),
    ("log", np.log, "positive", False),
    ("log2", np.log2, "positive", False),
    ("log10", np.log10, "positive", False),
    ("log1p", np.log1p, "positive", False),
    ("sin", np.sin, "normal", False),
    ("cos", np.cos, "normal", False),
    ("tan", np.tan, "unit", False),
    ("tanh", np.tanh, "normal", False),
    ("sinh", np.sinh, "normal", False),
    ("cosh", np.cosh, "normal", False),
    ("atan", np.arctan, "normal", False),
    ("cbrt", np.cbrt, "normal", False),
]
BINARY = [
    ("min", np.minimum, "normal", True),
    ("max", np.maximum, "normal", True),
    ("copysign", np.copysign, "normal", True),
    ("rem", np.fmod, "normal", True),
    ("mod", lambda a, b: a % b, "normal", True),
    ("pow", np.power, "positive", False),
    ("hypot", np.hypot, "normal", False),
]


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("name,f,dom,exact", UNARY, ids=[u[0] for u in UNARY])
def test_unary_function(gpu, name, f, dom, exact, dtype):
    x = data((3000, 2), dtype, kind=dom)
    tol = F64_TOL if dtype == np.float64 else F32_TOL
    check(gpu, lambda: OperateOn(f, Signal(x, 8 * kHz)), tol=tol, exact=exact)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("name,f,dom,exact", BINARY, ids=[b[0] for b in BINARY])
def test_binary_function(gpu, name, f, dom, exact, dtype):
    x, y = data((2500, 2), dtype, 1, dom), data((2500, 2), dtype, 2, dom)
    tol = F64_TOL if dtype == np.float64 else F32_TOL
    check(gpu, lambda: OperateOn(f, Signal(x, 8 * kHz), Signal(y, 8 * kHz)), tol=tol, exact=exact)
    # a constant on either side (FN2 on a CONST leaf, or PUSH ... POPFN2)
    check(gpu, lambda: OperateOn(lambda v: f(v, 0.75), Signal(x, 8 * kHz)), tol=tol, exact=exact)
    check(gpu, lambda: OperateOn(lambda v: f(1.5, v), Signal(x, 8 * kHz)), tol=tol, exact=exact)


@pytest.mark.parametrize("name,f", [("abs", abs), ("sign", np.sign), ("max", lambda v: np.maximum(v, 0)),
                                    ("min", lambda a: np.minimum(a, 3)), ("clip", lambda v: np.clip(v, -5, 5)),
                                    ("square", lambda v: v ** 2), ("affine", lambda v: 3 * v - 1)])
def test_int64_exact(gpu, name, f):
    x = data((2000, 2), np.int64)
    check(gpu, lambda: OperateOn(f, Signal(x, 8 * kHz)), exact=True)


def test_closure_with_shared_subexpressions(gpu):
    a, b, c = (data((4000, 2), seed=k) for k in (3, 4, 5))
    fs = 8 * kHz
    check(gpu, lambda: OperateOn(lambda u, v: np.tanh(u * v) + u * v - np.maximum(u, v), Signal(a, fs), Signal(b, fs)))
    check(gpu, lambda: OperateOn(lambda u, v, w: (u - v) / (1 + (u - v) ** 2) + np.hypot(w, u - v),
                                 Signal(a, fs), Signal(b, fs), Signal(c, fs)))
    check(gpu, lambda: OperateOn(lambda u: 1.0 / (1.0 + np.exp(-u)), Signal(a, fs)))
    check(gpu, lambda: OperateOn(lambda u: 2.0 - u, Signal(a, fs)), exact=True)


def test_argument_expressions_materialised_when_too_long(gpu):
    """An argument used many times that is an expression of its own: computed once into a temp, read back."""
    a, b = data((4000, 1), seed=6), data((4000, 1), seed=8)
    fs = 8 * kHz

    def make():
        u = OperateOn(lambda p, q: np.tanh(p) * np.cos(q) + np.sin(p * q) - np.abs(q), Signal(a, fs), Signal(b, fs))
        return OperateOn(lambda v: v * v * v * v * v * v + v * v * v * v * v - v * v * v + v, u)
    check(gpu, make)


def test_mid_side(gpu):
    x = data((6000, 2), seed=9)
    ms = lambda f: (0.5 * (f[0] + f[1]), 0.5 * (f[0] - f[1]))   # noqa: E731
    got = check(gpu, lambda: OperateOn(ms, Signal(x, 8 * kHz), bychannel=False), exact=True)
    assert np.array_equal(got[:, 1], 0.5 * (x[:, 0] - x[:, 1]))


def test_normpower_after_nonlinear_map(gpu):
    x = data((8000, 2), seed=10)
    check(gpu, lambda: OperateOn(np.tanh, Signal(x, 8 * kHz)) >> Normpower)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_functions_around_filters_and_resamplers(gpu, dtype):
    x = data((9600, 2), dtype, seed=11)
    tol = F64_TOL if dtype == np.float64 else F32_TOL
    fs = 48 * kHz
    check(gpu, lambda: OperateOn(abs, Signal(x, fs)) >> Filt(Lowpass, 50 * Hz), tol=tol)
    check(gpu, lambda: Signal(x, fs) >> Filt(Bandpass, 500 * Hz, 4 * kHz) >> Operate(np.tanh), tol=tol)
    check(gpu, lambda: OperateOn(lambda v: np.clip(v, -1, 1), Signal(x, fs)) >> Filt(Lowpass, 4 * kHz)
          >> Operate(lambda v: np.maximum(v, 0.0)), tol=tol)
    check(gpu, lambda: ToFramerate(Signal(x, fs), 44.1 * kHz) >> Operate(np.tanh), tol=tol)


# ---- dispatch: which kernel the planner picks (SIGOPS_DEBUG lines, as in test_gpu_dispatch.py) ----------------------

LINE = re.compile(r"^\[sigops\] (IIR|FIR) stage \d+: (.+?) rows=.*$", re.M)


@pytest.fixture
def fresh_sink(monkeypatch):
    monkeypatch.setenv("SIGOPS_DEBUG", "1")
    monkeypatch.setenv("SIGOPS_HOST_WAVES", "1")
    g = GPUSink([0])
    yield g
    g.close()


def iir_kernels(capfd):
    return [m.group(2) for m in LINE.finditer(capfd.readouterr().err) if m.group(1) == "IIR"]


def batch_parity(g, chain, xs):
    got = sink_batch([chain(x) for x in xs], g)
    for x, (y, _) in zip(xs, got):
        want, _ = oracle.sink(chain(x))
        assert np.max(np.abs(y - want)) <= F64_TOL * rms(want)
    return g.last_stats


@pytest.mark.parametrize("where", ["before", "after"])
def test_fused_function_stays_on_tensor_map_kernel(fresh_sink, capfd, where):
    """Full-wave rectification before the filter (an envelope follower's first half) or a soft clip (tanh after it) on a
    strided batch of 96 rows: one tensor-map launch with the function fused into its row-invariant programs."""
    rng = np.random.default_rng(12)
    xs = [np.asfortranarray(rng.standard_normal((48000, 32))) for _ in range(3)]
    if where == "before":
        chain = lambda x: OperateOn(abs, Signal(x, 48 * kHz)) >> Filt(Lowpass, 4 * kHz, order=8)   # noqa: E731
    else:
        chain = lambda x: Signal(x, 48 * kHz) >> Filt(Lowpass, 4 * kHz, order=8) >> Operate(np.tanh)   # noqa: E731
    stats = batch_parity(fresh_sink, chain, xs)
    assert iir_kernels(capfd) == ["tensor-map (fused row-invariant programs)"]
    assert stats["launches"] == 1


def test_max_of_two_buffers_takes_the_per_lane_path(fresh_sink, capfd):
    """An input program that reads two buffers has no tensor-map or TMA form: the per-lane generic kernel runs it."""
    rng = np.random.default_rng(13)
    xs = [np.asfortranarray(rng.standard_normal((24000, 32))) for _ in range(3)]
    ys = [np.asfortranarray(rng.standard_normal((24000, 32))) for _ in range(3)]

    def chain(xy):
        x, y = xy
        return OperateOn(np.maximum, Signal(x, 48 * kHz), Signal(y, 48 * kHz)) >> Filt(Lowpass, 4 * kHz)
    batch_parity(fresh_sink, chain, list(zip(xs, ys)))
    assert iir_kernels(capfd) == ["generic"]
