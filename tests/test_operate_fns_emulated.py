"""CPU check of traced OperateOn closures: the parity cases of test_gpu_operate_fns.py lowered to plan bytes and run on
the plan emulator (tests/plan_emulator.py, with the closure functions of tests/plan_emulator_fns.py) against the
oracle, plus the tracer itself (which closures trace, what is refused and how), Julia's NaN and signed-zero rules of
min / max / clamp, and the programs of the existing operator chains."""
import math
import operator

import numpy as np
import pytest

import test_gpu_operate_fns as T
from plan_emulator_fns import EmulatedFnsSink, efn
from signalops import (AddChannel, Amplify, Filt, Hz, Lowpass, Mix, Operate, OperateOn, Signal, ToChannels, kHz, sink)
from signalops.graph import reverse
from signalops import lowering as L
from signalops.lowering import LoweringError, lower
from signalops.trace import TraceError, trace


@pytest.fixture(scope="module")
def gpu():
    return EmulatedFnsSink()


for _name in dir(T):
    if _name.startswith("test_") and "fresh_sink" not in getattr(T, _name).__code__.co_varnames:
        globals()[_name] = getattr(T, _name)


def ops(chain):
    return [(I.op, I.leaf, I.fn) for st in lower(chain).stages for prog in [p.prog for p in st.pieces] +
            [st.in_prog, st.epi_prog] for I in prog]


X = np.zeros((64, 2))


# ---- the tracer -------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("f,expect", [
    (abs, "abs(arg0)"),
    (np.tanh, "tanh(arg0)"),
    (math.floor, "floor(arg0)"),
    (round, "round(arg0)"),
    (lambda v: np.clip(v, -1, 1), "clamp(arg0)"),
    (lambda v: v ** 2, "*(arg0, arg0)"),
    (lambda v: v ** 3, "pow(arg0, 3.0)"),
    (lambda v: 2 - v, "-(2.0, arg0)"),
    (lambda v: v % 1.5, "mod(arg0, 1.5)"),
    (lambda v: np.maximum(v, 0), "max(arg0, 0.0)"),
    (lambda v: -np.square(v), "neg(*(arg0, arg0))"),
])
def test_closures_that_trace(f, expect):
    assert repr(trace(f, 1)) == expect


def test_whole_frame_closure_traces_per_channel():
    ms = trace(lambda f: (0.5 * (f[0] + f[1]), 0.5 * (f[0] - f[1])), 1, [2])
    assert [repr(n) for n in ms] == ["*(0.5, +(arg(0, 0), arg(0, 1)))", "*(0.5, -(arg(0, 0), arg(0, 1)))"]


@pytest.mark.parametrize("f,needle", [
    (lambda v: v if v > 0 else -v, "comparison"),
    (lambda v: 1.0 if v else 0.0, "branching"),
    (lambda v: max(v, 0.0), "builtin min/max"),
    (lambda v: min(v, 1.0), "builtin min/max"),
    (lambda v: math.sqrt(v), "math.sqrt"),
    (lambda v: float(v) * 2, "float()"),
    (lambda v: v // 2, "floor division"),
    (lambda v: np.greater(v, 0), "greater"),
])
def test_refused_constructs_are_named(f, needle):
    with pytest.raises(TraceError, match=needle.replace("(", r"\(").replace(")", r"\)")):
        trace(f, 1)
    with pytest.raises(LoweringError, match=needle.replace("(", r"\(").replace(")", r"\)")):
        lower(OperateOn(f, Signal(X, 10 * Hz)))


# ---- Julia's corner cases (numpy's minimum / maximum / clip differ at the signed zeros) ---------------------------

NAN, INF = float("nan"), float("inf")


def same(a, b):
    return (math.isnan(a) and math.isnan(b)) or (a == b and math.copysign(1, a) == math.copysign(1, b))


@pytest.mark.parametrize("a,b,lo,hi", [
    (-0.0, 0.0, -0.0, 0.0), (0.0, -0.0, -0.0, 0.0), (NAN, 1.0, NAN, NAN), (1.0, NAN, NAN, NAN),
    (-INF, 2.0, -INF, 2.0), (3.0, 2.0, 2.0, 3.0), (-0.0, -0.0, -0.0, -0.0)])
def test_min_max_are_julias(a, b, lo, hi):
    assert same(float(efn(L.EFN["min"], a, b)), lo)
    assert same(float(efn(L.EFN["max"], a, b)), hi)


@pytest.mark.parametrize("x,lo,hi,want", [
    (NAN, -1.0, 1.0, NAN), (-0.0, 0.0, 1.0, -0.0), (0.0, -1.0, -0.0, 0.0), (2.0, -1.0, 1.0, 1.0), (-2.0, -1.0, 1.0, -1.0)])
def test_clamp_is_julias(x, lo, hi, want):
    assert same(float(efn(L.EFN["clamp"], x, lo, hi)), want)


@pytest.mark.parametrize("f,args,want", [
    ("sign", (-0.0,), -0.0), ("sign", (NAN,), NAN), ("round", (2.5,), 2.0), ("round", (-0.5,), -0.0),
    ("mod", (-1.0, 3.0), 2.0), ("mod", (3.0, -2.0), -1.0), ("mod", (-3.0, 3.0), 0.0), ("mod", (3.0, -3.0), -0.0),
    ("rem", (-1.0, 3.0), -1.0), ("sqrt", (-1.0,), NAN), ("log", (-1.0,), NAN), ("pow", (-2.0, 0.5), NAN)])
def test_exact_corners(f, args, want):
    assert same(float(efn(L.EFN[f], *args)), want)


def test_device_results_at_the_corners(gpu):
    """Through the lowering and the emulated device: Julia's values, not numpy's, at signed zeros and NaNs."""
    a = np.array([[-0.0], [0.0], [NAN], [1.0], [-0.0]])
    b = np.array([[0.0], [-0.0], [1.0], [NAN], [-0.0]])
    got, _ = sink(OperateOn(np.minimum, Signal(a, 10 * Hz), Signal(b, 10 * Hz)), gpu)
    assert all(same(g, w) for g, w in zip(got[:, 0], [-0.0, -0.0, NAN, NAN, -0.0]))
    got, _ = sink(OperateOn(np.maximum, Signal(a, 10 * Hz), Signal(b, 10 * Hz)), gpu)
    assert all(same(g, w) for g, w in zip(got[:, 0], [0.0, 0.0, NAN, NAN, -0.0]))
    got, _ = sink(OperateOn(lambda v: np.clip(v, 0.0, 1.0), Signal(a, 10 * Hz)), gpu)
    assert all(same(g, w) for g, w in zip(got[:, 0], [-0.0, 0.0, NAN, 1.0, -0.0]))


# ---- lowering -----------------------------------------------------------------------------------------------------

def test_existing_operator_chains_keep_their_programs():
    """Arithmetic operators, reverse and the channel functions do not go through the tracer."""
    x = Signal(X, 10 * Hz)
    for chain in (Mix(x, x), Amplify(x, 2), OperateOn(operator.sub, x, 1), OperateOn(operator.neg, x),
                  OperateOn(operator.truediv, x, 3), OperateOn(reverse, x, bychannel=False), AddChannel(x, x) >> ToChannels(1)):
        assert all(op < L.OP_FN1 for op, _, _ in ops(chain))


def test_programs_of_traced_closures():
    x = Signal(X, 10 * Hz)
    B, C = L.LEAF_BUF, L.LEAF_CONST
    assert ops(OperateOn(abs, x)) == [(L.OP_LOAD, B, 0), (L.OP_FN1, 0, L.EFN["abs"])]
    assert ops(OperateOn(lambda v: 2 - v, x)) == [(L.OP_LOAD, C, 0), (L.OP_SUB, B, 0)]
    assert ops(OperateOn(lambda v: 2 - np.tanh(v), x)) == [(L.OP_LOAD, B, 0), (L.OP_FN1, 0, L.EFN["tanh"]),
                                                           (L.OP_NEG, 0, 0), (L.OP_ADD, C, 0)]
    assert ops(OperateOn(lambda v: 2 / v, x)) == [(L.OP_LOAD, C, 0), (L.OP_DIV, B, 0)]
    assert ops(OperateOn(lambda v: 2 / abs(v), x)) == [(L.OP_LOAD, C, 0), (L.OP_PUSH, 0, 0), (L.OP_LOAD, B, 0),
                                                       (L.OP_FN1, 0, L.EFN["abs"]), (L.OP_POPDIV, 0, 0)]
    assert ops(OperateOn(lambda v: np.maximum(0, v), x)) == [(L.OP_LOAD, B, 0), (L.OP_FN2, C, L.EFN["max"])]
    assert ops(OperateOn(lambda v: 3 * v + 1, x)) == [(L.OP_LOAD, B, 0), (L.OP_MUL, C, 0), (L.OP_ADD, C, 0)]
    assert ops(OperateOn(lambda v: v ** 2, x)) == [(L.OP_LOAD, B, 0), (L.OP_MUL, B, 0)]
    # Float32: rounded after every operation, constants meet the samples as Float32
    x32 = Signal(X.astype(np.float32), 10 * Hz)
    p = lower(OperateOn(lambda v: np.tanh(v * 0.1), x32)).stages[0].pieces[0].prog
    assert [I.op for I in p] == [L.OP_LOAD, L.OP_MUL, L.OP_CAST_F32, L.OP_FN1, L.OP_CAST_F32]
    assert p[1].d0 == float(np.float32(0.1))
    # Int64 results end with the integer conversion
    p = lower(OperateOn(abs, Signal(X.astype(np.int64), 10 * Hz))).stages[0].pieces[0].prog
    assert [I.op for I in p] == [L.OP_LOAD, L.OP_FN1, L.OP_CAST_I64]


def test_generator_operand_of_a_function_goes_through_the_stack():
    from signalops import sin, Until, s
    g = Signal(sin, 10 * Hz, ω=1 * Hz) >> Until(6.4 * s)
    assert ops(OperateOn(np.copysign, Signal(X, 10 * Hz), g)) == [
        (L.OP_LOAD, L.LEAF_BUF, 0), (L.OP_PUSH, 0, 0), (L.OP_LOAD, L.LEAF_GEN, L.FN_SIN), (L.OP_POPFN2, 0, L.EFN["copysign"])]
    # min / max swap their operands (exact) to keep the buffer as the leaf
    assert ops(OperateOn(np.minimum, Signal(X, 10 * Hz), g)) == [(L.OP_LOAD, L.LEAF_GEN, L.FN_SIN),
                                                                 (L.OP_FN2, L.LEAF_BUF, L.EFN["min"])]


def test_functions_fuse_into_filter_programs():
    x = Signal(np.zeros((4800, 2)), 48 * kHz)
    st = lower(OperateOn(abs, x) >> Filt(Lowpass, 4 * kHz) >> Operate(np.tanh)).stages
    assert len(st) == 1 and st[0].kind == L.STAGE_IIR
    assert [I.op for I in st[0].in_prog] == [L.OP_LOAD, L.OP_FN1]
    assert [(I.op, I.leaf) for I in st[0].epi_prog] == [(L.OP_LOAD, L.LEAF_STAGE), (L.OP_FN1, 0)]


def test_too_long_expression_is_refused():
    x = Signal(X, 10 * Hz)
    with pytest.raises(LoweringError, match="more than"):
        lower(OperateOn(lambda v: sum([np.tanh(v * k) for k in range(1, 40)], v), x))
