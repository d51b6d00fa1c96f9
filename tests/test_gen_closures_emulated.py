"""CPU check of traced generator closures: the parity cases of test_gpu_gen_closures.py lowered to plan bytes and run on
the plan emulator against the oracle, plus what the lowering emits (the enumerated generator shapes, what stays on the
host and why, the fallbacks over the device limits, batches)."""
import math
import os
import sys

import numpy as np
import pytest

import test_gpu_gen_closures as T
from plan_emulator_fns import EmulatedFnsSink
from signalops import Amplify, Filt, Hz, Lowpass, Mix, Signal, Until, kHz, s, sin, sink_batch
from signalops import lowering as L
from signalops.functors import FN_AFFINE_COS, FN_AFFINE_SIN, FN_COS, FN_IDENTITY, FN_SAW, generator_shape
from signalops.gpusink import _build_prefix
from signalops.lowering import Lowerer, lower
from signalops.trace import trace_generator

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden", "plans"))
import make_plans  # noqa: E402


@pytest.fixture(scope="module")
def gpu():
    return EmulatedFnsSink()


for _name in dir(T):
    if _name.startswith("test_") and not {"fresh_sink", "monkeypatch"} & set(getattr(T, _name).__code__.co_varnames):
        globals()[_name] = getattr(T, _name)


def leaves(x):
    """(op, leaf, fn) of every instruction of every program of the plan of `x`, and its number of input buffers."""
    p = lower(x)
    return [(I.op, I.leaf, I.fn) for st in p.stages for prog in [q.prog for q in st.pieces] + [st.in_prog, st.epi_prog]
            for I in prog], len(p.inputs)


def gen(f, **kw):
    return Signal(f, 8 * kHz, **kw) >> Until(0.1 * s)


# ---- the enumerated shapes ------------------------------------------------------------------------------------------

@pytest.mark.parametrize("f,shape", [
    (lambda p: p, (FN_IDENTITY, 0.0, 0.0)),
    (lambda p: p / np.pi - 1, (FN_SAW, 0.0, 0.0)),
    (lambda p: p / math.pi - 1, (FN_SAW, 0.0, 0.0)),
    (np.cos, (FN_COS, 0.0, 0.0)),
    (lambda p: np.cos(p), (FN_COS, 0.0, 0.0)),
    (lambda p: np.sin(p), (FN_AFFINE_SIN, 1.0, 0.0)),
    (lambda p: 0.5 * np.sin(p) + 0.5, (FN_AFFINE_SIN, 0.5, 0.5)),
    (lambda p: np.sin(p) * 0.5 + 0.5, (FN_AFFINE_SIN, 0.5, 0.5)),
    (lambda p: 0.25 + 0.5 * np.sin(p), (FN_AFFINE_SIN, 0.5, 0.25)),
    (lambda p: 0.25 + np.sin(p) * 0.5, (FN_AFFINE_SIN, 0.5, 0.25)),
    (lambda p: 2 * np.sin(p) - 0.125, (FN_AFFINE_SIN, 2.0, -0.125)),
    (lambda p: np.sin(p) + 3, (FN_AFFINE_SIN, 1.0, 3.0)),
    (lambda p: 0.5 * np.cos(p) + 0.5, (FN_AFFINE_COS, 0.5, 0.5)),
    (lambda p: 0.1 + np.cos(p) * -2, (FN_AFFINE_COS, -2.0, 0.1)),
    (lambda p: np.cos(p) * 3 - 1, (FN_AFFINE_COS, 3.0, -1.0)),
])
def test_enumerated_shapes(f, shape):
    assert generator_shape(trace_generator(f, 1)[0]) == shape
    ops, n_in = leaves(gen(f, ω=10 * Hz))
    assert n_in == 0 and ops == [(L.OP_LOAD, L.LEAF_GEN, shape[0])]


@pytest.mark.parametrize("f", [lambda p: 0.5 * np.sin(2 * p) + 0.5, lambda p: np.sin(p) / 2, lambda p: 2 - np.cos(p),
                               lambda p: p / np.pi - 2, lambda p: 0.5 * np.sin(p) * 0.5 + 1, lambda p: np.sin(p + 1)])
def test_other_expressions_are_programs(f):
    assert generator_shape(trace_generator(f, 1)[0]) is None
    ops, n_in = leaves(gen(f, ω=10 * Hz))
    assert n_in == 0 and len(ops) > 1 and ops[0] == (L.OP_LOAD, L.LEAF_GEN, FN_IDENTITY)


def test_generator_argument():
    """The argument is the FN_IDENTITY generator leaf: 2π((k/fs·ω + ϕ) % 1) with ω, k/fs + ϕ without."""
    p = lower(Signal(lambda p: np.tanh(p), 8 * kHz, ω=10 * Hz, phi=np.pi / 2) >> Until(0.1 * s))
    I = p.stages[0].pieces[0].prog[0]
    assert (I.leaf, I.fn, I.flags, I.i0, I.d0, I.d1, I.d2) == (L.LEAF_GEN, FN_IDENTITY, L.FLAG_HAS_OMEGA, 1, 8000.0, 10.0, 0.25)
    p = lower(Signal(lambda t: np.tanh(t), 8 * kHz) >> Until(0.1 * s))
    I = p.stages[0].pieces[0].prog[0]
    assert (I.leaf, I.fn, I.flags, I.d0, I.d2) == (L.LEAF_GEN, FN_IDENTITY, 0, 8000.0, 0.0)


def test_tuple_generator_gives_one_piece_per_channel():
    p = lower(Signal(lambda p: (np.sin(p), np.tanh(p)), 8 * kHz, ω=10 * Hz) >> Until(0.1 * s))
    assert not p.inputs
    pcs = p.stages[-1].pieces
    assert [(q.clo, q.chi) for q in pcs] == [(0, 1), (1, 2)]
    assert pcs[0].prog == [L._gen_leaf(Signal(np.sin, 8 * kHz, ω=10 * Hz), 0, FN_AFFINE_SIN, 1.0, 0.0)]


def test_float32_rounds_after_every_operation_and_integers_cast():
    ops, _ = leaves(gen(lambda p: np.sin(np.float32(2) * p), ω=10 * Hz))
    assert ops == [(L.OP_LOAD, L.LEAF_GEN, FN_IDENTITY), (L.OP_MUL, L.LEAF_CONST, 0), (L.OP_CAST_F32, 0, 0),
                   (L.OP_FN1, 0, L.EFN["sin"]), (L.OP_CAST_F32, 0, 0)]
    ops, _ = leaves(gen(lambda p: round(10 * p), ω=10 * Hz))
    assert ops[-2:] == [(L.OP_FN1, 0, L.EFN["round"]), (L.OP_CAST_I64, 0, 0)]


# ---- what stays on the host -------------------------------------------------------------------------------------------

def host_evaluated(x):
    ops, n_in = leaves(x)
    return n_in == 1 and ops == [(L.OP_LOAD, L.LEAF_BUF, 0)]


def test_impure_closures_stay_on_the_host(gpu):
    rng = np.random.default_rng(3)
    assert host_evaluated(gen(lambda p: np.sin(p) + 0.01 * rng.standard_normal(), ω=10 * Hz))
    assert host_evaluated(gen(lambda _: rng.uniform(-1, 1), ω=10 * Hz))
    assert host_evaluated(gen(lambda _: 0.5, ω=10 * Hz))


@pytest.mark.parametrize("f", [lambda p: 1.0 if p < math.pi else -1.0, lambda p: math.sin(p), lambda p: min(p, 1.0),
                               lambda p: float(p) * 2, lambda p: np.sin(p).item()],
                         ids=["comparison", "math.sin", "min", "float", "attribute"])
def test_refused_closures_stay_on_the_host(gpu, f):
    assert host_evaluated(gen(f, ω=10 * Hz))
    T.check(gpu, lambda: gen(f, ω=10 * Hz))


def many_partials(p):
    return sum((0.1 / k) * np.sin(k * p) for k in range(1, 14))


def test_expression_over_the_program_limit_stays_on_the_host(gpu):
    assert host_evaluated(gen(many_partials, ω=10 * Hz))
    T.check(gpu, lambda: gen(many_partials, ω=10 * Hz))


def test_long_program_around_a_generator_materialises_it(gpu):
    """A generator program that fits alone, inside a mix that then exceeds MAX_PROG: it is computed into a temp by a
    MAP stage of its own, the mix reads it back as a buffer."""
    f = lambda p: sum((0.1 / k) * np.sin(k * p) for k in range(1, 8))   # noqa: E731
    x = np.random.default_rng(4).standard_normal((800, 1))

    def make():
        return Mix(*[Signal(x * (k + 1), 8 * kHz) for k in range(8)], Signal(f, 8 * kHz, ω=10 * Hz)) >> Until(0.1 * s)
    p = lower(make())
    assert len(p.inputs) == 8 and len(p.temps) == 1 and len(p.stages) == 2
    T.check(gpu, make)
    # the same through sink!'s prefix lowering
    p = _build_prefix(Lowerer(), make(), 800, np.float64)
    assert len(p.inputs) == 8 and len(p.temps) == 1 and len(p.stages) == 2


# ---- the README closures give the committed plan bytes -----------------------------------------------------------------

@pytest.mark.parametrize("name", ["cfg4", "cfg5"])
def test_readme_closures_lower_to_committed_bytes(monkeypatch, name):
    monkeypatch.setattr(make_plans, "Sawtooth", lambda: (lambda p: p / np.pi - 1))
    monkeypatch.setattr(make_plans, "AffineSin", lambda a, b: (lambda p: a * np.sin(p) + b))
    with open(os.path.join(HERE, "golden", "plans", name + ".bin"), "rb") as f:
        assert lower(getattr(make_plans, name)()).tobytes() == f.read()


# ---- batches -----------------------------------------------------------------------------------------------------------

class _Capture(EmulatedFnsSink):
    def compiled(self, plan_bytes):
        self.blob = plan_bytes
        return super().compiled(plan_bytes)


def test_batch_of_identical_closures_has_no_generator_inputs():
    g = _Capture()
    sink_batch([Signal(lambda p: np.tanh(np.sin(p)), 8 * kHz, ω=5 * Hz) >> Until(0.1 * s) for _ in range(4)], g)
    assert g.blob == lower(Signal(lambda p: np.tanh(np.sin(p)), 8 * kHz, ω=5 * Hz) >> Until(0.1 * s)).tobytes()
    assert int.from_bytes(g.blob[8:12], "little") == 0          # n_inputs


def test_batch_with_different_omegas_is_host_evaluated():
    g = _Capture()
    xs = [Signal(lambda p: np.tanh(np.sin(p)), 8 * kHz, ω=w * Hz) >> Until(0.1 * s) for w in (3, 5)]
    sink_batch(xs, g)
    assert g.blob == Lowerer(generators="host").build(xs[0]).tobytes()
    assert int.from_bytes(g.blob[8:12], "little") == 1


def test_functor_generators_are_unchanged():
    assert leaves(gen(sin, ω=10 * Hz))[0] == [(L.OP_LOAD, L.LEAF_GEN, L.FN_SIN)]
    x = np.zeros((800, 2))
    p = lower(Amplify(Signal(x, 8 * kHz), Signal(lambda p: 0.5 * np.sin(p) + 0.5, 8 * kHz, ω=5 * Hz)) >> Until(0.1 * s)
              >> Filt(Lowpass, 1 * kHz))
    assert [(I.op, I.leaf, I.fn) for I in p.stages[0].in_prog] == [(L.OP_LOAD, L.LEAF_BUF, 0), (L.OP_MUL, L.LEAF_GEN, FN_AFFINE_SIN)]
