"""Generator closures `Signal(ϕ -> …)` traced into device programs, against the CPU oracle, which calls the Python
closure once per frame.

Tolerances are BASELINE.json's (Float64 1e-9 of the RMS, Float32 1e-5).  The `test_*` functions that take the `gpu`
fixture also run on the plan emulator (tests/test_gen_closures_emulated.py); the dispatch cases at the end need the
device."""
import re

import numpy as np
import pytest

import oracle
from signalops import (Amplify, Bandpass, Filt, GPUSink, Hz, Lowpass, Mix, Normpower, Ramp, Signal, ToFramerate, Until, kHz,
                       ms, s, sink, sink_batch)

pytestmark = pytest.mark.gpu

F64_TOL = 1e-9
F32_TOL = 1e-5


def rms(a):
    a = np.asarray(a, dtype=np.float64)
    return float(np.sqrt(np.mean(a ** 2))) if a.size else 0.0


def rel_err(got, want):
    return float(np.max(np.abs(got.astype(np.float64) - want.astype(np.float64)))) / max(rms(want), 1e-300)


def check(gpu, make, tol=F64_TOL):
    want, fs = oracle.sink(make())
    got, fs2 = sink(make(), gpu)
    assert fs == fs2 and got.shape == want.shape and got.dtype == want.dtype
    err = rel_err(got, want)
    assert err <= tol, f"max err / rms = {err:g}"
    return got


def envelope(p):
    """An AM envelope that is none of the enumerated generators: two partials and an offset."""
    return 0.5 * np.sin(p) + 0.25 * np.sin(2 * p) + 0.25


def tone(p):
    return 0.3 * np.sin(p) + 0.1 * np.cos(3 * p)


def data(shape, seed=7):
    return np.random.default_rng(seed).standard_normal(shape)


@pytest.mark.parametrize("kw", [dict(ω=5 * Hz), dict(ω=440 * Hz, phi=np.pi / 3), dict()], ids=["omega", "omega-phi", "time"])
def test_closure_generator(gpu, kw):
    f = envelope if kw else (lambda t: np.exp(-3 * t) * np.sin(2 * np.pi * 440 * t))
    check(gpu, lambda: Signal(f, 48 * kHz, **kw) >> Until(0.5 * s))


def test_readme_closures(gpu):
    check(gpu, lambda: Signal(lambda p: p / np.pi - 1, 8 * kHz, ω=100 * Hz) >> Until(1 * s))
    check(gpu, lambda: Signal(lambda p: 0.5 * np.sin(p) + 0.5, 8 * kHz, ω=5 * Hz) >> Until(1 * s))


def test_stereo_tuple_generator(gpu):
    check(gpu, lambda: Signal(lambda p: (np.sin(p), 0.5 * np.cos(p) + 0.1 * np.sin(5 * p)), 48 * kHz, ω=300 * Hz)
          >> Until(0.5 * s))


def test_float32_and_integer_generators(gpu):
    got = check(gpu, lambda: Signal(lambda p: np.sin(np.float32(2) * p) * np.float32(0.5), 8 * kHz, ω=50 * Hz)
                >> Until(1 * s), tol=F32_TOL)
    assert got.dtype == np.float32
    got = check(gpu, lambda: Signal(lambda p: round(10 * p), 8 * kHz, ω=7 * Hz) >> Until(1 * s))
    assert got.dtype == np.int64


def test_closure_mixed_into_a_buffer(gpu):
    x = data((24000, 2))
    check(gpu, lambda: Mix(Signal(x, 48 * kHz), Signal(tone, 48 * kHz, ω=1 * kHz) >> Until(0.5 * s)))
    check(gpu, lambda: Amplify(Signal(x, 48 * kHz), Signal(envelope, 48 * kHz, ω=5 * Hz)) >> Until(0.5 * s))


def test_closures_around_a_filter(gpu):
    """A closure modulator in the filter's input program and a closure tone in its epilogue (config 5's shape)."""
    x = data((48000, 4), seed=8)

    def make():
        am = Amplify(Signal(x, 48 * kHz), Signal(envelope, 48 * kHz, ω=5 * Hz)) >> Until(1 * s)
        return am >> Filt(Bandpass, 500 * Hz, 4 * kHz) >> Ramp(10 * ms) >> Mix(Signal(tone, 48 * kHz, ω=1 * kHz) >> Until(1 * s))
    check(gpu, make)


def test_sixty_seconds(gpu):
    check(gpu, lambda: Signal(envelope, 48 * kHz, ω=3 * Hz) >> Until(60 * s))


def test_normpower_after_closure_generator(gpu):
    check(gpu, lambda: Signal(tone, 48 * kHz, ω=200 * Hz) >> Until(1 * s) >> Normpower)


def test_closure_generator_before_resampling(gpu):
    check(gpu, lambda: Signal(tone, 48 * kHz, ω=300 * Hz) >> Until(1 * s) >> ToFramerate(44.1 * kHz))


def test_batch_of_identical_closures(gpu):
    make = lambda: Signal(lambda p: 0.5 * np.sin(p) + 0.25 * np.sin(2 * p), 48 * kHz, ω=5 * Hz) >> Until(0.25 * s)  # noqa: E731
    want, _ = oracle.sink(make())
    for got, _ in sink_batch([make() for _ in range(64)], gpu):
        assert rel_err(got, want) <= F64_TOL


def test_batch_with_different_omegas(gpu):
    makes = [lambda w=w: Signal(envelope, 48 * kHz, ω=w * Hz) >> Until(0.25 * s) for w in (3, 5, 7, 11)]
    for make, (got, _) in zip(makes, sink_batch([m() for m in makes], gpu)):
        assert rel_err(got, oracle.sink(make())[0]) <= F64_TOL


def test_several_host_waves(monkeypatch):
    """A small workspace budget splits a batch of closure signals into several host waves."""
    monkeypatch.setenv("SIGOPS_WS_BYTES", str(16 << 20))
    g = GPUSink([0])
    try:
        make = lambda: Signal(envelope, 48 * kHz, ω=5 * Hz) >> Until(10 * s)   # noqa: E731
        got = sink_batch([make() for _ in range(16)], g)
        assert g.last_stats["launches"] > 1
        want, _ = oracle.sink(make())
        for y, _ in got:
            assert rel_err(y, want) <= F64_TOL
    finally:
        g.close()


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


def strided_batch(seed=12):
    rng = np.random.default_rng(seed)
    return [np.asfortranarray(rng.standard_normal((48000, 32))) for _ in range(3)]


def modulated(env):
    return lambda x: (Amplify(Signal(x, 48 * kHz), Signal(env, 48 * kHz, ω=5 * Hz)) >> Until(1 * s) >> Filt(Lowpass, 4 * kHz, order=8)
                      >> Mix(Signal(tone, 48 * kHz, ω=1 * kHz) >> Until(1 * s)))


def test_closure_modulator_stays_on_tensor_map_kernel(fresh_sink, capfd, monkeypatch):
    """A closure AM envelope before the filter and a closure tone after it, on a strided batch of 96 rows: ONE launch of
    the tensor-map kernel, the closures fused into its row-invariant programs as sub-programs, equal to the per-lane
    path (SIGOPS_NO_TMAP_LEAVES=1) up to the generators' angle addition there."""
    xs = strided_batch()
    chain = modulated(envelope)
    got = sink_batch([chain(x) for x in xs], fresh_sink)
    assert iir_kernels(capfd) == ["tensor-map (fused row-invariant programs)"]
    assert fresh_sink.last_stats["launches"] == 1
    for x, (y, _) in zip(xs, got):
        assert rel_err(y, oracle.sink(chain(x))[0]) <= F64_TOL
    monkeypatch.setenv("SIGOPS_NO_TMAP_LEAVES", "1")
    g = GPUSink([0])
    try:
        ref = sink_batch([chain(x) for x in xs], g)
    finally:
        g.close()
    assert iir_kernels(capfd) == ["generic"]
    for (y, _), (r, _) in zip(got, ref):
        assert rel_err(y, r) <= 1e-12


def test_sub_program_over_the_cap_takes_the_per_lane_path(fresh_sink, capfd):
    """A modulator whose sub-program is longer than the fused kernel takes (24 instructions): the per-lane path."""
    xs = strided_batch(13)[:2]
    chain = modulated(lambda p: (0.2 * np.sin(p) + 0.2 * np.sin(2 * p) + 0.2 * np.sin(3 * p) + 0.2 * np.sin(4 * p)
                                 + 0.1 * np.cos(p) + 0.1))
    got = sink_batch([chain(x) for x in xs], fresh_sink)
    assert iir_kernels(capfd) == ["generic"]
    for x, (y, _) in zip(xs, got):
        assert rel_err(y, oracle.sink(chain(x))[0]) <= F64_TOL
