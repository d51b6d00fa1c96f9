"""CPU check of the plans behind test_gpu_fir_long.py: strong down-sampling and long `FIRFilter` banks lowered to plan
bytes and evaluated by tests/plan_emulator.py (numpy) against the oracle, or against `scipy.signal.upfirdn` where the
oracle has no such filter.  This pins what the long-bank FIR stages mean without a GPU."""
from fractions import Fraction

import numpy as np
import pytest
from scipy import signal as sps

import oracle
from plan_emulator import Emulator
from signalops import Amplify, Filt, Hz, Normpower, Signal, ToFramerate, dB, dspjl, kHz
from signalops.lowering import STAGE_FIR, lower


def rms(a):
    return float(np.sqrt(np.mean(np.asarray(a, dtype=np.float64) ** 2)))


def emulate(sig, x):
    plan = lower(sig)
    (y,) = Emulator(plan.tobytes()).run([np.asfortranarray(x)])
    return np.asarray(y).reshape(len(y), -1), plan


def fir_stage(plan):
    (st,) = [s for s in plan.stages if s.kind == STAGE_FIR]
    return st


@pytest.mark.parametrize("fi,fo,taps", [(48000, 8000, 219), (48000, 11025, 159), (48000, 12000, 147), (44100, 8000, 201),
                                        (192000, 48000, 147), (48000, 1000, 1742)])
def test_strong_downsampling(fi, fo, taps):
    x = np.random.default_rng(fo).standard_normal((int(fi) // 8, 2))
    chain = lambda v: ToFramerate(Signal(v, fi * Hz), fo * Hz)   # noqa: E731
    got, plan = emulate(chain(x), x)
    assert fir_stage(plan).taps_per_phase == taps
    want, _ = oracle.sink(chain(x))
    assert got.shape == want.shape and np.max(np.abs(got - want)) <= 1e-12 * rms(want)


@pytest.mark.parametrize("ntaps", [202, 1025, 4097])
def test_single_rate_fir_filter(ntaps):
    h = sps.firwin(ntaps, 0.2)
    x = np.random.default_rng(ntaps).standard_normal((6000, 1))
    chain = lambda v: Signal(v, 48 * kHz) >> Filt(dspjl.FIRFilter(h)) >> Amplify(-6 * dB)   # noqa: E731
    got, plan = emulate(chain(x), x)
    assert fir_stage(plan).taps_per_phase == ntaps and fir_stage(plan).epi_prog       # the gain is the stage's epilogue
    want, _ = oracle.sink(chain(x))
    assert np.max(np.abs(got - want)) <= 1e-12 * rms(want)
    ref = sps.lfilter(h, 1.0, x[:, 0]) * 10 ** (-6 / 20)
    assert np.max(np.abs(got[:, 0] - ref)) <= 1e-12 * rms(ref)


@pytest.mark.parametrize("ntaps,ratio,up,down,per_phase", [(1500, Fraction(1, 5), 1, 5, 1500), (2048, 4, 4, 1, 512),
                                                           (1200, Fraction(2, 7), 2, 7, 600)])
def test_resampling_fir_filter(ntaps, ratio, up, down, per_phase):
    h = sps.firwin(ntaps, 0.8 / max(up, down))
    x = np.random.default_rng(ntaps).standard_normal((5001, 1))
    got, plan = emulate(Signal(x, 48 * kHz) >> Filt(dspjl.FIRFilter(h, ratio)), x)
    assert fir_stage(plan).taps_per_phase == per_phase
    u = sps.upfirdn(h, x[:, 0], up, down)
    n = min(len(u), len(got))
    assert np.max(np.abs(got[:n, 0] - u[:n])) <= 1e-12 * rms(u[:n])
    assert not np.any(got[n:])


def test_normpower_after_strong_downsampling():
    x = np.random.default_rng(3).standard_normal((9000, 2))
    chain = lambda v: ToFramerate(Signal(v, 48 * kHz), 12 * kHz) >> Normpower >> Amplify(-20 * dB)   # noqa: E731
    got, plan = emulate(chain(x), x)
    assert fir_stage(plan).sumsq_slot >= 0
    want, _ = oracle.sink(chain(x))
    assert np.max(np.abs(got - want)) <= 1e-12 * rms(want)
