"""Plan-byte fixtures of traced generator closures `Signal(ϕ -> …)` for the Julia glue, next to the fixtures of
make_plans.py and checked the same way: julia/test_gen_plans.jl builds each graph below with the reference's API and
`GPUSinks.lower`, and compares its plan with the committed <name>.bin; tests/test_gen_plan_fixtures.py checks that
host/lowering.py still emits those bytes.

usage: python tests/golden/plans/make_gen_plans.py   (rewrites the .bin files of the cases below)"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(HERE))))

from signalops import Amplify, Bandpass, Filt, Hz, Mix, Ramp, Signal, Until, kHz, ms, s  # noqa: E402
from signalops.lowering import lower  # noqa: E402

Z = np.zeros


def gen_am():
    """Config 5's shape with a closure AM envelope (a sub-program of the filter's input program) and a closure tone."""
    am = Amplify(Signal(Z((48000, 2)), 48 * kHz), Signal(lambda p: 0.5 * np.sin(p) + 0.25 * np.sin(2 * p) + 0.25, ω=5 * Hz))
    tone = Signal(lambda p: 0.3 * np.sin(p) + 0.1 * np.cos(3 * p), ω=1 * kHz) >> Until(1 * s)
    return am >> Until(1 * s) >> Filt(Bandpass, 500 * Hz, 4 * kHz) >> Ramp(10 * ms) >> Mix(tone)


def gen_readme():
    """The README's closures `ϕ -> ϕ/π - 1` and `ϕ -> 0.5sin(ϕ) + 0.5`: the enumerated generator leaves."""
    saw = Signal(lambda p: p / np.pi - 1, 10 * kHz, ω=100 * Hz)
    return Mix(saw, Signal(lambda p: 0.5 * np.sin(p) + 0.5, 10 * kHz, ω=5 * Hz, phi=np.pi / 2)) >> Until(100 * ms)


def gen_stereo():
    """A two-channel closure: one program per channel."""
    return Signal(lambda p: (np.sin(p), 0.5 * np.cos(p) + 0.1 * np.sin(5 * p)), 10 * kHz, ω=300 * Hz) >> Until(100 * ms)


def gen_time():
    """A closure of time (no ω): its argument is k/fs."""
    return Signal(lambda t: np.exp(-3 * t) * np.sin(2 * np.pi * 440 * t), 10 * kHz) >> Until(100 * ms)


CASES = {"gen_am": gen_am, "gen_readme": gen_readme, "gen_stereo": gen_stereo, "gen_time": gen_time}


def plan_bytes(name):
    return lower(CASES[name]()).tobytes()


if __name__ == "__main__":
    for name in CASES:
        with open(os.path.join(HERE, name + ".bin"), "wb") as f:
            f.write(plan_bytes(name))
        print(name, os.path.getsize(os.path.join(HERE, name + ".bin")), "bytes")
