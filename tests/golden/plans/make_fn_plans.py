"""Plan-byte fixtures of traced OperateOn closures (SIGOPS_OP_FN1 / FN2 / POPFN2) for the Julia glue, next to the
fixtures of make_plans.py and checked the same way: julia/test_plans.jl builds each graph below with the reference's
API and `GPUSinks.Traced`, and compares its plan with the committed <name>.bin; tests/test_fn_plan_fixtures.py checks
that host/lowering.py still emits those bytes.

usage: python tests/golden/plans/make_fn_plans.py   (rewrites the .bin files of the cases below)"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(HERE))))

from signalops import Bandpass, Filt, Hz, Lowpass, Mix, Operate, OperateOn, Signal, kHz  # noqa: E402
from signalops.lowering import lower  # noqa: E402

Z = np.zeros


def envelope():
    """Envelope follower: full-wave rectification, then a 50 Hz lowpass (`OperateOn(abs, x) |> Filt(Lowpass, 50Hz)`)."""
    return OperateOn(abs, Signal(Z((48000, 2)), 48 * kHz)) >> Filt(Lowpass, 50 * Hz)


def softclip():
    """Soft saturation after a filter, Float32 (rounded after every traced operation)."""
    x = Signal(Z((48000, 2), dtype=np.float32), 48 * kHz)
    return x >> Filt(Bandpass, 500 * Hz, 4 * kHz) >> Operate(lambda v: np.tanh(np.float32(2) * v))


def clamp():
    """Clipping to [-1, 1], and `max(x, 0)`, of a mix."""
    x = Signal(Z((1000, 1)), 10 * kHz)
    return Mix(OperateOn(lambda v: np.clip(v, -1, 1), x), OperateOn(lambda v: np.maximum(v, 0), x))


def midside():
    """Mid/side of a stereo signal: a whole-frame closure, one expression per output channel."""
    return OperateOn(lambda f: (0.5 * (f[0] + f[1]), 0.5 * (f[0] - f[1])), Signal(Z((1000, 2)), 10 * kHz), bychannel=False)


CASES = {"envelope": envelope, "softclip": softclip, "clamp": clamp, "midside": midside}


def plan_bytes(name):
    return lower(CASES[name]()).tobytes()


if __name__ == "__main__":
    for name in CASES:
        with open(os.path.join(HERE, name + ".bin"), "wb") as f:
            f.write(plan_bytes(name))
        print(name, os.path.getsize(os.path.join(HERE, name + ".bin")), "bytes")
