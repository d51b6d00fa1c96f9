"""Test-only extension of tests/plan_emulator.py: the OperateOn closure functions of include/signalops.h
(SIGOPS_OP_FN1 / FN2 / POPFN2, SIGOPS_EFN_*) with Julia's NaN and signed-zero rules, in numpy.  Like the emulator it
extends, nothing in the product imports it."""
import numpy as np

from plan_emulator import Emulator
from test_lowering_emulated import EmulatedSink, _EmuPlan

OP_FN1, OP_FN2, OP_POPFN2 = 14, 15, 16
LEAVES_READING_FN = (4, 5, 6)          # LEAF_GEN, LEAF_RAMP_ON, LEAF_RAMP_OFF: not allowed under FN2


def _jl_min(a, b):
    """Julia's `min`: a NaN operand wins, -0.0 orders below 0.0 (numpy's minimum differs at the signed zeros)."""
    a, b = np.broadcast_arrays(np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64))
    r = np.where(a == b, np.where(np.signbit(a), a, b), np.where(a < b, a, b))
    return np.where(np.isnan(a) | np.isnan(b), a + b, r)


def _jl_max(a, b):
    a, b = np.broadcast_arrays(np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64))
    r = np.where(a == b, np.where(np.signbit(a), b, a), np.where(a > b, a, b))
    return np.where(np.isnan(a) | np.isnan(b), a + b, r)


def _jl_mod(a, b):
    r = np.fmod(a, b)
    return np.where(r == 0, np.copysign(r, b), np.where((r > 0) != (b > 0), r + b, r))


def _jl_sign(a):
    return np.where(a > 0, 1.0, np.where(a < 0, -1.0, a))


# SIGOPS_EFN_*: unary codes 1.., binary codes 32..
EFN1 = {1: np.abs, 2: _jl_sign, 3: np.floor, 4: np.ceil, 5: np.trunc, 6: np.rint, 7: np.sqrt, 8: None, 9: np.exp,
        10: np.exp2, 11: np.expm1, 12: np.log, 13: np.log2, 14: np.log10, 15: np.log1p, 16: np.sin, 17: np.cos,
        18: np.tan, 19: np.tanh, 20: np.sinh, 21: np.cosh, 22: np.arctan, 23: np.cbrt}
EFN2 = {32: _jl_min, 33: _jl_max, 34: np.copysign, 35: np.fmod, 36: _jl_mod, 37: np.power, 38: np.hypot}


def efn(fn, a, b=None, c=None):
    """Function `fn` of an FN1 (b, c = the instruction's d0, d1) or FN2 / POPFN2 instruction, on Float64 arrays;
    domain errors give NaN like the device (numpy's warnings are silenced)."""
    with np.errstate(all="ignore"):
        a = np.asarray(a, dtype=np.float64)
        if fn == 8:                                   # clamp(x, lo, hi): NaN stays NaN, -0.0 is inside [0, 1]
            return np.where(a > c, c, np.where(a < b, b, a))
        if fn in EFN1:
            return EFN1[fn](a)
        return EFN2[fn](a, np.asarray(b, dtype=np.float64))


class EmulatorFns(Emulator):
    """The plan emulator with the closure-function opcodes.  A program without them is evaluated by the base class."""

    def run_prog(self, start, ln, n, c, stage=None):
        prog = self.instrs[start:start + ln]
        if not any(I[0] >= OP_FN1 for I in prog):
            return super().run_prog(start, ln, n, c, stage)
        acc, stack = None, []
        for I in prog:
            op = I[0]
            if op <= 5:
                v = self.leaf(I, n, c, stage)
                acc = v if op == 1 else acc + v if op == 2 else acc - v if op == 3 else acc * v if op == 4 else acc / v
            elif op == 6:
                stack.append(acc)
            elif op <= 10:
                l = stack.pop()
                acc = l + acc if op == 7 else l - acc if op == 8 else l * acc if op == 9 else l / acc
            elif op == 11:
                acc = -acc
            elif op == 12:
                acc = acc.astype(np.float32).astype(np.float64)
            elif op == 13:
                acc = acc.astype(np.int64).astype(np.float64)
            elif op == OP_FN1:                 # acc = f(acc)
                acc = efn(I[2], acc, I[10], I[11])
            elif op == OP_FN2:                 # acc = g(acc, leaf)
                assert I[1] not in LEAVES_READING_FN, "FN2 on a leaf that reads fn"
                acc = efn(I[2], acc, self.leaf(I, n, c, stage))
            elif op == OP_POPFN2:              # acc = g(popped, acc)
                acc = efn(I[2], stack.pop(), acc)
        return acc


class _EmuFnsPlan(_EmuPlan):
    def run_host(self, ninst, ins, outs):
        n_in = len(ins) // ninst
        n_out = len(outs) // ninst
        for i in range(ninst):
            res = EmulatorFns(self.blob).run(ins[i * n_in:(i + 1) * n_in], inst=i)
            for o, r in zip(outs[i * n_out:(i + 1) * n_out], res):
                o = o.raw if hasattr(o, "raw") else o
                o.reshape(r.shape)[...] = r
        return {"launches": 0}


class EmulatedFnsSink(EmulatedSink):
    def compiled(self, plan_bytes):
        return _EmuFnsPlan(plan_bytes)
