"""Ragged batches on the CPU: `sink([x1, x2, ...], GPUSink())` over signals of different lengths, with the plan bytes
the GPU would receive evaluated by tests/ragged_emulator.py under the runtime's rules (max plan, zero tails, masked sums
of squares, waves of sorted instances computing prefixes, per-instance copy-out), against `oracle.sink` of each element
alone; plus the batches that must be refused, and equal-length batches keeping the ordinary path."""
import numpy as np
import pytest

import oracle
from plan_emulator import Emulator
from ragged_emulator import RaggedEmulator
from signalops import (After, Amplify, Append, Filt, GPUSink, Highpass, Hz, Lowpass, Mix, Normpower, Pad, Ramp,
                       Signal, ToFramerate, Until, dB, kHz, randn, s, sin, sink)
from signalops.lowering import Lowerer
from signalops.philox import PhiloxRNG
from signalops import graph as G


class _EmuPlan:
    def __init__(self, blob, log):
        self.blob, self.log = blob, log

    def run_host(self, ninst, ins, outs):
        self.log.append("ordinary")
        n_in, n_out = len(ins) // ninst, len(outs) // ninst
        for i in range(ninst):
            res = Emulator(self.blob).run(ins[i * n_in:(i + 1) * n_in], inst=i)
            for o, r in zip(outs[i * n_out:(i + 1) * n_out], res):
                o.reshape(r.shape)[...] = r
        return {}

    def run_ragged(self, ninst, ins, outs, temp_frames):
        self.log.append("ragged")
        n_in, n_out = len(ins) // ninst, len(outs) // ninst
        emu = RaggedEmulator(self.blob)
        res = emu.run_ragged([ins[i * n_in:(i + 1) * n_in] for i in range(ninst)],
                             [outs[i * n_out].shape[0] for i in range(ninst)], temp_frames)
        for i in range(ninst):
            for o, r in zip(outs[i * n_out:(i + 1) * n_out], res[i]):
                if o.size:
                    o.reshape(r.shape)[...] = r
        return {}


class RaggedEmulatedSink(GPUSink):
    def __init__(self):
        super().__init__()
        self.log = []

    def compiled(self, plan_bytes):
        return _EmuPlan(plan_bytes, self.log)

    def alloc_result(self, shape, dtype):
        return np.empty(shape, dtype=dtype, order="F")


def rms(a):
    return float(np.sqrt(np.mean(np.asarray(a, dtype=np.float64) ** 2))) if np.size(a) else 1.0


CHAINS = {
    "up_441_48": (44100, 1, lambda v: ToFramerate(Signal(v, 44.1 * kHz), 48 * kHz)),
    "down_48_441": (48000, 1, lambda v: ToFramerate(Signal(v, 48 * kHz), 44.1 * kHz)),
    "two_thirds": (48000, 1, lambda v: ToFramerate(Signal(v, 48 * kHz), 32 * kHz)),
    "strong_down": (48000, 1, lambda v: ToFramerate(Signal(v, 48 * kHz), 1 * kHz)),
    "lowpass": (48000, 1, lambda v: Signal(v, 48 * kHz) >> Filt(Lowpass, 4 * kHz, order=8)),
    "slow_highpass": (48000, 1, lambda v: Signal(v, 48 * kHz) >> Filt(Highpass, 0.5 * Hz, order=4)),
    "filt_resample": (48000, 1, lambda v: Signal(v, 48 * kHz) >> Filt(Lowpass, 8 * kHz) >> ToFramerate(44.1 * kHz)),
    "norm_iir_stereo": (48000, 2, lambda v: Signal(v, 48 * kHz) >> Filt(Lowpass, 3 * kHz) >> Normpower >> Amplify(-20 * dB)),
    "norm_fir_stereo": (44100, 2, lambda v: Signal(v, 44.1 * kHz) >> ToFramerate(48 * kHz) >> Normpower >> Amplify(-20 * dB)),
    "corpus": (44100, 2, lambda v: Signal(v, 44.1 * kHz) >> ToFramerate(48 * kHz) >> Filt(Lowpass, 8 * kHz) >> Normpower
               >> Amplify(-20 * dB)),
    "after": (48000, 1, lambda v: Signal(v, 48 * kHz) >> After(0.01 * s) >> Filt(Lowpass, 2 * kHz)),
    "until_ramp": (48000, 1, lambda v: Signal(v, 48 * kHz) >> Until(0.01 * s) >> Ramp(0.005 * s)),
}
LENGTHS = [1500, 4100, 700, 2917, 2200]          # unsorted; 700 < 0.015 s < the rest


def batch(name, lengths, dtype=np.float64, seed=0):
    fs, C, chain = CHAINS[name]
    rng = np.random.default_rng(seed)
    xs = [np.asfortranarray(rng.standard_normal((n, C)).astype(dtype)) for n in lengths]
    return [chain(x) for x in xs]


def check(sigs, f32=False, log=None):
    gpu = RaggedEmulatedSink()
    outs = sink(sigs, gpu)
    assert gpu.log == ["ragged"] if log is None else gpu.log == log
    for x, (got, fs) in zip(sigs, outs):
        want, fs2 = oracle.sink(x)
        assert fs == fs2 and got.shape == want.shape and got.dtype == want.dtype
        tol = (1e-5 if f32 else 1e-9) * rms(want)
        assert np.max(np.abs(got.astype(np.float64) - want), initial=0.0) <= tol
    return outs


@pytest.mark.parametrize("name", sorted(CHAINS))
def test_ragged_chain_matches_each_element_alone(name):
    check(batch(name, LENGTHS))


def test_float32_inputs():
    check(batch("lowpass", LENGTHS, np.float32), f32=True)
    check(batch("norm_fir_stereo", LENGTHS, np.float32), f32=True)


def test_zero_pad_extensions_of_ragged_signals():
    # a fixed-length tone mixed in that ends inside some elements and past others, and every element padded with zeros
    # to one length: where an element reads a constant zero past its end, the plan reads its zero-padded buffer
    tone = lambda: Signal(sin, ω=1 * kHz) >> Until(0.02 * s) >> Amplify(0.5)          # 960 frames  # noqa: E731
    xs = [np.random.default_rng(n).standard_normal((n, 1)) for n in (1500, 300, 2600, 959, 961)]
    check([Mix(Signal(x, 48 * kHz), tone()) for x in xs])
    check([Mix(tone(), Signal(x, 48 * kHz)) >> Filt(Lowpass, 2 * kHz) for x in xs])
    check([Pad(Signal(x, 48 * kHz), 0.0) >> Until(0.05 * s) for x in xs])
    check([Mix(Signal(x, 48 * kHz), tone()) >> Normpower for x in xs])


def test_device_noise_keeps_caller_order():
    fs = 8000
    lens = [800, 2400, 1600]
    xs = [np.random.default_rng(n).standard_normal((n, 1)) for n in lens]
    sigs = [Mix(Signal(x, fs * Hz), Signal(randn, fs * Hz, rng=PhiloxRNG(42, stream=10 + k)) >> Until(n / fs * s)
                >> Amplify(0.1)) >> Filt(Lowpass, 1 * kHz) for k, (x, n) in enumerate(zip(xs, lens))]
    check(sigs)


def test_zero_length_and_single_element():
    sigs = batch("corpus", [1800, 0, 1000])
    outs = check(sigs)
    assert outs[1][0].shape == (0, 2)
    check(batch("corpus", [1800]), log=["ordinary"])
    gpu = RaggedEmulatedSink()
    assert [o[0].shape for o in sink(batch("lowpass", [0, 0]), gpu)] == [(0, 1), (0, 1)] and gpu.log == []


def test_equal_lengths_take_the_ordinary_path():
    sigs = batch("corpus", [1500, 1500, 1500])
    blobs = [Lowerer(instance_index=k).build(x).tobytes() for k, x in enumerate(sigs)]
    assert all(b == blobs[0] for b in blobs)
    check(sigs, log=["ordinary"])


def refused(sigs, match):
    with pytest.raises(G.SignalError, match=match):
        sink(sigs, RaggedEmulatedSink())


def test_refusals_name_the_operator():
    xs = [np.random.default_rng(n).standard_normal((n, 1)) for n in (1500, 900)]
    S = lambda x: Signal(x, 48 * kHz)                                               # noqa: E731
    tone = Signal(sin, ω=1 * kHz) >> Until(0.02 * s)
    refused([S(x) >> Ramp(0.005 * s) for x in xs], "Ramp, RampOff or FadeTo")
    refused([S(x) >> Append(tone) for x in xs], "Append after a signal of ragged length")
    refused([Pad(S(x), 1.0) >> Until(0.05 * s) for x in xs], "a pad with the constant 1 ")
    y = np.random.default_rng(0).standard_normal((1000, 1))
    refused([Amplify(S(x), S(y)) for x in xs], "a pad with the constant 1 ")      # the `one` pad of the 900-frame clip
    for pad, name in (("cycle", "cycle"), ("mirror", "mirror"), ("lastframe", "lastframe")):
        refused([Pad(S(x), getattr(G, pad)) >> Until(0.05 * s) for x in xs], f"Pad\\(x, {name}\\)")
    # other constants, filters or channel counts: the existing message
    refused([S(x) >> Amplify(g) for x, g in zip(xs, (0.5, 0.25))], "does not lower to the same plan")
    refused([S(xs[0]) >> Filt(Lowpass, 2 * kHz), S(xs[1]) >> Filt(Lowpass, 3 * kHz)], "does not lower to the same plan")
    refused([S(xs[0]), S(np.hstack([xs[1], xs[1]]))], "does not lower to the same plan")


def test_ramp_inside_a_fixed_cut_is_fine():
    xs = [np.random.default_rng(n).standard_normal((n, 1)) for n in (1500, 900, 2000)]
    # (the inputs differ in length, the fade-out starts at the same frame for all)
    check([Signal(x, 48 * kHz) >> Until(0.015 * s) >> Ramp(0.002 * s) for x in xs])

