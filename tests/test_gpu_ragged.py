"""Ragged batches on the B200: `sink([x1, x2, ...], GPUSink())` over signals of different lengths, per element against
the oracle and against `sink(x, GPUSink())` of the element alone, on every IIR and FIR kernel path, over several waves,
on a workspace a previous batch left full of NaN, and over two devices when there are two."""
import numpy as np
import pytest

import oracle
from signalops import GPUSink, Filt, Hz, Lowpass, Mix, Normpower, Pad, Signal, ToFramerate, Until, Amplify, kHz, randn, s, sin, sink
from signalops.philox import PhiloxRNG
from signalops.cabi import load
from test_ragged_batch import CHAINS

pytestmark = pytest.mark.gpu


def rms(a):
    return float(np.sqrt(np.mean(np.asarray(a, dtype=np.float64) ** 2))) if np.size(a) else 1.0


def signals(name, lengths, seed=0, dtype=np.float64):
    fs, C, chain = CHAINS[name]
    rng = np.random.default_rng(seed)
    return [chain(np.asfortranarray(rng.standard_normal((n, C)).astype(dtype))) for n in lengths]


def lengths_for(n, lo, hi, seed=1):
    return [int(v) for v in np.random.default_rng(seed).integers(lo, hi, n)]


def check(gpu, sigs, against_sink=None, f32=False):
    """Every element against the oracle; with `against_sink` (a tolerance relative to RMS) also against `sink` of the
    element alone, which runs the same kernels except where a chunking follows the length (IIR carry chunks)."""
    try:
        outs = sink(sigs, gpu)
        assert gpu.last_stats["out_samples"] == sum(o[0].size for o in outs)
        for x, (got, fs) in zip(sigs, outs):
            want, fs2 = oracle.sink(x)
            assert fs == fs2 and got.shape == want.shape and got.dtype == want.dtype
            assert np.all(np.isfinite(got))
            assert np.max(np.abs(got.astype(np.float64) - want), initial=0.0) <= (1e-5 if f32 else 1e-9) * rms(want)
            if against_sink is not None and got.size:
                own = sink(x, gpu)[0]
                assert np.max(np.abs(got.astype(np.float64) - own)) <= against_sink * rms(own)
        return outs
    finally:
        gpu.close()


# 72 elements of 0.02 - 1 s: enough rows for the tensor-map kernels
@pytest.mark.parametrize("name", ["up_441_48", "down_48_441", "two_thirds", "strong_down", "lowpass", "slow_highpass",
                                  "filt_resample", "norm_iir_stereo", "norm_fir_stereo", "corpus", "after"])
def test_ragged_chain(name):
    # Against the element alone: the same kernels on the same plan lengths' recurrences, except the slow high-pass,
    # which runs MAIN + CARRY + FIX with a chunk length that follows the frames of the wave (2e-10 measured).
    check(GPUSink(), signals(name, lengths_for(72, 960, 48000)), against_sink=1e-9 if name == "slow_highpass" else 1e-12)


def test_zero_pad_extensions():
    # a fixed-length tone that ends inside some elements and past others; every element padded with zeros to one length
    tone = lambda: Signal(sin, ω=1 * kHz) >> Until(0.5 * s) >> Amplify(0.5)          # 24 000 frames  # noqa: E731
    xs = [np.asfortranarray(np.random.default_rng(n).standard_normal((n, 2))) for n in lengths_for(72, 960, 48000, seed=3)]
    check(GPUSink(), [Mix(Signal(x, 48 * kHz), tone()) >> Filt(Lowpass, 4 * kHz) >> Normpower for x in xs], against_sink=1e-12)
    check(GPUSink(), [Pad(Signal(x, 48 * kHz), 0.0) >> Until(1 * s) >> ToFramerate(44.1 * kHz) for x in xs], against_sink=1e-12)


def test_device_noise_keeps_each_elements_stream(monkeypatch):
    # unsorted lengths over many waves: a plan with device noise runs in the caller's order, so that element k draws
    # stream 10 + k
    monkeypatch.setenv("SIGOPS_WS_BYTES", str(64 << 20))
    fs = 8000
    # (lengths whose time `n / fs` gives back n frames: the noise then ends with its element)
    lens = [n for n in lengths_for(60, 400, 40000, seed=13) if (Signal(randn, fs * Hz) >> Until(n / fs * s)).nframes == n][:48]
    xs = [np.random.default_rng(n).standard_normal((n, 1)) for n in lens]
    sigs = [Mix(Signal(x, fs * Hz), Signal(randn, fs * Hz, rng=PhiloxRNG(42, stream=10 + k)) >> Until(n / fs * s))
            >> Filt(Lowpass, 1 * kHz) >> Normpower for k, (x, n) in enumerate(zip(xs, lens))]
    check(GPUSink(), sigs, against_sink=1e-12)


def test_float32():
    check(GPUSink(), signals("corpus", lengths_for(40, 960, 30000), dtype=np.float32), f32=True)


@pytest.mark.parametrize("knob", ["SIGOPS_NO_TMAP", "SIGOPS_NO_FIR_TMAP", "SIGOPS_NO_FIR_MMA", "SIGOPS_NO_FIR_BANDS"])
def test_kernel_paths(knob, monkeypatch):
    monkeypatch.setenv(knob, "1")
    name = "norm_iir_stereo" if knob == "SIGOPS_NO_TMAP" else "corpus"
    check(GPUSink(), signals(name, lengths_for(72, 960, 30000, seed=5)))


def test_many_waves_lengths_over_100x(monkeypatch):
    monkeypatch.setenv("SIGOPS_WS_BYTES", str(64 << 20))
    lens = lengths_for(60, 480, 48000, seed=7) + [480, 48000]
    check(GPUSink(), signals("corpus", lens))


def test_stale_workspace_reads_zero_tails():
    gpu = GPUSink()
    fs, C, chain = CHAINS["corpus"]
    junk = [np.full((44100, C), np.nan, order="F") for _ in range(64)]
    sink([chain(x) for x in junk], gpu)                                   # leaves NaN in every temp of the workspace
    check(gpu, signals("corpus", lengths_for(64, 441, 44100, seed=9) + [0]))


def test_two_devices():
    import ctypes
    n = ctypes.c_int()
    load().sigops_device_count(ctypes.byref(n))
    if n.value < 2:
        pytest.skip("one device")
    check(GPUSink([0, 1]), signals("corpus", lengths_for(48, 960, 30000, seed=11)))
