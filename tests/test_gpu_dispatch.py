"""Which kernel the launch planner of csrc/runtime.cu picks for a stage, read from its SIGOPS_DEBUG line
(`[sigops] IIR stage 0: tma rows=… matrix=1`).  The line is printed when a wave's launches are prepared, not when
they are replayed, so every case runs on a sink of its own.

IIR: tensor-map (Float64, Float32, fused row-invariant programs), per-lane TMA (WARM and MAIN + CARRY + FIX),
cp.async, generic.  FIR: tensor-map (with and without the period tables), per-row tensor-core, scalar.  The two
paths only device-resident rows off a 16-byte boundary take (cp.async, scalar) are also checked against the oracle."""
import re

import numpy as np
import pytest

import oracle
from signalops import (AffineSin, Amplify, Bandpass, Bandstop, Filt, GPUSink, Hz, Lowpass, Mix, Normpower, Ramp, Signal,
                       ToFramerate, Until, cabi, dB, kHz, ms, s, sin, sink_batch)
from signalops.lowering import lower

pytestmark = pytest.mark.gpu
LINE = re.compile(r"^\[sigops\] (IIR|FIR) stage \d+: (.+?) rows=.*$", re.M)


def rms(a):
    return float(np.sqrt(np.mean(np.asarray(a, dtype=np.float64) ** 2)))


@pytest.fixture
def fresh_sink(monkeypatch):
    """A sink of its own (nothing prepared yet), with planner debug lines on and each batch in one wave."""
    monkeypatch.setenv("SIGOPS_DEBUG", "1")
    monkeypatch.setenv("SIGOPS_HOST_WAVES", "1")
    g = GPUSink([0])
    yield g
    g.close()


def stage_lines(capfd, kind):
    """(kernel, whole line) of every `kind` stage line printed since the last call."""
    return [(m.group(2), m.group(0)) for m in LINE.finditer(capfd.readouterr().err) if m.group(1) == kind]


def kernels(capfd, kind):
    return {k for k, _ in stage_lines(capfd, kind)}


def run_device_misaligned(g, chain, xs):
    """xs: (ninst, nch, n) Float64.  The inputs sit one element past a 16-byte boundary in device memory."""
    import torch
    ninst, nch, n = xs.shape
    plan = lower(chain(np.zeros((n, nch))))
    cp = g.compiled(plan.tobytes())
    n_out = plan.outputs[0].nframes
    store = torch.zeros(xs.size + 1, dtype=torch.float64, device="cuda")
    x = store[1:].view(ninst, nch, n)
    x.copy_(torch.from_numpy(xs))
    y = torch.zeros((ninst, nch, n_out), dtype=torch.float64, device="cuda")
    assert x.data_ptr() % 16 == 8
    ins = (cabi.Buffer * ninst)(*[cabi.Buffer(x[i].data_ptr(), n, nch, cabi.F64, n) for i in range(ninst)])
    outs = (cabi.Buffer * ninst)(*[cabi.Buffer(y[i].data_ptr(), n_out, nch, cabi.F64, n_out) for i in range(ninst)])
    torch.cuda.synchronize()
    cp.run_device(ninst, ins, outs)
    torch.cuda.synchronize()
    return y.cpu().numpy()


def lowpass(x, fs=48 * kHz):
    return Signal(x, fs) >> Filt(Lowpass, 4 * kHz, order=8) >> Amplify(-20 * dB)


def test_iir_tensor_map_f64(fresh_sink, capfd):
    rng = np.random.default_rng(1)
    sink_batch([lowpass(rng.standard_normal((48000, 2))) for _ in range(16)], fresh_sink)     # 32 rows
    assert kernels(capfd, "IIR") == {"tensor-map"}


def test_iir_tensor_map_f32(fresh_sink, capfd):
    rng = np.random.default_rng(2)
    chain = lambda x: Signal(x, 48 * kHz) >> Filt(Lowpass, 4 * kHz, order=8) >> Amplify(np.float32(-20) * dB)   # noqa: E731
    sink_batch([chain(rng.standard_normal((48000, 2)).astype(np.float32)) for _ in range(16)], fresh_sink)
    assert kernels(capfd, "IIR") == {"tensor-map (Float32)"}


def test_iir_tensor_map_fused_row_invariant_programs(fresh_sink, capfd):
    rng = np.random.default_rng(3)

    def chain(x):
        am = Amplify(Signal(x, 96 * kHz), Signal(AffineSin(0.5, 0.5), ω=5 * Hz)) >> Until(0.5 * s)
        return am >> Filt(Bandpass, 500 * Hz, 4 * kHz) >> Ramp(10 * ms) >> Mix(Signal(sin, ω=1 * kHz) >> Until(0.5 * s))
    sink_batch([chain(np.asfortranarray(rng.standard_normal((48000, 32)))) for _ in range(3)], fresh_sink)   # 96 rows
    assert kernels(capfd, "IIR") == {"tensor-map (fused row-invariant programs)"}


def test_iir_per_lane_tma_warm(fresh_sink, capfd):
    """3 rows: too few to fill the tensor-map kernel's warps; the filter decays within a short chunk."""
    rng = np.random.default_rng(4)
    sink_batch([lowpass(rng.standard_normal((48000, 1))) for _ in range(3)], fresh_sink)
    (k, line), = stage_lines(capfd, "IIR")
    assert k == "tma" and line.endswith("matrix=0")


def test_iir_per_lane_tma_carry_pass(fresh_sink, capfd):
    """A band-stop that takes ~3300 frames to decay, on 80 rows: chunks far shorter than the decay, MAIN + CARRY + FIX."""
    rng = np.random.default_rng(5)
    chain = lambda x: Signal(x, 44.1 * kHz) >> Filt(Bandstop, 0.5 * kHz, 2 * kHz) >> Normpower >> Amplify(-20 * dB)   # noqa: E731
    sink_batch([chain(rng.standard_normal((44100, 2))) for _ in range(40)], fresh_sink)
    (k, line), = stage_lines(capfd, "IIR")
    assert k == "tma" and line.endswith("matrix=1")


def test_iir_cp_async_on_unaligned_device_rows(fresh_sink, capfd):
    rng = np.random.default_rng(6)
    xs = rng.standard_normal((3, 2, 48000))
    y = run_device_misaligned(fresh_sink, lowpass, xs)
    assert kernels(capfd, "IIR") == {"cp.async"}
    for k in (0, 2):
        want, _ = oracle.sink(lowpass(xs[k].T))
        assert np.max(np.abs(y[k].T - want)) <= 1e-9 * rms(want)


def test_iir_generic(fresh_sink, capfd):
    """Float32 on one row: no tensor-map kernel (too few rows), no Float64 fast path."""
    rng = np.random.default_rng(7)
    chain = lambda x: Signal(x, 48 * kHz) >> Filt(Lowpass, 4 * kHz, order=8) >> Amplify(np.float32(-20) * dB)   # noqa: E731
    sink_batch([chain(rng.standard_normal((16000, 1)).astype(np.float32))], fresh_sink)
    assert kernels(capfd, "IIR") == {"generic"}


def test_fir_tensor_map_with_period_tables(fresh_sink, capfd):
    """44.1 -> 48 kHz repeats every 160 outputs; 80 rows."""
    rng = np.random.default_rng(8)
    sink_batch([ToFramerate(Signal(rng.standard_normal((30000, 2)), 44.1 * kHz), 48 * kHz) for _ in range(40)], fresh_sink)
    (k, line), = stage_lines(capfd, "FIR")
    assert k == "tensor-map" and line.endswith(" (tap bands from the period tables)")


def test_fir_tensor_map_without_period_tables(fresh_sink, capfd):
    """44.1 kHz -> 47 999 Hz has no period within the table limit; 72 rows."""
    rng = np.random.default_rng(9)
    sink_batch([ToFramerate(Signal(rng.standard_normal((20000, 2)), 44100 * Hz), 47999 * Hz) for _ in range(36)], fresh_sink)
    (k, line), = stage_lines(capfd, "FIR")
    assert k == "tensor-map" and line.endswith(" outputs")


def test_fir_mma_up_to_64_rows(fresh_sink, capfd):
    rng = np.random.default_rng(10)
    sink_batch([ToFramerate(Signal(rng.standard_normal((5003, 2)), 48 * kHz), 44.1 * kHz) for _ in range(20)], fresh_sink)
    (k, line), = stage_lines(capfd, "FIR")
    assert k == "mma" and "rows=40 " in line and "rows/block=64 " in line


def test_fir_scalar_on_unaligned_device_rows(fresh_sink, capfd):
    rng = np.random.default_rng(11)
    xs = rng.standard_normal((3, 2, 4410))
    chain = lambda x: ToFramerate(Signal(x, 44.1 * kHz), 48 * kHz)   # noqa: E731
    y = run_device_misaligned(fresh_sink, chain, xs)
    assert kernels(capfd, "FIR") == {"scalar"}
    for k in (0, 2):
        want, _ = oracle.sink(chain(xs[k].T))
        assert y[k].shape == want.T.shape
        assert np.max(np.abs(y[k].T - want)) <= 1e-9 * rms(want)
