"""FIR stages whose filter bank does not fit in shared memory (csrc/k_fir_long.cuh): strong down-sampling
(`ToFramerate` below ~0.29 of the input rate) and long `FIRFilter` banks of every kind, sample for sample against
the oracle and, where they apply, `scipy.signal.lfilter` / `upfirdn`.

Shapes: one row, three rows, more than 64 rows in one strided batch, a signal shorter than the filter, output lengths
that are not a multiple of the 64-output tile, several host waves, device rows off a 16-byte boundary and outputs
pre-filled with NaN.  Epilogues: a constant gain (folded into the taps) and the sum of squares of a following
`Normpower`.  The planner's debug line names the kernel: `long` for these stages, the kernel they always had for the
shapes that planned before."""
import re
from fractions import Fraction

import numpy as np
import pytest
from scipy import signal as sps

import oracle
from signalops import Amplify, Filt, GPUSink, Hz, Normpower, Signal, ToFramerate, cabi, dB, dspjl, kHz, sink, sink_batch
from signalops.lowering import LEAF_CONST, LEAF_STAGE, OP_ADD, OP_LOAD, STAGE_FIR, Instr, lower

pytestmark = pytest.mark.gpu
F64_TOL = 1e-9
SCIPY_TOL = 1e-12
LINE = re.compile(r"^\[sigops\] FIR stage \d+: (\S+) rows=.*$", re.M)


def rms(a):
    return float(np.sqrt(np.mean(np.asarray(a, dtype=np.float64) ** 2)))


def rel_err(got, want):
    return float(np.max(np.abs(np.asarray(got, dtype=np.float64) - want))) / rms(want)


def resample(fi, fo):
    return lambda x: ToFramerate(Signal(x, fi * Hz), fo * Hz)


def fir(h, ratio=1, fs=48 * kHz):
    return lambda x: Signal(x, fs) >> Filt(dspjl.FIRFilter(h, ratio))


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


def run_device_nan_filled(g, chain, xs):
    """As above on aligned rows, with every output sample NaN before the run: a sample the kernel skips stays NaN."""
    import torch
    ninst, nch, n = xs.shape
    plan = lower(chain(np.zeros((n, nch))))
    cp = g.compiled(plan.tobytes())
    n_out = plan.outputs[0].nframes
    x = torch.from_numpy(xs).to("cuda")
    y = torch.full((ninst, nch, n_out), float("nan"), dtype=torch.float64, device="cuda")
    ins = (cabi.Buffer * ninst)(*[cabi.Buffer(x[i].data_ptr(), n, nch, cabi.F64, n) for i in range(ninst)])
    outs = (cabi.Buffer * ninst)(*[cabi.Buffer(y[i].data_ptr(), n_out, nch, cabi.F64, n_out) for i in range(ninst)])
    torch.cuda.synchronize()
    cp.run_device(ninst, ins, outs)
    torch.cuda.synchronize()
    return y.cpu().numpy()


@pytest.fixture
def fresh_sink(monkeypatch):
    """A sink of its own, with planner debug lines on and each batch in one wave."""
    monkeypatch.setenv("SIGOPS_DEBUG", "1")
    monkeypatch.setenv("SIGOPS_HOST_WAVES", "1")
    g = GPUSink([0])
    yield g
    g.close()


def fir_kernels(capfd):
    return [m.group(1) for m in LINE.finditer(capfd.readouterr().err)]


# ---- strong down-sampling: ToFramerate on data signals ---------------------------------------------------------

@pytest.mark.parametrize("fi,fo,n,nch,ninst", [
    (48000, 8000, 20011, 1, 1),          # speech rate, 219 taps/phase; one row
    (48000, 11025, 20000, 3, 1),         # three rows
    (48000, 12000, 9001, 2, 40),         # 80 rows in one strided batch
    (44100, 8000, 30000, 1, 3),          # 201 taps/phase
    (192000, 48000, 40000, 2, 2),
    (48000, 1000, 96000, 1, 2),          # 1742 taps/phase: beyond the former cap of 1024
])
def test_strong_downsampling_matches_oracle(gpu, fi, fo, n, nch, ninst):
    rng = np.random.default_rng(n + nch)
    xs = [rng.standard_normal((n, nch)) for _ in range(ninst)]
    chain = resample(fi, fo)
    got = sink_batch([chain(x) for x in xs], gpu)
    for k in sorted({0, ninst - 1}):
        want, fs = oracle.sink(chain(xs[k]))
        assert got[k][1] == fs == float(fo) and got[k][0].shape == want.shape
        assert rel_err(got[k][0], want) <= F64_TOL, k


def test_tone_survives_48k_to_8k_at_unit_gain(gpu):
    """A 1 kHz tone, under the new Nyquist frequency, comes out as the same tone at 8 kHz with unit gain and zero delay
    (the 60 dB design spec of `resample_filter`, as in test_resample_analytic.py)."""
    fi, fo, f = 48000.0, 8000.0, 1000.0
    x = np.sin(2 * np.pi * f * np.arange(int(fi)) / fi)
    y, fs = sink(ToFramerate(Signal(x, fi * Hz), fo * Hz), gpu)
    assert fs == fo and y.shape == (8000, 1)
    m = np.arange(8000)
    ref = np.sin(2 * np.pi * f * m / fo)
    sl = slice(500, 7500)
    assert np.max(np.abs(y[sl, 0] - ref[sl])) < 10 ** (-60 / 20) * 1.2


# ---- long FIRFilter banks --------------------------------------------------------------------------------------

@pytest.mark.parametrize("ntaps,n,nch", [(202, 20000, 2), (1025, 12345, 1), (4097, 30000, 3), (4097, 3000, 1)])
def test_single_rate_fir_filter_matches_lfilter(gpu, ntaps, n, nch):
    """`Filt(x, FIRFilter(h))` with firwin designs; (4097, 3000): a signal shorter than the filter."""
    h = sps.firwin(ntaps, 0.2)
    x = np.random.default_rng(ntaps + n).standard_normal((n, nch))
    chain = fir(h)
    got, _ = sink(chain(x), gpu)
    want, _ = oracle.sink(chain(x))
    ref = np.stack([sps.lfilter(h, 1.0, x[:, c]) for c in range(nch)], axis=1)
    assert got.shape == want.shape == (n, nch)
    assert rel_err(got, want) <= F64_TOL
    err = rel_err(got, ref)
    print(f"FIRFilter {ntaps} taps: max error / rms against lfilter {err:.2e}")
    assert err <= SCIPY_TOL


@pytest.mark.parametrize("ntaps,ratio,up,down", [
    (1500, Fraction(1, 5), 1, 5),        # decimator, 1500 taps
    (2048, 4, 4, 1),                     # interpolator, 512 taps/phase
    (1200, Fraction(2, 7), 2, 7),        # rational, 600 taps/phase
])
def test_resampling_fir_filter_matches_upfirdn(gpu, ntaps, ratio, up, down):
    """`Filt(x, FIRFilter(h, p//q))`: the oracle has no such filter; `upfirdn` computes the same stream."""
    h = sps.firwin(ntaps, 0.8 / max(up, down))
    xs = [np.random.default_rng(ntaps + k).standard_normal((9001, 2)) for k in range(36)]     # 72 rows
    got = sink_batch([fir(h, ratio)(x) for x in xs], gpu)
    for k in (0, 35):
        y = got[k][0]
        for c in range(2):
            u = sps.upfirdn(h, xs[k][:, c], up, down)
            nn = min(len(u), len(y))
            assert rel_err(y[:nn, c], u[:nn]) <= SCIPY_TOL
            assert not np.any(y[nn:, c])             # past the stream the input is zero padding


# ---- epilogues -------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("chain", [
    lambda x: ToFramerate(Signal(x, 48 * kHz), 8 * kHz) >> Amplify(-6 * dB),
    lambda x: fir(sps.firwin(1025, 0.3))(x) >> Amplify(-6 * dB),
    lambda x: ToFramerate(Signal(x, 48 * kHz), 12 * kHz) >> Normpower >> Amplify(-20 * dB),
    lambda x: fir(sps.firwin(1025, 0.3))(x) >> Normpower,
], ids=["resample-gain", "fir-gain", "resample-normpower", "fir-normpower"])
@pytest.mark.parametrize("ninst", [1, 40])
def test_gain_and_normpower(gpu, chain, ninst):
    xs = [np.random.default_rng(100 + k).standard_normal((7003, 2)) * (1 + k) for k in range(ninst)]
    got = sink_batch([chain(x) for x in xs], gpu)
    for k in sorted({0, ninst - 1}):
        want, _ = oracle.sink(chain(xs[k]))
        assert rel_err(got[k][0], want) <= F64_TOL


def test_rational_normpower_sum_of_squares(gpu):
    """The oracle has no rational FIRFilter: check the Normpower scale against upfirdn."""
    h = sps.firwin(1200, 0.1)
    x = np.random.default_rng(5).standard_normal((7003, 2))
    y, _ = sink(Signal(x, 48 * kHz) >> Filt(dspjl.FIRFilter(h, Fraction(2, 7))) >> Normpower, gpu)
    u = np.zeros_like(y)                             # the stream, then the zero padding of the input
    for c in range(2):
        v = sps.upfirdn(h, x[:, c], 2, 7)[:len(y)]
        u[:len(v), c] = v
    ref = u / np.sqrt(np.mean(u ** 2))               # one power over all channels
    assert rel_err(y, ref) <= 1e-11


# ---- input kinds and batch shapes ------------------------------------------------------------------------------

def test_float32_input(gpu):
    x = np.random.default_rng(6).standard_normal((20000, 2)).astype(np.float32)
    chain = resample(48000, 8000)
    got, _ = sink(chain(x), gpu)
    want, _ = oracle.sink(chain(x))
    assert got.dtype == want.dtype == np.float32
    # widened on the way in, rounded once on the way out: one Float32 rounding of the same value
    assert np.max(np.abs(got.astype(np.float64) - want)) <= 2.0 ** -23 * np.max(np.abs(want))


def test_several_waves(monkeypatch):
    """A small workspace budget splits the batch into several host waves."""
    monkeypatch.setenv("SIGOPS_WS_BYTES", str(64 << 20))
    g = GPUSink([0])
    try:
        xs = [np.random.default_rng(200 + k).standard_normal((120000, 2)) for k in range(40)]
        chain = resample(48000, 8000)
        got = sink_batch([chain(x) for x in xs], g)
        assert g.last_stats["launches"] > 1          # one launch per wave
        for k in (0, 21, 39):
            want, _ = oracle.sink(chain(xs[k]))
            assert rel_err(got[k][0], want) <= F64_TOL
    finally:
        g.close()


@pytest.mark.parametrize("chain", [resample(48000, 8000), fir(sps.firwin(1025, 0.25))], ids=["resample", "fir"])
def test_unaligned_device_rows(fresh_sink, capfd, chain):
    xs = np.random.default_rng(7).standard_normal((3, 2, 12001))
    y = run_device_misaligned(fresh_sink, chain, xs)
    assert fir_kernels(capfd) == ["long"]
    for k in (0, 2):
        want, _ = oracle.sink(chain(xs[k].T))
        assert rel_err(y[k].T, want) <= F64_TOL


@pytest.mark.parametrize("chain,n", [(resample(48000, 8000), 12001), (resample(192000, 48000), 40003),
                                     (fir(sps.firwin(4097, 0.25)), 5001)], ids=["48k-8k", "192k-48k", "fir4097"])
def test_every_output_sample_is_written(fresh_sink, capfd, chain, n):
    xs = np.random.default_rng(8).standard_normal((70, 1, n))     # 70 rows; n_out not a multiple of 64
    y = run_device_nan_filled(fresh_sink, chain, xs)
    assert fir_kernels(capfd) == ["long"]
    assert not np.isnan(y).any()
    for k in (0, 69):
        want, _ = oracle.sink(chain(xs[k].T))
        assert rel_err(y[k].T, want) <= F64_TOL


# ---- dispatch and limits ---------------------------------------------------------------------------------------

@pytest.mark.parametrize("fi,fo,nch,ninst,kernel", [
    (48000, 8000, 1, 1, "long"),
    (48000, 1000, 2, 3, "long"),
    (44100, 8000, 2, 40, "long"),
    (44100, 48000, 2, 40, "tensor-map"),    # 80 rows
    (44100, 48000, 2, 20, "mma"),           # 40 rows
    (48000, 44100, 2, 20, "mma"),
])
def test_dispatch_resample(fresh_sink, capfd, fi, fo, nch, ninst, kernel):
    rng = np.random.default_rng(9)
    sink_batch([resample(fi, fo)(rng.standard_normal((20000, nch))) for _ in range(ninst)], fresh_sink)
    assert fir_kernels(capfd) == [kernel]


@pytest.mark.parametrize("make,kernel", [
    (lambda x: ToFramerate(Signal(x, 48 * kHz), 16 * kHz), "mma"),     # decimator 1/3
    (fir(sps.firwin(201, 0.3)), "scalar"),                                # the longest bank k_fir holds
    (fir(sps.firwin(202, 0.3)), "long"),
    (fir(sps.firwin(4097, 0.3)), "long"),
    (lambda x: Signal(x, 48 * kHz) >> Filt(dspjl.FIRFilter(sps.firwin(1500, 0.1), Fraction(1, 5))), "long"),
])
def test_dispatch_fir(fresh_sink, capfd, make, kernel):
    sink(make(np.random.default_rng(10).standard_normal((20000, 2))), fresh_sink)
    assert fir_kernels(capfd) == [kernel]


def test_bank_over_the_cap_is_unsupported(gpu):
    plan = lower(fir(np.ones(65537) / 65537)(np.zeros((70000, 1))))
    with pytest.raises(cabi.SigopsError) as e:
        gpu.compiled(plan.tobytes())
    assert e.value.code == -2 and "65536" in e.value.msg


def test_long_bank_with_a_richer_epilogue_is_unsupported(gpu):
    """A hand-built plan: a long bank followed by `y + 1` (the lowering keeps that a separate pass)."""
    plan = lower(resample(48000, 8000)(np.zeros((20000, 1))))
    st = next(s for s in plan.stages if s.kind == STAGE_FIR)
    st.epi_prog = [Instr(OP_LOAD, LEAF_STAGE, buf=0), Instr(OP_ADD, LEAF_CONST, d0=1.0)]
    with pytest.raises(cabi.SigopsError) as e:
        gpu.compiled(plan.tobytes())
    assert e.value.code == -2 and "shared memory per block" in e.value.msg
