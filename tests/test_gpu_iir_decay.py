"""Every IIR kernel path (csrc/runtime.cu `plan_iir_stage`) on filters on both sides of the planner's decay-length
walk, which stops at 2^18 frames (`derive_iir`), sample for sample against the oracle's sequential DF2T.

A chunk of the WARM form starts Wc frames early from zero state, so it is exact only when the cascade's zero-input
response has died out within Wc; MAIN + CARRY + FIX is exact for any filter.  A response still alive at the walk's cap
has to be read as "never decays": a 0.5 Hz high-pass at 48 kHz needs ~1.8 M frames to fall to 2^-64, and a running
sum never does.  The inputs carry DC and a 0.3 Hz tone so that the slow states are loaded.

Shapes (one per kernel the planner can pick) and filters are crossed; each case checks every output sample of every
instance (the two fused shapes: the first and last instance), with the frame's offset in its chunk in the message.

Float64 bounds (max |err| / RMS against the oracle) are about 10x the worst case measured on a B200.  Two filters need
more than the 1e-11 of the others, and the reason is the carry pass, not a kernel: with MAIN + CARRY + FIX the chunk
start states come from s_in[k] = s_zs[k-1] + A^L s_in[k-1], and the same algorithm emulated in numpy (double) shows the
same error against a quad-precision DF2T:
- `under_cap` (8 poles near z = 1): A^L has entries up to 1.6e19 at L = 1200, so the carry's sums cancel.  Measured
  1.8e-10 (the sequential filter's own error against quad: 2e-11).
- `over_cap`: the rounding of A^L, which is computed once and applied at every chunk, adds up coherently over the
  800 chunks of a row.  Measured 7.7e-8 (the sequential filter's own error: 5.8e-10).
The two fused shapes also mix in a 1 kHz tone and a 5 Hz modulator.  At frame 840 000 the tone's phase is 1.1e5 rad,
one ulp of which is 1.5e-11, so two equally valid ways of computing it (n * (w / fs) or (n / fs) * w) already differ by
that much.  The per-lane program kernel measured 3.9e-11 there, away from any chunk boundary; those shapes get 4e-10.
Float32 output is rounded once from the Float64 result: |err| <= max(ulp32(ref), bound * RMS), where the floor is
1e-12 * RMS for the well-conditioned filters."""
import math
import re

import numpy as np
import pytest

import oracle
from signalops import (AffineSin, Amplify, Bandstop, Filt, GPUSink, Highpass, Hz, Lowpass, Mix, Normpower,
                       PolynomialRatio, Ramp, Signal, Until, dspjl, frames, kHz, ms, sin, sink_batch)
from signalops.graph import FilteredSignal
from test_gpu_dispatch import run_device_misaligned

N = 960_000                # 20 s at 48 kHz: past the walk's cap, several chunks of it per row
N_LONG = 4_423_680         # >= 16 * 2^18 with margin: choose_iir_chunking's long-chunk branch
CAP = 1 << 18
# max |err| / RMS allowed in Float64 (see the module docstring)
TOL = {"fast": 1e-11, "slow": 1e-11, "never": 1e-11, "under_cap": 2e-9, "over_cap": 1e-6}
FUSED_TOL = 4e-10
LINE = re.compile(r"^\[sigops\] IIR stage \d+: (.+?) (rows=.*)$", re.M)

FILTERS = {     # frame rate in Hz, filter
    "fast": (48000.0, lambda: Filt(Lowpass, 4 * kHz, order=8)),
    "slow": (44100.0, lambda: Filt(Bandstop, 0.5 * kHz, 2 * kHz)),
    "under_cap": (48000.0, lambda: Filt(Lowpass, 10 * Hz, order=8)),
    "over_cap": (48000.0, lambda: Filt(Highpass, 0.5 * Hz, order=4)),
    "never": (48000.0, lambda: Filt(PolynomialRatio([1.0], [1.0, -1.0]))),
}
# (kernel named by the debug line for `fast`, instances, channels, Float32, frames)
SHAPES = {
    "tmap_f64": ("tensor-map", 16, 2, False, N),
    "tmap_f32": ("tensor-map (Float32)", 16, 2, True, N),
    "tmap_fused": ("tensor-map (fused row-invariant programs)", 3, 32, False, N),
    "tma_prog": ("tma", 3, 32, False, N),
    "tma": ("tma", 3, 1, False, N),
    "tma_carry": ("tma", 40, 2, False, N),
    "cp_async": ("cp.async", 3, 2, False, N),
    "generic": ("generic", 1, 1, True, N),
    "generic_long": ("generic", 1, 1, True, N_LONG),
}
FUSED = ("tmap_fused", "tma_prog")


def rms(a):
    return float(np.sqrt(np.mean(np.asarray(a, dtype=np.float64) ** 2)))


def pole_frames(fid):
    """Frames for the slowest pole of the filter's sections to fall to 2^-64 (inf when |p| >= 1)."""
    fs, filt = FILTERS[fid]
    h = filt()(Signal(np.zeros((1, 1)), fs * Hz))
    assert isinstance(h, FilteredSignal)
    coef = dspjl.to_sos(h.fn(fs * Hz)).coef_table()
    r = max(abs(p) for b0, b1, b2, a1, a2 in coef for p in np.roots([1.0, a1, a2]))
    return math.inf if r >= 1.0 else 64 * math.log(2) / -math.log(r)


def test_pole_estimates_sit_on_their_side_of_the_cap():
    est = {fid: pole_frames(fid) for fid in FILTERS}
    assert est["fast"] < 1000 and 3000 < est["slow"] < 3600
    assert 150_000 < est["under_cap"] < CAP < N
    assert N < est["over_cap"] < math.inf and est["never"] == math.inf


def inputs(fid, ninst, nch, n, f32, seed):
    """White noise + 0.5 DC + 0.05 sin(2 pi 0.3 Hz t) ((n, nch) each); integers in [-8, 8] for the running sum."""
    rng = np.random.default_rng(seed)
    fs = FILTERS[fid][0]
    if fid == "never":
        xs = [rng.integers(-8, 9, size=(n, nch)).astype(np.float64) for _ in range(ninst)]
    else:
        drift = 0.5 + 0.05 * np.sin(2 * np.pi * 0.3 * np.arange(n) / fs)[:, None]
        xs = [rng.standard_normal((n, nch)) + drift for _ in range(ninst)]
    return [x.astype(np.float32) if f32 else x for x in xs]


def chain_for(fid, shape, normpower=False):
    fs, filt = FILTERS[fid]

    def plain(x):
        y = Signal(x, fs * Hz) >> filt()
        return y >> Normpower if normpower else y

    def fused(x):
        """BASELINE config 5's chain with the filter swapped: AM noise |> Filt |> Ramp |> Mix(tone)."""
        n = x.shape[0]
        am = Amplify(Signal(x, fs * Hz), Signal(AffineSin(0.5, 0.5), ω=5 * Hz)) >> Until(n * frames)
        return am >> filt() >> Ramp(10 * ms) >> Mix(Signal(sin, ω=1 * kHz) >> Until(n * frames))
    return fused if shape in FUSED else plain


@pytest.fixture
def fresh_sink(monkeypatch):
    """A sink of its own (planner lines are printed when a wave is prepared), each batch in one wave."""
    monkeypatch.setenv("SIGOPS_DEBUG", "1")
    monkeypatch.setenv("SIGOPS_HOST_WAVES", "1")
    g = GPUSink([0])
    yield g
    g.close()


def iir_lines(capfd):
    """[(kernel, {field: int})] of the IIR stage lines printed since the last read."""
    return [(m.group(1), {k: int(v) for k, v in re.findall(r"([\w/]+)=(\d+)", m.group(2))})
            for m in LINE.finditer(capfd.readouterr().err)]


def run(shape, g, chain, xs, monkeypatch):
    if shape == "tma_prog":
        monkeypatch.setenv("SIGOPS_NO_TMAP_LEAVES", "1")
    if shape == "cp_async":
        return [y.T for y in run_device_misaligned(g, chain, np.stack([x.T for x in xs]))]
    return [y for y, _ in sink_batch([chain(x) for x in xs], g)]


def compare(got, want, f32, tol, Ls, what):
    """Every sample; the message names the worst one's channel and frame, and the frame's offset in its chunk."""
    assert got.shape == want.shape and got.dtype == want.dtype, what
    g, w = got.astype(np.float64), want.astype(np.float64)
    err = np.abs(g - w)
    r = rms(w)
    if f32:
        floor = 1e-12 if tol <= 1e-11 else tol
        bound = np.maximum(np.spacing(np.abs(want)).astype(np.float64), floor * r)
    else:
        bound = np.full_like(w, tol * r)
    bad = err > bound
    if bad.any() or not np.isfinite(g).all():
        n, ch = np.unravel_index(np.argmax(np.where(np.isfinite(err), err / bound, np.inf)), err.shape)
        mods = ", ".join(f"frame mod {L} = {n % L}" for L in Ls)
        pytest.fail(f"{what}: {int(bad.sum())} samples off; worst at channel {ch}, frame {n} ({mods}): got {g[n, ch]!r}, want {w[n, ch]!r}, |err|/rms = {err[n, ch] / r:.3e}")
    return float(err.max() / r) if r else 0.0


_fused_refs = {}


def reference(chain, x, key):
    """oracle.sink; with a key, the last fused case's references are kept for the other fused shape."""
    if key is None:
        return oracle.sink(chain(x))[0]
    if key not in _fused_refs:
        if any(k[0] != key[0] for k in _fused_refs):
            _fused_refs.clear()
        _fused_refs[key] = oracle.sink(chain(x))[0]
    return _fused_refs[key]


def check_case(fid, shape, g, capfd, monkeypatch, normpower=False):
    kernel, ninst, nch, f32, n = SHAPES[shape]
    # (the two fused shapes take the same inputs and share the oracle's slow references)
    seed = 100 * list(FILTERS).index(fid) + list(SHAPES).index(FUSED[0] if shape in FUSED else shape) + 50 * normpower
    xs = inputs(fid, ninst, nch, n, f32, seed)
    chain = chain_for(fid, shape, normpower)
    got = run(shape, g, chain, xs, monkeypatch)
    lines = iir_lines(capfd)        # one per wave: a large batch may be split
    assert lines
    for k, f in lines:
        print(f"{fid}/{shape}: {k} {f}")
        if fid == "fast":
            assert k == kernel, f"{shape} was meant for the {kernel} kernel, got: {k} {f}"
        if fid in ("over_cap", "never"):
            assert not k.startswith("tensor-map") and (f["matrix"] == 1 or f["chunks/row"] == 1), f"WARM over chunks: {k} {f}"
            assert f["W"] >= min(pole_frames(fid), n), f
    Ls = sorted({f["L"] for _, f in lines})
    checked = (0, ninst - 1) if shape in FUSED else range(ninst)
    worst = 0.0
    for i in checked:
        want = reference(chain, xs[i], (fid, i) if shape in FUSED else None)
        worst = max(worst, compare(got[i], want, f32, max(TOL[fid], FUSED_TOL) if shape in FUSED else TOL[fid], Ls, f"{fid}/{shape} instance {i}"))
        if fid == "never" and shape not in FUSED and not normpower:
            # integer partial sums: exact in any order, on the carry path too (A^L = [[1, 1], [0, 0]])
            exact = np.cumsum(xs[i].astype(np.int64), axis=0).astype(got[i].dtype)
            assert np.array_equal(got[i], exact), f"{fid}/{shape} instance {i}: running sum not bit-exact"
    print(f"{fid}/{shape}: max |err|/rms = {worst:.3e}")


@pytest.mark.gpu
@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("fid", list(FILTERS))
def test_iir_paths_match_the_sequential_filter(fid, shape, fresh_sink, capfd, monkeypatch):
    check_case(fid, shape, fresh_sink, capfd, monkeypatch)


@pytest.mark.gpu
@pytest.mark.parametrize("fid", ["over_cap", "never"])
def test_normpower_sums_every_fixed_frame(fid, fresh_sink, capfd, monkeypatch):
    """Normpower after MAIN + CARRY + FIX: the sum of squares has to take the frames FIX rewrites over a whole chunk."""
    check_case(fid, "tma_carry", fresh_sink, capfd, monkeypatch, normpower=True)
