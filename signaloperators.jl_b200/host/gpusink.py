"""`sink(x, GPUSink())` — the drop-in for the reference's CPU `sink` (src/sink.jl).

Follows the reference's custom-sink contract (docs/src/custom_sink.md:1-18) and
the shape of its non-`Type` sink method `sink(x,to::String)` (src/sink.jl:139-142):
`process_sink_params`, then hand the signal to the backend, then wrap the data
like `initsink(x,T,data)` (src/sink.jl:120-121).  It never goes through
`nextblock`/`frame`/`sink_helper!`: the graph is lowered once (lowering.py) and
run by libsignalops_cuda.so.
"""
from __future__ import annotations

import hashlib

import numpy as np

from . import cabi, graph as G
from .lowering import Lowerer, np_dtype, ragged_plan
from .wav import WavRaw, write_wav
from .lowering import dtype_code as dtype_code_of


class Array:
    """Sink-type token: return a bare array (Julia `Array`)."""


class Tuple:
    """Sink-type token: return `(array, framerate)` (Julia `Tuple`)."""


class GPUSink:
    """Materialise on B200s.  `devices`: CUDA ordinals to shard batches over."""

    def __init__(self, devices=None, container=None, pin_results=False):
        self.devices = list(devices) if devices else [0]
        self.container = container
        # Page-locked result arrays are written by the DMA engines directly (2.5x the end-to-end rate of pageable
        # ones) but page-locking itself costs ~0.6 s per GB (measured), so it only pays when result blocks are
        # recycled: a sink that serves a steady stream of batches and drops each result before the next call.
        # Off by default; pageable results go through the library's own pinned staging ring.
        self.pin_results = bool(pin_results)
        self._ctx = None
        self._plans = {}
        self.last_stats = None

    @property
    def ctx(self):
        if self._ctx is None:
            self._ctx = cabi.Context(self.devices)
        return self._ctx

    def compiled(self, plan_bytes):
        key = hashlib.sha1(plan_bytes).digest()
        cp = self._plans.get(key)
        if cp is None:
            cp = cabi.CompiledPlan(self.ctx, plan_bytes)
            self._plans[key] = cp
        return cp

    def alloc_result(self, shape, dtype):
        """The array `sink` returns (`initsink`, src/sink.jl:115-121).  The sink allocates it, so it may be
        page-locked (`pin_results`): the device then writes it without the staged copy pageable memory needs."""
        nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        if self.pin_results and nbytes >= _PIN_MIN_BYTES:
            return cabi.pinned_empty(shape, dtype, order="F")      # from the pool of recycled blocks when there is one
        return np.empty(shape, dtype=dtype, order="F")

    def close(self):
        for cp in self._plans.values():
            cp.close()
        self._plans.clear()
        if self._ctx is not None:
            self._ctx.close()
            self._ctx = None


def _wrap(plan, data, to):
    container = to.container
    if container is Array:
        return data
    if container is Tuple or plan.wants_tuple:
        return data, plan.framerate
    return data


def _colmajor(a):
    if isinstance(a, WavRaw):
        return a
    return _colmajor_array(a)


def _colmajor_array(a):
    """Dense channel-planar view of `a` for the C ABI (element (n,c) at ptr[c*ld + n]): strided
    1-D / (N,1) views (`x[::2]`, `stereo[:,0]` of a C-ordered array, `x[::-1]`) and C-ordered
    matrices are copied; anything already dense in Julia's column-major layout is passed as is."""
    if a.ndim == 1 or a.shape[1] == 1:
        return a if a.size <= 1 or a.strides[0] == a.itemsize else np.ascontiguousarray(a)
    # column-major with any leading dimension >= nframes (a view of the first rows of a taller matrix) is fine
    ok = a.shape[0] <= 1 or (a.strides[0] == a.itemsize and a.strides[1] >= a.shape[0] * a.itemsize
                             and a.strides[1] % a.itemsize == 0)
    return a if ok else np.asfortranarray(a)


_PIN_MIN_BYTES = 1 << 20


# sample types the plan can write straight into the caller's array
_DIRECT_RESULT_DTYPES = (np.dtype(np.float32), np.dtype(np.float64), np.dtype(np.int64))


def sink(x=None, to=None):
    """`sink(x, GPUSink())`; `sink(GPUSink())` curries like `sink(to)` at src/sink.jl:29.
    A list/tuple of signals is a batch (one plan, many instances; additive API,
    SURVEY.md §8b)."""
    if isinstance(x, GPUSink) and to is None:
        return lambda y: sink(y, x)
    if not isinstance(to, GPUSink):
        raise G.SignalError(
            "this package only implements the GPU sink: call sink(x, GPUSink()). The CPU "
            "`sink` belongs to the reference (restated under oracle/ for tests).")
    if isinstance(x, list):
        return sink_batch(x, to)
    plan = Lowerer().build(x)
    out = plan.outputs[0]
    data = to.alloc_result((out.nframes, out.nchannels), np_dtype(out.dtype))
    if out.nframes > 0:
        cp = to.compiled(plan.tobytes())
        to.last_stats = cp.run_host(1, [_colmajor(a) for a in plan.input_arrays], [data])
    return _wrap(plan, data, to)


def sink_wav(x, path, to, encoding=None):
    """`sink(x, "file.wav")` (src/sink.jl:139-142 + src/WAV.jl:3-7) on the GPU sink: the root stage's output is
    transposed to frame-interleaved order and converted to the file's sample encoding on the device
    (csrc/k_wav.cuh), so the host only prepends the RIFF header.  `encoding`: "float64" (default for Float64
    signals, what WAV.jl writes for a Float64 matrix), "float32" (default for Float32 signals) or "pcm16"
    (round(clamp(x,-1,1)*32767)).  Returns the frame rate written, `round(Int, framerate(x))`."""
    if not isinstance(to, GPUSink):
        raise G.SignalError("sink_wav needs a GPUSink")
    plan = Lowerer().build(x)
    out = plan.outputs[0]
    if np_dtype(out.dtype) not in (np.float32, np.float64):
        raise G.SignalError("only floating-point signals are written as WAV by the GPU sink")
    enc = encoding or ("float32" if np_dtype(out.dtype) == np.float32 else "float64")
    dt = {"float64": np.float64, "float32": np.float32, "pcm16": np.int16}.get(enc)
    if dt is None:
        raise G.SignalError(f"unknown WAV encoding {enc!r}")
    nbytes = out.nframes * out.nchannels * np.dtype(dt).itemsize
    raw = (cabi.pinned_empty((out.nframes, out.nchannels), dt, order="C") if to.pin_results and nbytes >= _PIN_MIN_BYTES
           else np.empty((out.nframes, out.nchannels), dtype=dt))
    if out.nframes > 0:
        cp = to.compiled(plan.tobytes())
        to.last_stats = cp.run_host(1, [_colmajor(a) for a in plan.input_arrays], [WavRaw(raw)])
    fs = int(round(plan.framerate))
    write_wav(path, raw, fs)
    return fs


def sink_into(result, x, to):
    """`sink!(result, x)` (src/sink.jl:158-168): write size(result,1) frames — a
    prefix of `x` — into the caller's array, forcing the channel count."""
    if isinstance(result, tuple):
        return sink_into(result[0], x, to), result[1]
    x = G.Signal(x)
    n = result.shape[0]
    nch = 1 if result.ndim == 1 else result.shape[1]
    xn = x.nframes
    if xn is not None and not G.isknowninf(xn) and xn < n:
        raise G.SignalError(f"Signal is too short to fill buffer of length {n}.")
    lw = Lowerer()
    x = G.ToChannels(x, nch)
    # The reference's `sink!` accepts any result eltype (each frame is converted on assignment).
    # The device writes Float32/Float64/Int64; every other eltype (Int32, Int16, UInt8, Bool, ...) is
    # sunk in the signal's own sample type and converted on the host.
    direct = result.dtype in _DIRECT_RESULT_DTYPES
    plan_dtype = result.dtype if direct else np_dtype(dtype_code_of(x.sampletype))
    # the plan covers only the requested prefix, so infinite signals are fine here
    plan = _build_prefix(lw, x, n, plan_dtype)
    if n == 0:
        return result
    cp = to.compiled(plan.tobytes())
    dense = _colmajor(result) is result
    if direct and dense:
        to.last_stats = cp.run_host(1, [_colmajor(a) for a in plan.input_arrays], [result])
    elif (direct and result.ndim == 2 and result.shape[1] > 1 and result.flags.c_contiguous
          and result.dtype in (np.float32, np.float64)):
        # numpy's own (nframes, nchannels) layout is frame-interleaved: the device writes it directly (SIGOPS_INTERLEAVED)
        to.last_stats = cp.run_host(1, [_colmajor(a) for a in plan.input_arrays], [WavRaw(result)])
    else:
        # strided / C-ordered / narrow-integer results: run into a dense temporary and copy back
        tmp = np.empty(result.shape, dtype=plan_dtype, order="F")
        to.last_stats = cp.run_host(1, [_colmajor(a) for a in plan.input_arrays], [tmp])
        if direct or np.dtype(plan_dtype).kind in "iu":
            result[...] = tmp
        else:
            if result.dtype.kind in "iub" and not np.all(tmp == np.trunc(tmp)):
                raise G.SignalError(f"InexactError: cannot convert non-integral samples to {result.dtype}")
            result[...] = tmp.astype(result.dtype)
    return result


def _build_prefix(lw, x, n, dtype):
    from .lowering import STAGE_MAP, BufDesc, LoweringError, Stage, dtype_code
    C = x.nchannels
    try:
        lw.plan.outputs.append(BufDesc(n, C, dtype_code(dtype)))
        lw.plan.framerate = x.framerate
        pieces = lw.lower(x, 0, 0, n, 1, 0, 0, C) if n > 0 else []
        lw.plan.stages.append(Stage(STAGE_MAP, ("out", 0), pieces=pieces, nchannels=C, n_out=n))
        lw._fuse_epilogues()
        lw._check_limits()
    except LoweringError:
        nxt = lw.fallback()          # traced generators over a device limit: lower them the next way
        if nxt is None:
            raise
        return _build_prefix(nxt, x, n, dtype)
    return lw.plan


def sink_batch(xs, to):
    """Materialise many structurally identical graphs in one call.  Every graph is
    lowered; the plans must agree byte for byte (same operators, lengths and
    constants) and differ only in the arrays they read — or differ in lengths alone
    (a ragged batch: `_sink_ragged`)."""
    if not xs:
        return []
    lws = [Lowerer(instance_index=k) for k in range(len(xs))]
    plans = [lw.build(x) for lw, x in zip(lws, xs)]
    ref = plans[0].tobytes()
    if any(lw.traced_generators for lw in lws) and any(_unlike(p, plans[0]) for p in plans[1:]):
        # closure generators whose traced programs differ between elements (other ω, ϕ or constants): evaluated on
        # the host, their frames are input buffers and the plans agree again
        plans = [Lowerer(instance_index=k, generators="host").build(x) for k, x in enumerate(xs)]
        ref = plans[0].tobytes()
    if any(p.tobytes() != ref for p in plans[1:]):
        return _sink_ragged(plans, to)
    out = plans[0].outputs[0]
    datas = [to.alloc_result((out.nframes, out.nchannels), np_dtype(out.dtype)) for _ in xs]
    if out.nframes > 0:
        cp = to.compiled(ref)
        ins = [_colmajor(a) for p in plans for a in p.input_arrays]
        to.last_stats = cp.run_host(len(xs), ins, datas)
    return [_wrap(plans[0], d, to) for d in datas]


def _unlike(p, ref):
    """Do two plans differ in more than their lengths?"""
    try:
        ragged_plan([ref, p])
        return False
    except G.SignalError:
        return True


def _sink_ragged(plans, to):
    """Elements whose plans differ in lengths alone (include/signalops.h `sigops_plan_run_ragged`): one plan, the
    field-wise maximum of theirs, runs every element at its own lengths; each result has its own frame count.
    Elements of no frames take no part in the comparison (their plans have no pieces): they run as instances whose
    buffers are all empty, which keeps every other element's index in the call (its noise stream)."""
    live = [k for k, p in enumerate(plans) if p.outputs[0].nframes > 0]
    if not live:
        return [_wrap(p, to.alloc_result((0, p.outputs[0].nchannels), np_dtype(p.outputs[0].dtype)), to) for p in plans]
    mplan, tf = ragged_plan([plans[k] for k in live])
    if any(isinstance(a, WavRaw) for p in plans for a in p.input_arrays):
        raise G.SignalError("a batch of signals of different lengths cannot read WAV-layout buffers (WAV files, C-ordered "
                            "matrices): give the elements one length, or pass column-major arrays")
    temp_frames = np.zeros((len(plans), len(mplan.temps)), dtype=np.int64)
    temp_frames[live] = tf
    ins, datas = [], []
    for k, p in enumerate(plans):
        if k in live:
            ins += [_colmajor(a) for a in p.input_arrays]
        else:
            ins += [np.empty((0, b.nchannels), dtype=np_dtype(b.dtype), order="F") for b in mplan.inputs]
        o = mplan.outputs[0]
        datas.append(to.alloc_result((p.outputs[0].nframes, o.nchannels), np_dtype(o.dtype)))
    cp = to.compiled(mplan.tobytes())
    to.last_stats = cp.run_ragged(len(plans), ins, datas, temp_frames)
    return [_wrap(p, d, to) for p, d in zip(plans, datas)]
