"""Lower a finished lazy signal graph to the kernel plan `libsignalops_cuda.so` runs.

This is the GPU-side replacement for what the reference does *inside* `sink!`:
instead of pulling blocks through `nextblock`/`frame` (src/sink.jl:225-267 and
the per-node block types of SURVEY.md §8 row a3) the graph is cut at its
materialisation barriers {Filt, ToFramerate-on-data, Normpower, root} and every
region between two barriers becomes one elementwise program.  All lengths and
offsets (Until/After/Pad/Append plumbing, src/cutting.jl:130-214,
src/padding.jl:200-235, src/appending.jl:92-110, src/mapsignal.jl:219-244) are
resolved here, on the host, as exact integers.

The byte layout produced by `Plan.tobytes()` is the one documented in
include/signalops.h; julia/GPUSink.jl emits the same bytes from the reference's
own node types.
"""
from __future__ import annotations

import math
import struct
from dataclasses import dataclass, field, replace

import numpy as np

from . import dspjl, graph as G
from .functors import functor_code
from .philox import PhiloxRNG
from .trace import TraceError, trace
from .wav import WavSignal

# ---- constants mirrored from include/signalops.h -------------------------------
F32, F64, I64 = 1, 2, 3
OP_LOAD, OP_ADD, OP_SUB, OP_MUL, OP_DIV = 1, 2, 3, 4, 5
OP_PUSH, OP_POPADD, OP_POPSUB, OP_POPMUL, OP_POPDIV = 6, 7, 8, 9, 10
OP_NEG, OP_CAST_F32, OP_CAST_I64 = 11, 12, 13
OP_FN1, OP_FN2, OP_POPFN2 = 14, 15, 16
LEAF_NONE, LEAF_CONST, LEAF_BUF, LEAF_CHANSUM, LEAF_GEN = 0, 1, 2, 3, 4
LEAF_RAMP_ON, LEAF_RAMP_OFF, LEAF_RMS, LEAF_STAGE, LEAF_RANDN = 5, 6, 7, 8, 9
PAD_CONST, PAD_CYCLE, PAD_MIRROR, PAD_LAST = 0, 1, 2, 3
FLAG_HAS_OMEGA = 1
FN_SIN, FN_COS, FN_SAW, FN_AFFINE_SIN, FN_AFFINE_COS, FN_IDENTITY, FN_SINRAMP = 1, 2, 3, 4, 5, 6, 7
# closure functions (SIGOPS_EFN_*): unary codes for FN1, binary codes (from 32) for FN2 / POPFN2
EFN = {"abs": 1, "sign": 2, "floor": 3, "ceil": 4, "trunc": 5, "round": 6, "sqrt": 7, "clamp": 8, "exp": 9, "exp2": 10,
       "expm1": 11, "log": 12, "log2": 13, "log10": 14, "log1p": 15, "sin": 16, "cos": 17, "tan": 18, "tanh": 19,
       "sinh": 20, "cosh": 21, "atan": 22, "cbrt": 23,
       "min": 32, "max": 33, "copysign": 34, "rem": 35, "mod": 36, "pow": 37, "hypot": 38}
# leaves FN2 may take: the ones that do not read `fn` (generators and ramps keep their function there)
FN2_LEAVES = (LEAF_CONST, LEAF_BUF, LEAF_CHANSUM, LEAF_RMS, LEAF_STAGE, LEAF_RANDN)
STAGE_MAP, STAGE_IIR, STAGE_FIR = 1, 2, 3
FIR_ARBITRARY, FIR_RATIONAL, FIR_DECIMATOR = 1, 2, 3
MAX_STACK, MAX_PROG, MAX_PIECES, MAX_BUFS, MAX_SECTIONS = 4, 48, 64, 32, 8
MAGIC, PLAN_VERSION = 0x504F4753, 1

_ARITH_OPS = {"+": (OP_ADD, OP_POPADD), "-": (OP_SUB, OP_POPSUB),
              "*": (OP_MUL, OP_POPMUL), "/": (OP_DIV, OP_POPDIV)}


class LoweringError(G.SignalError):
    """The graph is valid but contains something the GPU path does not lower."""


def dtype_code(dt):
    dt = np.dtype(dt)
    if dt == np.float32:
        return F32
    if dt == np.float64:
        return F64
    if dt.kind in "iub":
        return I64
    raise LoweringError(f"sample type {dt} is not supported by the GPU sink")


def np_dtype(code):
    return {F32: np.float32, F64: np.float64, I64: np.int64}[code]


@dataclass(frozen=True)
class Instr:
    op: int = OP_LOAD
    leaf: int = LEAF_NONE
    fn: int = 0
    flags: int = 0
    buf: int = 0
    c_mul: int = 1
    c_off: int = 0
    i0: int = 0
    i1: int = 0
    i2: int = 0
    d0: float = 0.0
    d1: float = 0.0
    d2: float = 0.0
    d3: float = 0.0
    d4: float = 0.0

    def pack(self):
        return struct.pack("<4B3i3q5d", self.op, self.leaf, self.fn, self.flags, self.buf,
                           self.c_mul, self.c_off, self.i0, self.i1, self.i2,
                           self.d0, self.d1, self.d2, self.d3, self.d4)


@dataclass
class Piece:
    lo: int
    hi: int
    clo: int
    chi: int
    prog: list


@dataclass
class Stage:
    kind: int
    out_buf: int
    sumsq_slot: int = -1
    pieces: list = field(default_factory=list)      # MAP
    in_prog: list = field(default_factory=list)     # IIR/FIR
    epi_prog: list = field(default_factory=list)
    nchannels: int = 0
    n_in: int = 0
    n_out: int = 0
    n_sections: int = 0
    coef_table: int = -1
    gain: float = 1.0
    fir_kind: int = 0
    n_phases: int = 0
    taps_per_phase: int = 0
    pfb_table: int = -1
    dpfb_table: int = -1
    interpolation: int = 0
    decimation: int = 0
    input_deficit: int = 0
    rate: float = 0.0
    phase0: float = 0.0


@dataclass
class BufDesc:
    nframes: int
    nchannels: int
    dtype: int


class Plan:
    """The lowered form of one graph: stages + the host arrays that feed it."""

    def __init__(self):
        self.inputs: list[BufDesc] = []
        self.input_arrays: list[np.ndarray] = []    # (N,C) arrays, order of `inputs`
        self.temps: list[BufDesc] = []
        self.outputs: list[BufDesc] = []
        self.n_scalars = 0
        self.tables: list[np.ndarray] = []
        self.stages: list[Stage] = []
        self.framerate = None
        self.wants_tuple = True

    # buffer ids: inputs, then temps, then outputs — fixed up in tobytes()
    def tobytes(self):
        n_in, n_tmp = len(self.inputs), len(self.temps)

        def bid(tag):
            kind, k = tag
            return k if kind == "in" else (n_in + k if kind == "tmp" else n_in + n_tmp + k)

        def fix(prog):
            return [replace(I, buf=bid(I.buf)) if I.leaf in (LEAF_BUF, LEAF_CHANSUM) and
                    isinstance(I.buf, tuple) else I for I in prog]

        instrs, pieces, stages = [], [], []
        for st in self.stages:
            p_start = len(pieces)
            in_start = in_len = epi_start = epi_len = 0
            if st.kind == STAGE_MAP:
                for pc in st.pieces:
                    prog = fix(pc.prog)
                    pieces.append(struct.pack("<2q4i", pc.lo, pc.hi - pc.lo, pc.clo, pc.chi - pc.clo,
                                              len(instrs), len(prog)))
                    instrs += prog
            else:
                prog = fix(st.in_prog)
                in_start, in_len = len(instrs), len(prog)
                instrs += prog
                prog = fix(st.epi_prog)
                epi_start, epi_len = len(instrs), len(prog)
                instrs += prog
            stages.append(struct.pack(
                "<10i2q2id8iq2d", st.kind, bid(st.out_buf), st.sumsq_slot, p_start,
                len(st.pieces), in_start, in_len, epi_start, epi_len, st.nchannels,
                st.n_in, st.n_out, st.n_sections, st.coef_table, st.gain,
                st.fir_kind, st.n_phases, st.taps_per_phase, st.pfb_table, st.dpfb_table,
                st.interpolation, st.decimation, 0, st.input_deficit, st.rate, st.phase0))
        blob = np.concatenate([t.ravel() for t in self.tables]) if self.tables else np.zeros(0)
        offs, o = [], 0
        for t in self.tables:
            offs.append((o, t.size))
            o += t.size
        out = [struct.pack("<10IQ", MAGIC, PLAN_VERSION, n_in, n_tmp, len(self.outputs),
                           self.n_scalars, len(self.tables), len(instrs), len(pieces),
                           len(stages), blob.size)]
        for b in self.inputs + self.temps + self.outputs:
            out.append(struct.pack("<q2i", b.nframes, b.nchannels, b.dtype))
        for off, cnt in offs:
            out.append(struct.pack("<2q", off, cnt))
        out += [I.pack() for I in instrs]
        out += pieces
        out += stages
        out.append(np.ascontiguousarray(blob, dtype="<f8").tobytes())
        return b"".join(out)


def _isleaf(prog):
    return len(prog) == 1 and prog[0].op == OP_LOAD


def _as_operand(prog, op):
    """Program that combines the running accumulator with `prog` (right operand)."""
    direct, popop = _ARITH_OPS[op]
    if _isleaf(prog):
        return [replace(prog[0], op=direct)]
    return [Instr(op=OP_PUSH)] + list(prog) + [Instr(op=popop)]


def _stack_depth(prog):
    sp = mx = 0
    for I in prog:
        if I.op == OP_PUSH:
            sp += 1
            mx = max(mx, sp)
        elif OP_POPADD <= I.op <= OP_POPDIV or I.op == OP_POPFN2:
            sp -= 1
    return mx


class _TooLong(Exception):
    pass


def _traced_program(node, argprog, f32):
    """Accumulator program computing the traced expression `node` (host/trace.py) from the programs of its
    arguments.  IEEE results are kept: operands are never reassociated, only the exact swap of `+ * min max`
    operands is used, and `c - v` becomes `-v + c` (the definition of subtraction).  A Float32 map rounds after
    every operation, as the reference's Float32 arithmetic does.  Shared subexpressions are evaluated again."""
    rnd = [Instr(op=OP_CAST_F32)] if f32 else []

    def const(v):
        return float(np.float32(v)) if f32 else float(v)     # numpy: a Python float meets Float32 samples as Float32

    def leaf(p, ok=None):
        return _isleaf(p) and (ok is None or p[0].leaf in ok)

    def emit(nd):
        out = _emit(nd)
        if len(out) > MAX_PROG:
            raise _TooLong
        return out

    def _emit(nd):
        k = nd.kind
        if k == "arg":
            return list(argprog[nd.key])
        if k == "const":
            return [Instr(OP_LOAD, LEAF_CONST, d0=const(nd.value))]
        if k == "neg":
            return emit(nd.args[0]) + [Instr(op=OP_NEG)]
        if k == "clamp":
            lo, hi = nd.value
            return emit(nd.args[0]) + [Instr(op=OP_FN1, fn=EFN[k], d0=const(lo), d1=const(hi))] + rnd
        if len(nd.args) == 1:
            return emit(nd.args[0]) + [Instr(op=OP_FN1, fn=EFN[k])] + rnd
        pa, pb = emit(nd.args[0]), emit(nd.args[1])
        if k in ("+", "*", "min", "max") and leaf(pa, (LEAF_CONST,)) and not leaf(pb, (LEAF_CONST,)):
            pa, pb = pb, pa            # the sample first (`max(0, v)` as `max(v, 0)`): the fused filter forms want it so
        if k in _ARITH_OPS:
            direct, popop = _ARITH_OPS[k]
            if leaf(pb):
                return pa + [replace(pb[0], op=direct)] + rnd
            if leaf(pa) and k in "+*":
                return pb + [replace(pa[0], op=direct)] + rnd
            if leaf(pa) and k == "-":
                return pb + [Instr(op=OP_NEG), replace(pa[0], op=OP_ADD)] + rnd
            return pa + [Instr(op=OP_PUSH)] + pb + [Instr(op=popop)] + rnd
        code = EFN[k]
        if leaf(pb, FN2_LEAVES):
            return pa + [replace(pb[0], op=OP_FN2, fn=code)] + rnd
        if leaf(pa, FN2_LEAVES) and k in ("min", "max"):
            return pb + [replace(pa[0], op=OP_FN2, fn=code)] + rnd
        return pa + [Instr(op=OP_PUSH)] + pb + [Instr(op=OP_POPFN2, fn=code)] + rnd

    return emit(node)


def _node_args(node, out):
    if node.kind == "arg":
        out.add(node.key)
    for a in node.args:
        _node_args(a, out)
    return out


def _intersect(a: Piece, b: Piece):
    lo, hi = max(a.lo, b.lo), min(a.hi, b.hi)
    clo, chi = max(a.clo, b.clo), min(a.chi, b.chi)
    if lo < hi and clo < chi:
        return lo, hi, clo, chi
    return None


class Lowerer:
    def __init__(self, instance_index=0):
        self.instance_index = instance_index     # position of this graph in a batch call (device noise streams)
        self.plan = Plan()
        self._input_ids = {}      # id(ndarray) -> input index
        self._barrier_memo = {}   # id(node) -> (buf tag, frames materialised, stage)
        self._keepalive = []

    # ---- buffers -------------------------------------------------------------
    def add_input(self, arr):
        arr = np.asarray(arr)
        m = arr.reshape(-1, 1) if arr.ndim == 1 else arr
        key = id(arr)
        if key in self._input_ids:
            return ("in", self._input_ids[key])
        if m.dtype.kind in "iub":
            m = m.astype(np.int64)
        elif m.dtype not in (np.float32, np.float64):
            m = m.astype(np.float64)
        # numpy's own layout of an (nframes, nchannels) matrix is frame-interleaved — exactly a WAV data chunk, which the
        # C ABI takes as it is (SIGOPS_INTERLEAVED: the device transposes).  No host-side transposition: numpy needs
        # 45 ms for a one-minute stereo signal, eight times what the rest of the call costs
        if m.ndim == 2 and m.shape[0] > 1 and m.shape[1] > 1 and m.flags.c_contiguous and m.dtype in (np.float32, np.float64):
            from .wav import WavRaw
            k = len(self.plan.inputs)
            self.plan.inputs.append(BufDesc(m.shape[0], m.shape[1], dtype_code(m.dtype)))
            self.plan.input_arrays.append(WavRaw(m))
            self._input_ids[key] = k
            self._keepalive.append(arr)
            return ("in", k)
        # strided views (x[::2], stereo[:,0] of a C-ordered array, x[::-1]) become dense copies here:
        # the C ABI only describes rows that are contiguous in time
        if m.shape[0] > 1 and m.strides[0] != m.itemsize:
            m = np.asfortranarray(m) if m.shape[1] > 1 else np.ascontiguousarray(m)
        k = len(self.plan.inputs)
        self.plan.inputs.append(BufDesc(m.shape[0], m.shape[1], dtype_code(m.dtype)))
        self.plan.input_arrays.append(m)
        self._input_ids[key] = k
        self._keepalive.append(arr)
        return ("in", k)

    def add_wav_input(self, wav):
        key = id(wav)
        if key in self._input_ids:
            return ("in", self._input_ids[key])
        k = len(self.plan.inputs)
        self.plan.inputs.append(BufDesc(wav.shape[0], wav.shape[1], F64))
        self.plan.input_arrays.append(wav)
        self._input_ids[key] = k
        self._keepalive.append(wav)
        return ("in", k)

    def add_temp(self, nframes, nch, dtype):
        self.plan.temps.append(BufDesc(int(nframes), int(nch), dtype_code(dtype)))
        return ("tmp", len(self.plan.temps) - 1)

    def add_table(self, arr):
        self.plan.tables.append(np.ascontiguousarray(arr, dtype=np.float64))
        return len(self.plan.tables) - 1

    def new_scalar(self):
        self.plan.n_scalars += 1
        return self.plan.n_scalars - 1

    # ---- entry point ------------------------------------------------------------
    def build(self, x, nframes=None, nchannels=None, out_dtype=None):
        x = G.process_sink_params(x)
        N = x.nframes if nframes is None else int(nframes)
        if nchannels is not None:
            x = G.ToChannels(x, nchannels)           # sink! semantics, src/sink.jl:164
        C = x.nchannels
        dt = x.sampletype if out_dtype is None else out_dtype
        self.plan.outputs.append(BufDesc(N, C, dtype_code(dt)))
        self.plan.framerate = x.framerate
        self.plan.wants_tuple = G.result_wants_tuple(x)
        out = ("out", 0)
        pieces = self.lower(x, 0, 0, N, 1, 0, 0, C) if N > 0 else []
        if N == 0:
            self._probe_cuts(x)
        st = Stage(STAGE_MAP, out, pieces=pieces, nchannels=C, n_out=N)
        self.plan.stages.append(st)
        self._fuse_epilogues()
        self._check_limits()
        return self.plan

    def _probe_cuts(self, x):
        """The reference calls `nextblock(x,0,false)` even for an empty result, so an
        `After` that skips past the end of its child still throws (cutting.jl:174-181)."""
        while isinstance(x, G.WrappedSignal):
            if isinstance(x, G.CutApply) and x.kind == "after":
                cn, k = x.signal.nframes, x.resolvelen()
                if k is not None and cn is not None and not G.isknowninf(cn) and cn < k:
                    raise G.SignalError(f"Signal is too short to skip {x.time}")
            x = x.child()

    # ---- recursive lowering -------------------------------------------------------
    # Produce programs for consumer frames n in [lo,hi) and consumer channels
    # c in [clo,chi), where the node's own (0-based) frame is n+shift and its
    # channel is c*cm+co.
    def lower(self, x, shift, lo, hi, cm, co, clo, chi):
        if lo >= hi or clo >= chi:
            return []
        if isinstance(x, WavSignal):
            # samples still in file layout (frame-interleaved PCM16 / float): decoded on the device
            tag = self.add_wav_input(x.wav)
            return [Piece(lo, hi, clo, chi, [Instr(OP_LOAD, LEAF_BUF, buf=tag, c_mul=cm, c_off=co,
                                                   i0=shift, i1=x.wav.shape[0])])]
        if isinstance(x, G.ArraySignal):
            tag = self.add_input(x.data)
            n = x.data.shape[0]
            return [Piece(lo, hi, clo, chi, [Instr(OP_LOAD, LEAF_BUF, buf=tag, c_mul=cm, c_off=co,
                                                   i0=shift, i1=n)])]
        if isinstance(x, G.NumberSignal):
            return [Piece(lo, hi, clo, chi, [Instr(OP_LOAD, LEAF_CONST, d0=float(x.val))])]
        if isinstance(x, G.SignalFunction):
            return self._lower_function(x, shift, lo, hi, cm, co, clo, chi)
        if isinstance(x, G.CutApply):
            if x.kind == "until":
                return self.lower(x.signal, shift, lo, hi, cm, co, clo, chi)
            k = max(0, x.resolvelen())
            cn = x.signal.nframes
            if not G.isknowninf(cn) and cn < k:
                raise G.SignalError(f"Signal is too short to skip {x.time}")     # cutting.jl:174-181
            return self.lower(x.signal, shift + k, lo, hi, cm, co, clo, chi)
        if isinstance(x, G.PaddedSignal):
            return self._lower_pad(x, shift, lo, hi, cm, co, clo, chi)
        if isinstance(x, G.AppendSignals):
            out, start = [], 0
            for j, ch in enumerate(x.signals):
                n = ch.nframes
                last = j == len(x.signals) - 1
                end = None if G.isknowninf(n) else start + n
                a = max(lo, start - shift)
                b = hi if (end is None) else min(hi, end - shift)
                if a < b:
                    out += self.lower(ch, shift - start, a, b, cm, co, clo, chi)
                if end is None:
                    break
                start = end
                if last and hi > end - shift:
                    raise G.SignalError("internal: read past the end of an appended signal")
            return out
        if isinstance(x, G.RampSignal):
            return self._lower_ramp(x, shift, lo, hi, clo, chi)
        if isinstance(x, G.NormedSignal):
            return self._lower_normed(x, shift, lo, hi, cm, co, clo, chi)
        if isinstance(x, G.FilteredSignal):
            tag, n = self._materialize_filter(x, hi + shift)
            return [Piece(lo, hi, clo, chi, [Instr(OP_LOAD, LEAF_BUF, buf=tag, c_mul=cm, c_off=co,
                                                   i0=shift, i1=n)])]
        if isinstance(x, G.MapSignal):
            return self._lower_map(x, shift, lo, hi, cm, co, clo, chi)
        raise LoweringError(f"cannot lower node of type {type(x).__name__}")

    # ---- leaves ---------------------------------------------------------------------
    def _lower_function(self, x, shift, lo, hi, cm, co, clo, chi):
        fs = x.framerate
        if fs is None:
            raise G.SignalError("Unknown frame rate for a function signal.")
        if isinstance(x.fn, G.RandFn) and isinstance(x.fn.rng, PhiloxRNG):
            # device noise (src/functions.jl:98-114 with a counter-based generator): frame k of stream
            # `stream base + index of the instance in the call`; the base makes the graphs of a batch (streams
            # s, s+1, ...) lower to the same bytes
            rng = x.fn.rng
            seed = rng.seed - (1 << 64) if rng.seed >= (1 << 63) else rng.seed
            return [Piece(lo, hi, clo, chi, [Instr(OP_LOAD, LEAF_RANDN, i0=shift + 1, i1=seed,
                                                   i2=rng.stream - self.instance_index)])]
        code = None if isinstance(x.fn, G.RandFn) else functor_code(x.fn)
        if code is not None and x.nchannels == 1:
            fn, a, b = code
            return [Piece(lo, hi, clo, chi, [Instr(
                OP_LOAD, LEAF_GEN, fn=fn, flags=FLAG_HAS_OMEGA if x.omega is not None else 0,
                i0=shift + 1, d0=float(fs), d1=float(x.omega or 0.0), d2=x.phi, d3=a, d4=b)])]
        # not expressible on the device: evaluate this leaf on the host with the
        # reference's formula and feed it as an input buffer (SURVEY.md §7.3-5/6)
        vals = host_function_frames(x, lo + shift + 1, hi + shift + 1)
        tag = self.add_input(vals)
        return [Piece(lo, hi, clo, chi, [Instr(OP_LOAD, LEAF_BUF, buf=tag, c_mul=cm, c_off=co,
                                               i0=-lo, i1=hi - lo)])]

    def _lower_ramp(self, x, shift, lo, hi, clo, chi):
        L = x.resolvelen()
        if L is None:
            raise G.SignalError("Unknown frame rate for a ramp.")
        if x.fn is G.sinramp:
            fn = FN_SINRAMP
        elif x.fn is G.identity:
            fn = FN_IDENTITY
        else:
            fn = None
        if x.direction == "on":
            if fn is None:
                env = np.array([float(x.fn(k / L)) for k in range(L)], dtype=np.float64)
                tag = self.add_input(env)
                return [Piece(lo, hi, clo, chi, [Instr(OP_LOAD, LEAF_BUF, buf=tag, c_mul=0, c_off=0,
                                                       i0=shift, i1=L, d0=1.0)])]
            return [Piece(lo, hi, clo, chi, [Instr(OP_LOAD, LEAF_RAMP_ON, fn=fn, i0=shift + 1, i1=L)])]
        N = x.nframes
        if G.isknowninf(N):
            return [Piece(lo, hi, clo, chi, [Instr(OP_LOAD, LEAF_CONST, d0=1.0)])]
        n0 = N - L
        if n0 < 0:
            raise G.SignalError("Ramp is longer than the signal it is applied to.")   # SURVEY App. C-10
        if fn is None:
            env = np.array([float(x.fn(1 - k / L)) for k in range(1, L + 1)], dtype=np.float64)
            tag = self.add_input(env)
            return [Piece(lo, hi, clo, chi, [Instr(OP_LOAD, LEAF_BUF, buf=tag, c_mul=0, c_off=0,
                                                   i0=shift - n0, i1=L, d0=1.0)])]
        return [Piece(lo, hi, clo, chi, [Instr(OP_LOAD, LEAF_RAMP_OFF, fn=fn, i0=shift + 1, i1=n0, i2=L)])]

    def _lower_pad(self, x, shift, lo, hi, cm, co, clo, chi):
        child = x.signal
        nc = child.nframes
        b = nc - shift                       # first padded consumer frame
        p = x.pad
        T = x.sampletype
        if any(p is q for q in (G.cycle, G.mirror, G.lastframe)):
            if p is not G.lastframe and not isinstance(child, G.ArraySignal):
                raise G.SignalError("Attemped to specify an indexing pad function for a signal "
                                    "which is not known to support `getindex`.")     # padding.jl:172-181
            if nc == 0:
                raise G.SignalError("Signal is length zero; there is no last frame to pad with.")
            mode = {G.cycle: PAD_CYCLE, G.mirror: PAD_MIRROR, G.lastframe: PAD_LAST}[p]
            if isinstance(child, G.ArraySignal):
                tag = self.add_input(child.data)
            else:
                tag = self._materialize(child, nc)
            return [Piece(lo, hi, clo, chi, [Instr(OP_LOAD, LEAF_BUF, flags=mode << 1, buf=tag,
                                                   c_mul=cm, c_off=co, i0=shift, i1=nc)])]
        out = []
        if lo < min(hi, b):
            out += self.lower(child, shift, lo, min(hi, b), cm, co, clo, chi)
        if max(lo, b) < hi:
            a = max(lo, b)
            if G._isnumber(p):
                prog = [Instr(OP_LOAD, LEAF_CONST, d0=float(np.dtype(T).type(p)))]
            elif isinstance(p, (tuple, list, np.ndarray)):
                vals = np.asarray(p, dtype=np.dtype(T)).reshape(1, -1)
                if vals.shape[1] != x.nchannels:
                    raise G.SignalError("padding tuple must have one value per channel")
                tag = self.add_input(vals)
                prog = [Instr(OP_LOAD, LEAF_BUF, flags=PAD_LAST << 1, buf=tag, c_mul=cm, c_off=co,
                              i0=0, i1=1)]
            elif p is G.zero or p is G.one:
                prog = [Instr(OP_LOAD, LEAF_CONST, d0=float(p(T)))]
            elif callable(p):
                try:
                    v = p(np.dtype(T))
                except TypeError:
                    raise G.SignalError(f"Pad function ({p}) must take 1 or 3 arguments. "
                                        "Refer to `Pad` documentation.") from None
                prog = [Instr(OP_LOAD, LEAF_CONST, d0=float(v))]
            else:
                raise G.SignalError(f"unsupported padding value {p!r}")
            out.append(Piece(a, hi, clo, chi, prog))
        return out

    # ---- barriers ------------------------------------------------------------------------
    def _materialize(self, x, n):
        """Frames [0,n) of `x` in a buffer; reuses a producing stage when there is one."""
        if isinstance(x, G.ArraySignal) and x.data.shape[0] >= n:
            return self.add_input(x.data)
        if isinstance(x, G.FilteredSignal):
            return self._materialize_filter(x, n)[0]
        key = id(x)
        memo = self._barrier_memo.get(key)
        if memo and memo[1] >= n:
            return memo[0]
        C = x.nchannels
        tag = self.add_temp(n, C, x.sampletype)
        pieces = self.lower(x, 0, 0, n, 1, 0, 0, C)
        st = Stage(STAGE_MAP, tag, pieces=pieces, nchannels=C, n_out=n)
        self.plan.stages.append(st)
        self._barrier_memo[key] = (tag, n, st)
        self._keepalive.append(x)
        return tag

    def _stage_of(self, tag):
        for st in self.plan.stages:
            if st.out_buf == tag:
                return st
        return None

    def _lower_normed(self, x, shift, lo, hi, cm, co, clo, chi):
        child = x.signal
        N = child.nframes
        if G.isknowninf(N):
            raise G.SignalError("Cannot normalize an infinite-length signal. Please "
                                "use `Until` to take a prefix of the signal")     # filters.jl:297-300
        C = child.nchannels
        key = ("norm", id(x))
        memo = self._barrier_memo.get(key)
        if memo is None:
            if isinstance(child, G.ArraySignal):
                # raw data still needs its sum of squares: copy through a MAP stage
                tag = self.add_temp(N, C, x.sampletype)
                st = Stage(STAGE_MAP, tag, pieces=self.lower(child, 0, 0, N, 1, 0, 0, C),
                           nchannels=C, n_out=N)
                self.plan.stages.append(st)
            else:
                tag = self._materialize(child, N)
                st = self._stage_of(tag)
                if st is None or st.n_out != N or st.sumsq_slot >= 0:
                    # a longer prefix was materialised for someone else: take an exact copy
                    src = tag
                    tag = self.add_temp(N, C, x.sampletype)
                    st = Stage(STAGE_MAP, tag, nchannels=C, n_out=N, pieces=[Piece(
                        0, N, 0, C, [Instr(OP_LOAD, LEAF_BUF, buf=src, i0=0, i1=N)])])
                    self.plan.stages.append(st)
            slot = self.new_scalar()
            st.sumsq_slot = slot
            memo = (tag, slot)
            self._barrier_memo[key] = memo
            self._keepalive.append(x)
        tag, slot = memo
        prog = [Instr(OP_LOAD, LEAF_BUF, buf=tag, c_mul=cm, c_off=co, i0=shift, i1=N),
                Instr(OP_DIV, LEAF_RMS, buf=slot, d0=float(N * C))]
        if np.dtype(x.sampletype) == np.float32:
            prog.append(Instr(op=OP_CAST_F32))       # `vals ./= rms` is stored as Float32 before anything reads it
        return [Piece(lo, hi, clo, chi, prog)]

    def _materialize_filter(self, x, need):
        """Stage(s) computing frames [0,n) of a FilteredSignal into a temp."""
        N = x.nframes
        n = need if G.isknowninf(N) else N       # causal: a prefix needs only a prefix
        key = id(x)
        memo = self._barrier_memo.get(key)
        if memo and memo[1] >= n:
            return memo[0], memo[1]
        child = x.signal
        C = child.nchannels
        fs = x.framerate
        if fs is None:
            raise G.SignalError("Unknown frame rate for a filtered signal.")
        h = x.fn(fs)
        T = x.sampletype
        if isinstance(h, dspjl.FIRFilter):
            tag = self._emit_fir(x, h, child, n, C, T)
        else:
            tag = self._emit_iir(x, dspjl.to_sos(h), child, n, C, T)
        self._barrier_memo[key] = (tag, n, None)
        self._keepalive.append(x)
        return tag, n

    def _input_program(self, child, n_in, C):
        """Single program giving frames [0,n_in) of `child` followed by zeros
        (`Pad(x.signal,zero)`, src/filters.jl:240); materialises when piecewise."""
        cn = child.nframes
        avail = n_in if G.isknowninf(cn) else min(cn, n_in)
        pieces = self.lower(child, 0, 0, avail, 1, 0, 0, C) if avail > 0 else []
        if len(pieces) == 1 and _isleaf(pieces[0].prog) and pieces[0].prog[0].leaf == LEAF_BUF \
                and pieces[0].prog[0].i0 == 0 and (pieces[0].prog[0].flags >> 1) == PAD_CONST \
                and pieces[0].prog[0].c_mul == 1 and pieces[0].prog[0].c_off == 0:
            I = pieces[0].prog[0]
            return [replace(I, i1=min(I.i1, avail), d0=0.0)], True
        if len(pieces) == 1 and avail == n_in and not any(
                I.leaf == LEAF_BUF and (I.flags >> 1) != PAD_CONST for I in pieces[0].prog):
            return pieces[0].prog, False
        if avail == 0:
            return [Instr(OP_LOAD, LEAF_CONST, d0=0.0)], False
        tag = self.add_temp(avail, C, child.sampletype)
        self.plan.stages.append(Stage(STAGE_MAP, tag, pieces=pieces, nchannels=C, n_out=avail))
        return [Instr(OP_LOAD, LEAF_BUF, buf=tag, i0=0, i1=avail, d0=0.0)], True

    def _emit_iir(self, x, sos, child, n, C, T):
        prog, _ = self._input_program(child, n, C)
        biquads = list(sos.biquads)
        groups = [biquads[i:i + MAX_SECTIONS] for i in range(0, len(biquads), MAX_SECTIONS)] or [[]]
        tag = None
        for gi, grp in enumerate(groups):
            lastg = gi == len(groups) - 1
            if not grp:
                grp = [dspjl.Biquad(1, 0, 0, 0, 0)]
            tag = self.add_temp(n, C, T if lastg else np.float64)
            tbl = self.add_table(np.array([b.astuple() for b in grp]))
            self.plan.stages.append(Stage(
                STAGE_IIR, tag, in_prog=prog, nchannels=C, n_in=n, n_out=n,
                n_sections=len(grp), coef_table=tbl, gain=sos.g if lastg else 1.0))
            prog = [Instr(OP_LOAD, LEAF_BUF, buf=tag, i0=0, i1=n, d0=0.0)]
        return tag

    def _emit_fir(self, x, f, child, n_out, C, T):
        cn = child.nframes
        if G.isknowninf(cn):
            n_in = int(math.ceil(n_out / f.rate)) + f.input_deficit + f.tapsper + 2
        else:
            n_in = cn
        prog, plain = self._input_program(child, n_in, C)
        # The tensor-core kernel (csrc/k_fir_mma.cuh) wants plain Float64 rows on both sides.  Float32
        # signals are widened once on the way in and rounded once on the way out — the rounding the
        # reference's Float32 output block performs (src/filters.jl:213-214) — which costs two light
        # elementwise passes and still beats the scalar kernel by a wide margin.
        f32 = np.dtype(T) == np.float32
        if not plain or np.dtype(child.sampletype) == np.float32:
            tag_in = self.add_temp(n_in, C, np.float64 if np.dtype(child.sampletype) == np.float32 else child.sampletype)
            self.plan.stages.append(Stage(STAGE_MAP, tag_in, nchannels=C, n_out=n_in,
                                          pieces=[Piece(0, n_in, 0, C, prog)]))
            prog = [Instr(OP_LOAD, LEAF_BUF, buf=tag_in, i0=0, i1=n_in, d0=0.0)]
        tag = self.add_temp(n_out, C, np.float64 if f32 else T)
        st = Stage(STAGE_FIR, tag, in_prog=prog, nchannels=C, n_in=n_in, n_out=n_out,
                   rate=float(f.rate), input_deficit=int(f.input_deficit))
        if f.kind == "arbitrary":
            st.fir_kind = FIR_ARBITRARY
            st.n_phases, st.taps_per_phase = f.nphases, f.tapsper
            st.pfb_table = self.add_table(f.pfb.T)       # [phase][tap], window order
            st.dpfb_table = self.add_table(f.dpfb.T)
            st.phase0 = float(f.phi_acc)
        elif f.kind in ("rational", "interpolator"):
            st.fir_kind = FIR_RATIONAL
            st.n_phases, st.taps_per_phase = f.nphases, f.tapsper
            st.interpolation, st.decimation = f.nphases, f.decimation
            st.pfb_table = self.add_table(f.pfb.T)
            st.phase0 = float(f.phi_idx)
        elif f.kind == "decimator":
            st.fir_kind = FIR_DECIMATOR
            st.n_phases, st.taps_per_phase = 1, f.hlen
            st.interpolation, st.decimation = 1, f.decimation
            st.pfb_table = self.add_table(f.hrev.reshape(1, -1))
            st.phase0 = 1.0
        elif f.kind == "standard":
            # single-rate FIR (`Filt(x, FIRFilter(h))`, DSP.jl FIRStandard): the decimator kernel with step 1
            st.fir_kind = FIR_DECIMATOR
            st.n_phases, st.taps_per_phase = 1, f.hlen
            st.interpolation, st.decimation = 1, 1
            st.pfb_table = self.add_table(f.hrev.reshape(1, -1))
            st.phase0 = 1.0
        else:
            raise LoweringError(f"FIR kernel kind {f.kind!r} is not lowered to the GPU path")
        self.plan.stages.append(st)
        if f32:
            tag32 = self.add_temp(n_out, C, T)
            self.plan.stages.append(Stage(STAGE_MAP, tag32, nchannels=C, n_out=n_out, pieces=[Piece(
                0, n_out, 0, C, [Instr(OP_LOAD, LEAF_BUF, buf=tag, i0=0, i1=n_out, d0=0.0), Instr(op=OP_CAST_F32)])]))
            return tag32
        return tag

    # ---- maps ---------------------------------------------------------------------------
    def _lower_map(self, x, shift, lo, hi, cm, co, clo, chi):
        fn = x.fn
        kids = x.padded_signals
        if x.bychannel:
            if isinstance(fn, G.ToEltypeFn):
                ps = self.lower(kids[0], shift, lo, hi, cm, co, clo, chi)
                code = dtype_code(fn.T)
                if code == F64 or (code == F32 and kids[0].sampletype == np.float32):
                    return ps
                cast = OP_CAST_F32 if code == F32 else OP_CAST_I64
                return [Piece(p.lo, p.hi, p.clo, p.chi, p.prog + [Instr(op=cast)]) for p in ps]
            if x.op == "neg":
                ps = self.lower(kids[0], shift, lo, hi, cm, co, clo, chi)
                return [Piece(p.lo, p.hi, p.clo, p.chi, p.prog + [Instr(op=OP_NEG)]) for p in ps]
            if x.op not in _ARITH_OPS:
                return self._lower_traced(x, shift, lo, hi, cm, co, clo, chi)
            acc = self.lower(kids[0], shift, lo, hi, cm, co, clo, chi)
            if len(kids) == 1 and x.op == "-":
                return [Piece(p.lo, p.hi, p.clo, p.chi, p.prog + [Instr(op=OP_NEG)]) for p in acc]
            f32 = np.dtype(x.sampletype) == np.float32
            for k in kids[1:]:
                rhs = self.lower(k, shift, lo, hi, cm, co, clo, chi)
                nxt = []
                for a in acc:
                    for b in rhs:
                        r = _intersect(a, b)
                        if r:
                            nxt.append(Piece(*r, a.prog + _as_operand(b.prog, x.op)))
                acc = nxt
            if f32:
                # Float32 arithmetic rounds after every operation in the reference
                acc = [Piece(p.lo, p.hi, p.clo, p.chi, p.prog + [Instr(op=OP_CAST_F32)]) for p in acc]
            return acc
        # ---- whole-frame functions (bychannel=false)
        if isinstance(fn, G.AsNChannels):
            return self.lower(kids[0], shift, lo, hi, 0, 0, clo, chi)
        if isinstance(fn, G.GetChanFn):
            if not 1 <= fn.n <= kids[0].nchannels:
                raise G.SignalError(f"channel {fn.n} out of range")
            return self.lower(kids[0], shift, lo, hi, 0, fn.n - 1, clo, chi)
        if isinstance(fn, G.As1Channel):
            k = kids[0]
            nc = k.nchannels
            acc = self.lower(k, shift, lo, hi, 0, 0, clo, chi)
            for ch in range(1, nc):
                rhs = self.lower(k, shift, lo, hi, 0, ch, clo, chi)
                nxt = []
                for a in acc:
                    for b in rhs:
                        r = _intersect(a, b)
                        if r:
                            nxt.append(Piece(*r, a.prog + _as_operand(b.prog, "+")))
                acc = nxt
            if any(len(p.prog) > MAX_PROG or _stack_depth(p.prog) > MAX_STACK for p in acc):
                n = k.nframes
                if G.isknowninf(n):
                    n = hi + shift
                tag = self._materialize(k, n)
                return [Piece(lo, hi, clo, chi, [Instr(OP_LOAD, LEAF_CHANSUM, buf=tag, i0=shift,
                                                       i1=n, i2=nc)])]
            return acc
        if isinstance(fn, G.TupleCat):
            out, off = [], 0
            for k in kids:
                kc = k.nchannels
                if cm == 0:
                    if off <= co < off + kc:
                        out += self.lower(k, shift, lo, hi, 0, co - off, clo, chi)
                else:
                    a, b = max(clo, off - co), min(chi, off + kc - co)
                    if a < b:
                        out += self.lower(k, shift, lo, hi, 1, co - off, a, b)
                off += kc
            return out
        if fn is G.reverse and len(kids) == 1:
            # channel c of the result is channel C-1-c of the child: one piece per channel
            C = kids[0].nchannels
            out = []
            for c in range(clo, chi):
                src = c * cm + co if cm else co
                out += self.lower(kids[0], shift, lo, hi, 0, C - 1 - src, c, c + 1)
            return out
        return self._lower_traced(x, shift, lo, hi, cm, co, clo, chi)

    def _lower_traced(self, x, shift, lo, hi, cm, co, clo, chi):
        """OperateOn with any other function: trace it (host/trace.py) and compile the expression.  By channel, one
        expression serves every channel; a whole-frame closure (bychannel=false) gives one expression per output
        channel, which becomes one piece per channel like `reverse`."""
        kids = x.padded_signals
        name = getattr(x.fn, "__name__", repr(x.fn))
        try:
            if x.bychannel:
                roots = trace(x.fn, len(kids))
            else:
                roots = trace(x.fn, len(kids), [k.nchannels for k in kids])
        except TraceError as e:
            raise LoweringError(f"OperateOn({name}) cannot be compiled for the GPU sink: {e}") from None
        T = np.dtype(x.sampletype)
        f32 = T == np.float32
        tail = [Instr(op=OP_CAST_I64)] if T.kind in "iub" else []
        # (consumer channels, node channel map, expression) of each group of output channels
        if x.bychannel:
            groups = [(clo, chi, cm, co, roots)]
        else:
            groups = [(c, c + 1, 0, c * cm + co if cm else co, roots[c * cm + co if cm else co]) for c in range(clo, chi)]

        def arg_pieces(key, a, b, gcm, gco, materialise):
            k, ch = (key, None) if x.bychannel else key
            kcm, kco = (gcm, gco) if ch is None else (0, ch)
            kid = kids[k]
            if materialise:
                n = kid.nframes
                if G.isknowninf(n):
                    n = hi + shift
                tag = self._materialize(kid, n)
                return [Piece(lo, hi, a, b, [Instr(OP_LOAD, LEAF_BUF, buf=tag, c_mul=kcm, c_off=kco, i0=shift, i1=n)])]
            return self.lower(kid, shift, lo, hi, kcm, kco, a, b)

        def build(materialise):
            out = []
            for a, b, gcm, gco, root in groups:
                combos = [(lo, hi, a, b, {})]
                for key in sorted(_node_args(root, set()), key=repr):
                    ps = arg_pieces(key, a, b, gcm, gco, key in materialise)
                    if any(not _isleaf(p.prog) for p in ps):
                        expressions.add(key)
                    nxt = []
                    for c0 in combos:
                        for p in ps:
                            r = _intersect(Piece(*c0[:4], None), p)
                            if r:
                                nxt.append((*r, {**c0[4], key: p.prog}))
                    combos = nxt
                for (plo, phi, pclo, pchi, argprog) in combos:
                    prog = _traced_program(root, argprog, f32) + tail
                    if len(prog) > MAX_PROG or _stack_depth(prog) > MAX_STACK:
                        raise _TooLong
                    out.append(Piece(plo, phi, pclo, pchi, prog))
            return out

        expressions = set()
        try:
            return build(set())
        except _TooLong:
            pass
        # an argument used several times is evaluated each time: when that does not fit, the arguments that are
        # expressions of their own are computed once into temps (as As1Channel does) and read back as buffers
        try:
            return build(set(expressions))
        except _TooLong:
            raise LoweringError(f"OperateOn({name}): the traced expression needs more than {MAX_PROG} operations "
                                f"or nests deeper than the device stack ({MAX_STACK})") from None

    # ---- post passes -----------------------------------------------------------------------
    def _fuse_epilogues(self):
        """MAP stage that only post-processes the full output of the IIR/FIR stage
        right before it -> becomes that stage's epilogue (one HBM round trip)."""
        changed = True
        while changed:
            changed = False
            for i, st in enumerate(self.plan.stages):
                if st.kind != STAGE_MAP or len(st.pieces) != 1:
                    continue
                pc = st.pieces[0]
                refs = [I for I in pc.prog if I.leaf in (LEAF_BUF, LEAF_CHANSUM) and
                        isinstance(I.buf, tuple) and I.buf[0] == "tmp"]
                cands = {I.buf for I in refs}
                for tag in cands:
                    prod = next((s for s in self.plan.stages[:i] if s.out_buf == tag), None)
                    if prod is None or prod.epi_prog or prod.sumsq_slot >= 0:
                        continue
                    bare_copy = (len(pc.prog) == 1 and pc.prog[0].op == OP_LOAD and
                                 self._desc(st.out_buf).dtype == self._desc(tag).dtype)
                    # an elementwise producer only absorbs a bare copy of its whole output (it then
                    # writes straight into the copy's destination)
                    if prod.kind == STAGE_MAP and not bare_copy:
                        continue
                    # resamplers take a bare store or a constant gain (`ToFramerate |> Amplify(c)`: the
                    # tensor-core kernels fold it into the taps); anything richer stays a separate
                    # elementwise pass, which costs far less than the scalar FIR kernel
                    const_gain = (2 <= len(pc.prog) <= 3 and pc.prog[0].op == OP_LOAD and all(
                        I.op == OP_MUL and I.leaf == LEAF_CONST for I in pc.prog[1:]) and
                        self._desc(st.out_buf).dtype == self._desc(tag).dtype == F64)
                    if prod.kind == STAGE_FIR and not (bare_copy or const_gain):
                        continue
                    uses = [I for I in refs if I.buf == tag]
                    elsewhere = any(I.leaf in (LEAF_BUF, LEAF_CHANSUM) and I.buf == tag
                                    for s2 in self.plan.stages if s2 is not st
                                    for prog in ([p.prog for p in s2.pieces] + [s2.in_prog, s2.epi_prog])
                                    for I in prog)
                    I0 = uses[0]
                    if (len(uses) != 1 or elsewhere or I0.leaf != LEAF_BUF or I0.i0 != 0 or I0.c_mul != 1
                            or I0.c_off != 0 or (I0.flags >> 1) != PAD_CONST
                            or pc.lo != 0 or pc.hi != prod.n_out or pc.clo != 0
                            or pc.chi != prod.nchannels or I0.i1 != prod.n_out):
                        continue
                    obuf = st.out_buf
                    ob = self._desc(obuf)
                    if ob.nframes != prod.n_out or ob.nchannels != prod.nchannels:
                        continue
                    if prod.kind == STAGE_MAP:
                        prod.out_buf = obuf
                        prod.sumsq_slot = st.sumsq_slot
                        self.plan.stages.pop(i)
                        changed = True
                        break
                    prod.epi_prog = [replace(I, leaf=LEAF_STAGE, buf=0) if I is I0 else I for I in pc.prog]
                    prod.out_buf = obuf
                    prod.sumsq_slot = st.sumsq_slot
                    # the fused stage runs where the MAP stage stood, so every other
                    # buffer/scalar its epilogue reads has been produced by then
                    self.plan.stages[i] = prod
                    self.plan.stages.remove(prod)
                    changed = True
                    break
                if changed:
                    break
        self._drop_unused_temps()

    def _desc(self, tag):
        kind, k = tag
        return {"in": self.plan.inputs, "tmp": self.plan.temps, "out": self.plan.outputs}[kind][k]

    def _drop_unused_temps(self):
        used = set()
        for st in self.plan.stages:
            if st.out_buf[0] == "tmp":
                used.add(st.out_buf[1])
        remap, temps = {}, []
        for k, t in enumerate(self.plan.temps):
            if k in used:
                remap[k] = len(temps)
                temps.append(t)
        self.plan.temps = temps

        def fix_tag(tag):
            return ("tmp", remap[tag[1]]) if isinstance(tag, tuple) and tag[0] == "tmp" else tag

        for st in self.plan.stages:
            st.out_buf = fix_tag(st.out_buf)
            for pc in st.pieces:
                pc.prog = [replace(I, buf=fix_tag(I.buf)) for I in pc.prog]
            st.in_prog = [replace(I, buf=fix_tag(I.buf)) for I in st.in_prog]
            st.epi_prog = [replace(I, buf=fix_tag(I.buf)) for I in st.epi_prog]

    def _check_limits(self):
        p = self.plan
        if len(p.inputs) + len(p.temps) + len(p.outputs) > MAX_BUFS:
            raise LoweringError(f"graph needs more than {MAX_BUFS} buffers")
        for st in p.stages:
            if len(st.pieces) > MAX_PIECES:
                raise LoweringError(f"stage has {len(st.pieces)} pieces (max {MAX_PIECES})")
            for prog in [pc.prog for pc in st.pieces] + [st.in_prog, st.epi_prog]:
                if len(prog) > MAX_PROG:
                    raise LoweringError(f"fused expression of {len(prog)} operations exceeds {MAX_PROG}")
                if _stack_depth(prog) > MAX_STACK:
                    raise LoweringError("expression nests deeper than the device stack")


def host_function_frames(x, k_lo, k_hi):
    """Frames k_lo..k_hi-1 (1-based) of a SignalFunction evaluated on the host, with
    the formulas of src/functions.jl:53-60,113-114. Used only for leaves the device
    cannot express (arbitrary callables, `randn`)."""
    n = k_hi - k_lo
    if isinstance(x.fn, G.RandFn):
        if hasattr(x.fn.rng, "frames"):
            return x.fn.rng.frames(k_lo, k_hi).reshape(-1, 1)
        return x.fn.rng.standard_normal(n).reshape(-1, 1)
    k = np.arange(k_lo, k_hi, dtype=np.float64)
    t = k / x.framerate
    if x.omega is not None:
        arg = 2 * math.pi * np.fmod(t * x.omega + x.phi, 1.0)
    else:
        arg = t + x.phi
    C = x.nchannels
    out = np.empty((n, C), dtype=np.float64)
    for i, a in enumerate(arg):
        v = x.fn(float(a))
        out[i, :] = v if isinstance(v, tuple) else (v,)
    return out


def lower(x, **kw):
    return Lowerer().build(x, **kw)
