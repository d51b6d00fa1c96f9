# GPUSink.jl — the reference-side binding for libsignalops_cuda.so.
#
# NOT EXECUTED IN THIS REPOSITORY'S CI: the build image has no Julia.  This file is the
# glue a SignalOperators.jl maintainer adds (e.g. as src/GPUSink.jl behind a `Requires`
# hook next to src/SignalOperators.jl:45-72).  It is a transcription, method by method,
# of the Python host layer that IS exercised here: `Lowerer` below follows
# signaloperators.jl_b200/host/lowering.py line for line and must emit the same plan bytes
# (include/signalops.h; tests/plan_emulator.py documents their meaning).  The byte-for-byte
# check a maintainer runs is julia/test_plans.jl against tests/golden/plans/*.bin.
#
# Plug-in point: the documented custom-sink interface (docs/src/custom_sink.md:1-18):
# `sink(x, to)` dispatches on `to`, exactly like `sink(x, to::String)` at
# src/sink.jl:139-142.  Nothing of the block-pull machinery (`nextblock`, `frame`,
# `sink_helper!`) is used.

module GPUSinks

using SignalOperators
using SignalOperators: AbstractSignal, CutApply, PaddedSignal, AppendSignals, FilteredSignal,
    NormedSignal, MapSignal, RampSignal, SignalFunction, NumberSignal, FilterFn, RawFilterFn,
    ResamplerFn, FnBr, ToEltypeFn, AsNChannels, As1Channel, GetChanFn, tuplecat, RandFn,
    process_sink_params, initsink, refineroot, root, resolvelen, child, sinramp, inflen,
    isknowninf, cycle, mirror, lastframe
using DSP
using Random

export GPUSink, Sawtooth, AffineSin, AffineCos, PhiloxRNG, lower

const libsignalops = "libsignalops_cuda"

# ---- C ABI (include/signalops.h) -------------------------------------------------------
struct SigopsBuffer
    ptr::Ptr{Cvoid}
    nframes::Int64
    nchannels::Int32
    dtype::Int32          # 1 = Float32, 2 = Float64, 3 = Int64
    ld::Int64
end

mutable struct SigopsStats
    gpu_ms::Float64; h2d_ms::Float64; d2h_ms::Float64; wall_ms::Float64
    launches::Int64; h2d_bytes::Int64; d2h_bytes::Int64; out_samples::Int64
    SigopsStats() = new(0, 0, 0, 0, 0, 0, 0, 0)
end

lasterror(ctx) = unsafe_string(ccall((:sigops_last_error, libsignalops), Cstring, (Ptr{Cvoid},), ctx))

mutable struct GPUSink
    devices::Vector{Cint}
    ctx::Ptr{Cvoid}
    plans::Dict{Vector{UInt8},Ptr{Cvoid}}
    pin_results::Bool       # page-lock the arrays `sink` returns (0.6 s per GB: only for sinks that recycle results)
    function GPUSink(devices = [0]; pin_results = false)
        ctx = Ref{Ptr{Cvoid}}(C_NULL)
        devs = Cint.(devices)
        rc = ccall((:sigops_ctx_create, libsignalops), Cint, (Ptr{Cint}, Cint, Ref{Ptr{Cvoid}}),
                   devs, length(devs), ctx)
        rc == 0 || error(lasterror(C_NULL))
        s = new(devs, ctx[], Dict{Vector{UInt8},Ptr{Cvoid}}(), pin_results)
        finalizer(s) do s
            foreach(p -> ccall((:sigops_plan_destroy, libsignalops), Cvoid, (Ptr{Cvoid},), p), values(s.plans))
            ccall((:sigops_ctx_destroy, libsignalops), Cvoid, (Ptr{Cvoid},), s.ctx)
        end
    end
end

check(to::GPUSink, rc) = rc == 0 || error(lasterror(to.ctx))

function compiled(to::GPUSink, bytes::Vector{UInt8})
    get!(to.plans, bytes) do
        p = Ref{Ptr{Cvoid}}(C_NULL)
        check(to, ccall((:sigops_plan_create, libsignalops), Cint,
                        (Ptr{Cvoid}, Ptr{UInt8}, Csize_t, Ref{Ptr{Cvoid}}), to.ctx, bytes, length(bytes), p))
        p[]
    end
end

# Page-locked result arrays (opt-in, `GPUSink(pin_results = true)`): the sink allocates what it returns (`initsink`,
# src/sink.jl:115-121), so the result can live where the device writes directly (include/signalops.h
# `sigops_host_alloc`).  Page-locking costs ~0.6 s per GB, so this only pays for sinks whose results are recycled
# (a pool behind the finalizer is the natural next step; host/cabi.py has one).  Caller arrays (inputs, `sink!`
# results) and default results are ordinary pageable Julia arrays; the library stages those through its own pinned ring.
function pinned_matrix(to::GPUSink, ::Type{T}, n, c) where T
    (!to.pin_results || n * c * sizeof(T) < (1 << 20)) && return Array{T,2}(undef, n, c)
    p = Ref{Ptr{Cvoid}}(C_NULL)
    rc = ccall((:sigops_host_alloc, libsignalops), Cint, (Csize_t, Ref{Ptr{Cvoid}}), n * c * sizeof(T), p)
    rc == 0 || error(lasterror(C_NULL))
    a = unsafe_wrap(Array, Ptr{T}(p[]), (n, c); own = false)
    finalizer(_ -> ccall((:sigops_host_free, libsignalops), Cint, (Ptr{Cvoid},), p[]), a)
    a
end

# ---- the sink methods ---------------------------------------------------------------------
# Same shape as `sink(x,to::String)` (src/sink.jl:139-142): validate, hand to the backend,
# wrap like `initsink(x,T,data)` (src/sink.jl:120-121).
SignalOperators.sink(to::GPUSink) = x -> sink(x, to)
function SignalOperators.sink(x, to::GPUSink; as = nothing)
    x = process_sink_params(x)                                   # src/sink.jl:94-99
    plan = lower(x)                                              # graph -> stages (below)
    result = pinned_matrix(to, plan.outtype, nframes(x), nchannels(x))   # initsink, src/sink.jl:115-117
    nframes(x) > 0 && run!(to, [plan], [result])
    wrapresult(x, as === nothing ? refineroot(root(x)) : as, result)
end
SignalOperators.sink(x, ::Type{T}, to::GPUSink) where T = sink(x, to; as = T)    # `sink(x, AxisArray)` etc.

# `initsink(x,T,data)` exists for Array and Tuple (src/sink.jl:120-121).  Container sinks — AxisArray
# (src/AxisArrays.jl:41-46), DimensionalArray (src/DimensionalData.jl:36-42), SampleBuf (src/SampledSignals.jl:17-18) —
# only define the allocating `initsink(x,T)`: build the container with the reference's own method and fill it.
# Sample types the device does not compute in (`Fixed{Int16,15}`, src/FixedPointNumbers.jl) are computed in
# Float64 and converted on the way into the container, as `sink!` does per frame (src/sink.jl:262-267).
function wrapresult(x, ::Type{T}, data) where T
    if T <: Union{Array,Tuple} && eltype(data) === sampletype(x)
        return initsink(x, T, data)
    end
    out = initsink(x, T)
    dest = out isa Tuple ? out[1] : out
    dest .= data
    out
end

# `sink!(result, x)` semantics of src/sink.jl:158-168: a prefix of x, forced channel count.
function SignalOperators.sink!(result::Union{AbstractVector,AbstractMatrix}, x, to::GPUSink)
    x = Signal(x)
    n = size(result, 1)
    (!isknowninf(nframes(x)) && nframes(x) < n) && error("Signal is too short to fill buffer of length $n.")
    x = ToChannels(x, size(result, 2))
    T = eltype(result)
    if (T === Float32 || T === Float64 || T === Int64) && stride(result, 1) == 1
        n > 0 && run!(to, [lower(x; nframes = n, outtype = T)], [result])
    else                                                         # any other eltype: convert on the host (src/sink.jl:262-267)
        S = sampletype(x) <: Integer ? Int64 : sampletype(x)
        tmp = Array{S,2}(undef, n, size(result, 2))
        n > 0 && run!(to, [lower(x; nframes = n, outtype = S)], [tmp])
        result .= reshape(tmp, size(result))                     # throws InexactError like the reference
    end
    result
end

# Additive API: a batch of structurally identical graphs = one plan, many instances.
function SignalOperators.sink(xs::AbstractVector, to::GPUSink)
    xs = process_sink_params.(xs)
    plans = [lower(x; instance_index = i - 1) for (i, x) in enumerate(xs)]
    all(p -> p.bytes == plans[1].bytes, plans) || error("batch elements do not lower to the same plan")
    results = [pinned_matrix(to, p.outtype, nframes(x), nchannels(x)) for (x, p) in zip(xs, plans)]
    (isempty(xs) || nframes(xs[1]) == 0) || run!(to, plans, results)
    [wrapresult(x, refineroot(root(x)), r) for (x, r) in zip(xs, results)]
end

# `sink(x, "file.wav")` (src/sink.jl:139-142, src/WAV.jl:3-7) on the GPU sink: the device transposes the result to
# frame-interleaved order (a C x N column-major Julia matrix IS a WAV data chunk) and converts the samples
# (Float64 / Float32 / PCM16), so the host only writes the RIFF header in front of the bytes.
const SIGOPS_INTERLEAVED = Int32(0x100)
function SignalOperators.sink(x, to::GPUSink, filename::String; encoding::Type = sampletype(x) === Float32 ? Float32 : Float64)
    x = process_sink_params(x)
    plan = lower(x)
    n, c = nframes(x), nchannels(x)
    raw = Array{encoding,2}(undef, c, n)
    enc = encoding === Int16 ? Int32(4) : dtypecode(encoding)
    if n > 0
        handle = compiled(to, plan.bytes)
        ins = [buffer(a) for a in plan.inputs]
        outs = [SigopsBuffer(pointer(raw), n, c, enc | SIGOPS_INTERLEAVED, n)]
        stats = SigopsStats()
        GC.@preserve plan raw check(to, ccall((:sigops_plan_run, libsignalops), Cint,
            (Ptr{Cvoid}, Int64, Ptr{SigopsBuffer}, Ptr{SigopsBuffer}, Ref{SigopsStats}), handle, 1, ins, outs, stats))
    end
    fs = round(Int, framerate(x))                                 # src/WAV.jl:5
    isfloat = encoding <: AbstractFloat
    open(filename, "w") do io
        fmt = IOBuffer()
        foreach(v -> write(fmt, htol(v)), (UInt16(isfloat ? 3 : 1), UInt16(c), UInt32(fs), UInt32(fs * c * sizeof(encoding)),
                                          UInt16(c * sizeof(encoding)), UInt16(8 * sizeof(encoding))))
        isfloat && write(fmt, htol(UInt16(0)))
        fmtb = take!(fmt)
        fact = isfloat ? vcat(Vector{UInt8}("fact"), reinterpret(UInt8, [htol(UInt32(4)), htol(UInt32(n))])) : UInt8[]
        nbytes = sizeof(raw)
        write(io, "RIFF", htol(UInt32(4 + 8 + length(fmtb) + length(fact) + 8 + nbytes)), "WAVE", "fmt ", htol(UInt32(length(fmtb))), fmtb,
              fact, "data", htol(UInt32(nbytes)), raw)
    end
    fs
end

dtypecode(::Type{Float32}) = Int32(1)
dtypecode(::Type{Float64}) = Int32(2)
dtypecode(::Type{<:Integer}) = Int32(3)
dtypecode(::Type{Bool}) = Int32(3)
dtypecode(T::Type) = error("sample type $T is not supported by the GPU sink")
juliatype(code) = (Float32, Float64, Int64)[code]
buffer(a::AbstractVecOrMat{T}) where T =
    SigopsBuffer(pointer(a), size(a, 1), size(a, 2), dtypecode(T), max(size(a, 1), size(a, 2) > 1 ? stride(a, 2) : size(a, 1)))

function run!(to::GPUSink, plans, results)
    handle = compiled(to, plans[1].bytes)
    ins = [buffer(a) for p in plans for a in p.inputs]
    outs = [buffer(r) for r in results]
    stats = SigopsStats()
    GC.@preserve plans results begin                              # caller owns every host buffer
        check(to, ccall((:sigops_plan_run, libsignalops), Cint,
                        (Ptr{Cvoid}, Int64, Ptr{SigopsBuffer}, Ptr{SigopsBuffer}, Ref{SigopsStats}),
                        handle, length(results), ins, outs, stats))
    end
    stats
end

# ---- constants of include/signalops.h ---------------------------------------------------------------------
const MAGIC = 0x504F4753; const PLAN_VERSION = UInt32(1)
const F32, F64, I64 = Int32(1), Int32(2), Int32(3)
const OP_LOAD, OP_ADD, OP_SUB, OP_MUL, OP_DIV = UInt8(1), UInt8(2), UInt8(3), UInt8(4), UInt8(5)
const OP_PUSH, OP_POPADD, OP_POPSUB, OP_POPMUL, OP_POPDIV = UInt8(6), UInt8(7), UInt8(8), UInt8(9), UInt8(10)
const OP_NEG, OP_CAST_F32, OP_CAST_I64 = UInt8(11), UInt8(12), UInt8(13)
const OP_FN1, OP_FN2, OP_POPFN2 = UInt8(14), UInt8(15), UInt8(16)
# closure functions (SIGOPS_EFN_*): unary codes for FN1, binary codes (from 32) for FN2 / POPFN2
const EFN = Dict{Symbol,UInt8}(:abs => 1, :sign => 2, :floor => 3, :ceil => 4, :trunc => 5, :round => 6, :sqrt => 7,
    :clamp => 8, :exp => 9, :exp2 => 10, :expm1 => 11, :log => 12, :log2 => 13, :log10 => 14, :log1p => 15, :sin => 16,
    :cos => 17, :tan => 18, :tanh => 19, :sinh => 20, :cosh => 21, :atan => 22, :cbrt => 23,
    :min => 32, :max => 33, :copysign => 34, :rem => 35, :mod => 36, :pow => 37, :hypot => 38)
const LEAF_NONE, LEAF_CONST, LEAF_BUF, LEAF_CHANSUM, LEAF_GEN = UInt8(0), UInt8(1), UInt8(2), UInt8(3), UInt8(4)
const LEAF_RAMP_ON, LEAF_RAMP_OFF, LEAF_RMS, LEAF_STAGE, LEAF_RANDN = UInt8(5), UInt8(6), UInt8(7), UInt8(8), UInt8(9)
const PAD_CONST, PAD_CYCLE, PAD_MIRROR, PAD_LAST = 0, 1, 2, 3
const FLAG_HAS_OMEGA = UInt8(1)
const FN_SIN, FN_COS, FN_SAW, FN_AFFINE_SIN, FN_AFFINE_COS, FN_IDENTITY, FN_SINRAMP =
    UInt8(1), UInt8(2), UInt8(3), UInt8(4), UInt8(5), UInt8(6), UInt8(7)
const STAGE_MAP, STAGE_IIR, STAGE_FIR = Int32(1), Int32(2), Int32(3)
const FIR_ARBITRARY, FIR_RATIONAL, FIR_DECIMATOR = Int32(1), Int32(2), Int32(3)
const MAX_STACK, MAX_PROG, MAX_PIECES, MAX_BUFS, MAX_SECTIONS = 4, 48, 64, 32, 8

struct LoweringError <: Exception
    msg::String
end
Base.showerror(io::IO, e::LoweringError) = print(io, "GPUSinks: ", e.msg)

# ---- GPU-aware generator functions (host/functors.py) -------------------------------------------------------
# `Signal(fn, ω=...)` with one of these lowers to a device generator; any other callable is evaluated on the
# host with the reference's own formula (src/functions.jl:53-60) and fed as an input buffer.
struct Sawtooth end
(::Sawtooth)(x) = x / π - 1
struct AffineSin; a::Float64; b::Float64; end
(f::AffineSin)(x) = f.a * sin(x) + f.b
struct AffineCos; a::Float64; b::Float64; end
(f::AffineCos)(x) = f.a * cos(x) + f.b
functor_code(::typeof(sin)) = (FN_SIN, 0.0, 0.0)
functor_code(::typeof(cos)) = (FN_COS, 0.0, 0.0)
functor_code(::Sawtooth) = (FN_SAW, 0.0, 0.0)
functor_code(f::AffineSin) = (FN_AFFINE_SIN, f.a, f.b)
functor_code(f::AffineCos) = (FN_AFFINE_COS, f.a, f.b)
functor_code(::typeof(identity)) = (FN_IDENTITY, 0.0, 0.0)
functor_code(_) = nothing

# ---- plan objects ------------------------------------------------------------------------------------------------
const Tag = Tuple{Symbol,Int}          # (:in | :tmp | :out, 0-based index); plain Int for scalar slots

struct Instr                           # sigops_instr, 80 bytes
    op::UInt8; leaf::UInt8; fn::UInt8; flags::UInt8
    buf::Union{Int,Tag}; c_mul::Int32; c_off::Int32
    i0::Int64; i1::Int64; i2::Int64
    d0::Float64; d1::Float64; d2::Float64; d3::Float64; d4::Float64
end
Instr(op, leaf = LEAF_NONE; fn = 0x00, flags = 0x00, buf = 0, c_mul = 1, c_off = 0, i0 = 0, i1 = 0, i2 = 0,
      d0 = 0.0, d1 = 0.0, d2 = 0.0, d3 = 0.0, d4 = 0.0) =
    Instr(op, leaf, fn, flags, buf, Int32(c_mul), Int32(c_off), Int64(i0), Int64(i1), Int64(i2),
          Float64(d0), Float64(d1), Float64(d2), Float64(d3), Float64(d4))
withop(I::Instr, op) = Instr(op, I.leaf, I.fn, I.flags, I.buf, I.c_mul, I.c_off, I.i0, I.i1, I.i2, I.d0, I.d1, I.d2, I.d3, I.d4)
withbuf(I::Instr, buf; leaf = I.leaf) = Instr(I.op, leaf, I.fn, I.flags, buf, I.c_mul, I.c_off, I.i0, I.i1, I.i2, I.d0, I.d1, I.d2, I.d3, I.d4)
withlen(I::Instr, i1, d0) = Instr(I.op, I.leaf, I.fn, I.flags, I.buf, I.c_mul, I.c_off, I.i0, i1, I.i2, d0, I.d1, I.d2, I.d3, I.d4)
padmode(I::Instr) = Int(I.flags >> 1)

mutable struct Piece
    lo::Int; hi::Int; clo::Int; chi::Int
    prog::Vector{Instr}
end

Base.@kwdef mutable struct Stage
    kind::Int32
    out_buf::Tag
    sumsq_slot::Int = -1
    pieces::Vector{Piece} = Piece[]
    in_prog::Vector{Instr} = Instr[]
    epi_prog::Vector{Instr} = Instr[]
    nchannels::Int = 0
    n_in::Int = 0
    n_out::Int = 0
    n_sections::Int = 0
    coef_table::Int = -1
    gain::Float64 = 1.0
    fir_kind::Int32 = 0
    n_phases::Int = 0
    taps_per_phase::Int = 0
    pfb_table::Int = -1
    dpfb_table::Int = -1
    interpolation::Int = 0
    decimation::Int = 0
    input_deficit::Int = 0
    rate::Float64 = 0.0
    phase0::Float64 = 0.0
end

struct BufDesc
    nframes::Int; nchannels::Int; dtype::Int32
end

struct Plan
    bytes::Vector{UInt8}
    inputs::Vector{Array}
    outtype::Type
end

mutable struct Lowerer
    inputs::Vector{BufDesc}
    input_arrays::Vector{Array}
    temps::Vector{BufDesc}
    outputs::Vector{BufDesc}
    n_scalars::Int
    tables::Vector{Vector{Float64}}
    stages::Vector{Stage}
    input_ids::Dict{UInt,Int}
    memo::Dict{Any,Any}
    instance_index::Int          # position of this graph in a batch call (device noise streams)
    Lowerer(instance_index = 0) = new(BufDesc[], Array[], BufDesc[], BufDesc[], 0, Vector{Float64}[], Stage[], Dict{UInt,Int}(),
                                      Dict{Any,Any}(), instance_index)
end

# `Signal(randn; rng = PhiloxRNG(seed, stream))`: noise drawn ON THE DEVICE (src/functions.jl:98-114 with a
# counter-based generator).  Frame k of the stream is a pure function of (seed, stream, k) — Philox4x32-10 +
# Box-Muller, host/philox.py is the executable definition — so nothing crosses the link and the numbers do not
# depend on block scheduling.  In a batch, element i must carry stream = (stream of element 1) + i - 1.
# On the CPU sink the object works as an AbstractRNG through `randn(rng)` (one draw per frame, in order).
mutable struct PhiloxRNG <: Random.AbstractRNG
    seed::UInt64
    stream::Int64
    pos::Int64                   # frames drawn so far by the CPU sink
    PhiloxRNG(seed = 0, stream = 0) = new(UInt64(seed), Int64(stream), 0)
end
function philox4x32_10(c0::UInt32, c1::UInt32, c2::UInt32, c3::UInt32, k0::UInt32, k1::UInt32)
    for _ in 1:10
        p0, p1 = UInt64(0xD2511F53) * c0, UInt64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = ((p1 >> 32) % UInt32) ⊻ c1 ⊻ k0, p1 % UInt32, ((p0 >> 32) % UInt32) ⊻ c3 ⊻ k1, p0 % UInt32
        k0 += 0x9E3779B9
        k1 += 0xBB67AE85
    end
    c0, c1, c2, c3
end
function noiseframe(rng::PhiloxRNG, k::Integer)          # frame k (1-based) of the stream: host/philox.py `frames`
    pair, st = UInt64(k - 1) >> 1, reinterpret(UInt64, rng.stream)
    x0, x1, x2, x3 = philox4x32_10(pair % UInt32, (pair >> 32) % UInt32, st % UInt32, (st >> 32) % UInt32,
                                   rng.seed % UInt32, (rng.seed >> 32) % UInt32)
    unit(lo, hi) = (Float64(((UInt64(hi) << 32) | lo) >> 11) + 0.5) / 9007199254740992.0
    u1, u2 = unit(x0, x1), unit(x2, x3)
    r = sqrt(-2log(u1))
    isodd(k) ? r * cospi(2u2) : r * sinpi(2u2)
end
Random.randn(rng::PhiloxRNG) = noiseframe(rng, rng.pos += 1)   # the CPU sink draws frame by frame, in order

# ---- buffers (lowering.py `add_input` ... `new_scalar`) -------------------------------------------------------
function add_input!(lw::Lowerer, arr::AbstractArray)
    key = objectid(arr)
    haskey(lw.input_ids, key) && return (:in, lw.input_ids[key])
    m = arr isa AbstractVector ? reshape(arr, :, 1) : arr
    T = eltype(m)
    m = T <: Union{Float32,Float64} ? m : (T <: Union{Integer,Bool} ? Int64.(m) : Float64.(m))
    m = m isa Array && (size(m, 2) == 1 || stride(m, 2) >= size(m, 1)) ? m : Array(m)      # dense columns
    k = length(lw.inputs)
    push!(lw.inputs, BufDesc(size(m, 1), size(m, 2), dtypecode(eltype(m))))
    push!(lw.input_arrays, m)
    lw.input_ids[key] = k
    (:in, k)
end
add_temp!(lw, n, c, T) = (push!(lw.temps, BufDesc(Int(n), Int(c), dtypecode(T))); (:tmp, length(lw.temps) - 1))
add_table!(lw, a) = (push!(lw.tables, vec(collect(Float64, a))); length(lw.tables) - 1)
new_scalar!(lw) = (lw.n_scalars += 1; lw.n_scalars - 1)
desc(lw, tag::Tag) = (tag[1] === :in ? lw.inputs : tag[1] === :tmp ? lw.temps : lw.outputs)[tag[2] + 1]

isleaf(prog) = length(prog) == 1 && prog[1].op == OP_LOAD
const ARITH = Dict{Any,Tuple{UInt8,UInt8}}((+) => (OP_ADD, OP_POPADD), (-) => (OP_SUB, OP_POPSUB),
                                           (*) => (OP_MUL, OP_POPMUL), (/) => (OP_DIV, OP_POPDIV))
# program that combines the running accumulator with `prog` (right operand)
as_operand(prog, f) = isleaf(prog) ? [withop(prog[1], ARITH[f][1])] : vcat([Instr(OP_PUSH)], prog, [Instr(ARITH[f][2])])
function stack_depth(prog)
    sp = mx = 0
    for I in prog
        I.op == OP_PUSH && (sp += 1; mx = max(mx, sp))
        (OP_POPADD <= I.op <= OP_POPDIV || I.op == OP_POPFN2) && (sp -= 1)
    end
    mx
end
withfn(I::Instr, op, fn) = Instr(op, I.leaf, UInt8(fn), I.flags, I.buf, I.c_mul, I.c_off, I.i0, I.i1, I.i2, I.d0, I.d1, I.d2, I.d3, I.d4)

# ---- traced OperateOn closures (host/trace.py) ----------------------------------------------------------------------
# The closure is called once with `Traced` values standing for the samples; what it returns is an expression DAG over
# the arguments (`:arg`, key = argument index or (argument, channel)) and Float64 constants.  Anything that needs a
# sample's value (a comparison, and so `if`, `ifelse`, `isless`) throws a LoweringError naming it.
struct TNode
    kind::Symbol
    args::Vector{TNode}
    value::Any
end
struct Traced <: Real
    node::TNode
end
tnode(x::Traced) = x.node
tnode(x::Real) = TNode(:const, TNode[], Float64(x))
traced(kind, xs...; value = nothing) = Traced(TNode(kind, TNode[tnode(x) for x in xs], value))
for (f, k) in ((:+, :+), (:-, :-), (:*, :*), (:/, :/), (:min, :min), (:max, :max), (:copysign, :copysign), (:rem, :rem),
               (:mod, :mod), (:hypot, :hypot), (:^, :pow))
    @eval Base.$f(a::Traced, b::Traced) = traced($(QuoteNode(k)), a, b)
    @eval Base.$f(a::Traced, b::Real) = traced($(QuoteNode(k)), a, b)
    @eval Base.$f(a::Real, b::Traced) = traced($(QuoteNode(k)), a, b)
end
Base.:-(a::Traced) = traced(:neg, a)
Base.:+(a::Traced) = a
for f in (:abs, :sign, :floor, :ceil, :trunc, :sqrt, :exp, :exp2, :expm1, :log, :log2, :log10, :log1p, :sin, :cos, :tan,
          :tanh, :sinh, :cosh, :atan, :cbrt)
    @eval Base.$f(a::Traced) = traced($(QuoteNode(f)), a)
end
Base.round(a::Traced) = traced(:round, a)
Base.round(a::Traced, ::RoundingMode{:Nearest}) = traced(:round, a)
Base.round(a::Traced, ::RoundingMode{:Down}) = traced(:floor, a)
Base.round(a::Traced, ::RoundingMode{:Up}) = traced(:ceil, a)
Base.round(a::Traced, ::RoundingMode{:ToZero}) = traced(:trunc, a)
Base.clamp(a::Traced, lo::Real, hi::Real) = Traced(TNode(:clamp, [tnode(a)], (Float64(lo), Float64(hi))))
Base.literal_pow(::typeof(^), a::Traced, ::Val{2}) = a * a                  # Julia's x^2 is x*x
Base.literal_pow(::typeof(^), a::Traced, ::Val{p}) where p = traced(:pow, a, p)
Base.promote_rule(::Type{Traced}, ::Type{<:Real}) = Traced
Base.float(a::Traced) = a
refuse(what) = throw(LoweringError("$what on a traced sample: the GPU sink compiles the closure once for all samples, " *
                                   "so it cannot depend on a sample's value"))
for f in (:<, :<=, :isless, :(==), :isequal)
    @eval Base.$f(::Traced, ::Traced) = refuse("a comparison ($($(string(f))), ifelse, if)")
    @eval Base.$f(::Traced, ::Real) = refuse("a comparison ($($(string(f))), ifelse, if)")
    @eval Base.$f(::Real, ::Traced) = refuse("a comparison ($($(string(f))), ifelse, if)")
end
Base.isnan(::Traced) = refuse("isnan")
Base.signbit(::Traced) = refuse("signbit")
Base.Bool(::Traced) = refuse("a conversion to Bool")

targs!(out, nd::TNode) = (nd.kind === :arg && push!(out, nd.value); foreach(a -> targs!(out, a), nd.args); out)

# accumulator program of a traced expression (lowering.py `_traced_program`): IEEE results kept, only the exact operand
# swap of + * min max, constants meet Float32 samples as Float32, a Float32 map rounds after every operation
function traced_program(nd::TNode, argprog, f32::Bool)
    rnd = f32 ? [Instr(OP_CAST_F32)] : Instr[]
    cval(v) = f32 ? Float64(Float32(v)) : Float64(v)
    leaf(p, ok = nothing) = isleaf(p) && (ok === nothing || p[1].leaf in ok)
    fn2ok = (LEAF_CONST, LEAF_BUF, LEAF_CHANSUM, LEAF_RMS, LEAF_STAGE, LEAF_RANDN)
    function emit(nd)
        out = emit1(nd)
        length(out) > MAX_PROG && throw(LoweringError("traced expression of more than $MAX_PROG operations"))
        out
    end
    function emit1(nd)
        k = nd.kind
        k === :arg && return copy(argprog[nd.value])
        k === :const && return [Instr(OP_LOAD, LEAF_CONST; d0 = cval(nd.value))]
        k === :neg && return vcat(emit(nd.args[1]), [Instr(OP_NEG)])
        k === :clamp && return vcat(emit(nd.args[1]), [Instr(OP_FN1; fn = EFN[k], d0 = cval(nd.value[1]), d1 = cval(nd.value[2]))], rnd)
        length(nd.args) == 1 && return vcat(emit(nd.args[1]), [Instr(OP_FN1; fn = EFN[k])], rnd)
        pa, pb = emit(nd.args[1]), emit(nd.args[2])
        if k in (:+, :*, :min, :max) && leaf(pa, (LEAF_CONST,)) && !leaf(pb, (LEAF_CONST,))
            pa, pb = pb, pa
        end
        if k in (:+, :-, :*, :/)
            f = k === :+ ? (+) : k === :- ? (-) : k === :* ? (*) : (/)
            leaf(pb) && return vcat(pa, [withop(pb[1], ARITH[f][1])], rnd)
            leaf(pa) && k in (:+, :*) && return vcat(pb, [withop(pa[1], ARITH[f][1])], rnd)
            leaf(pa) && k === :- && return vcat(pb, [Instr(OP_NEG), withop(pa[1], OP_ADD)], rnd)
            return vcat(pa, [Instr(OP_PUSH)], pb, [Instr(ARITH[f][2])], rnd)
        end
        leaf(pb, fn2ok) && return vcat(pa, [withfn(pb[1], OP_FN2, EFN[k])], rnd)
        leaf(pa, fn2ok) && k in (:min, :max) && return vcat(pb, [withfn(pa[1], OP_FN2, EFN[k])], rnd)
        vcat(pa, [Instr(OP_PUSH)], pb, [Instr(OP_POPFN2; fn = EFN[k])], rnd)
    end
    emit(nd)
end
function intersect_pieces(a::Piece, b::Piece)
    lo, hi, clo, chi = max(a.lo, b.lo), min(a.hi, b.hi), max(a.clo, b.clo), min(a.chi, b.chi)
    (lo < hi && clo < chi) ? (lo, hi, clo, chi) : nothing
end

# ---- entry point (`Lowerer.build`) -------------------------------------------------------------------------------
function lower(x; nframes = SignalOperators.nframes(x), outtype = nothing, instance_index = 0)
    lw = Lowerer(instance_index)
    N, C = Int(nframes), nchannels(x)
    S = sampletype(x)
    T = outtype !== nothing ? outtype : S <: Union{Integer,Bool} ? Int64 : S <: Union{Float32,Float64} ? S : Float64
    push!(lw.outputs, BufDesc(N, C, dtypecode(T)))
    pieces = N > 0 ? lower_node(lw, x, 0, 0, N, 1, 0, 0, C) : Piece[]
    push!(lw.stages, Stage(kind = STAGE_MAP, out_buf = (:out, 0), pieces = pieces, nchannels = C, n_out = N))
    fuse_epilogues!(lw)
    check_limits(lw)
    Plan(tobytes(lw), lw.input_arrays, T)
end

# ---- recursive lowering: programs for consumer frames n in [lo,hi) and channels c in [clo,chi), where the node's
# ---- own 0-based frame is n+shift and its channel is c*cm+co (`Lowerer.lower`) ------------------------------------
arraydata(x::AbstractArray) = x
arraydata(x::Tuple{<:AbstractArray,<:Number}) = x[1]
const ArrayLike = Union{AbstractArray,Tuple{<:AbstractArray,<:Number}}

function lower_node(lw, x::ArrayLike, shift, lo, hi, cm, co, clo, chi)                 # src/arrays.jl:118-132
    (lo >= hi || clo >= chi) && return Piece[]
    tag = add_input!(lw, arraydata(x))
    [Piece(lo, hi, clo, chi, [Instr(OP_LOAD, LEAF_BUF; buf = tag, c_mul = cm, c_off = co, i0 = shift, i1 = size(arraydata(x), 1))])]
end

lower_node(lw, x::NumberSignal, shift, lo, hi, cm, co, clo, chi) =                      # src/numbers.jl:62-64
    (lo >= hi || clo >= chi) ? Piece[] : [Piece(lo, hi, clo, chi, [Instr(OP_LOAD, LEAF_CONST; d0 = Float64(x.val))])]

function lower_node(lw, x::SignalFunction, shift, lo, hi, cm, co, clo, chi)            # src/functions.jl:53-60
    (lo >= hi || clo >= chi) && return Piece[]
    fs = framerate(x)
    ismissing(fs) && error("Unknown frame rate for a function signal.")
    if x.fn isa RandFn && x.fn.rng isa PhiloxRNG
        rng = x.fn.rng
        return [Piece(lo, hi, clo, chi, [Instr(OP_LOAD, LEAF_RANDN; i0 = shift + 1, i1 = reinterpret(Int64, rng.seed),
                                               i2 = rng.stream - lw.instance_index)])]
    end
    code = x.fn isa RandFn ? nothing : functor_code(x.fn)
    if code !== nothing && nchannels(x) == 1
        fn, a, b = code
        return [Piece(lo, hi, clo, chi, [Instr(OP_LOAD, LEAF_GEN; fn = fn, flags = ismissing(x.ω) ? 0x00 : FLAG_HAS_OMEGA,
                                               i0 = shift + 1, d0 = Float64(fs), d1 = ismissing(x.ω) ? 0.0 : Float64(x.ω),
                                               d2 = x.ϕ, d3 = a, d4 = b)])]
    end
    # not expressible on the device: frames lo+shift+1 .. hi+shift by the reference's own CPU sink
    vals = sink(Until(x, (hi + shift) * SignalOperators.frames), Array)[lo + shift + 1:hi + shift, :]
    tag = add_input!(lw, vals)
    [Piece(lo, hi, clo, chi, [Instr(OP_LOAD, LEAF_BUF; buf = tag, c_mul = cm, c_off = co, i0 = -lo, i1 = hi - lo)])]
end

function lower_node(lw, x::CutApply{<:Any,<:Any,K}, shift, lo, hi, cm, co, clo, chi) where K   # src/cutting.jl:130-214
    K <: Val{:Until} && return lower_node(lw, x.signal, shift, lo, hi, cm, co, clo, chi)
    k = max(0, resolvelen(x))
    cn = nframes(x.signal)
    (!isknowninf(cn) && cn < k) && error("Signal is too short to skip $(x.time)")
    lower_node(lw, x.signal, shift + k, lo, hi, cm, co, clo, chi)
end

function lower_node(lw, x::AppendSignals, shift, lo, hi, cm, co, clo, chi)             # src/appending.jl:92-110
    out, start = Piece[], 0
    for ch in x.signals
        n = nframes(ch)
        stop = isknowninf(n) ? nothing : start + n
        a = max(lo, start - shift)
        b = stop === nothing ? hi : min(hi, stop - shift)
        a < b && append!(out, lower_node(lw, ch, shift - start, a, b, cm, co, clo, chi))
        stop === nothing && break
        start = stop
    end
    out
end

function lower_node(lw, x::RampSignal{D}, shift, lo, hi, cm, co, clo, chi) where D     # src/ramps.jl:56-119
    (lo >= hi || clo >= chi) && return Piece[]
    L = resolvelen(x)
    fn = x.fn === sinramp ? FN_SINRAMP : x.fn === identity ? FN_IDENTITY : nothing
    if D === :on
        if fn === nothing                     # custom ramp function: its L values as a table, 1 beyond
            tag = add_input!(lw, Float64[x.fn(k / L) for k in 0:L-1])
            return [Piece(lo, hi, clo, chi, [Instr(OP_LOAD, LEAF_BUF; buf = tag, c_mul = 0, c_off = 0, i0 = shift, i1 = L, d0 = 1.0)])]
        end
        return [Piece(lo, hi, clo, chi, [Instr(OP_LOAD, LEAF_RAMP_ON; fn = fn, i0 = shift + 1, i1 = L)])]
    end
    N = nframes(x)
    isknowninf(N) && return [Piece(lo, hi, clo, chi, [Instr(OP_LOAD, LEAF_CONST; d0 = 1.0)])]
    n0 = N - L
    n0 < 0 && error("Ramp is longer than the signal it is applied to.")
    if fn === nothing
        tag = add_input!(lw, Float64[x.fn(1 - k / L) for k in 1:L])
        return [Piece(lo, hi, clo, chi, [Instr(OP_LOAD, LEAF_BUF; buf = tag, c_mul = 0, c_off = 0, i0 = shift - n0, i1 = L, d0 = 1.0)])]
    end
    [Piece(lo, hi, clo, chi, [Instr(OP_LOAD, LEAF_RAMP_OFF; fn = fn, i0 = shift + 1, i1 = n0, i2 = L)])]
end

function lower_node(lw, x::PaddedSignal, shift, lo, hi, cm, co, clo, chi)              # src/padding.jl:150-235
    (lo >= hi || clo >= chi) && return Piece[]
    ch = x.signal
    nc = nframes(ch)
    b = nc - shift                                 # first padded consumer frame
    p = x.Pad
    T = sampletype(x)
    if p === cycle || p === mirror || p === lastframe
        (p !== lastframe && !(ch isa ArrayLike)) &&
            error("Attemped to specify an indexing pad function for a signal which is not known to support `getindex`.")
        nc == 0 && error("Signal is length zero; there is no last frame to pad with.")
        mode = p === cycle ? PAD_CYCLE : p === mirror ? PAD_MIRROR : PAD_LAST
        tag = ch isa ArrayLike ? add_input!(lw, arraydata(ch)) : materialize!(lw, ch, nc)
        return [Piece(lo, hi, clo, chi, [Instr(OP_LOAD, LEAF_BUF; flags = UInt8(mode << 1), buf = tag, c_mul = cm, c_off = co,
                                               i0 = shift, i1 = nc)])]
    end
    out = Piece[]
    lo < min(hi, b) && append!(out, lower_node(lw, ch, shift, lo, min(hi, b), cm, co, clo, chi))
    if max(lo, b) < hi
        a = max(lo, b)
        prog = if p isa Number
            [Instr(OP_LOAD, LEAF_CONST; d0 = Float64(convert(T, p)))]
        elseif p isa Union{Tuple,AbstractArray}
            length(p) == nchannels(x) || error("padding tuple must have one value per channel")
            tag = add_input!(lw, reshape(T[convert(T, v) for v in p], 1, :))
            [Instr(OP_LOAD, LEAF_BUF; flags = UInt8(PAD_LAST << 1), buf = tag, c_mul = cm, c_off = co, i0 = 0, i1 = 1)]
        elseif p isa Function
            [Instr(OP_LOAD, LEAF_CONST; d0 = Float64(p(T)))]       # `zero`, `one`, any fn(T) (src/padding.jl:186-190)
        else
            error("unsupported padding value $p")
        end
        push!(out, Piece(a, hi, clo, chi, prog))
    end
    out
end

function lower_node(lw, x::NormedSignal, shift, lo, hi, cm, co, clo, chi)              # src/filters.jl:296-309
    (lo >= hi || clo >= chi) && return Piece[]
    ch = x.signal
    N = nframes(ch)
    isknowninf(N) && error("Cannot normalize an infinite-length signal. Please use `Until` to take a prefix of the signal")
    C = nchannels(ch)
    key = (:norm, objectid(x))
    if !haskey(lw.memo, key)
        local tag, st
        if ch isa ArrayLike                       # raw data still needs its sum of squares: copy through a MAP stage
            tag = add_temp!(lw, N, C, sampletype(x))
            st = Stage(kind = STAGE_MAP, out_buf = tag, pieces = lower_node(lw, ch, 0, 0, N, 1, 0, 0, C), nchannels = C, n_out = N)
            push!(lw.stages, st)
        else
            tag = materialize!(lw, ch, N)
            st = stage_of(lw, tag)
            if st === nothing || st.n_out != N || st.sumsq_slot >= 0
                src = tag                          # a longer prefix was materialised for someone else: take an exact copy
                tag = add_temp!(lw, N, C, sampletype(x))
                st = Stage(kind = STAGE_MAP, out_buf = tag, nchannels = C, n_out = N,
                           pieces = [Piece(0, N, 0, C, [Instr(OP_LOAD, LEAF_BUF; buf = src, i0 = 0, i1 = N)])])
                push!(lw.stages, st)
            end
        end
        slot = new_scalar!(lw)
        st.sumsq_slot = slot
        lw.memo[key] = (tag, slot)
    end
    tag, slot = lw.memo[key]
    prog = [Instr(OP_LOAD, LEAF_BUF; buf = tag, c_mul = cm, c_off = co, i0 = shift, i1 = N),
            Instr(OP_DIV, LEAF_RMS; buf = slot, d0 = Float64(N * C))]
    sampletype(x) === Float32 && push!(prog, Instr(OP_CAST_F32))      # `vals ./= rms` is stored as Float32
    [Piece(lo, hi, clo, chi, prog)]
end

function lower_node(lw, x::FilteredSignal, shift, lo, hi, cm, co, clo, chi)            # src/filters.jl:204-262
    (lo >= hi || clo >= chi) && return Piece[]
    tag, n = materialize_filter!(lw, x, hi + shift)
    [Piece(lo, hi, clo, chi, [Instr(OP_LOAD, LEAF_BUF; buf = tag, c_mul = cm, c_off = co, i0 = shift, i1 = n)])]
end

unwrapfn(f::FnBr) = f.fn
unwrapfn(f) = f

function lower_node(lw, x::MapSignal, shift, lo, hi, cm, co, clo, chi)                 # src/mapsignal.jl:219-272
    (lo >= hi || clo >= chi) && return Piece[]
    fn = unwrapfn(x.fn)
    kids = x.padded_signals
    if x.bychannel
        if fn isa ToEltypeFn
            El = typeof(fn).parameters[1]
            ps = lower_node(lw, kids[1], shift, lo, hi, cm, co, clo, chi)
            code = dtypecode(El)
            (code == F64 || (code == F32 && sampletype(kids[1]) === Float32)) && return ps
            cast = code == F32 ? OP_CAST_F32 : OP_CAST_I64
            return [Piece(p.lo, p.hi, p.clo, p.chi, vcat(p.prog, [Instr(cast)])) for p in ps]
        end
        haskey(ARITH, fn) || return lower_traced(lw, x, fn, kids, shift, lo, hi, cm, co, clo, chi)
        acc = lower_node(lw, kids[1], shift, lo, hi, cm, co, clo, chi)
        (length(kids) == 1 && fn === (-)) &&
            return [Piece(p.lo, p.hi, p.clo, p.chi, vcat(p.prog, [Instr(OP_NEG)])) for p in acc]
        for k in Base.tail(kids)
            rhs = lower_node(lw, k, shift, lo, hi, cm, co, clo, chi)
            nxt = Piece[]
            for a in acc, b in rhs
                r = intersect_pieces(a, b)
                r === nothing || push!(nxt, Piece(r..., vcat(a.prog, as_operand(b.prog, fn))))
            end
            acc = nxt
        end
        # Float32 arithmetic rounds after every operation in the reference
        sampletype(x) === Float32 && (acc = [Piece(p.lo, p.hi, p.clo, p.chi, vcat(p.prog, [Instr(OP_CAST_F32)])) for p in acc])
        return acc
    end
    # ---- whole-frame functions (bychannel=false), src/reformatting.jl:148-184, src/mapsignal.jl:359-391
    fn isa AsNChannels && return lower_node(lw, kids[1], shift, lo, hi, 0, 0, clo, chi)
    if fn isa GetChanFn
        1 <= fn.n <= nchannels(kids[1]) || error("channel $(fn.n) out of range")
        return lower_node(lw, kids[1], shift, lo, hi, 0, fn.n - 1, clo, chi)
    end
    if fn isa As1Channel
        k = kids[1]
        nc = nchannels(k)
        acc = lower_node(lw, k, shift, lo, hi, 0, 0, clo, chi)
        for ch in 1:nc-1
            rhs = lower_node(lw, k, shift, lo, hi, 0, ch, clo, chi)
            nxt = Piece[]
            for a in acc, b in rhs
                r = intersect_pieces(a, b)
                r === nothing || push!(nxt, Piece(r..., vcat(a.prog, as_operand(b.prog, +))))
            end
            acc = nxt
        end
        if any(p -> length(p.prog) > MAX_PROG || stack_depth(p.prog) > MAX_STACK, acc)
            n = isknowninf(nframes(k)) ? hi + shift : nframes(k)
            tag = materialize!(lw, k, n)
            return [Piece(lo, hi, clo, chi, [Instr(OP_LOAD, LEAF_CHANSUM; buf = tag, i0 = shift, i1 = n, i2 = nc)])]
        end
        return acc
    end
    if fn === tuplecat
        out, off = Piece[], 0
        for k in kids
            kc = nchannels(k)
            if cm == 0
                off <= co < off + kc && append!(out, lower_node(lw, k, shift, lo, hi, 0, co - off, clo, chi))
            else
                a, b = max(clo, off - co), min(chi, off + kc - co)
                a < b && append!(out, lower_node(lw, k, shift, lo, hi, 1, co - off, a, b))
            end
            off += kc
        end
        return out
    end
    lower_traced(lw, x, fn, kids, shift, lo, hi, cm, co, clo, chi)
end

# any other OperateOn function: trace it, compile the expression (lowering.py `_lower_traced`)
function lower_traced(lw, x, fn, kids, shift, lo, hi, cm, co, clo, chi)
    if x.bychannel
        r = fn((Traced(TNode(:arg, TNode[], k - 1)) for k in eachindex(kids))...)
        r isa Traced || throw(LoweringError("OperateOn($fn) did not return one traced value per sample"))
        groups = [(clo, chi, cm, co, r.node)]
    else
        r = fn((Tuple(Traced(TNode(:arg, TNode[], (k - 1, c))) for c in 0:nchannels(kids[k])-1) for k in eachindex(kids))...)
        roots = r isa Traced ? [r.node] : [tnode(v) for v in r]
        groups = [(c, c + 1, 0, cm == 0 ? co : c * cm + co, roots[(cm == 0 ? co : c * cm + co) + 1]) for c in clo:chi-1]
    end
    T = sampletype(x)
    f32 = T === Float32
    tail = T <: Integer ? [Instr(OP_CAST_I64)] : Instr[]
    function argpieces(key, a, b, gcm, gco, mat)
        k, ch = x.bychannel ? (key, nothing) : key
        kcm, kco = ch === nothing ? (gcm, gco) : (0, ch)
        kid = kids[k+1]
        if mat
            n = isknowninf(nframes(kid)) ? hi + shift : nframes(kid)
            tag = materialize!(lw, kid, n)
            return [Piece(lo, hi, a, b, [Instr(OP_LOAD, LEAF_BUF; buf = tag, c_mul = kcm, c_off = kco, i0 = shift, i1 = n)])]
        end
        lower_node(lw, kid, shift, lo, hi, kcm, kco, a, b)
    end
    exprs = Set{Any}()
    function build(mat)
        out = Piece[]
        for (a, b, gcm, gco, root) in groups
            combos = [(lo, hi, a, b, Dict{Any,Vector{Instr}}())]
            for key in sort!(collect(targs!(Set{Any}(), root)); by = repr)
                ps = argpieces(key, a, b, gcm, gco, key in mat)
                any(p -> !isleaf(p.prog), ps) && push!(exprs, key)
                nxt = []
                for c0 in combos, p in ps
                    r = intersect_pieces(Piece(c0[1], c0[2], c0[3], c0[4], Instr[]), p)
                    r === nothing || push!(nxt, (r..., merge(c0[5], Dict{Any,Vector{Instr}}(key => p.prog))))
                end
                combos = nxt
            end
            for (plo, phi, pclo, pchi, argprog) in combos
                prog = vcat(traced_program(root, argprog, f32), tail)
                (length(prog) > MAX_PROG || stack_depth(prog) > MAX_STACK) && return nothing
                push!(out, Piece(plo, phi, pclo, pchi, prog))
            end
        end
        out
    end
    out = try build(Set{Any}()) catch e; e isa LoweringError ? nothing : rethrow() end
    out === nothing || return out
    # an argument used several times is evaluated each time: when that does not fit, the arguments that are
    # expressions of their own are computed once into temps and read back as buffers
    out = try build(copy(exprs)) catch e; e isa LoweringError ? nothing : rethrow() end
    out === nothing && throw(LoweringError("OperateOn($fn): the traced expression needs more than $MAX_PROG operations " *
                                           "or nests deeper than the device stack ($MAX_STACK)"))
    out
end

lower_node(lw, x, args...) = throw(LoweringError("cannot lower node of type $(typeof(x))"))

# ---- barriers ----------------------------------------------------------------------------------------------------------
stage_of(lw, tag) = (i = findfirst(s -> s.out_buf == tag, lw.stages); i === nothing ? nothing : lw.stages[i])

# frames [0,n) of `x` in a buffer; reuses a producing stage when there is one (`_materialize`)
function materialize!(lw, x, n)
    (x isa ArrayLike && size(arraydata(x), 1) >= n) && return add_input!(lw, arraydata(x))
    x isa FilteredSignal && return materialize_filter!(lw, x, n)[1]
    key = objectid(x)
    m = get(lw.memo, key, nothing)
    (m !== nothing && m[2] >= n) && return m[1]
    C = nchannels(x)
    tag = add_temp!(lw, n, C, sampletype(x))
    push!(lw.stages, Stage(kind = STAGE_MAP, out_buf = tag, pieces = lower_node(lw, x, 0, 0, n, 1, 0, 0, C), nchannels = C, n_out = n))
    lw.memo[key] = (tag, n)
    tag
end

# stage(s) computing frames [0,n) of a FilteredSignal into a temp (`_materialize_filter`)
function materialize_filter!(lw, x::FilteredSignal, need)
    N = nframes(x)
    n = isknowninf(N) ? need : N               # causal: a prefix needs only a prefix
    key = objectid(x)
    m = get(lw.memo, key, nothing)
    (m !== nothing && m[2] >= n) && return m
    ch = x.signal
    C = nchannels(ch)
    fs = framerate(x)
    ismissing(fs) && error("Unknown frame rate for a filtered signal.")
    h = x.fn(fs)                                # design at sink time, src/filters.jl:205 (once, not per channel)
    T = sampletype(x)
    tag = h isa DSP.Filters.FIRFilter ? emit_fir!(lw, h, ch, n, C, T) : emit_iir!(lw, h, ch, n, C, T)
    lw.memo[key] = (tag, n)
    (tag, n)
end

# single program giving frames [0,n_in) of `child` followed by zeros (`Pad(x.signal,zero)`, src/filters.jl:240);
# materialises when piecewise (`_input_program`)
function input_program!(lw, ch, n_in, C)
    cn = nframes(ch)
    avail = isknowninf(cn) ? n_in : min(cn, n_in)
    pieces = avail > 0 ? lower_node(lw, ch, 0, 0, avail, 1, 0, 0, C) : Piece[]
    if length(pieces) == 1 && isleaf(pieces[1].prog)
        I = pieces[1].prog[1]
        if I.leaf == LEAF_BUF && I.i0 == 0 && padmode(I) == PAD_CONST && I.c_mul == 1 && I.c_off == 0
            return [withlen(I, min(I.i1, avail), 0.0)], true
        end
    end
    if length(pieces) == 1 && avail == n_in && !any(I -> I.leaf == LEAF_BUF && padmode(I) != PAD_CONST, pieces[1].prog)
        return pieces[1].prog, false
    end
    avail == 0 && return [Instr(OP_LOAD, LEAF_CONST; d0 = 0.0)], false
    tag = add_temp!(lw, avail, C, sampletype(ch))
    push!(lw.stages, Stage(kind = STAGE_MAP, out_buf = tag, pieces = pieces, nchannels = C, n_out = avail))
    [Instr(OP_LOAD, LEAF_BUF; buf = tag, i0 = 0, i1 = avail, d0 = 0.0)], true
end

# DSP.jl coefficient object -> second-order sections (what `DF2TFilter(h)` runs, src/filters.jl:94).
# PolynomialRatio above order 2 is factored (roots of numerator and denominator) into sections; the
# cascade equals the direct form up to rounding.
tosos(h::DSP.SecondOrderSections) = h
tosos(h::DSP.Biquad) = DSP.SecondOrderSections([h], 1.0)
tosos(h) = convert(DSP.SecondOrderSections, h)

function emit_iir!(lw, h, ch, n, C, T)                                          # SURVEY.md App. B.2
    prog, _ = input_program!(lw, ch, n, C)
    sos = tosos(h)
    biquads = collect(sos.biquads)
    groups = isempty(biquads) ? [DSP.Biquad{Float64}[]] : [biquads[i:min(i + MAX_SECTIONS - 1, end)] for i in 1:MAX_SECTIONS:length(biquads)]
    tag = (:tmp, -1)
    for (gi, grp) in enumerate(groups)
        lastg = gi == length(groups)
        rows = isempty(grp) ? Float64[1, 0, 0, 0, 0] : reduce(vcat, [Float64[b.b0, b.b1, b.b2, b.a1, b.a2] for b in grp])
        tag = add_temp!(lw, n, C, lastg ? T : Float64)
        tbl = add_table!(lw, rows)
        push!(lw.stages, Stage(kind = STAGE_IIR, out_buf = tag, in_prog = prog, nchannels = C, n_in = n, n_out = n,
                               n_sections = max(1, length(grp)), coef_table = tbl, gain = lastg ? Float64(sos.g) : 1.0))
        prog = [Instr(OP_LOAD, LEAF_BUF; buf = tag, i0 = 0, i1 = n, d0 = 0.0)]
    end
    tag
end

function emit_fir!(lw, h, ch, n_out, C, T)                                      # src/reformatting.jl:92-99, App. B.4
    k = h.kernel
    cn = nframes(ch)
    rate = k isa DSP.Filters.FIRArbitrary ? Float64(k.rate) : Float64(h.ratio)
    tapsper = k isa Union{DSP.Filters.FIRDecimator,DSP.Filters.FIRStandard} ? length(k.h) : Int(k.tapsPerϕ)
    n_in = isknowninf(cn) ? ceil(Int, n_out / rate) + Int(k.inputDeficit) + tapsper + 2 : cn
    prog, plain = input_program!(lw, ch, n_in, C)
    f32 = T === Float32
    if !plain || sampletype(ch) === Float32          # the tensor-core kernels want plain Float64 rows on both sides
        tag_in = add_temp!(lw, n_in, C, sampletype(ch) === Float32 ? Float64 : sampletype(ch))
        push!(lw.stages, Stage(kind = STAGE_MAP, out_buf = tag_in, nchannels = C, n_out = n_in, pieces = [Piece(0, n_in, 0, C, prog)]))
        prog = [Instr(OP_LOAD, LEAF_BUF; buf = tag_in, i0 = 0, i1 = n_in, d0 = 0.0)]
    end
    tag = add_temp!(lw, n_out, C, f32 ? Float64 : T)
    st = Stage(kind = STAGE_FIR, out_buf = tag, in_prog = prog, nchannels = C, n_in = n_in, n_out = n_out, rate = rate,
               input_deficit = Int(k.inputDeficit))
    if k isa DSP.Filters.FIRArbitrary
        st.fir_kind = FIR_ARBITRARY
        st.n_phases, st.taps_per_phase = Int(k.Nϕ), Int(k.tapsPerϕ)
        st.pfb_table = add_table!(lw, k.pfb)              # Julia column ϕ = row [phase][tap] of the C layout
        st.dpfb_table = add_table!(lw, k.dpfb)
        st.phase0 = Float64(k.ϕAccumulator)
    elseif k isa Union{DSP.Filters.FIRRational,DSP.Filters.FIRInterpolator}
        st.fir_kind = FIR_RATIONAL
        st.n_phases, st.taps_per_phase = Int(k.Nϕ), Int(k.tapsPerϕ)
        st.interpolation = Int(k.Nϕ)
        st.decimation = k isa DSP.Filters.FIRRational ? Int(denominator(k.ratio)) : 1
        st.pfb_table = add_table!(lw, k.pfb)
        st.phase0 = Float64(k.ϕIdx)
    elseif k isa DSP.Filters.FIRDecimator
        st.fir_kind = FIR_DECIMATOR
        st.n_phases, st.taps_per_phase = 1, length(k.h)
        st.interpolation, st.decimation = 1, Int(k.decimation)
        st.pfb_table = add_table!(lw, k.h)                 # stored reversed by DSP.jl: window order
        st.phase0 = 1.0
    else                                                   # FIRStandard: a decimator with step 1
        st.fir_kind = FIR_DECIMATOR
        st.n_phases, st.taps_per_phase = 1, length(k.h)
        st.interpolation, st.decimation = 1, 1
        st.pfb_table = add_table!(lw, k.h)
        st.phase0 = 1.0
    end
    push!(lw.stages, st)
    if f32
        tag32 = add_temp!(lw, n_out, C, T)
        push!(lw.stages, Stage(kind = STAGE_MAP, out_buf = tag32, nchannels = C, n_out = n_out, pieces = [Piece(0, n_out, 0, C,
              [Instr(OP_LOAD, LEAF_BUF; buf = tag, i0 = 0, i1 = n_out, d0 = 0.0), Instr(OP_CAST_F32)])]))
        return tag32
    end
    tag
end

# ---- post passes (`_fuse_epilogues`, `_drop_unused_temps`, `_check_limits`) -------------------------------------------
bufrefs(prog) = [I for I in prog if (I.leaf == LEAF_BUF || I.leaf == LEAF_CHANSUM) && I.buf isa Tag]
allprogs(s::Stage) = vcat([p.prog for p in s.pieces], [s.in_prog, s.epi_prog])

# a MAP stage that only post-processes the full output of the IIR/FIR stage right before it becomes that stage's
# epilogue (one HBM round trip)
function fuse_epilogues!(lw)
    changed = true
    while changed
        changed = false
        for (i, st) in enumerate(lw.stages)
            (st.kind == STAGE_MAP && length(st.pieces) == 1) || continue
            pc = st.pieces[1]
            refs = [I for I in bufrefs(pc.prog) if I.buf[1] === :tmp]
            for tag in unique(I.buf for I in refs)
                j = findfirst(s -> s.out_buf == tag, lw.stages[1:i-1])
                j === nothing && continue
                prod = lw.stages[j]
                (!isempty(prod.epi_prog) || prod.sumsq_slot >= 0) && continue
                bare = length(pc.prog) == 1 && pc.prog[1].op == OP_LOAD && desc(lw, st.out_buf).dtype == desc(lw, tag).dtype
                (prod.kind == STAGE_MAP && !bare) && continue
                const_gain = 2 <= length(pc.prog) <= 3 && pc.prog[1].op == OP_LOAD &&
                             all(I -> I.op == OP_MUL && I.leaf == LEAF_CONST, pc.prog[2:end]) &&
                             desc(lw, st.out_buf).dtype == desc(lw, tag).dtype == F64
                (prod.kind == STAGE_FIR && !(bare || const_gain)) && continue
                uses = [I for I in refs if I.buf == tag]
                elsewhere = any(I.buf == tag for s2 in lw.stages if s2 !== st for pr in allprogs(s2) for I in bufrefs(pr))
                I0 = uses[1]
                (length(uses) != 1 || elsewhere || I0.leaf != LEAF_BUF || I0.i0 != 0 || I0.c_mul != 1 || I0.c_off != 0 ||
                 padmode(I0) != PAD_CONST || pc.lo != 0 || pc.hi != prod.n_out || pc.clo != 0 || pc.chi != prod.nchannels ||
                 I0.i1 != prod.n_out) && continue
                ob = desc(lw, st.out_buf)
                (ob.nframes != prod.n_out || ob.nchannels != prod.nchannels) && continue
                if prod.kind == STAGE_MAP
                    prod.out_buf = st.out_buf
                    prod.sumsq_slot = st.sumsq_slot
                    deleteat!(lw.stages, i)
                else
                    prod.epi_prog = [I === I0 ? withbuf(I, 0; leaf = LEAF_STAGE) : I for I in pc.prog]
                    prod.out_buf = st.out_buf
                    prod.sumsq_slot = st.sumsq_slot
                    lw.stages[i] = prod             # the fused stage runs where the MAP stage stood
                    deleteat!(lw.stages, j)
                end
                changed = true
                break
            end
            changed && break
        end
    end
    drop_unused_temps!(lw)
end

function drop_unused_temps!(lw)
    used = Set(s.out_buf[2] for s in lw.stages if s.out_buf[1] === :tmp)
    remap, temps = Dict{Int,Int}(), BufDesc[]
    for (k, t) in enumerate(lw.temps)
        if (k - 1) in used
            remap[k - 1] = length(temps)
            push!(temps, t)
        end
    end
    lw.temps = temps
    fixtag(t) = (t isa Tag && t[1] === :tmp) ? (:tmp, remap[t[2]]) : t
    fixprog(pr) = [withbuf(I, fixtag(I.buf)) for I in pr]
    for s in lw.stages
        s.out_buf = fixtag(s.out_buf)
        foreach(pc -> pc.prog = fixprog(pc.prog), s.pieces)
        s.in_prog = fixprog(s.in_prog)
        s.epi_prog = fixprog(s.epi_prog)
    end
end

function check_limits(lw)
    length(lw.inputs) + length(lw.temps) + length(lw.outputs) > MAX_BUFS && throw(LoweringError("graph needs more than $MAX_BUFS buffers"))
    for s in lw.stages
        length(s.pieces) > MAX_PIECES && throw(LoweringError("stage has $(length(s.pieces)) pieces (max $MAX_PIECES)"))
        for pr in allprogs(s)
            length(pr) > MAX_PROG && throw(LoweringError("fused expression of $(length(pr)) operations exceeds $MAX_PROG"))
            stack_depth(pr) > MAX_STACK && throw(LoweringError("expression nests deeper than the device stack"))
        end
    end
end

# ---- plan bytes (`Plan.tobytes`; layout in include/signalops.h) -------------------------------------------------------
function tobytes(lw::Lowerer)
    n_in, n_tmp = length(lw.inputs), length(lw.temps)
    bid(t::Tag) = t[1] === :in ? t[2] : t[1] === :tmp ? n_in + t[2] : n_in + n_tmp + t[2]
    bid(t::Int) = t
    instrs, pieces, stages = Instr[], IOBuffer(), IOBuffer()
    npieces = 0
    w(io, T, v) = write(io, htol(convert(T, v)))
    for st in lw.stages
        p_start = npieces
        in_start = in_len = epi_start = epi_len = 0
        if st.kind == STAGE_MAP
            for pc in st.pieces
                w(pieces, Int64, pc.lo); w(pieces, Int64, pc.hi - pc.lo)
                w(pieces, Int32, pc.clo); w(pieces, Int32, pc.chi - pc.clo)
                w(pieces, Int32, length(instrs)); w(pieces, Int32, length(pc.prog))
                append!(instrs, pc.prog)
                npieces += 1
            end
        else
            in_start, in_len = length(instrs), length(st.in_prog)
            append!(instrs, st.in_prog)
            epi_start, epi_len = length(instrs), length(st.epi_prog)
            append!(instrs, st.epi_prog)
        end
        foreach(v -> w(stages, Int32, v), (st.kind, bid(st.out_buf), st.sumsq_slot, p_start, length(st.pieces), in_start, in_len,
                                           epi_start, epi_len, st.nchannels))
        w(stages, Int64, st.n_in); w(stages, Int64, st.n_out)
        w(stages, Int32, st.n_sections); w(stages, Int32, st.coef_table); w(stages, Float64, st.gain)
        foreach(v -> w(stages, Int32, v), (st.fir_kind, st.n_phases, st.taps_per_phase, st.pfb_table, st.dpfb_table,
                                           st.interpolation, st.decimation, 0))
        w(stages, Int64, st.input_deficit); w(stages, Float64, st.rate); w(stages, Float64, st.phase0)
    end
    blob = reduce(vcat, lw.tables; init = Float64[])
    io = IOBuffer()
    foreach(v -> w(io, UInt32, v), (MAGIC, PLAN_VERSION, n_in, n_tmp, length(lw.outputs), lw.n_scalars, length(lw.tables),
                                    length(instrs), npieces, length(lw.stages)))
    w(io, UInt64, length(blob))
    for b in vcat(lw.inputs, lw.temps, lw.outputs)
        w(io, Int64, b.nframes); w(io, Int32, b.nchannels); w(io, Int32, b.dtype)
    end
    off = 0
    for t in lw.tables
        w(io, Int64, off); w(io, Int64, length(t)); off += length(t)
    end
    for I in instrs
        write(io, I.op, I.leaf, I.fn, I.flags)
        w(io, Int32, bid(I.buf)); w(io, Int32, I.c_mul); w(io, Int32, I.c_off)
        w(io, Int64, I.i0); w(io, Int64, I.i1); w(io, Int64, I.i2)
        foreach(v -> w(io, Float64, v), (I.d0, I.d1, I.d2, I.d3, I.d4))
    end
    write(io, take!(pieces)); write(io, take!(stages))
    foreach(v -> w(io, Float64, v), blob)
    take!(io)
end

end # module
