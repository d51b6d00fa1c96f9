# test_plans.jl — byte-for-byte check of GPUSinks.lower against the plans host/lowering.py emits.
#
# Run by a maintainer who has Julia, SignalOperators.jl 0.5 and DSP.jl 0.6 (none of which exist in this
# repository's build image):
#     julia --project -e 'include("signaloperators.jl_b200/julia/test_plans.jl")'
# Each graph below is the Julia spelling of the graph of the same name in tests/golden/plans/make_plans.py
# (traced OperateOn closures: tests/golden/plans/make_fn_plans.py).
# Everything the lowering decides (buffer shapes, instructions, pieces, stage wiring, integer fields) must
# match exactly; numbers that DSP.jl produces on the Julia side and host/dspjl.py on the Python side (biquad
# coefficients, polyphase banks, and the gain / rate / phase0 fields of a stage) must agree to 1e-12.
using Test, SignalOperators, SignalOperators.Units, DSP
include(joinpath(@__DIR__, "GPUSink.jl"))
using .GPUSinks: lower, Sawtooth, AffineSin, PhiloxRNG

const PLANS = normpath(joinpath(@__DIR__, "..", "..", "tests", "golden", "plans"))
Z(dims...) = zeros(dims...)

graphs = Dict(
    "noise" => () -> begin
        x = Signal(sin, ω = 1kHz) |> Until(1s) |> Ramp |> Normpower |> Amplify(-20dB + 5dB)
        y = Signal(randn, 44.1kHz, rng = PhiloxRNG(UInt64(2)^63 + 1983, 3)) |> After(0.5s) |> Until(1s) |>
            Filt(Bandstop, 0.5kHz, 2kHz) |> Normpower |> Amplify(-20dB)
        Mix(x, y)
    end,
    "cfg1" => () -> begin
        x = Signal(sin, ω = 1kHz) |> Until(1s) |> Ramp |> Normpower |> Amplify(-20dB + 5dB)
        y = Signal(Z(44100), 44.1kHz) |> Until(1s) |> Filt(Bandstop, 0.5kHz, 2kHz) |> Normpower |> Amplify(-20dB)
        Mix(x, y) |> ToFramerate(44.1kHz)
    end,
    "cfg2" => () -> Signal(Z(480000, 2), 48kHz) |> Filt(Lowpass, 4kHz, order = 8) |> Amplify(-20dB),
    "cfg3" => () -> ToFramerate(Signal(Z(2646000, 2), 44.1kHz), 48kHz),
    "cfg3_gain" => () -> ToFramerate(Signal(Z(2646000, 2), 44.1kHz), 48kHz) |> Amplify(-6dB),
    "cfg4" => () -> begin
        fs = 44.1kHz
        s1 = Signal(sin, ω = 1kHz) |> Until(5s) |> Ramp |> Normpower |> Amplify(-20dB)
        s2 = Signal(Z(88200), fs) |> Normpower |> Amplify(-20dB)
        s3 = Signal(Sawtooth(), ω = 1kHz) |> Until(2s) |> Ramp |> Normpower |> Amplify(-20dB)
        s4 = Signal(Z(220500), fs) |> Amplify(Signal(AffineSin(0.5, 0.5), ω = 5Hz)) |> Until(5s) |> Normpower |> Amplify(-20dB)
        x = Signal(sin, ω = 1kHz) |> Until(1s) |> Ramp |> Normpower |> Amplify(-20dB + 5dB)
        y = Signal(Z(44100), fs) |> Until(1s) |> Filt(Bandstop, 0.5kHz, 2kHz) |> Normpower |> Amplify(-20dB)
        Append(s1, s2, s3, s4, Mix(x, y)) |> Normpower |> Amplify(-20dB) |> ToFramerate(fs)
    end,
    "cfg5" => () -> begin
        am = Amplify(Signal(Z(576000, 4), 96kHz), Signal(AffineSin(0.5, 0.5), ω = 5Hz)) |> Until(6s)
        am |> Filt(Bandpass, 500Hz, 4kHz) |> Ramp(10ms) |> Mix(Signal(sin, ω = 1kHz) |> Until(6s))
    end,
    "plumbing" => () -> begin
        a = Signal(Z(100, 2), 10Hz)
        b = Signal(Z(40, 2), 10Hz)
        x = a |> After(2s) |> Append(b |> Pad(zero) |> Until(60frames)) |> RampOn(5frames)
        Mix(x, Signal(Z(30, 2), 10Hz) |> Pad(cycle) |> Until(140frames)) |> Amplify(0.5)
    end,
    "channels" => () -> begin
        a = Signal(Z(50, 3), 10Hz)
        AddChannel(a |> SelectChannel(2), a |> ToChannels(1)) |> ToChannels(2) |> Amplify(2)
    end,
    "envelope" => () -> OperateOn(abs, Signal(Z(48000, 2), 48kHz)) |> Filt(Lowpass, 50Hz),
    "softclip" => () -> Signal(zeros(Float32, 48000, 2), 48kHz) |> Filt(Bandpass, 500Hz, 4kHz) |> Operate(v -> tanh(2f0 * v)),
    "clamp" => () -> begin
        x = Signal(Z(1000, 1), 10kHz)
        Mix(OperateOn(v -> clamp(v, -1, 1), x), OperateOn(v -> max(v, 0), x))
    end,
    "midside" => () -> OperateOn(f -> (0.5(f[1] + f[2]), 0.5(f[1] - f[2])), Signal(Z(1000, 2), 10kHz), bychannel = false),
)

# section offsets of a plan (include/signalops.h)
function sections(b::Vector{UInt8})
    u32(i) = ltoh(reinterpret(UInt32, b[4i+1:4i+4])[1])
    n_in, n_tmp, n_out, n_tab, n_instr, n_piece, n_stage = u32(2), u32(3), u32(4), u32(6), u32(7), u32(8), u32(9)
    n_dbl = ltoh(reinterpret(UInt64, b[41:48])[1])
    stages0 = 48 + 16 * (n_in + n_tmp + n_out) + 16 * n_tab + 80 * n_instr + 32 * n_piece
    blob0 = stages0 + 128 * n_stage
    @assert length(b) == blob0 + 8 * n_dbl
    (stages0 = Int(stages0), n_stage = Int(n_stage), blob0 = Int(blob0))
end
f64(b, off) = ltoh(reinterpret(Float64, b[off+1:off+8])[1])

@testset "GPUSinks.lower emits the plans of host/lowering.py" begin
    for (name, build) in graphs
        want = read(joinpath(PLANS, name * ".bin"))
        got = lower(SignalOperators.process_sink_params(build())).bytes
        @test length(got) == length(want)
        length(got) == length(want) || continue
        s = sections(want)
        @test got[1:s.stages0] == want[1:s.stages0]                       # header, buffers, tables, instructions, pieces
        for k in 0:s.n_stage-1                                           # stages: integers exactly, DSP.jl numbers to 1e-12
            o = s.stages0 + 128k
            dbl = (o + 64, o + 112, o + 120)                              # gain, rate, phase0
            mask = trues(128)
            foreach(d -> mask[d-o+1:d-o+8] .= false, dbl)
            @test got[o+1:o+128][mask] == want[o+1:o+128][mask]
            foreach(d -> @test(isapprox(f64(got, d), f64(want, d); rtol = 1e-12, atol = 1e-300)), dbl)
        end
        gb = reinterpret(Float64, got[s.blob0+1:end]); wb = reinterpret(Float64, want[s.blob0+1:end])
        @test all(isapprox.(ltoh.(gb), ltoh.(wb); rtol = 1e-12, atol = 1e-15))
    end
end
