# test_gen_plans.jl — byte-for-byte check of GPUSinks.lower on traced generator closures `Signal(ϕ -> …)` against the
# plans host/lowering.py emits (tests/golden/plans/make_gen_plans.py, each graph below is the Julia spelling of the
# graph of the same name there).
#
# Run by a maintainer who has Julia, SignalOperators.jl 0.5 and DSP.jl 0.6 (none of which exist in this
# repository's build image):
#     julia --project -e 'include("signaloperators.jl_b200/julia/test_gen_plans.jl")'
# Everything the lowering decides must match exactly; the biquad coefficients and the gain / rate / phase0 fields of a
# stage, which DSP.jl computes on the Julia side, to 1e-12 (as in test_plans.jl).
using Test, SignalOperators, SignalOperators.Units, DSP
include(joinpath(@__DIR__, "GPUSink.jl"))
using .GPUSinks: lower

const PLANS = normpath(joinpath(@__DIR__, "..", "..", "tests", "golden", "plans"))

graphs = Dict(
    "gen_am" => () -> begin
        am = Amplify(Signal(zeros(48000, 2), 48kHz), Signal(ϕ -> 0.5sin(ϕ) + 0.25sin(2ϕ) + 0.25, ω = 5Hz))
        tone = Signal(ϕ -> 0.3sin(ϕ) + 0.1cos(3ϕ), ω = 1kHz) |> Until(1s)
        am |> Until(1s) |> Filt(Bandpass, 500Hz, 4kHz) |> Ramp(10ms) |> Mix(tone)
    end,
    "gen_readme" => () -> Mix(Signal(ϕ -> ϕ / π - 1, 10kHz, ω = 100Hz), Signal(ϕ -> 0.5sin(ϕ) + 0.5, 10kHz, ω = 5Hz, ϕ = π / 2)) |>
                          Until(100ms),
    "gen_stereo" => () -> Signal(ϕ -> (sin(ϕ), 0.5cos(ϕ) + 0.1sin(5ϕ)), 10kHz, ω = 300Hz) |> Until(100ms),
    "gen_time" => () -> Signal(t -> exp(-3t) * sin(2π * 440 * t), 10kHz) |> Until(100ms),
)

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

@testset "GPUSinks.lower traces generator closures as host/lowering.py does" begin
    for (name, build) in graphs
        want = read(joinpath(PLANS, name * ".bin"))
        got = lower(SignalOperators.process_sink_params(build())).bytes
        @test length(got) == length(want)
        length(got) == length(want) || continue
        s = sections(want)
        @test got[1:s.stages0] == want[1:s.stages0]                       # header, buffers, tables, instructions, pieces
        for k in 0:s.n_stage-1
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
