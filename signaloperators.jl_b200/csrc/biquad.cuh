// The biquad-cascade core shared by the IIR kernels (k_iir*.cuh): coefficients and state of up to
// kIirMaxSections second-order sections, one section update, the software-pipelined loop over a run
// of frames, and the hand-over of chunk states between the MAIN and FIX passes.
#pragma once
#include <cstdint>

namespace sigops {

constexpr int kIirMaxSections = 8;

template <int M>
struct Cascade;

// One section update (DSP.jl `_filt!` inner body for SecondOrderSections (DF2T), SURVEY.md App. B.2).
// UNITB: the section has b0 == 1 and b2 == 1 exactly (every zero on the unit circle, which is what the
// Butterworth/Chebyshev designs give), so `b0*x` and `b2*x` are skipped without changing a single bit
// of the result.
template <int M, bool UNITB>
__device__ __forceinline__ double biquad_step(Cascade<M>& f, int j, double xi) {
    double y;
    if (UNITB) {
        y = xi + f.s1[j];
        f.s1[j] = fma(-f.a1[j], y, fma(f.b1[j], xi, f.s2[j]));
        f.s2[j] = fma(-f.a2[j], y, xi);
    } else {
        y = fma(f.b0[j], xi, f.s1[j]);
        f.s1[j] = fma(-f.a1[j], y, fma(f.b1[j], xi, f.s2[j]));
        f.s2[j] = fma(-f.a2[j], y, f.b2[j] * xi);
    }
    return y;
}

template <int M>
struct Cascade {
    double b0[M], b1[M], b2[M], a1[M], a2[M];
    double s1[M], s2[M];
    // coef[j] = {b0, b1, b2, a1, a2} of section j; zero state
    __device__ __forceinline__ void init(const double (&coef)[kIirMaxSections][5]) {
#pragma unroll
        for (int j = 0; j < M; ++j) {
            b0[j] = coef[j][0]; b1[j] = coef[j][1]; b2[j] = coef[j][2];
            a1[j] = coef[j][3]; a2[j] = coef[j][4];
            s1[j] = 0.0; s2[j] = 0.0;
        }
    }
    // one frame through every section in turn
    __device__ __forceinline__ double step(double x) {
        double y = x;
#pragma unroll
        for (int j = 0; j < M; ++j) y = biquad_step<M, false>(*this, j, y);
        return y;
    }
};

// NT frames through the cascade, software-pipelined across sections: at step t section j works on
// frame t-j, so the M updates of a step are mutually independent (M-way ILP on the FP64 pipe) while
// every frame still sees exactly the sequential recurrence.  ZERO_IN: the first section's input is 0
// (FIX pass: the zero-input response of the carried-in state).  emit(k, y) receives the cascade output
// of frame k.  pipe holds the sections' in-flight outputs; the caller declares it after its input
// array, because an array declared in here would come first once inlined, which renumbers the
// compiler's registers and changes the register assignment of the largest kernels.
template <int M, int NT, bool ZERO_IN, bool UNITB, class Emit>
__device__ __forceinline__ void cascade_frames(Cascade<M>& f, const double (&xr)[NT], double (&pipe)[M], Emit&& emit) {
#pragma unroll
    for (int t = 0; t < NT + M - 1; ++t) {
#pragma unroll
        for (int j = M - 1; j >= 0; --j) {     // descending: section j reads pipe[j-1] of step t-1
            const int k = t - j;
            if (k >= 0 && k < NT) {
                const double in = (j == 0) ? (ZERO_IN ? 0.0 : xr[k]) : pipe[j - 1];
                pipe[j] = biquad_step<M, UNITB>(f, j, in);
                if (j == M - 1) emit(k, pipe[j]);
            }
        }
    }
}

// Chunk states of the MAIN + CARRY + FIX decomposition (k_iir.cuh), stored [2M][nslots] in the
// kernel's IirParams P: FIX starts chunk `slot` from s_in[k] (P.state_in), or from s_zs[k-1]
// (P.state_zs[slot - 1]) when the carry is a plain shift; MAIN records the chunk's final zero-state
// state s_zs[k].
template <int M, class Params>
__device__ __forceinline__ void load_carried_state(Cascade<M>& f, const Params& P, int64_t nslots, int64_t slot) {
    const double* sin_ = P.carry_is_shift ? P.state_zs : P.state_in;
    const int64_t src = P.carry_is_shift ? slot - 1 : slot;
#pragma unroll
    for (int j = 0; j < M; ++j) {
        f.s1[j] = sin_[(2 * j) * nslots + src];
        f.s2[j] = sin_[(2 * j + 1) * nslots + src];
    }
}
template <int M>
__device__ __forceinline__ void store_final_state(const Cascade<M>& f, double* state_zs, int64_t nslots, int64_t slot) {
#pragma unroll
    for (int j = 0; j < M; ++j) {
        state_zs[(2 * j) * nslots + slot] = f.s1[j];
        state_zs[(2 * j + 1) * nslots + slot] = f.s2[j];
    }
}

}  // namespace sigops
