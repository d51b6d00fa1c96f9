// Cross-chunk state propagation for the MAIN + CARRY + FIX decomposition (see k_iir.cuh).
#pragma once
#include "biquad.cuh"

namespace sigops {

// CARRY: one thread per row walks its chunks in order.
//   s_in[0] = 0;  s_in[k] = s_zs[k-1] + AL * s_in[k-1]
// `AL` is the (2M x 2M) L-step state transition matrix (row-major) or nullptr
// when the zero-input response has fully decayed within one chunk (Wc < L).
struct CarryParams {
    const double* state_zs;
    double* state_in;
    const double* AL;
    int64_t nrows, slots_per_row, nchunks;
    int M2;     // 2M
};

__global__ void k_iir_carry(const CarryParams P) {
    // one warp per row; lane i owns state component i (2M <= 16 lanes busy), so a chunk step is
    // one coalesced load, 2M shuffles + FMAs and one coalesced store instead of (2M)^2 scalar loads
    const int lane = threadIdx.x & 31;
    const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row >= P.nrows) return;
    const int64_t nslots = P.nrows * P.slots_per_row;
    const bool on = lane < P.M2;
    double a_row[2 * kIirMaxSections];
#pragma unroll
    for (int j = 0; j < 2 * kIirMaxSections; ++j) a_row[j] = (P.AL && on && j < P.M2) ? P.AL[lane * P.M2 + j] : 0.0;
    double s = 0.0;
    // software prefetch: the zero-state results do not depend on the carry
    double zs_next = (on && P.nchunks > 0) ? P.state_zs[(int64_t)lane * nslots + row * P.slots_per_row] : 0.0;
    for (int64_t k = 0; k < P.nchunks; ++k) {
        const int64_t slot = row * P.slots_per_row + k;
        const double zs = zs_next;
        if (k + 1 < P.nchunks && on) zs_next = P.state_zs[(int64_t)lane * nslots + slot + 1];
        if (on) P.state_in[(int64_t)lane * nslots + slot] = s;
        double t = zs;
#pragma unroll
        for (int j = 0; j < 2 * kIirMaxSections; ++j) {
            const double sj = __shfl_sync(0xffffffffu, s, j);
            if (j < P.M2) t = fma(a_row[j], sj, t);
        }
        s = t;
    }
}

}  // namespace sigops
