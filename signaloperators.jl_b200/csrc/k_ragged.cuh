// Kernels of ragged runs (sigops_plan_run_ragged): instances of one plan whose buffers hold fewer valid frames
// than the plan declares.  Every stage is prefix-stable, so an instance is computed inside the plan of the
// longest one as long as every buffer reads zero past the instance's valid frames and each Normpower sums only
// those frames.  Both need the per-instance valid lengths, which only these two kernels read.
#pragma once
#include "interp.cuh"

namespace sigops {

constexpr int kRgThreads = 256;
constexpr int kRgPer = 4;                        // elements per thread and block pass
constexpr int kRgSpan = kRgThreads * kRgPer;     // frames one block covers

struct RaggedParams {
    const BufRef* bufrefs;      // [ninst][nbuf]
    const int64_t* valid;       // [ninst][nbuf] valid frames of every buffer of every instance
    double* scalars;            // [ninst][nscalars]
    int nbuf, nscalars, buf, slot;
    int64_t ninst;
    double d0;                  // divisor the plan's LEAF_RMS applies to the slot (N * C of the longest instance)
};

// Frames [valid, ld) of every row (instance x channel) of buffer `buf` set to zero.  Block (x, y) covers frames
// [valid + x*kRgSpan, +kRgSpan) of the rows y, y + gridDim.y, ...; consecutive threads store consecutive frames.
__global__ void __launch_bounds__(kRgThreads) k_tail_zero(RaggedParams P) {
    for (int64_t i = blockIdx.y; i < P.ninst; i += gridDim.y) {
        const BufRef r = P.bufrefs[i * P.nbuf + P.buf];
        const int64_t lo = P.valid[i * P.nbuf + P.buf] + (int64_t)blockIdx.x * kRgSpan;
        if (lo >= r.ld) continue;
        const int64_t hi = min(r.ld, lo + (int64_t)kRgSpan);
        for (int c = 0; c < r.nch; ++c) {
            if (r.dtype == SIGOPS_F32) {
                float* row = (float*)r.ptr + (int64_t)c * r.ld;
                for (int64_t n = lo + threadIdx.x; n < hi; n += kRgThreads) row[n] = 0.0f;
            } else {
                int64_t* row = (int64_t*)r.ptr + (int64_t)c * r.ld;      // F64 and I64: all-zero bits
                for (int64_t n = lo + threadIdx.x; n < hi; n += kRgThreads) row[n] = 0;
            }
        }
    }
}

// Sum of squares of frames [0, valid) of all channels of buffer `buf`, per instance, added to the instance's slot
// scaled by d0 / (valid * C): LEAF_RMS then yields sqrt(sum / (valid * C)), the instance's own Normpower divisor.
// Block (x, y) sums frames [x*kRgSpan, +kRgSpan) of instance y (and y + gridDim.y, ...).
__global__ void __launch_bounds__(kRgThreads) k_sumsq_rows(RaggedParams P) {
    __shared__ double part[kRgThreads / 32];
    for (int64_t i = blockIdx.y; i < P.ninst; i += gridDim.y) {
        const BufRef r = P.bufrefs[i * P.nbuf + P.buf];
        const int64_t v = P.valid[i * P.nbuf + P.buf];
        const int64_t lo = (int64_t)blockIdx.x * kRgSpan;
        if (lo >= v) continue;                                   // (uniform across the block)
        const int64_t hi = min(v, lo + (int64_t)kRgSpan);
        double s = 0.0;
        for (int c = 0; c < r.nch; ++c)
            for (int64_t n = lo + threadIdx.x; n < hi; n += kRgThreads) {
                const int64_t k = (int64_t)c * r.ld + n;
                const double x = r.dtype == SIGOPS_F32 ? (double)((const float*)r.ptr)[k]
                               : r.dtype == SIGOPS_F64 ? ((const double*)r.ptr)[k] : (double)((const int64_t*)r.ptr)[k];
                s = fma(x, x, s);
            }
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = s;
        __syncthreads();
        if (threadIdx.x == 0) {
            double t = 0.0;
            for (int w = 0; w < kRgThreads / 32; ++w) t += part[w];
            atomicAdd(&P.scalars[i * P.nscalars + P.slot], t * (P.d0 / ((double)v * r.nch)));
        }
        __syncthreads();
    }
}

}  // namespace sigops
