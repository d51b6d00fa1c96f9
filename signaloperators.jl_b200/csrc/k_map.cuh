// K1 — fused elementwise / generator kernel.
//
// One launch materialises a whole MAP stage: every piece (Append segment /
// AddChannel channel group) of the stage's output, all channels, all instances
// of the batch.  Replaces the `sink!` block loop + `sink_helper!` inner loop
// (src/sink.jl:225-267) for graphs without filters, and the three memory
// passes of `initblock(::NormedSignal)` (src/filters.jl:296-309): the sum of
// squares is accumulated while the producer stores, the division by the RMS is
// a leaf of the consumer's program.
//
// HBM-bound: 8(k+1) bytes per output sample for k buffer leaves (SURVEY.md §8d).
// Layout: a block walks an 8192-frame tile in four passes; in each, thread t owns frames
// t, t+256, ..., t+1792 of a 2048-frame span, so every warp access is a fully coalesced
// 256-byte row and the eight frames share one decode of each program instruction.
#pragma once
#include "interp.cuh"

namespace sigops {

constexpr int kMapThreads = 256;
constexpr int kMapV = 8;
constexpr int kMapSub = kMapThreads * kMapV;   // frames one pass of a block covers
constexpr int kMapPasses = 4;                  // passes per block: the per-block set-up (program copy, folded
                                               // constants, piece search) is paid once per 8192 frames
constexpr int kMapTile = kMapSub * kMapPasses;  // frames per block when the launch is large
constexpr int kMaxPieces = 64;
constexpr int kMaxBufs = 32;

struct MapParams {
    const sigops_instr* instrs;     // whole plan's instruction array (device)
    const BufRef* bufrefs;          // [ninst][nbuf]
    double* scalars;                // [ninst][nscalars]
    int nbuf, nscalars;
    int out_buf, sumsq_slot, out_nch;
    int n_pieces;
    int passes;                     // 2048-frame passes per block (kMapPasses, or 1 for small launches)
    int64_t inst0;                  // index of the wave's first instance in the whole call (noise streams)
    sigops_piece pieces[kMaxPieces];
    int tile_prefix[kMaxPieces + 1];
};

template <bool FN>      // the plan holds closure functions (eval_program)
__global__ void __launch_bounds__(kMapThreads, 4)
k_map(const __grid_constant__ MapParams P) {
    __shared__ sigops_instr sprog[SIGOPS_MAX_PROG];
    __shared__ double leafconst[SIGOPS_MAX_PROG];
    __shared__ double2 leafrot[SIGOPS_MAX_PROG];
    __shared__ BufRef sbufs[kMaxBufs];
    __shared__ double red[kMapThreads / 32];
    extern __shared__ double stack[];

    const int inst = blockIdx.z, c = blockIdx.y;
    // which piece this tile belongs to: the lanes of each warp compare one prefix each
    int p = 0;       // = number of piece boundaries at or below this tile
    for (int base = 1; base < P.n_pieces; base += 32) {
        const int i = base + (threadIdx.x & 31);
        const bool past = i < P.n_pieces && (int)blockIdx.x >= P.tile_prefix[i];
        p += __popc(__ballot_sync(0xffffffffu, past));
    }
    const sigops_piece pc = P.pieces[p];
    if (c < pc.ch_start || c >= pc.ch_start + pc.ch_count) return;

    for (int i = threadIdx.x; i < P.nbuf; i += blockDim.x) sbufs[i] = P.bufrefs[(size_t)inst * P.nbuf + i];
    Env env{sbufs, P.scalars + (size_t)inst * P.nscalars, P.inst0 + inst};
    prepare_program(P.instrs + pc.prog_start, pc.prog_len, sprog, leafconst, leafrot, env, kMapThreads);
    __syncthreads();

    const int64_t tile = (int64_t)blockIdx.x - P.tile_prefix[p];
    const int64_t nend = pc.out_start + pc.out_len;
    const BufRef ob = sbufs[P.out_buf];
    double ss = 0.0;
#pragma unroll 1
    for (int pass = 0; pass < P.passes; ++pass) {
        const int64_t n0 = pc.out_start + (tile * P.passes + pass) * (int64_t)kMapSub + threadIdx.x;
        if (n0 - threadIdx.x >= nend) break;
        double acc[kMapV];
        eval_program<kMapV, FN>(sprog, leafconst, leafrot, pc.prog_len, env, n0, kMapThreads, c, nullptr, acc,
                            stack + threadIdx.x, kMapThreads);
        if (ob.dtype == SIGOPS_F64) {
            double* op = reinterpret_cast<double*>(ob.ptr) + (int64_t)c * ob.ld + n0;
#pragma unroll
            for (int j = 0; j < kMapV; ++j)
                if (n0 + (int64_t)j * kMapThreads < nend) {
                    op[j * kMapThreads] = acc[j];
                    ss = fma(acc[j], acc[j], ss);
                }
        } else if (ob.dtype == SIGOPS_F32) {
            float* op = reinterpret_cast<float*>(ob.ptr) + (int64_t)c * ob.ld + n0;
#pragma unroll
            for (int j = 0; j < kMapV; ++j)
                if (n0 + (int64_t)j * kMapThreads < nend) {
                    const float v = (float)acc[j];
                    op[j * kMapThreads] = v;
                    ss = fma((double)v, (double)v, ss);
                }
        } else {
#pragma unroll
            for (int j = 0; j < kMapV; ++j) {
                const int64_t n = n0 + (int64_t)j * kMapThreads;
                if (n < nend) {
                    const double v = store_elem(ob.ptr, ob.dtype, (int64_t)c * ob.ld + n, acc[j]);
                    ss += v * v;
                }
            }
        }
    }
    if (P.sumsq_slot >= 0) {
        ss = warp_sum(ss);
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
        __syncthreads();
        if (threadIdx.x == 0) {
            double t = 0.0;
            for (int w = 0; w < kMapThreads / 32; ++w) t += red[w];
            atomicAdd(P.scalars + (size_t)inst * P.nscalars + P.sumsq_slot, t);
        }
    }
}

}  // namespace sigops
