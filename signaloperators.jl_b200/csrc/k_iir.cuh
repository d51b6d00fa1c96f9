// K3 — biquad-cascade (SOS, DF2T) filtering as a chunked parallel scan.
//
// Replaces DSP.jl's sequential `filt!(out, DF2TFilter{SOS}, x)` called per
// channel per 4096-frame block at src/filters.jl:252-255 (recurrence restated
// in SURVEY.md App. B.2), plus the two block copies around it
// (src/filters.jl:240-244, 213-214).
//
// Parallel decomposition (the filter is linear and time-invariant):
//   1. MAIN   every channel is cut into chunks of L frames; each lane runs the
//             cascade over one chunk from ZERO state (zero-state response) and
//             records its final state.  Lanes of a warp own 32 consecutive chunks
//             of one channel; data moves through a per-warp 32x32 shared-memory
//             tile so every global access is a coalesced 256-byte row.
//   2. CARRY  s_in[k] = s_zs[k-1] + A^L s_in[k-1]   (cross-chunk / cross-block
//             carry of the 2M-vector state; A^L is the cascade's L-step state
//             transition matrix, precomputed on the host).
//   3. FIX    chunk k >= 1 adds the zero-input response of s_in[k] to its first
//             Wc frames, where Wc is the number of frames after which that
//             response has decayed below 2^-64 of its peak (Wc = L if it never
//             does).  MAIN leaves those frames un-finalised; FIX applies the
//             fused epilogue to them.  The generic kernel k_iir instead leaves
//             them unwritten and FIX reruns the cascade over them from s_in[k]:
//             its output may be Float32, which cannot hold the zero-state
//             values exactly until FIX adds the rest.
// Superposition makes 1+3 equal to the sequential filter up to rounding.
//
// Roofline: 16 B/sample HBM (8 in + 8 out); 5 FP64 instructions per section per
// sample (SURVEY.md §8d: "FP64 pipe ~ HBM").
#pragma once
#include "biquad.cuh"
#include "interp.cuh"
#include "ptx.cuh"

namespace sigops {

constexpr int kIirWarps = 4;
constexpr int kIirThreads = kIirWarps * 32;
constexpr int kIirV = 4;
constexpr int kTilePitch = 33;

struct IirParams {
    const sigops_instr* instrs;
    const BufRef* bufrefs;     // [ninst][nbuf]
    double* scalars;           // [ninst][nscalars]
    int nbuf, nscalars;
    int out_buf, sumsq_slot;
    int in_prog_start, in_prog_len;
    int epi_prog_start, epi_prog_len;
    int plain_in_buf;          // >= 0: input program is a bare zero-padded buffer load
    int64_t plain_in_len;
    int nch;                   // channels (rows) per instance
    int blocks_per_row;
    int64_t N, L, Wc;          // frames, chunk length, un-finalised prefix (both multiples of 32)
    int64_t slots_per_row;     // blocks_per_row * kIirThreads
    double* state_zs;          // [2M][rows*slots_per_row]  MAIN out
    double* state_in;          // [2M][rows*slots_per_row]  CARRY out, FIX in
    int M;
    double gain;
    double coef[kIirMaxSections][5];
    // FAST path: Float64 plain input buffer, Float64 output, epilogue = up to two
    // constant multipliers applied in order (Amplify chains)
    int n_epi_scale;
    double epi_scale[2];
    int carry_is_shift;        // FIX reads s_in[k] = state_zs[k-1] directly (no CARRY launch)
    int64_t inst0;             // index of the wave's first instance in the whole call (noise streams)
};

enum { IIR_MAIN = 0, IIR_FIX = 1, IIR_WARM = 2 };

// NT frames of one chunk through the cascade (cascade_frames), in place in the lane's shared-memory row.
// out = in_tile + (cascade * gain) for FIX, (cascade * gain) * sc for MAIN.
template <int M, int NT, bool ZERO_IN, bool UNITB>
__device__ __forceinline__ void cascade_tile(Cascade<M>& f, double* myrow, double gain, double sc) {
    // pull the lane's NT frames into registers first: the shared-memory latency is paid
    // once per tile instead of once per frame on the critical path
    double xr[NT];
#pragma unroll
    for (int k = 0; k < NT; ++k) xr[k] = myrow[k];
    double pipe[M];
    cascade_frames<M, NT, ZERO_IN, UNITB>(f, xr, pipe, [&](int k, double y) {
        myrow[k] = ZERO_IN ? fma(y, gain, xr[k]) * sc : (y * gain) * sc;
    });
}

constexpr int kHalfCols = 16;          // frames per half-tile
constexpr int kHalfPitch = 17;         // doubles; odd pitch keeps lane=row accesses conflict-free
constexpr int kHalfElems = 32 * kHalfPitch;

// FAST kernel: same decomposition as k_iir below, specialised for the common case
// (Float64 buffer in, Float64 buffer out, constant-gain epilogue): no interpreter.
// Each warp streams its 32 chunks through two 32x16 shared-memory half-tiles:
// while it runs the cascade on one, cp.async is already filling the other, so every
// warp always has 4 KB of reads in flight (global rows are 128-byte segments).
template <int M, int MODE, bool UNITB>
__global__ void __launch_bounds__(kIirThreads, 5)
k_iir_fast(const __grid_constant__ IirParams P) {
    __shared__ double tiles[kIirWarps][2][kHalfElems];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t row = blockIdx.x / P.blocks_per_row;
    const int brow = blockIdx.x % P.blocks_per_row;
    const int inst = (int)(row / P.nch), c = (int)(row % P.nch);
    const BufRef ib = P.bufrefs[(size_t)inst * P.nbuf + P.plain_in_buf];
    const BufRef ob = P.bufrefs[(size_t)inst * P.nbuf + P.out_buf];
    const double* __restrict__ xin = reinterpret_cast<const double*>(ib.ptr) + (int64_t)c * ib.ld;
    double* yout = reinterpret_cast<double*>(ob.ptr) + (int64_t)c * ob.ld;
    const int64_t nvalid = P.plain_in_len < P.N ? P.plain_in_len : P.N;

    const int64_t chunk0 = (int64_t)brow * kIirThreads + warp * 32;
    const int64_t mychunk = chunk0 + lane;
    const int64_t slot = row * P.slots_per_row + mychunk;
    const int64_t nslots = (int64_t)gridDim.x / P.blocks_per_row * P.slots_per_row;
    if (chunk0 * P.L >= P.N) return;
    // every frame of the warp's 32 chunks exists in both buffers: no bounds checks needed
    const bool interior = (chunk0 + 32) * P.L <= nvalid;

    Cascade<M> f;
    f.init(P.coef);
    if (MODE == IIR_FIX && mychunk >= 1) load_carried_state(f, P, nslots, slot);
    const int64_t L = P.L;
    const int64_t nh_raw = P.Wc / kHalfCols;
    const int64_t nh = (MODE == IIR_FIX) ? nh_raw : L / kHalfCols;
    const double sc_final = P.epi_scale[0] * P.epi_scale[1];
    // copy mapping: instruction i moves rows 2i and 2i+1; lanes 0-15 / 16-31 take one row each
    const int crow = lane >> 4, ccol = lane & 15;
    const int64_t cbase = (chunk0 + crow) * L + ccol;      // frame of (row crow, col ccol) in half-tile 0
    double ss = 0.0;

    auto issue_loads = [&](int64_t h, double* buf) {
        const double* gsrc = (MODE == IIR_MAIN) ? xin : yout;
        const int64_t n0 = cbase + h * kHalfCols;
        double* dst = buf + crow * kHalfPitch + ccol;
        if (interior && (MODE == IIR_MAIN || chunk0 >= 1)) {
#pragma unroll
            for (int i = 0; i < 16; ++i) cp_async8(dst + 2 * i * kHalfPitch, gsrc + n0 + 2 * i * L, true);
        } else {
#pragma unroll 4
            for (int i = 0; i < 16; ++i) {
                const int64_t n = n0 + 2 * i * L;
                const bool ok = (MODE == IIR_MAIN) ? (n < nvalid) : (n < P.N && chunk0 + 2 * i + crow >= 1);
                cp_async8(dst + 2 * i * kHalfPitch, gsrc + (ok ? n : 0), ok);
            }
        }
        cp_async_commit();
    };

    issue_loads(0, tiles[warp][0]);
    for (int64_t h = 0; h < nh; ++h) {
        double* buf = tiles[warp][h & 1];
        if (h + 1 < nh) {
            issue_loads(h + 1, tiles[warp][(h + 1) & 1]);
            cp_async_wait_group<1>();
        } else {
            cp_async_wait_group<0>();
        }
        __syncwarp();
        // MAIN leaves the first Wc frames of chunks >= 1 un-scaled (raw zero-state
        // response): FIX adds the carried-in state's response and applies the gain.
        const bool raw_phase = (MODE == IIR_MAIN) && (h < nh_raw);
        const double sc = (raw_phase && mychunk >= 1) ? 1.0 : sc_final;
        cascade_tile<M, kHalfCols, MODE == IIR_FIX, UNITB>(f, buf + lane * kHalfPitch, P.gain, sc);
        __syncwarp();
        // ---- store: rows as 128-byte segments
        const int64_t n0 = cbase + h * kHalfCols;
        const double* srcs = buf + crow * kHalfPitch + ccol;
        if (interior && chunk0 >= 1) {
            double v[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = srcs[2 * i * kHalfPitch];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                yout[n0 + 2 * i * L] = v[i];
                if (!raw_phase) ss = fma(v[i], v[i], ss);
            }
        } else {
#pragma unroll 4
            for (int i = 0; i < 16; ++i) {
                const int64_t n = n0 + 2 * i * L;
                const int64_t chunk = chunk0 + 2 * i + crow;
                const double w = srcs[2 * i * kHalfPitch];
                const bool skip = (MODE == IIR_FIX) && chunk < 1;
                if (n < P.N && !skip) {
                    yout[n] = w;
                    if (!(raw_phase && chunk >= 1)) ss = fma(w, w, ss);
                }
            }
        }
        __syncwarp();
    }

    if (MODE == IIR_MAIN) store_final_state(f, P.state_zs, nslots, slot);
    if (P.sumsq_slot >= 0) {
        ss = warp_sum(ss);
        if (lane == 0) atomicAdd(P.scalars + (size_t)inst * P.nscalars + P.sumsq_slot, ss);
    }
}

template <int M, int MODE>
__global__ void __launch_bounds__(kIirThreads)
k_iir(const __grid_constant__ IirParams P) {
    __shared__ sigops_instr sprog_in[SIGOPS_MAX_PROG];
    __shared__ sigops_instr sprog_epi[SIGOPS_MAX_PROG];
    __shared__ double lc_in[SIGOPS_MAX_PROG], lc_epi[SIGOPS_MAX_PROG];
    __shared__ double2 lr_in[SIGOPS_MAX_PROG], lr_epi[SIGOPS_MAX_PROG];
    __shared__ BufRef sbufs[32];
    __shared__ double tiles[kIirWarps][32 * kTilePitch];
    extern __shared__ double stack[];

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t row = blockIdx.x / P.blocks_per_row;
    const int brow = blockIdx.x % P.blocks_per_row;
    const int inst = (int)(row / P.nch), c = (int)(row % P.nch);

    for (int i = threadIdx.x; i < P.nbuf; i += blockDim.x) sbufs[i] = P.bufrefs[(size_t)inst * P.nbuf + i];
    Env env{sbufs, P.scalars + (size_t)inst * P.nscalars, P.inst0 + inst};
    prepare_program(P.instrs + P.in_prog_start, P.in_prog_len, sprog_in, lc_in, lr_in, env, P.L);
    prepare_program(P.instrs + P.epi_prog_start, P.epi_prog_len, sprog_epi, lc_epi, lr_epi, env, P.L);
    __syncthreads();

    double* tile = tiles[warp];
    const int64_t chunk0 = (int64_t)brow * kIirThreads + warp * 32;  // first chunk of this warp
    const int64_t mychunk = chunk0 + lane;
    const int64_t slot = row * P.slots_per_row + mychunk;
    const int64_t nslots = (int64_t)gridDim.x / P.blocks_per_row * P.slots_per_row;
    if (chunk0 * P.L >= P.N) return;      // whole warp past the end (warp-uniform)

    Cascade<M> f;
    f.init(P.coef);
    if (MODE == IIR_FIX && mychunk >= 1) load_carried_state(f, P, nslots, slot);

    const BufRef ob = sbufs[P.out_buf];
    const int64_t nsub_all = P.L / 32, nsub_raw = P.Wc / 32;
    const int64_t nsub = (MODE == IIR_FIX) ? nsub_raw : nsub_all;
    double ss = 0.0;

    for (int64_t s = 0; s < nsub; ++s) {
        // ---- load phase: rows of the tile = chunks, columns = 32 consecutive frames
#pragma unroll 1
        for (int r = 0; r < 32; r += kIirV) {
            const int64_t n0 = (chunk0 + r) * P.L + s * 32 + lane;
            double v[kIirV];
            if (P.plain_in_buf >= 0) {
                const BufRef ib = sbufs[P.plain_in_buf];
#pragma unroll
                for (int j = 0; j < kIirV; ++j) {
                    const int64_t n = n0 + j * P.L;
                    v[j] = (n < P.plain_in_len) ? load_elem(ib.ptr, ib.dtype, (int64_t)c * ib.ld + n) : 0.0;
                }
            } else {
                eval_program<kIirV>(sprog_in, lc_in, lr_in, P.in_prog_len, env, n0, P.L, c, nullptr, v,
                                    stack + threadIdx.x, kIirThreads);
            }
#pragma unroll
            for (int j = 0; j < kIirV; ++j) tile[(r + j) * kTilePitch + lane] = v[j];
        }
        __syncwarp();

        // ---- compute phase: lane = chunk, 32 sequential frames
        {
            double* myrow = tile + lane * kTilePitch;
#pragma unroll
            for (int k = 0; k < 32; ++k) myrow[k] = f.step(myrow[k]) * P.gain;
        }
        __syncwarp();

        // ---- store phase
#pragma unroll 1
        for (int r = 0; r < 32; r += kIirV) {
            const int64_t n0 = (chunk0 + r) * P.L + s * 32 + lane;
            double y[kIirV], o[kIirV];
#pragma unroll
            for (int j = 0; j < kIirV; ++j) y[j] = tile[(r + j) * kTilePitch + lane];
            if (P.epi_prog_len > 0)
                eval_program<kIirV>(sprog_epi, lc_epi, lr_epi, P.epi_prog_len, env, n0, P.L, c, y, o,
                                    stack + threadIdx.x, kIirThreads);
            else {
#pragma unroll
                for (int j = 0; j < kIirV; ++j) o[j] = y[j];
            }
#pragma unroll
            for (int j = 0; j < kIirV; ++j) {
                const int64_t n = n0 + j * P.L;
                const int64_t chunk = chunk0 + r + j;
                // MAIN leaves the first Wc frames of chunks >= 1 to FIX; FIX writes nothing else
                const bool fix_frame = (chunk >= 1) && (s < nsub_raw);
                if (n >= P.N || fix_frame != (MODE == IIR_FIX)) continue;
                const double w = store_elem(ob.ptr, ob.dtype, (int64_t)c * ob.ld + n, o[j]);
                ss += w * w;
            }
        }
        __syncwarp();
    }

    if (MODE == IIR_MAIN) store_final_state(f, P.state_zs, nslots, slot);
    if (P.sumsq_slot >= 0) {
        ss = warp_sum(ss);
        if (lane == 0) atomicAdd(P.scalars + (size_t)inst * P.nscalars + P.sumsq_slot, ss);
    }
}

}  // namespace sigops
