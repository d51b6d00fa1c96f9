// K4/K5 — polyphase FIR resampling (ToFramerate on data signals).
//
// Replaces DSP.jl's `filt!(out, FIRFilter{FIRArbitrary|FIRRational|FIRDecimator|
// FIRInterpolator}, x)` reached from src/filters.jl:252-255 with the filter
// built at src/reformatting.jl:92-99 (kernels restated in SURVEY.md App. B.4).
// One-shot semantics (SURVEY.md App. C-2): the input is the child followed by
// zeros and the first n_out outputs of the stream are kept.
//
// For every output m the host replayed the kernel's own index recurrence once
// (bit-exact Float64 phase accumulator) into two tables shared by every channel
// and instance of the batch:
//     xi0[m]  0-based index of the newest input sample in the window
//     phi[m]  FIRArbitrary phase accumulator (phiIdx = floor, alpha = frac) or
//             the integer phase of the rational kernels
// so  y[m] = sum_t (pfb[phiIdx][t] + alpha*dpfb[phiIdx][t]) * x[xi0 - tapsPerPhi + 1 + t].
//
// Block = tile of 64 outputs x RB = 32*G rows (a row = one channel of one instance).
//   * merged taps of the tile's outputs: built once in shared memory, shared by all rows,
//     each row of the table placed so that tap pairs are 16-byte aligned with the
//     (even) window position they multiply
//   * input window: cp.async global -> shared, layout [row][position] (coalesced 256-byte
//     reads, conflict-free 128-bit reads with lanes = rows)
//   * thread = 8 outputs x G rows register tile; per pair of window positions it issues
//     G 128-bit sample loads + 8 128-bit broadcast tap loads for 16*G FMAs
//   * results staged [row][output] and written back as coalesced 512-byte rows, through
//     the fused epilogue program when there is one.
//
// Roofline (44.1k -> 48k): 15.35 B per output sample of HBM traffic, 38 FP64
// FMAs per sample after merging (SURVEY.md §8d).
#pragma once
#include "interp.cuh"
#include "ptx.cuh"

namespace sigops {

constexpr int kFirR = 8;                    // outputs per thread
constexpr int kFirMaxWarps = 8;
// W warps per block: tile of T = 8*W outputs (W = 8: 64 outputs, W = 4: 32 outputs — the smaller
// tile lets two 128-row blocks share an SM so one block's copies overlap the other's FMAs)

struct FirParams {
    const sigops_instr* instrs;
    const BufRef* bufrefs;
    double* scalars;
    int nbuf, nscalars;
    int out_buf, sumsq_slot;
    int in_buf;                // input is always a materialised buffer, zero padded past in_len
    int64_t in_len;
    int epi_prog_start, epi_prog_len;
    int nch;
    int64_t nrows;
    int64_t n_out;
    int tapsper;
    int hbase;                 // even, > max window shift inside a group of 8 outputs
    int tpad;                  // doubles per merged-tap row (even)
    int xpitch;                // doubles per window row, = 2 mod 4, >= max positions of a tile + 2
    const double* pfb;         // [nphases][tapsper]
    const double* dpfb;        // or nullptr
    const int64_t* xi0;        // [ceil(n_out/T)*T], tail repeats the last entry
    const double* phi;
    int64_t inst0;             // index of the wave's first instance in the whole call (noise streams)
};

template <int G, int W>
__global__ void __launch_bounds__(W * 32)
k_fir(const __grid_constant__ FirParams P) {
    constexpr int RB = 32 * G;
    constexpr int kFirWarps = W, kFirThreads = W * 32, kFirT = W * kFirR;
    constexpr int kFirYPitch = kFirT + 2;       // doubles; = 2 mod 4 keeps lane=row 128-bit stores conflict free
    __shared__ sigops_instr sprog_epi[SIGOPS_MAX_PROG];
    __shared__ double lc_epi[W][SIGOPS_MAX_PROG];
    __shared__ double2 lr_epi[SIGOPS_MAX_PROG];
    __shared__ int s_ws[kFirT];                           // window start of output m relative to the tile
    extern __shared__ __align__(16) double smem[];
    double* hm = smem;                                    // [T][tpad]
    double* xs = smem + (size_t)kFirT * P.tpad;           // [RB][xpitch]; reused as ys[RB][kFirYPitch]
    const int xrows = P.xpitch > kFirYPitch ? P.xpitch : kFirYPitch;
    double* stack = xs + (size_t)RB * xrows;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t m0 = (int64_t)blockIdx.x * kFirT;
    const int64_t row0 = (int64_t)blockIdx.y * RB;
    // Everything the block needs from global memory before it can start copying is requested
    // up front, so the dependent-load chain at block start is one memory latency long:
    // my output's index/phase (4 threads per output), the tile's first/last index, my row's buffers.
    const int my_m = tid >> 2;
    const int64_t my_xi0 = __ldg(P.xi0 + m0 + my_m);
    const double my_phi = __ldg(P.phi + m0 + my_m);
    const int64_t xi_first = __ldg(P.xi0 + m0), xi_last = __ldg(P.xi0 + m0 + kFirT - 1);
    BufRef my_ib{}, my_ob{};
    int my_inst = 0, my_c = 0;
    const bool my_row_live = tid < RB && row0 + tid < P.nrows;
    if (my_row_live) {
        const int64_t row = row0 + tid;
        const int64_t inst = row / P.nch;
        my_inst = (int)inst;
        my_c = (int)(row - inst * P.nch);
        my_ib = P.bufrefs[(size_t)inst * P.nbuf + P.in_buf];
        my_ob = P.bufrefs[(size_t)inst * P.nbuf + P.out_buf];
    }
    // tile window: even start so that position pairs stay 16-byte aligned
    const int64_t p_first = xi_first - P.tapsper + 1;
    const int64_t p0 = p_first & ~int64_t(1);
    const int npos = (int)(xi_last - p0 + 1);

    // ---- 0. per-row addressing, once per block (one thread per row)
    __shared__ const double* s_src[32 * 4];     // row base + p0 for Float64 rows, else nullptr
    __shared__ int s_rowkind[32 * 4];           // 0 = no such row, 1 = Float64 (cp.async), 2 = other types
    __shared__ double* s_dst[32 * 4];           // output row base when it takes aligned Float64 pair stores
    __shared__ int s_inst[32 * 4], s_chan[32 * 4];
    if (tid < RB) {
        const double* src = nullptr;
        double* dstp = nullptr;
        int kind = 0;
        if (my_row_live) {
            kind = my_ib.dtype == SIGOPS_F64 ? 1 : 2;
            if (kind == 1) src = reinterpret_cast<const double*>(my_ib.ptr) + (int64_t)my_c * my_ib.ld + p0;
            if (my_ob.dtype == SIGOPS_F64 && ((((uintptr_t)my_ob.ptr) | (uintptr_t)(my_ob.ld * 8)) & 15) == 0)
                dstp = reinterpret_cast<double*>(my_ob.ptr) + (int64_t)my_c * my_ob.ld;
        }
        s_src[tid] = src;
        s_rowkind[tid] = kind;
        s_dst[tid] = dstp;
        s_inst[tid] = my_inst;
        s_chan[tid] = my_c;
    }
    // positions [jlo, jhi) of the tile exist in the signal; the rest is zero padding / history
    const int ncopy = npos + 1;
    // the 16-byte copies below move position PAIRS: they own cells [0, ncopy_e); the zeroed slack starts after them
    // (racecheck: the slack used to start at `ncopy` and overlap the last pair of an odd-length window)
    const int ncopy_e = (ncopy + 1) & ~1;
    const int jlo = p0 < 0 ? (int)(-p0 < ncopy ? -p0 : ncopy) : 0;
    const int64_t avail = P.in_len - p0;
    const int jhi = avail < 0 ? 0 : (avail < ncopy ? (int)avail : ncopy);
    __syncthreads();

    // ---- 1. start the window copy: rows x positions, lanes along positions
    for (int r = warp; r < RB; r += kFirWarps) {
        double* dst = xs + (size_t)r * P.xpitch;
        const int kind = s_rowkind[r];
        if (kind == 1) {
            const double* src = s_src[r];
            if ((((uintptr_t)src) & 15) == 0) {
                // two positions per lane; positions outside the signal (history before it, zero padding after it)
                // are plain zero stores — not zero-size cp.async copies, which the sanitizer tools do not model
                for (int j = 2 * lane; j < ncopy; j += 64) {
                    const bool in0 = j >= jlo && j < jhi, in1 = j + 1 >= jlo && j + 1 < jhi;
                    if (in0 && in1) cp_async16(dst + j, src + j, 16);
                    else {
                        if (in0) cp_async8(dst + j, src + j, true);
                        else dst[j] = 0.0;
                        if (in1) cp_async8(dst + j + 1, src + j + 1, true);
                        else dst[j + 1] = 0.0;
                    }
                }
            } else {
                for (int j = lane; j < ncopy_e; j += 32) {
                    if (j >= jlo && j < jhi) cp_async8(dst + j, src + j, true);
                    else dst[j] = 0.0;
                }
            }
        } else if (kind == 2) {
            const int64_t row = row0 + r;
            const int64_t inst = row / P.nch;
            const int c = (int)(row - inst * P.nch);
            const BufRef ib = P.bufrefs[(size_t)inst * P.nbuf + P.in_buf];
            for (int j = lane; j < ncopy_e; j += 32)
                dst[j] = (j >= jlo && j < jhi) ? load_elem(ib.ptr, ib.dtype, (int64_t)c * ib.ld + p0 + j) : 0.0;
        } else {
            for (int j = lane; j < ncopy_e; j += 32) dst[j] = 0.0;
        }
    }
    for (int i = tid; i < RB * 8; i += kFirThreads) xs[(size_t)(i >> 3) * P.xpitch + ncopy_e + (i & 7)] = 0.0;
    cp_async_commit();

    // ---- 2. merged taps while the copies fly: 4 threads per output
    for (int i = tid; i < P.epi_prog_len; i += kFirThreads) {
        const sigops_instr I = P.instrs[P.epi_prog_start + i];
        sprog_epi[i] = I;
        double2 rot = make_double2(0.0, 1.0);
        if (I.leaf == SIGOPS_LEAF_GEN && gen_is_trig(I)) {       // one-frame phase advance (see prepare_program)
            const double w = (I.flags & SIGOPS_FLAG_HAS_OMEGA) ? I.d1 : 1.0;
            double cyc = 1.0 / I.d0 * w;
            if (!(I.flags & SIGOPS_FLAG_HAS_OMEGA) && I.fn != SIGOPS_FN_SIN) cyc *= 0.15915494309189535;
            sincospi(2.0 * cyc, &rot.x, &rot.y);
        }
        lr_epi[i] = rot;
    }
    {
        const int m = my_m, sub = tid & 3;
        const int ws = (int)(my_xi0 - P.tapsper + 1 - p0);            // >= 0
        if (sub == 0) s_ws[m] = ws;
        double* hrow = hm + (size_t)m * P.tpad;
        const int base = P.hbase + (ws & 1);                          // tap t lives at hrow[base + t]
        for (int i = sub; i < P.tpad; i += 4)
            if (i < base || i >= base + P.tapsper) hrow[i] = 0.0;
        if (m0 + m < P.n_out) {
            const double acc = my_phi;
            const double fl = floor(acc);
            const double alpha = acc - fl;
            const double* pf = P.pfb + ((int64_t)fl - 1) * P.tapsper;
            const double* dpf = P.dpfb ? P.dpfb + ((int64_t)fl - 1) * P.tapsper : nullptr;
            for (int t = sub; t < P.tapsper; t += 4) {
                double h = __ldg(pf + t);
                if (dpf) h = fma(alpha, __ldg(dpf + t), h);
                hrow[base + t] = h;
            }
        } else {
            for (int t = sub; t < P.tapsper; t += 4) hrow[base + t] = 0.0;
        }
    }
    cp_async_commit();
    cp_async_wait_group<0>();
    __syncthreads();

    // ---- 3. register-tiled dot products: 8 outputs x G rows per thread, two positions per step
    double acc[kFirR][G];
#pragma unroll
    for (int r = 0; r < kFirR; ++r)
#pragma unroll
        for (int g = 0; g < G; ++g) acc[r][g] = 0.0;
    {
        const int mw = warp * kFirR;
        const int qs = s_ws[mw] & ~1;                                 // first (even) position of the group
        const int qe = s_ws[mw + kFirR - 1] + P.tapsper;              // one past the last position
        // one tap-row pointer per output (index arithmetic hoisted out of the loop)
        const double* hp[kFirR];
#pragma unroll
        for (int r = 0; r < kFirR; ++r) {
            const int ws = s_ws[mw + r];
            hp[r] = hm + (mw + r) * P.tpad + P.hbase + (ws & 1) + (qs - ws);
        }
        const double* xrow[G];
#pragma unroll
        for (int g = 0; g < G; ++g) xrow[g] = xs + (lane + 32 * g) * P.xpitch + qs;
        // four position pairs per iteration (immediate offsets, one pointer bump each); the
        // tail reads zero taps / zeroed slack, so no remainder loop is needed
        const int nquad = (qe - qs + 7) >> 3;
        for (int k = 0; k < nquad; ++k) {
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                double2 xv[G];
#pragma unroll
                for (int g = 0; g < G; ++g) xv[g] = *reinterpret_cast<const double2*>(xrow[g] + 2 * u);
#pragma unroll
                for (int r = 0; r < kFirR; ++r) {
                    // two 64-bit broadcast loads: a warp-uniform 128-bit load costs four shared-memory
                    // wavefronts (one per quarter warp), a uniform 64-bit load only one
                    const double h0 = hp[r][2 * u], h1 = hp[r][2 * u + 1];
#pragma unroll
                    for (int g = 0; g < G; ++g) {
                        acc[r][g] = fma(h0, xv[g].x, acc[r][g]);
                        acc[r][g] = fma(h1, xv[g].y, acc[r][g]);
                    }
                }
            }
#pragma unroll
            for (int g = 0; g < G; ++g) xrow[g] += 8;
#pragma unroll
            for (int r = 0; r < kFirR; ++r) hp[r] += 8;
        }
    }
    __syncthreads();

    // ---- 4. stage results [row][output] (reusing the window tile), then coalesced row stores
    double* ys = xs;
#pragma unroll
    for (int g = 0; g < G; ++g) {
        double* yr = ys + (size_t)(lane + 32 * g) * kFirYPitch + warp * kFirR;
#pragma unroll
        for (int r = 0; r < kFirR; r += 2) *reinterpret_cast<double2*>(yr + r) = make_double2(acc[r][g], acc[r + 1][g]);
    }
    __syncthreads();

    const bool plain_store = P.epi_prog_len == 0;
    if (plain_store) {
        // fast path: lanes 0-15 take row r, lanes 16-31 row r+1; each store instruction
        // writes one contiguous 256-byte span per row (outputs 32*q + 2l .. 2l+1)
        const int half = lane >> 4, l16 = lane & 15;
        constexpr int NQ = kFirT / 32;
        for (int r = 2 * warp + half; r < RB; r += 2 * kFirWarps) {
            if (s_rowkind[r] == 0) continue;
            const double* yp = ys + r * kFirYPitch + 2 * l16;
            double* dstp = s_dst[r];
            double ss = 0.0;
#pragma unroll
            for (int q = 0; q < NQ; ++q) {
                const double2 a = *reinterpret_cast<const double2*>(yp + 32 * q);
                const int64_t m = m0 + 32 * q + 2 * l16;
                if (dstp && m + 1 < P.n_out) {
                    *reinterpret_cast<double2*>(dstp + m) = a;
                    ss = fma(a.x, a.x, fma(a.y, a.y, ss));
                } else {
                    const int inst = s_inst[r], c = s_chan[r];
                    const BufRef ob = P.bufrefs[(size_t)inst * P.nbuf + P.out_buf];
                    if (m < P.n_out) { const double w = store_elem(ob.ptr, ob.dtype, (int64_t)c * ob.ld + m, a.x); ss = fma(w, w, ss); }
                    if (m + 1 < P.n_out) { const double w = store_elem(ob.ptr, ob.dtype, (int64_t)c * ob.ld + m + 1, a.y); ss = fma(w, w, ss); }
                }
            }
            if (P.sumsq_slot >= 0) {
                // reduce over the 16 lanes of this row
#pragma unroll
                for (int o = 8; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
                if (l16 == 0) atomicAdd(P.scalars + (size_t)s_inst[r] * P.nscalars + P.sumsq_slot, ss);
            }
        }
        return;
    }
    for (int r = warp; r < RB; r += kFirWarps) {
        if (s_rowkind[r] == 0) break;
        const int inst = s_inst[r], c = s_chan[r];
        const bool lane_on = 2 * lane < kFirT;
        const double2 yv = lane_on ? *reinterpret_cast<const double2*>(ys + (size_t)r * kFirYPitch + 2 * lane) : make_double2(0.0, 0.0);
        const int64_t m = m0 + 2 * lane;
        const BufRef* bufs = P.bufrefs + (size_t)inst * P.nbuf;
        Env env{bufs, P.scalars + (size_t)inst * P.nscalars, P.inst0 + inst};
        for (int i = lane; i < P.epi_prog_len; i += 32) {
            const sigops_instr& I = sprog_epi[i];
            double v = 0.0;
            if (I.leaf == SIGOPS_LEAF_CONST) v = I.d0;
            else if (I.leaf == SIGOPS_LEAF_RMS) v = sqrt(env.scalars[I.buf] / I.d0);
            lc_epi[warp][i] = v;
        }
        __syncwarp();
        const double y[2] = {yv.x, yv.y};
        double o[2];
        eval_program<2>(sprog_epi, lc_epi[warp], lr_epi, P.epi_prog_len, env, m, 1, c, y, o, stack + tid, kFirThreads);
        __syncwarp();
        double ss = 0.0;
        const BufRef ob = bufs[P.out_buf];
#pragma unroll
        for (int j = 0; j < 2; ++j)
            if (lane_on && m + j < P.n_out) {
                const double w = store_elem(ob.ptr, ob.dtype, (int64_t)c * ob.ld + m + j, o[j]);
                ss = fma(w, w, ss);
            }
        if (P.sumsq_slot >= 0) {
            ss = warp_sum(ss);
            if (lane == 0) atomicAdd(P.scalars + (size_t)inst * P.nscalars + P.sumsq_slot, ss);
        }
    }
}

}  // namespace sigops
