// K4/K5 (fast path) — polyphase FIR resampling on the FP64 tensor cores.
//
// Same arithmetic as k_fir.cuh (DSP.jl `filt!(out, FIRFilter{...}, x)` reached from
// src/filters.jl:252-255, filter built at src/reformatting.jl:92-99; the host replays the
// kernel's index recurrence into xi0[m], phi[m]):
//     y[m] = sum_t (pfb[phi][t] + alpha*dpfb[phi][t]) * x[xi0[m] - tapsPerPhi + 1 + t]
// restated for a group of 8 consecutive outputs as one small matrix product
//     Y[row][n] = sum_k X[row][q + k] * H[k][n],        k = 0 .. KS-1
// where q is the first window position of the group and H is the dense band of the eight
// outputs' merged taps (output n's taps start at row xi0[n] - xi0[0] of its column; zeros
// elsewhere).  `mma.sync.m8n8k4.f64` (DMMA) does 256 FMAs per warp instruction with one
// 64-bit operand load per lane, so the shared-memory pipe that bounds the FMA formulation
// (one broadcast tap load per G FMAs) is no longer the limit: measured on B200 the tensor
// pipe sustains 18.5 T FP64 FMA/s against 17.0 T for DFMA.
//
// The kernel is persistent along the time axis and warp-specialised:
//   * a block owns RB = 8*MF*RH rows (a row = one channel of one instance) and a contiguous
//     range of 32-output tiles; the rows' input windows live in a shared-memory RING indexed
//     by position mod `ring`, so every input sample is fetched from L2/HBM once per block
//   * the aux warps (second half of the block) prepare tile t+1 while tile t is multiplied.
//     Each owns a slice of the rows (lane = row) and extends their ring by the positions the
//     next tile adds: one TMA bulk copy per row, two where the ring wraps (cp.async.bulk ...
//     mbarrier::complete_tx; zero fill by hand outside [0, in_len): history before the signal /
//     the reference's zero padding).  It also builds a few columns of the tap bands (merging
//     pfb + alpha*dpfb, both banks staged in shared memory)
//   * warps 0-3 or 0-7 (warp = one 8-output group x one slice of the rows)
//     run the DMMA loop on the current tile and store their fragments straight to global
//     memory: a lane holds two consecutive outputs of one row, so every 32-byte sector is
//     written whole
//   * mbarriers: `data[t&3]` (every aux thread arrives once per ring extension, announcing its
//     copy's bytes with expect_tx; the extension for tile t+1 is
//     issued while tile t is multiplied, so HBM latency is off the critical path; four of them
//     because the producer runs ahead: a barrier is only reused after the compute warps are
//     known to have passed its previous phase), `taps[t&1]` (band of tile t built),
//     `done[t&1]` (compute warps; releases ring slots and the tap buffer two tiles later).
//
// Tried and dropped: staging the finished tile in shared memory and letting the aux warps write it
// out as whole 256-byte row pieces (the fragment stores cost the compute warps ~950 cycles per tile
// in the LSU).  It fits (tap bands at pitch 8), but the drain lengthens the aux path, which is
// the critical one: 1.92 ms against 1.76 ms.  Also dropped: building the B-fragment elements in the
// compute warps (no tap buffer, no taps barrier) — per k-step it costs a pipe switch each (2.30 ms),
// batched before the loop it is ~1000 cycles per tile that nothing overlaps (2.17 ms).  And a single
// lane issuing all of a warp's bulk copies in a scalar loop is slower than lane = row (~340 against
// ~110 cycles per copy): the per-row copies are bound by the TMA unit's issue rate, which only fewer,
// larger copies (a tensor map over all rows) would lift.
//
// Eligibility (checked by the host): Float64 in/out, 16-byte aligned rows, epilogue = none or a
// constant gain (folded into the taps; the sum of squares for a following Normpower is
// supported).  Everything else takes k_fir.cuh.  Batches whose rows sit at base + row*stride take
// k_fir_tmap.cuh instead (tensor-map loads and stores).
#pragma once
#include "interp.cuh"
#include "ptx.cuh"

namespace sigops {

constexpr int kFmT = 32;           // outputs per tile: 4 groups of 8
constexpr int kFmHbPitch = 12;     // doubles per position row of a tap band (8 used): the k-major
                                   // B-fragment load (k = lane&3, n = lane>>2) is then conflict free

struct FirMmaParams {
    const BufRef* bufrefs;
    double* scalars;
    int nbuf, nscalars;
    int in_buf, out_buf, sumsq_slot;
    int64_t in_len;
    int nch;
    int64_t nrows;
    int64_t n_out;
    int tapsper;
    int ks;                 // positions per 8-output group (multiple of 4)
    int ring;               // ring capacity in positions (even)
    int pitch;              // doubles per ring row: >= ring, = 4 mod 16 (conflict-free A-fragment loads)
    int64_t ntiles;         // ceil(n_out / 32)
    int64_t tiles_per_seg;  // tiles per block along x
    const double* pfb;      // [nphases][tapsper]
    const double* dpfb;     // or nullptr
    const int64_t* xi0;     // padded to a multiple of 64 entries
    const int32_t* poff;    // [m] (phase index - 1) * tapsper: row of output m in the banks
    const double* alpha;    // [m] fractional phase (0 for the rational kernels)
    int tab_doubles;        // nphases*tapsper: both banks are copied to shared memory
    double gain;            // constant-gain epilogue folded into the taps (1.0 = none)
};

// MF = 8-row fragments per compute warp, RH = compute warps per output group (row slices), SSQ =
// accumulate the sum of squares for a following Normpower (costs the compute warps 2*MF registers):
// RB = 8*MF*RH rows per block, 4*RH compute warps followed by 4*RH aux warps.
template <int MF, int RH, bool SSQ>
__global__ void __launch_bounds__(8 * RH * 32, 1)
k_fir_mma(const __grid_constant__ FirMmaParams P) {
    constexpr int RB = 8 * MF * RH;
    constexpr int NCW = 4 * RH;                  // compute warps
    constexpr int NAW = 4 * RH;                  // aux warps
    constexpr int kThreads = (NCW + NAW) * 32;
    constexpr int kAuxThreads = NAW * 32;
    extern __shared__ __align__(128) unsigned char fm_smem[];
    double* ring = reinterpret_cast<double*>(fm_smem);                       // [RB][pitch]
    double* hb = ring + (size_t)RB * P.pitch;                                // [2][4][ks][kFmHbPitch]
    double* tabs = hb + (size_t)2 * 4 * P.ks * kFmHbPitch;                   // pfb, dpfb copies when they fit
    __shared__ uint64_t bar_data[4], bar_taps[2], bar_done[2];
    __shared__ const double* s_src[RB];
    __shared__ double* s_dst[RB];
    __shared__ int s_inst[RB];

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t row0 = (int64_t)blockIdx.y * RB;
    const int64_t t0 = (int64_t)blockIdx.x * P.tiles_per_seg;
    const int64_t t1 = (t0 + P.tiles_per_seg < P.ntiles) ? t0 + P.tiles_per_seg : P.ntiles;
    if (t0 >= t1) return;

    if (tid < RB) {
        const int64_t row = row0 + tid;
        const double* src = nullptr;
        double* dst = nullptr;
        int inst = 0;
        if (row < P.nrows) {
            inst = (int)(row / P.nch);
            const int c = (int)(row - (int64_t)inst * P.nch);
            const BufRef ib = P.bufrefs[(size_t)inst * P.nbuf + P.in_buf];
            const BufRef ob = P.bufrefs[(size_t)inst * P.nbuf + P.out_buf];
            src = reinterpret_cast<const double*>(ib.ptr) + (int64_t)c * ib.ld;
            dst = reinterpret_cast<double*>(ob.ptr) + (int64_t)c * ob.ld;
        }
        s_src[tid] = src;
        s_dst[tid] = dst;
        s_inst[tid] = inst;
    }
    // both polyphase banks are staged in shared memory (the host only picks this kernel when they fit)
    for (int i = tid; i < P.tab_doubles; i += kThreads) {
        tabs[i] = __ldg(P.pfb + i);
        if (P.dpfb) tabs[P.tab_doubles + i] = __ldg(P.dpfb + i);
    }
    const double* const pf_tab = tabs;
    const double* const dpf_tab = P.dpfb ? tabs + P.tab_doubles : nullptr;
    if (tid == 0) {
        for (int i = 0; i < 4; ++i) mbar_init(&bar_data[i], kAuxThreads);
        mbar_init(&bar_taps[0], kAuxThreads);
        mbar_init(&bar_taps[1], kAuxThreads);
        mbar_init(&bar_done[0], NCW);
        mbar_init(&bar_done[1], NCW);
        fence_mbarrier_init();
    }
    fence_async_smem();
    __syncthreads();

    // position of ring slot 0: the (even) first window position of the block's first tile
    const int64_t pos_base = (__ldg(P.xi0 + t0 * kFmT) - P.tapsper + 1) & ~int64_t(1);
    const int hb_tile = 4 * P.ks * kFmHbPitch;          // doubles per tile buffer

    if (warp >= NCW) {
        // ---------------- ring loads + tap bands: aux warp x owns RB/NAW rows and 32/NAW band columns ----------------
        const int aux = warp - NCW;
        constexpr int RPA = RB / NAW;                   // rows per aux warp (lane = row)
        constexpr int NPW = kFmT / NAW;                 // outputs (band columns) per aux warp
        const int bg = (aux * NPW) >> 3, bn0 = (aux * NPW) & 7;   // my band: group, first column
        const int myrow = aux * RPA + lane;
        const double* const src = lane < RPA ? s_src[myrow] : nullptr;
        double* const rrow = ring + (size_t)(lane < RPA ? myrow : 0) * P.pitch;
        int64_t have = pos_base;                        // positions below `have` are in the ring (or on their way)
        int wi = 0;                                     // ring index of position `have`

        // Extend the ring to position `need` (exclusive, even); completion is signalled on `bar`, where
        // every aux thread arrives exactly once per call.  lane = row: one TMA bulk copy per row (two
        // where the ring wraps) — the fewest instructions on a sub-partition that also feeds DMMAs.
        auto extend = [&](int64_t need, uint64_t* bar) {
            if (need < have) need = have;
            // [a, b) comes from the signal by TMA, the rest of [have, need) is written by hand
            const int64_t a = have < 0 ? (need < 0 ? need : 0) : have;
            int64_t b = need < P.in_len ? need : (P.in_len & ~int64_t(1));
            if (b < a) b = a;
            const int cnt = (int)(b - a), total = (int)(need - have);
            if (lane < RPA && cnt < total) {
                int idx = wi;
                for (int64_t p = have; p < need; ++p) {
                    if (p < a || p >= b) rrow[idx] = (src && p >= 0 && p < P.in_len) ? src[p] : 0.0;
                    if (++idx == P.ring) idx = 0;
                }
            }
            if (cnt && src) {
                mbar_expect_tx(bar, (unsigned)cnt * 8u);           // arrive + announce my copy's bytes
                int ia = wi + (int)(a - have);
                if (ia >= P.ring) ia -= P.ring;
                const int first = cnt < P.ring - ia ? cnt : P.ring - ia;
                bulk_load(rrow + ia, src + a, (unsigned)first * 8u, bar);
                if (cnt > first) bulk_load(rrow, src + a + first, (unsigned)(cnt - first) * 8u, bar);
            } else
                mbar_arrive(bar);
            wi += total;
            if (wi >= P.ring) wi -= P.ring;
            have = need;
        };
        // (the k-steps of a group read ks positions from its window start: up to ks - tapsper past the window's end, times zero
        //  taps — they must be landed data all the same, 0 * NaN is NaN)
        auto need_of = [&](int64_t tile) { return (__ldg(P.xi0 + tile * kFmT + kFmT - 1) + 2 + (P.ks - P.tapsper)) & ~int64_t(1); };

        extend(need_of(t0), &bar_data[0]);              // the whole window of the first tile
        // index tables are read one tile ahead (they stream through L2 with everything else, so a
        // load issued and consumed in the same iteration would put DRAM latency on the aux path)
        int64_t need_nx = t0 + 1 < t1 ? need_of(t0 + 1) : 0;
        int64_t xi_nx = __ldg(P.xi0 + t0 * kFmT + lane);
        int po_nx = __ldg(P.poff + t0 * kFmT + lane);
        double al_nx = __ldg(P.alpha + t0 * kFmT + lane);
        for (int64_t t = t0; t < t1; ++t) {
            const int64_t u = t - t0;
            const int s = (int)(u & 1);
            // (a) where the next tile's window ends, (b) lane l: shift / bank row / phase fraction of output l
            const int64_t need = need_nx;
            const int64_t m_l = t * kFmT + lane;
            const int64_t xi_l = xi_nx;
            const int po_l = po_nx;
            const double alpha_l = al_nx;
            if (t + 2 < t1) need_nx = need_of(t + 2);
            if (t + 1 < t1) {
                xi_nx = __ldg(P.xi0 + m_l + kFmT);
                po_nx = __ldg(P.poff + m_l + kFmT);
                al_nx = __ldg(P.alpha + m_l + kFmT);
            }
            const int64_t xg = __shfl_sync(0xffffffffu, xi_l, lane & ~7);
            const int sh_l = (int)(xi_l - xg);
            const int off_l = po_l - sh_l;
            const int lo_l = m_l < P.n_out ? sh_l : P.ks;                 // band rows [lo, sh + tapsper) hold taps
            // tile t-2 must be finished: its ring slots and its tap buffer are about to be overwritten
            if (u >= 2) mbar_wait(&bar_done[s], (unsigned)((u >> 1) - 1) & 1u);

            // ---- ring: the positions tile t+1 adds, requested a whole tile ahead of their use
            if (t + 1 < t1) extend(need, &bar_data[(u + 1) & 3]);

            // ---- tap band of group `aux` for tile t: lanes along the band rows.  No FP64 instruction
            // other than the merges themselves, and those back to back: a DFMA issued from this warp
            // queues behind the DMMAs of the compute warp on the same sub-partition (measured: FP64
            // work of a second warp adds its full latency, integer / LDS work mostly overlaps).
            double* band = hb + (size_t)s * hb_tile + (size_t)bg * P.ks * kFmHbPitch + bn0;
            if (P.ks <= 64) {
                double pv[NPW][2], dv[NPW][2], al[NPW];
#pragma unroll
                for (int n = 0; n < NPW; ++n) {
                    const int o = aux * NPW + n;
                    const int off = __shfl_sync(0xffffffffu, off_l, o);
                    const int lo = __shfl_sync(0xffffffffu, lo_l, o);
                    const int hi = __shfl_sync(0xffffffffu, sh_l, o) + P.tapsper;
                    al[n] = __shfl_sync(0xffffffffu, alpha_l, o);
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        const int k = lane + 32 * j;
                        const bool in = k >= lo && k < hi;
                        pv[n][j] = in ? pf_tab[off + k] : 0.0;
                        dv[n][j] = (in && dpf_tab) ? dpf_tab[off + k] : 0.0;
                    }
                }
                if (dpf_tab) {
#pragma unroll
                    for (int n = 0; n < NPW; ++n)
#pragma unroll
                        for (int j = 0; j < 2; ++j) pv[n][j] = fma(al[n], dv[n][j], pv[n][j]);
                }
                if (P.gain != 1.0) {
#pragma unroll
                    for (int n = 0; n < NPW; ++n)
#pragma unroll
                        for (int j = 0; j < 2; ++j) pv[n][j] *= P.gain;
                }
#pragma unroll
                for (int n = 0; n < NPW; ++n)
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        const int k = lane + 32 * j;
                        if (k < P.ks) band[k * kFmHbPitch + n] = pv[n][j];
                    }
            } else {
#pragma unroll 1
                for (int n = 0; n < NPW; ++n) {
                    const int o = aux * NPW + n;
                    const int off = __shfl_sync(0xffffffffu, off_l, o);
                    const int lo = __shfl_sync(0xffffffffu, lo_l, o);
                    const int hi = __shfl_sync(0xffffffffu, sh_l, o) + P.tapsper;
                    const double alpha = __shfl_sync(0xffffffffu, alpha_l, o);
                    for (int k = lane; k < P.ks; k += 32) {
                        double h = 0.0;
                        if (k >= lo && k < hi) {
                            h = pf_tab[off + k];
                            if (dpf_tab) h = fma(alpha, dpf_tab[off + k], h);
                            h *= P.gain;
                        }
                        band[k * kFmHbPitch + n] = h;
                    }
                }
            }
            mbar_arrive(&bar_taps[s]);
        }
    } else {
        // ---------------- DMMA ----------------
        const int g = warp & 3, half = warp >> 2;
        const int kk = lane & 3, rr = lane >> 2;
        double ssq[SSQ ? MF : 1];
#pragma unroll
        for (int i = 0; i < (SSQ ? MF : 1); ++i) ssq[i] = 0.0;

        const int rbase = half * (RB / RH) + rr;          // my first row; fragment i holds row rbase + 8i
        const double* arow = ring + (size_t)rbase * P.pitch;
        // output row pointers stay in registers: a store then depends on nothing but its fragment
        double* dstp[MF];
#pragma unroll
        for (int i = 0; i < MF; ++i) dstp[i] = s_dst[rbase + 8 * i];
        int roff[MF];                                    // warp-uniform row offsets, kept out of the loop's address chain
#pragma unroll
        for (int i = 0; i < MF; ++i) roff[i] = i * 8 * P.pitch;
        const int nks = P.ks >> 2;
        int64_t qprev = pos_base;
        int qidx = 0;                                   // ring index of position qprev
        int64_t q_nx = __ldg(P.xi0 + t0 * kFmT + 8 * g) - P.tapsper + 1;   // read one tile ahead
        double prev[MF][2];                              // fragments of the previous tile, not yet stored
        int64_t mprev = -1;
        bool prev_full = false;                          // both outputs of the pending fragments exist
        // fragment (outputs m, m+1 of one row) -> global; predicated, no branch on the row pointer
        auto store_frag = [&](double* dst, int64_t m, bool full, double v0, double v1) {
            if (dst && full) __stcs(reinterpret_cast<double2*>(dst + m), make_double2(v0, v1));   // streaming: never re-read
            else if (dst && m < P.n_out) dst[m] = v0;
        };
        // Sum of squares for a following Normpower: only when asked for, and as one batch per tile —
        // every switch of the FP64 pipe between DMMA and scalar FP64 work costs a pipeline drain.
        for (int64_t t = t0; t < t1; ++t) {
            const int s = (int)((t - t0) & 1);
            // first window position of my group, as a ring index
            const int64_t q = q_nx;
            if (t + 1 < t1) q_nx = __ldg(P.xi0 + (t + 1) * kFmT + 8 * g) - P.tapsper + 1;
            qidx += (int)(q - qprev);
            qprev = q;
            while (qidx >= P.ring) qidx -= P.ring;
            int idx = qidx + kk;
            if (idx >= P.ring) idx -= P.ring;
            const double* bp = hb + (size_t)s * hb_tile + (size_t)g * P.ks * kFmHbPitch + kk * kFmHbPitch + rr;
            double acc[MF][2];
#pragma unroll
            for (int i = 0; i < MF; ++i) acc[i][0] = acc[i][1] = 0.0;
            mbar_wait(&bar_taps[s], (unsigned)((t - t0) >> 1) & 1u);
            mbar_wait(&bar_data[(t - t0) & 3], (unsigned)((t - t0) >> 2) & 1u);
            auto step = [&](int ks) {
                const double b = bp[ks * 4 * kFmHbPitch];
                const double* ap = arow + idx;
#pragma unroll
                for (int i = 0; i < MF; ++i) dmma884(acc[i][0], acc[i][1], ap[roff[i]], b);
                idx += 4;
                if (idx >= P.ring) idx -= P.ring;
            };
            // The previous tile's fragments go out one per k-step of this tile: the stores then
            // drain through the LSU underneath the DMMAs instead of holding both warps of the
            // sub-partition (which run in lockstep) in a store phase of their own.
#pragma unroll
            for (int i = 0; i < MF; ++i) {
                if (i < nks) step(i);
                if (mprev >= 0) store_frag(dstp[i], mprev, prev_full, prev[i][0], prev[i][1]);
            }
#pragma unroll 2
            for (int ks = MF; ks < nks; ++ks) step(ks);
            __syncwarp();
            if (lane == 0) mbar_arrive(&bar_done[s]);
            mprev = t * kFmT + 8 * g + 2 * kk;
            prev_full = mprev + 1 < P.n_out;
#pragma unroll
            for (int i = 0; i < MF; ++i) { prev[i][0] = acc[i][0]; prev[i][1] = acc[i][1]; }
            if (SSQ) {
                // outputs past n_out have all-zero taps, so their fragments are exactly 0
#pragma unroll
                for (int i = 0; i < MF; ++i) ssq[i] = fma(acc[i][0], acc[i][0], fma(acc[i][1], acc[i][1], ssq[i]));
            }
        }
#pragma unroll
        for (int i = 0; i < MF; ++i) store_frag(dstp[i], mprev, mprev + 1 < P.n_out, prev[i][0], prev[i][1]);
        if (SSQ) {
#pragma unroll
            for (int i = 0; i < (SSQ ? MF : 1); ++i) {
                const double v = quad_sum(ssq[i]);
                if (kk == 0 && dstp[i]) atomicAdd(P.scalars + (size_t)s_inst[rbase + 8 * i] * P.nscalars + P.sumsq_slot, v);
            }
        }
    }
}

}  // namespace sigops
