// K4/K5 (long banks) — FIR stages whose filter bank does not fit in shared memory: strong down-sampling
// (ToFramerate below ~0.29 of the input rate) and long `FIRFilter(h)` / `FIRFilter(h, p//q)` banks, up to
// 65 536 taps per phase, on the FP64 tensor cores.
//
// Same arithmetic as k_fir.cuh / k_fir_mma.cuh:
//     y[m] = sum_t h_m[t] * x[xi0[m] - tapsPerPhi + 1 + t],   h_m = pfb[phase] + alpha * dpfb[phase]
// restated for a group of 8 consecutive outputs as Y[row][n] = sum_k X[row][q + k] * Band[k][n], where q is the
// group's first window position and Band[k][n] = h_n[k - (xi0[n] - xi0[0])] (zero outside the taps).  The band is
// walked in CHUNKS of 8 positions, two `mma.sync.m8n8k4.f64` k-steps each: k-step 0 takes positions kk = 0..3 of the
// chunk, k-step 1 positions kk + 4.  The output accumulators stay in registers for the whole band.
//
// Neither the band nor a tile's window has to fit in shared memory:
//   * block = 8 warps = 8 output groups (a 64-output tile) x RB = 8*MF rows; one tile per block
//   * the tile's window [W0, Wend) is walked in SEGMENTS of kFlSeg positions through a ring of three segment
//     slots per row (one being multiplied, the next one, which the last chunks of a segment reach into, and one
//     in flight), so shared memory does not depend on the bank length.  A chunk belongs to the segment its first
//     position lies in.
//   * window loads: one thread per row, one bulk copy per segment on rows on a 16-byte boundary (mbarrier
//     complete_tx), 8-byte cp.async copies (cp.async.mbarrier.arrive) on rows off it, which only device-resident
//     callers produce; history before the signal and padding after it are written as zeros by hand.
//   * B fragments (lane = (rr, kk): Band[8c + kk][rr] and Band[8c + kk + 4][rr]):
//       BK_TAB   single-phase kinds (standard, decimator): output n of a group reads q*n positions after output 0,
//                so every group has the same band.  The host builds it once per plan as a table of fragments,
//                the constant gain folded in, and the compute warps stream it from L2 (one 16-byte load per lane
//                and chunk).
//       BK_BANK  multi-phase kinds without a derivative bank (rational, interpolator): gathered from pfb.
//       BK_MERGE arbitrary ratios: the merged taps pfb + alpha*dpfb are formed on the tensor pipe, not with
//                scalar DFMA (DESIGN.md §3: FP64 pipe switches cost the DMMA stream a drain).  With the chunk's
//                positions ordered sigma(2i) = i, sigma(2i+1) = i + 4, a DMMA accumulator fragment of the 8x8
//                matrix Band^T (outputs x positions) holds exactly the two B elements its lane needs, so
//                    C(= pfb band^T) += diag(alpha) * dpfb band^T
//                is two DMMAs per chunk (k = outputs 0..3, 4..7) that hand their result straight to the product.
//     The constant gain of the multi-phase kinds is applied to the finished outputs (once per output, not per tap).
#pragma once
#include "interp.cuh"
#include "ptx.cuh"

namespace sigops {

constexpr int kFlGroups = 8;                  // warps per block = 8-output groups per tile
constexpr int kFlT = 8 * kFlGroups;           // outputs per tile
constexpr int kFlSeg = 128;                   // positions per window segment
constexpr int kFlSlots = 3;                   // segment slots of the ring
constexpr int kFlRing = kFlSlots * kFlSeg;    // ring capacity in positions
constexpr int kFlPitch = kFlRing + 4;         // doubles per ring row, = 4 mod 16: conflict-free A-fragment loads

enum { BK_TAB = 0, BK_BANK = 1, BK_MERGE = 2 };

struct FirLongParams {
    const BufRef* bufrefs;
    double* scalars;
    int nbuf, nscalars;
    int in_buf, out_buf, sumsq_slot;
    int64_t in_len;
    int nch;
    int64_t nrows;
    int64_t n_out;
    int tapsper;
    int nchunks;            // 8-position chunks of a group's band (the longest band of any group)
    const int64_t* xi0;     // padded to a multiple of 64 entries
    const int32_t* poff;    // [m] (phase index - 1) * tapsper
    const double* alpha;    // [m] fractional phase
    const double* pfb;      // [nphases][tapsper]
    const double* dpfb;     // BK_MERGE only
    const double2* band;    // BK_TAB: [nchunks][32] B fragments of the common band, gain folded in
    double gain;            // constant-gain epilogue of the multi-phase kinds (1.0 = none)
};

template <int MF, int BK, bool SSQ>
__global__ void __launch_bounds__(kFlGroups * 32, 2)
k_fir_long(const __grid_constant__ FirLongParams P) {
    constexpr int RB = 8 * MF;
    extern __shared__ __align__(128) unsigned char fl_smem[];
    double* ring = reinterpret_cast<double*>(fl_smem);                       // [RB][kFlPitch]
    __shared__ uint64_t bar[kFlSlots];
    __shared__ const double* s_src[RB];
    __shared__ double* s_dst[RB];
    __shared__ int s_inst[RB];

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int kk = lane & 3, rr = lane >> 2;
    const int64_t m0 = (int64_t)blockIdx.x * kFlT;
    const int64_t row0 = (int64_t)blockIdx.y * RB;
    const int T = P.tapsper;

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
    if (tid == 0) {
        for (int i = 0; i < kFlSlots; ++i) mbar_init(&bar[i], RB);
        fence_mbarrier_init();
    }
    __syncthreads();

    // the tile's window: every group's band [q_g, q_g + 8*nchunks) lies inside [W0, Wend) (xi0 never decreases)
    const int64_t W0 = (__ldg(P.xi0 + m0) - T + 1) & ~int64_t(1);      // even: bulk copies start on 16-byte boundaries
    const int64_t Wend = __ldg(P.xi0 + m0 + kFlT - 8) - T + 1 + 8 * (int64_t)P.nchunks;
    const int nseg = (int)((Wend - W0 + kFlSeg - 1) / kFlSeg);         // segments multiplied; segment nseg is loaded too

    // Segment sg of my row into its slot; every row thread arrives once on the slot's barrier.
    auto load = [&](int sg) {
        if (tid >= RB) return;
        uint64_t* b = &bar[sg % kFlSlots];
        double* dst = ring + (size_t)tid * kFlPitch + (sg % kFlSlots) * kFlSeg;
        const double* src = s_src[tid];
        const int64_t a = W0 + (int64_t)sg * kFlSeg;
        // positions [lo, hi) come from the signal, the rest of the segment is zero
        int64_t lo = a < 0 ? 0 : a, hi = a + kFlSeg < P.in_len ? a + kFlSeg : P.in_len;
        if (!src || hi < lo) lo = hi = a;
        for (int j = 0; j < (int)(lo - a); ++j) dst[j] = 0.0;
        for (int j = (int)(hi - a); j < kFlSeg; ++j) dst[j] = 0.0;
        if ((((uintptr_t)src) & 15) == 0) {
            const int64_t pe = lo + ((hi - lo) & ~int64_t(1));          // whole 16-byte pairs by bulk copy
            if (hi > pe) dst[pe - a] = src[pe];
            if (pe > lo) {
                fence_async_smem();                                     // the slot was last read through the generic proxy
                mbar_expect_tx(b, (unsigned)(pe - lo) * 8u);
                bulk_load(dst + (lo - a), src + lo, (unsigned)(pe - lo) * 8u, b);
            } else
                mbar_arrive(b);
        } else {
            for (int64_t p = lo; p < hi; ++p) cp_async8(dst + (p - a), src + p, true);
            cp_async_mbar_arrive(b);                                    // counts the copies in, then completes them
            mbar_arrive(b);
        }
    };

    // my group: first output, first band position, and what the lane needs to form its B fragments
    const int64_t mg = m0 + 8 * warp;
    const int64_t xg = __ldg(P.xi0 + mg);
    const int64_t qg = xg - T + 1;
    const double* pf_r = nullptr;      // BK_BANK / BK_MERGE: taps of output rr, shifted by its window offset
    const double *dp_0 = nullptr, *dp_1 = nullptr;
    double al_0 = 0.0, al_1 = 0.0;
    int sh_r = 0, sh_0 = 0, sh_1 = 0;
    const int sig = (rr >> 1) + 4 * (rr & 1);
    if (BK != BK_TAB) {
        sh_r = (int)(__ldg(P.xi0 + mg + rr) - xg);
        pf_r = P.pfb + __ldg(P.poff + mg + rr);
    }
    if (BK == BK_MERGE) {
        const double al = __ldg(P.alpha + mg + rr);
        al_0 = rr == kk ? al : 0.0;                   // diag(alpha), k = outputs 0..3
        al_1 = rr == kk + 4 ? al : 0.0;               //              k = outputs 4..7
        sh_0 = (int)(__ldg(P.xi0 + mg + kk) - xg);
        sh_1 = (int)(__ldg(P.xi0 + mg + kk + 4) - xg);
        dp_0 = P.dpfb + __ldg(P.poff + mg + kk);
        dp_1 = P.dpfb + __ldg(P.poff + mg + kk + 4);
    }

    double acc[MF][2];
#pragma unroll
    for (int i = 0; i < MF; ++i) acc[i][0] = acc[i][1] = 0.0;
    const double* arow = ring + (size_t)rr * kFlPitch;

    load(0);
    load(1);
    for (int j = 0; j < nseg; ++j) {
        if (j > 0) __syncthreads();                   // segment j-1 is finished: its slot takes segment j+2
        if (j + 2 <= nseg) load(j + 2);
        mbar_wait(&bar[j % kFlSlots], (unsigned)(j / kFlSlots) & 1u);
        mbar_wait(&bar[(j + 1) % kFlSlots], (unsigned)((j + 1) / kFlSlots) & 1u);
        // my chunks whose first position lies in segment j
        const int64_t s0 = W0 + (int64_t)j * kFlSeg - qg;
        const int64_t ca = (s0 + 7) >> 3, cb = (s0 + kFlSeg + 7) >> 3;
        int c = (int)(ca < 0 ? 0 : ca);
        const int ce = (int)(cb < P.nchunks ? cb : P.nchunks);
        int idx = (int)((qg + 8 * (int64_t)c - W0) % kFlRing);
#pragma unroll 2
        for (; c < ce; ++c) {
            double b0, b1;
            if (BK == BK_TAB) {
                const double2 v = __ldg(P.band + (size_t)c * 32 + lane);
                b0 = v.x;
                b1 = v.y;
            } else {
                const int t0 = 8 * c + kk - sh_r, t1 = t0 + 4;
                b0 = (unsigned)t0 < (unsigned)T ? __ldg(pf_r + t0) : 0.0;
                b1 = (unsigned)t1 < (unsigned)T ? __ldg(pf_r + t1) : 0.0;
                if (BK == BK_MERGE) {
                    const int u0 = 8 * c + sig - sh_0, u1 = 8 * c + sig - sh_1;
                    const double d0 = (unsigned)u0 < (unsigned)T ? __ldg(dp_0 + u0) : 0.0;
                    const double d1 = (unsigned)u1 < (unsigned)T ? __ldg(dp_1 + u1) : 0.0;
                    dmma884(b0, b1, al_0, d0);
                    dmma884(b0, b1, al_1, d1);
                }
            }
            int i0 = idx + kk, i1 = idx + kk + 4;
            if (i0 >= kFlRing) i0 -= kFlRing;
            if (i1 >= kFlRing) i1 -= kFlRing;
#pragma unroll
            for (int i = 0; i < MF; ++i) dmma884(acc[i][0], acc[i][1], arow[i * 8 * kFlPitch + i0], b0);
#pragma unroll
            for (int i = 0; i < MF; ++i) dmma884(acc[i][0], acc[i][1], arow[i * 8 * kFlPitch + i1], b1);
            idx += 8;
            if (idx >= kFlRing) idx -= kFlRing;
        }
    }

    // lane (rr, kk) holds outputs mg + 2kk, mg + 2kk + 1 of rows rr + 8i
    const int64_t m = mg + 2 * kk;
#pragma unroll
    for (int i = 0; i < MF; ++i) {
        double* dst = s_dst[rr + 8 * i];
        double v0 = acc[i][0], v1 = acc[i][1];
        if (BK != BK_TAB && P.gain != 1.0) {
            v0 *= P.gain;
            v1 *= P.gain;
        }
        if (dst) {
            if (m + 1 < P.n_out && ((((uintptr_t)dst) & 15) == 0)) __stcs(reinterpret_cast<double2*>(dst + m), make_double2(v0, v1));
            else {
                if (m < P.n_out) dst[m] = v0;
                if (m + 1 < P.n_out) dst[m + 1] = v1;
            }
        }
        if (SSQ) {
            const double ss = quad_sum((m < P.n_out ? v0 * v0 : 0.0) + (m + 1 < P.n_out ? v1 * v1 : 0.0));
            if (kk == 0 && dst) atomicAdd(P.scalars + (size_t)s_inst[rr + 8 * i] * P.nscalars + P.sumsq_slot, ss);
        }
    }
}

}  // namespace sigops
