// K4/K5 (fastest path) — polyphase FIR resampling on the FP64 tensor cores, fed and drained by
// tensor-map TMA.
//
// Same arithmetic as k_fir_mma.cuh / k_fir.cuh (DSP.jl `filt!(out, FIRFilter{...}, x)` reached from
// src/filters.jl:252-255, filter built at src/reformatting.jl:92-99; the host replays the kernel's
// index recurrence into xi0[m], phi[m]):
//     y[m] = sum_t (pfb[phi][t] + alpha*dpfb[phi][t]) * x[xi0[m] - tapsPerPhi + 1 + t]
// as 8-output groups Y[row][n] = sum_k X[row][q + k] * H[k][n] on `mma.sync.m8n8k4.f64` (DMMA.8x8x4).
// What changes against k_fir_mma is who moves the data.  There, 128 lanes issue one bulk copy per
// row and tile (bound by the TMA unit's issue rate: ~1850 cycles per tile on the helper path) and
// the compute warps push their fragments to global memory themselves (~950 cycles per tile in the
// LSU).  Here the [rows][frames] matrices are described by tensor maps, so
//   * the input ring is made of SLOTS of 16 consecutive positions x 128 rows (a 16 KB box, 128-byte
//     swizzle), each filled by ONE `cp.async.bulk.tensor.2d` issued by a producer thread that runs
//     as far ahead as the ring allows (per-slot `full` barriers; a slot is reused once the last
//     tile that read it is done).  Slots start on 128-byte lines of the rows; positions before
//     the signal, past its end, and rows past the last one are zero-filled by the TMA unit —
//     the history before the first sample and the reference's zero padding (src/filters.jl:240);
//   * finished 32-output tiles are staged in shared memory (two 16-output swizzled boxes) and
//     written with `cp.async.bulk.tensor.2d` stores (16 outputs x 64 rows each) by one store thread per row half
//     (whole 128-byte lines; columns past n_out and rows past the last are clipped by the tensor bounds);
//   * the compute warps do nothing but LDS + DMMA + 8 shared-memory stores per tile: a k-step (block of 4 window
//     positions) is 9 LDS + 8 DMMA + a select and an add.  Shared memory is the co-critical resource (an m8n8k4
//     DMMA takes 256 bytes of A operand per 16 tensor cycles; ncu: tensor pipe 74 % active, the shared-memory pipe
//     about 70 %).
// A fragment rows are taken in bit-reversed order (fragment row r -> signal row {0,4,2,6,1,5,3,7}[r])
// which makes both the swizzled A-fragment loads (any position alignment) and the staging stores
// bank-conflict free.  The tap bands live at pitch 8 with an XOR on the column index (conflict-free
// B-fragment loads) and are merged by four helper warps ON THE TENSOR PIPE (see below).  A fused constant gain
// (`ToFramerate |> Amplify(c)` is one launch) is folded into the staged banks: g*(sum h x) becomes sum (g h) x, a
// rounding-level difference.  A band starts at its group's own first window position; groups whose eight outputs
// span fewer positions skip the last k-step (44.1 -> 48 kHz: 11.4 instead of 12 on average).
//
// Block = 16 warps in four warpgroups that re-balance their registers with setmaxnreg: 8 compute (two per
// sub-partition; each 8 row fragments = 64 rows x one output group, 176 registers), 4 helpers (tap bands, one per
// group), 1 producer (ring loads), 2 store threads (one per row half).  Barriers: full[slot], done[tile&3] (compute
// warps), taps[tile&1], stg_full / stg_free per row half (staging hand-over).
//
// Eligibility (host): Float64 in/out, every row of the wave at base + row*stride with 16-byte
// aligned base and stride (one batch tensor, or the library's own staging), epilogue = none or
// constant gain, band <= 64 positions, a tile's window within the ring.  Everything else takes
// k_fir_mma / k_fir.  SIGOPS_NO_FIR_TMAP=1 switches this kernel off.
#pragma once
#include <type_traits>

#include "k_fir_mma.cuh"   // kFmT
#include "ptx.cuh"

namespace sigops {

constexpr int kFtRows = 128;                    // rows per block
constexpr int kFtSlotPos = 16;                  // positions per ring slot (one 128-byte row piece)
constexpr int kFtSlotBytes = kFtRows * 128;     // 16 KB
constexpr int kFtMaxSlots = 10;
constexpr int kFtNCW = 8, kFtNAW = 4;           // compute / helper warps
constexpr int kFtThreads = 16 * 32;              // four warpgroups: compute x2, helpers, producer + store (+ 2 idle warps)
// registers per thread after the warpgroups re-balance the 128 they are launched with (setmaxnreg)
constexpr int kFtRegsCompute = 176, kFtRegsHelper = 112, kFtRegsMisc = 40;
constexpr int kFtMaxKs = 64;

struct FirTmParams {
    double* scalars;
    int nscalars, sumsq_slot, nch;
    int64_t nrows, n_out;
    int tapsper;
    int ks;                 // positions per 8-output band (multiple of 4, <= 64)
    int nslot;              // ring slots
    int64_t ntiles, tiles_per_seg;
    const double* pfb;      // [nphases][tapsper]
    const double* dpfb;     // or nullptr
    const int64_t* xi0;     // padded to a multiple of 64 entries
    const int32_t* poff;    // [m] (phase index - 1) * tapsper
    const double* alpha;    // [m] fractional phase
    int tab_doubles;
    double gain;            // folded into the taps
    const double* bands_g;  // periodic resamplers: merged tap bands of one period, [period_tiles][4][ks][8] (host-built), or nullptr
    int period_tiles;
    int64_t epoch_tiles;    // one period table per epoch of this many tiles (the phase accumulator's drift), n_epochs of them
    int n_epochs;
};

inline size_t fir_tm_smem_bytes(int nslot, int ks, int tab_doubles, bool has_dpfb) {
    return (size_t)nslot * kFtSlotBytes + 2 * 16384 + (size_t)2 * 4 * ks * 8 * sizeof(double) +
           (size_t)tab_doubles * sizeof(double) * (has_dpfb ? 2 : 1) + 1024;
}

// The dynamic shared memory of this kernel is addressed through 32-bit shared-window addresses and
// explicit ld.shared / st.shared (lds_f64, sts_f64, sts_v2f64): the 1024-byte alignment of the swizzled
// boxes is computed on the address, and a pointer rebuilt from it would make every access a generic LD/ST.
template <bool SSQ>
__global__ void __launch_bounds__(kFtThreads, 1)
k_fir_tmap(const __grid_constant__ FirTmParams P, const __grid_constant__ CUtensorMap tm_in,
           const __grid_constant__ CUtensorMap tm_out) {
    extern __shared__ unsigned char ft_smem_raw[];
    __shared__ uint64_t bar_full[kFtMaxSlots], bar_done[4], bar_taps[2], bar_stg_full[2], bar_stg_free[2];
    // tiles finished, counted once per compute warp: what the producer polls.  (A plain counter, not the
    // `done` barriers: with strong up-sampling the ring holds many tiles, the producer may trail the compute
    // warps by more than the two phases a parity wait can tell apart.)
    __shared__ unsigned done_count;

    const unsigned ring = (smem_u32(ft_smem_raw) + 1023u) & ~1023u;               // [nslot][128 rows][128 B], swizzled
    const unsigned stg = ring + (unsigned)P.nslot * kFtSlotBytes;                  // [2][128 rows][128 B], swizzled
    const unsigned bands = stg + 2 * 16384;                                        // [2][4][ks][8] doubles
    const unsigned tabs = bands + 2u * 4u * (unsigned)P.ks * 64u;                  // pfb, dpfb

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int row0 = (int)blockIdx.y * kFtRows;
    const int64_t t0 = (int64_t)blockIdx.x * P.tiles_per_seg;
    const int64_t t1 = (t0 + P.tiles_per_seg < P.ntiles) ? t0 + P.tiles_per_seg : P.ntiles;
    if (t0 >= t1) return;

    // both banks ride along in shared memory, with the constant-gain epilogue folded in once per block
    for (int i = tid; i < P.tab_doubles; i += kFtThreads) {
        sts_f64(tabs + 8u * i, __ldg(P.pfb + i) * P.gain);
        if (P.dpfb) sts_f64(tabs + 8u * (P.tab_doubles + i), __ldg(P.dpfb + i) * P.gain);
    }
    if (tid == 0) {
        done_count = 0u;
        for (int i = 0; i < P.nslot; ++i) mbar_init(&bar_full[i], 1);
        for (int i = 0; i < 4; ++i) mbar_init(&bar_done[i], kFtNCW);
        // (tap bands from the period table: the loader's arrive.expect_tx and its arrival once the window has landed)
        mbar_init(&bar_taps[0], P.bands_g ? 2 : kFtNAW * 32);
        mbar_init(&bar_taps[1], P.bands_g ? 2 : kFtNAW * 32);
        for (int i = 0; i < 2; ++i) {
            mbar_init(&bar_stg_full[i], kFtNCW / 2);
            mbar_init(&bar_stg_free[i], 1);
        }
        fence_mbarrier_init();
    }
    fence_async_smem();
    __syncthreads();

    // position of ring slot 0: the first window position of the block's first tile, rounded down to a
    // 128-byte line of the rows
    const int64_t pos_base = (__ldg(P.xi0 + t0 * kFmT) - P.tapsper + 1) & ~int64_t(kFtSlotPos - 1);
    const unsigned band_tile = 4u * (unsigned)P.ks * 64u;      // bytes per band buffer

    if (warp < kFtNCW) {
        // ---------------- DMMA: a warp owns 8 row fragments (64 rows) x one 8-output group of the tile ----------------
        // Two compute warps per sub-partition: a single one cannot hide its own index arithmetic and operand
        // loads behind its DMMAs (measured with 4 warps x 16 fragments: 39 cycles per DMMA instead of 16).
        // A warp issues in order, so every integer instruction between two DMMAs is time the tensor pipe may
        // idle (two warps at ~7 instructions per DMMA barely cover its 16 cycles): the k-loop below is written
        // so that a block of 4 positions costs 9 LDS + 8 DMMA + a select and an add.
        constexpr int F = 8;
        const int gw = warp & 3, rw = warp >> 2;                         // output group, row half
        asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kFtRegsCompute));
        const int kk = lane & 3, rr = lane >> 2;
        const int rmap = ((rr & 1) << 2) | (rr & 2) | (rr >> 2);        // 3-bit reversal
        const int rloc = rw * (8 * F) + rmap;                            // fragment i holds row rloc + 8i
        const int nn = rr ^ ((kk >> 1) << 2);                            // band column after the XOR
        // (opaque to the optimiser: otherwise ptxas re-derives these from the thread index inside the k-loop —
        //  S2R + a dozen integer instructions per k-step — instead of keeping a few registers)
        unsigned key = (unsigned)rmap << 4;                              // swizzle: 16-byte chunk ^= row & 7
        unsigned srow = stg + rloc * 128;
        unsigned bcol = (unsigned)((gw * P.ks + kk) * 64 + nn * 8);      // my B element of block 0 inside a band buffer
        unsigned arow1 = ring + rloc * 128;                              // my row of slot 0 (low 7 bits free for the offset)
        unsigned ring_end = arow1 + (unsigned)P.nslot * kFtSlotBytes;
        // barrier addresses and the lane-0 flag, kept in registers (re-derived per use they cost an S2R + LEA each)
        unsigned a_taps = smem_u32(&bar_taps[0]), a_free = smem_u32(&bar_stg_free[rw]), a_full = smem_u32(&bar_stg_full[rw]);
        unsigned a_done = smem_u32(&bar_done[0]), a_cnt = smem_u32(&done_count), lead = lane == 0 ? 1u : 0u;
        asm volatile("" : "+r"(key), "+r"(srow), "+r"(bcol), "+r"(arow1), "+r"(ring_end));
        asm volatile("" : "+r"(a_taps), "+r"(a_free), "+r"(a_full), "+r"(a_done), "+r"(a_cnt), "+r"(lead));
        const int nt = (int)(t1 - t0);                                   // tiles of this block
        const int64_t* xp = P.xi0 + t0 * kFmT + 8 * gw;                  // my group's entries of the index table
        double ssq[SSQ ? 8 : 1];
#pragma unroll
        for (int i = 0; i < (SSQ ? 8 : 1); ++i) ssq[i] = 0.0;

        // index tables, read one tile ahead: first / last output of my group
        int64_t xq_nx, x7_nx;
        auto fetch_idx = [&](int u) {
            xq_nx = __ldg(xp + (int64_t)u * kFmT);
            x7_nx = __ldg(xp + (int64_t)u * kFmT + 7);
        };
        fetch_idx(0);

        // The band starts at the group's own first window position, so every lane tracks its own position
        // p = first + kk + 4b.  Four blocks are 16 positions = one ring slot: within a tile, block b = 4c + J sits
        // at byte ((sub0 + 32J) & 127) of the lane's row, in slot c or c + 1 of the tile (w[J]) — per tile four
        // offsets (swizzle key folded in) and three flags, per block one select.
        unsigned cur = arow1, nxt = arow1;              // my row in the slots c, c + 1 of the tile
        int jcur = 0;                                   // global slot index behind `cur`
        unsigned off[4];
        bool w[4];
        unsigned bq = 0;                                // my B element of the next block to load
        int nbt = 0;                                    // blocks of the tile in flight
        struct Ops { double a[F], b; };
        Ops o0, o1;

        auto load_ops = [&](Ops& o, auto J) {
            const unsigned ap = (w[J.value] ? nxt : cur) + off[J.value];
#pragma unroll
            for (int i = 0; i < F; ++i) o.a[i] = lds_f64(ap + i * 1024);
            o.b = lds_f64(bq);
            bq += 256;
        };
        auto next_slot = [&]() {                         // c -> c + 1
            ++jcur;
            cur = nxt;
            nxt += kFtSlotBytes;
            if (nxt == ring_end) nxt = arow1;
        };
        // Set tile t up (index arithmetic, barrier wait) and load the operands of its first block into `o`.
        // Runs underneath the last block of the tile before it.
        auto setup = [&](int u, Ops& o) {
            const int s = u & 1;
            const int r = (int)(xq_nx - P.tapsper + 1 - pos_base) + kk;            // >= 0: my position of block 0
            int n = (int)(x7_nx - xq_nx) + P.tapsper + 3;
            n >>= 2;
            nbt = n < (P.ks >> 2) ? n : (P.ks >> 2);
            if (u + 1 < nt) fetch_idx(u + 1);
            // ring slot of the tile's first block, relative to the slot in use (windows overlap: a step back is normal)
            const int j_new = r >> 4;
            int slot = (int)((cur - arow1) / kFtSlotBytes) + (j_new - jcur);
            while (slot >= P.nslot) slot -= P.nslot;
            while (slot < 0) slot += P.nslot;
            jcur = j_new;
            cur = arow1 + (unsigned)slot * kFtSlotBytes;
            nxt = cur + kFtSlotBytes;
            if (nxt == ring_end) nxt = arow1;
            const unsigned sub0 = (unsigned)(r & 15) << 3;
#pragma unroll
            for (int J = 0; J < 4; ++J) {
                const unsigned q = sub0 + 32u * J;
                w[J] = q >= 128u;
                off[J] = (q & 127u) ^ key;
            }
            bq = bands + s * band_tile + bcol;
            // one barrier per tile: the helpers arrive on it once the tile's band is built AND its ring slots
            // have landed (they watch the `full` barriers, off the compute warps' path)
            mbar_wait(a_taps + 8u * s, (unsigned)(u >> 1) & 1u);
            load_ops(o, std::integral_constant<int, 0>{});
        };
        auto mma_block = [&](double (&acc)[F][2], const Ops& o) {
#pragma unroll
            for (int i = 0; i < F; ++i) dmma884(acc[i][0], acc[i][1], o.a[i], o.b);
        };
        // fragments of a finished tile -> staging (the store thread has read the tile before it out of it).  The
        // hand-over is split: the stores go out under the first block of the next tile, the proxy fence and the
        // arrival two blocks later — issued right behind the stores the fence would hold the warp (and its DMMAs)
        // until they have drained through the LSU queue (~400 cycles per tile, measured).
        auto stage_store = [&](double (&o)[F][2], int u_old) {
            if (u_old > 0) mbar_wait(a_free, (unsigned)(u_old - 1) & 1u);
            const unsigned sp = srow + (gw >> 1) * 16384 + ((unsigned)(((gw & 1) * 4 + kk) << 4) ^ key);
#pragma unroll
            for (int i = 0; i < F; ++i) sts_v2f64(sp + i * 1024, o[i][0], o[i][1]);
            if (SSQ) {
                // outputs past n_out have all-zero taps, rows past the last read zeros: exactly 0
#pragma unroll
                for (int i = 0; i < F; ++i) ssq[i] = fma(o[i][0], o[i][0], fma(o[i][1], o[i][1], ssq[i]));
            }
        };
        auto stage_signal = [&]() {
            fence_async_smem();
            __syncwarp();
            if (lead) mbar_arrive(a_full);
        };
        // One tile: its DMMAs accumulate into `acc` while the fragments of the tile before it (`old`) drain to
        // the staging boxes underneath its first block and, during the last block, the next tile is set up and its
        // first operands are fetched: the tensor pipe is never left waiting for a tile boundary.  On entry
        // o0 holds the operands of block 0; on exit it holds those of the next tile's.  Blocks alternate between
        // o0 (even) and o1 (odd); J = b mod 4 is a compile-time constant in every step.
        auto tile = [&](double (&acc)[F][2], double (&old)[F][2], int u) {
            const bool more = u + 1 < nt;
#pragma unroll
            for (int i = 0; i < F; ++i) acc[i][0] = acc[i][1] = 0.0;
            const int n = nbt;
            using I0 = std::integral_constant<int, 0>;
            using I1 = std::integral_constant<int, 1>;
            using I2 = std::integral_constant<int, 2>;
            using I3 = std::integral_constant<int, 3>;
            int b = 0;
            bool signalled = u == 0;
            while (true) {
                // J = 0 (o0)
                if (b + 1 < n) {
                    load_ops(o1, I1{});
                    mma_block(acc, o0);
                    if (b == 0 && u > 0) stage_store(old, u - 1);
                } else {
                    if (more) setup(u + 1, o1);
                    mma_block(acc, o0);
                    if (b == 0 && u > 0) stage_store(old, u - 1);
                    o0 = o1;
                    break;
                }
                ++b;
                // J = 1 (o1)
                if (b + 1 < n) {
                    load_ops(o0, I2{});
                    mma_block(acc, o1);
                } else {
                    if (more) setup(u + 1, o0);
                    mma_block(acc, o1);
                    break;
                }
                ++b;
                // J = 2 (o0)
                if (b + 1 < n) {
                    load_ops(o1, I3{});
                    mma_block(acc, o0);
                    if (b == 2 && u > 0) { stage_signal(); signalled = true; }
                } else {
                    if (more) setup(u + 1, o1);
                    mma_block(acc, o0);
                    o0 = o1;
                    break;
                }
                ++b;
                // J = 3 (o1)
                if (b + 1 < n) {
                    next_slot();
                    load_ops(o0, I0{});
                    mma_block(acc, o1);
                } else {
                    if (more) setup(u + 1, o0);
                    mma_block(acc, o1);
                    break;
                }
                ++b;
            }
            if (!signalled) stage_signal();               // (tiles of fewer than four blocks)
            __syncwarp();
            if (lead) {
                mbar_arrive(a_done + 8u * (u & 3));
                asm volatile("red.release.cta.shared::cta.add.u32 [%0], 1;" ::"r"(a_cnt) : "memory");
            }
        };

        double accA[F][2], accB[F][2];
        setup(0, o0);
        for (int u = 0; u < nt; u += 2) {
            tile(accA, accB, u);
            if (u + 1 < nt) tile(accB, accA, u + 1);
        }
        if (nt & 1) stage_store(accA, nt - 1);
        else stage_store(accB, nt - 1);
        stage_signal();
        if (SSQ) {
#pragma unroll
            for (int i = 0; i < F; ++i) {
                const double v = quad_sum(ssq[i]);
                const int64_t row = (int64_t)row0 + rloc + 8 * i;
                if (kk == 0 && row < P.nrows) atomicAdd(P.scalars + (size_t)(row / P.nch) * P.nscalars + P.sumsq_slot, v);
            }
        }
    } else if (warp < kFtNCW + kFtNAW) {
        // ---------------- tap bands: helper warp g merges the taps of output group g — on the tensor pipe ----------------
        // h[k][n] = pfb[phi_n][k - s_n] + alpha_n * dpfb[phi_n][k - s_n] for band rows k and the group's 8 outputs n
        // (s_n = where output n's taps start in the band, zero outside) is itself a small matrix product:
        // C (8 rows x 8 outputs, preloaded with the pfb values) += A (8 rows x 8: dpfb values) * B (diag(alpha)),
        // two DMMA.8x8x4 per 8 band rows.  Scalar FP64 instructions of a helper warp queue behind the DMMAs of
        // the compute warp on the same sub-partition (measured here: ~200 cycles per DFMA, 4500 cycles per tile
        // for one FMA per merged tap); DMMAs of another warp simply interleave, at 6 % more tensor work.
        // Operands are table look-ups and selects: no FP64 ALU instruction in this branch.  Whole band rows are
        // written (zeros included) as 16-byte pairs.  Band row 0 sits at the group's first window position.
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kFtRegsHelper));
        const int grp = warp - kFtNCW;
        if (P.bands_g) {
            // ---------------- periodic resampler: the tile's four bands are one bulk copy out of the period table ----------------
            // (L2-resident: 12 KB per tile).  No look-ups, no merge DMMAs, no helper traffic on the shared-memory pipe.
            if (grp == 0 && lane == 0) {
                const unsigned bytes = 4u * (unsigned)P.ks * 64u;
                int64_t jwait = 0;
                int jw_slot = 0;
                unsigned jw_par = 0;
                for (int64_t t = t0; t < t1; ++t) {
                    const int64_t u = t - t0;
                    const int s = (int)(u & 1);
                    // (+ 4: the last block of a group reads up to 3 positions past its window — times zero taps, but what is
                    //  multiplied must be landed data, not whatever the ring held: 0 * NaN is NaN)
                    const int64_t hi = (__ldg(P.xi0 + t * kFmT + kFmT - 1) + 4 - pos_base + (kFtSlotPos - 1)) >> 4;
                    if (u >= 2) mbar_wait(&bar_done[(u - 2) & 3], (unsigned)((u - 2) >> 2) & 1u);   // the buffer's last reader
                    mbar_expect_tx(&bar_taps[s], bytes);
                    int64_t ep = t / P.epoch_tiles;
                    ep = ep < P.n_epochs ? ep : P.n_epochs - 1;
                    const double* src = P.bands_g + (size_t)(ep * P.period_tiles + t % P.period_tiles) * (bytes / 8);
                    bulk_load(bands + (unsigned)s * band_tile, src, bytes, smem_u32(&bar_taps[s]));
                    while (jwait < hi) {                                                          // ... and the tile's window has landed
                        mbar_wait(&bar_full[jw_slot], jw_par);
                        ++jwait;
                        if (++jw_slot == P.nslot) { jw_slot = 0; jw_par ^= 1u; }
                    }
                    mbar_arrive(&bar_taps[s]);
                }
            }
            return;
        }
        const int kk = lane & 3, rr = lane >> 2;
        const unsigned pf_tab = tabs, dpf_tab = tabs + 8u * P.tab_doubles;
        const bool has_d = P.dpfb != nullptr;
        const int nblk = P.ks >> 3;                        // 8-row band blocks (ks is a multiple of 8 here)
        int64_t jwait = 0;                              // ring slots [0, jwait) have been seen to land
        int jw_slot = 0;
        unsigned jw_par = 0;
        int64_t xe_nx = __ldg(P.xi0 + t0 * kFmT + kFmT - 1);
        // lane l < 8 carries column l of the group (others mirror it)
        int64_t xi_nx = __ldg(P.xi0 + t0 * kFmT + 8 * grp + (lane & 7));
        int po_nx = __ldg(P.poff + t0 * kFmT + 8 * grp + (lane & 7));
        double al_nx = __ldg(P.alpha + t0 * kFmT + 8 * grp + (lane & 7));
        for (int64_t t = t0; t < t1; ++t) {
            const int64_t u = t - t0;
            const int s = (int)(u & 1);
            const int64_t m = t * kFmT + 8 * grp + (lane & 7);
            const int64_t xi = xi_nx;
            const bool live = m < P.n_out;
            const int po = po_nx;
            const double al = live ? al_nx : 0.0;
            const int64_t hi = (xe_nx + 4 - pos_base + (kFtSlotPos - 1)) >> 4;     // slots [0, hi) hold the tile's window (+ the 3 positions past it that the last blocks read, see band_loader)
            if (t + 1 < t1) {
                xi_nx = __ldg(P.xi0 + m + kFmT);
                po_nx = __ldg(P.poff + m + kFmT);
                al_nx = __ldg(P.alpha + m + kFmT);
                xe_nx = __ldg(P.xi0 + (t + 1) * kFmT + kFmT - 1);
            }
            const int64_t xg = __shfl_sync(0xffffffffu, xi, 0);
            // band rows [st, st + tapsper) hold column (lane & 7)'s taps; a dead column (past n_out) holds none
            const int st = live ? (int)(xi - xg) : (1 << 20);
            // what my fragment elements need: C columns 2kk, 2kk+1; A columns kk, 4+kk; B column rr
            const int st_c0 = __shfl_sync(0xffffffffu, st, 2 * kk), st_c1 = __shfl_sync(0xffffffffu, st, 2 * kk + 1);
            const int po_c0 = __shfl_sync(0xffffffffu, po, 2 * kk), po_c1 = __shfl_sync(0xffffffffu, po, 2 * kk + 1);
            const int st_a0 = __shfl_sync(0xffffffffu, st, kk), st_a1 = __shfl_sync(0xffffffffu, st, 4 + kk);
            const int po_a0 = __shfl_sync(0xffffffffu, po, kk), po_a1 = __shfl_sync(0xffffffffu, po, 4 + kk);
            const double al_b = __shfl_sync(0xffffffffu, al, rr);
            const double b0v = (kk == rr) ? al_b : 0.0, b1v = (4 + kk == rr) ? al_b : 0.0;
            const unsigned band = bands + s * band_tile + (unsigned)(grp * P.ks) * 64u;
            // tile t-2 must be finished: its band buffer is about to be overwritten
            if (u >= 2) mbar_wait(&bar_done[(u - 2) & 3], (unsigned)((u - 2) >> 2) & 1u);
            // batches of four 8-row blocks: all table look-ups first, then the (independent) DMMAs, then the stores —
            // a helper's instructions queue behind the compute warps' DMMA stream, so a dependent
            // look-up -> DMMA -> DMMA -> store chain per block would pay that queueing four times per block
            for (int b0 = 0; b0 < nblk; b0 += 4) {
                double cv0[4], cv1[4], a0[4], a1[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int k = 8 * (b0 + i) + rr;                                 // my band row
                    const bool on = b0 + i < nblk;
                    const unsigned tc0 = (unsigned)(k - st_c0), tc1 = (unsigned)(k - st_c1);   // tap indices (unsigned: one range test)
                    const unsigned ta0 = (unsigned)(k - st_a0), ta1 = (unsigned)(k - st_a1);
                    cv0[i] = on && tc0 < (unsigned)P.tapsper ? lds_f64(pf_tab + 8u * ((unsigned)po_c0 + tc0)) : 0.0;
                    cv1[i] = on && tc1 < (unsigned)P.tapsper ? lds_f64(pf_tab + 8u * ((unsigned)po_c1 + tc1)) : 0.0;
                    a0[i] = has_d && on && ta0 < (unsigned)P.tapsper ? lds_f64(dpf_tab + 8u * ((unsigned)po_a0 + ta0)) : 0.0;
                    a1[i] = has_d && on && ta1 < (unsigned)P.tapsper ? lds_f64(dpf_tab + 8u * ((unsigned)po_a1 + ta1)) : 0.0;
                }
                if (has_d) {
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        if (b0 + i < nblk) dmma884(cv0[i], cv1[i], a0[i], b0v);
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        if (b0 + i < nblk) dmma884(cv0[i], cv1[i], a1[i], b1v);
                }
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int k = 8 * (b0 + i) + rr;
                    // columns 2kk, 2kk+1 stay adjacent under the XOR on bit 2 of the column index
                    if (b0 + i < nblk) sts_v2f64(band + 8u * (unsigned)(k * 8 + ((2 * kk) ^ (((k >> 1) & 1) << 2))), cv0[i], cv1[i]);
                }
            }
            // ... and the tile's window has landed in the ring
            while (jwait < hi) {
                mbar_wait(&bar_full[jw_slot], jw_par);
                ++jwait;
                if (++jw_slot == P.nslot) { jw_slot = 0; jw_par ^= 1u; }
            }
            mbar_arrive(&bar_taps[s]);
        }
    } else {
      // (one setmaxnreg for the whole fourth warpgroup: producer, store and two warps that only give registers away)
      asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kFtRegsMisc));
      if (warp == kFtNCW + kFtNAW) {
        // ---------------- producer: one tensor copy per ring slot, as far ahead as the ring allows ----------------
        if (lane == 0) {
            const int64_t last_need = __ldg(P.xi0 + (t1 - 1) * kFmT + kFmT - 1) + 4;
            const int64_t nslots_total = (last_need - pos_base + (kFtSlotPos - 1)) >> 4;
            auto lo_of = [&](int64_t t) { return (__ldg(P.xi0 + t * kFmT) - P.tapsper + 1 - pos_base) >> 4; };
            int64_t tp = t0;
            int64_t lo_next = t0 + 1 < t1 ? lo_of(t0 + 1) : (int64_t(1) << 62);
            int s = 0;
            for (int64_t j = 0; j < nslots_total; ++j) {
                if (j >= P.nslot) {
                    // the last tile that reads slot j - nslot must be done before the slot is refilled
                    const int64_t k = j - P.nslot;
                    while (lo_next <= k) {
                        ++tp;
                        lo_next = tp + 1 < t1 ? lo_of(tp + 1) : (int64_t(1) << 62);
                    }
                    const unsigned target = (unsigned)(tp - t0 + 1) * kFtNCW;
                    unsigned seen;
                    // (polled in a tight spin, no pause between reads)
                    while (true) {
                        asm volatile("ld.acquire.cta.shared::cta.u32 %0, [%1];" : "=r"(seen) : "r"(smem_u32(&done_count)) : "memory");
                        if (seen >= target) break;
                    }
                }
                mbar_expect_tx(&bar_full[s], kFtSlotBytes);
                tmap_load_2d(ring + (unsigned)s * kFtSlotBytes, &tm_in, (int)(pos_base + j * kFtSlotPos), row0, &bar_full[s]);
                if (++s == P.nslot) s = 0;
            }
        }
      } else {
        // ---------------- store: one thread per row half, two tensor stores (16 outputs x 64 rows) per tile ----------------
        const int h = warp - (kFtNCW + kFtNAW + 1);
        if (h < 2 && lane == 0) {
            const bool rows_live = (int64_t)row0 + 64 * h < P.nrows;
            for (int64_t t = t0; t < t1; ++t) {
                const int64_t u = t - t0;
                mbar_wait(&bar_stg_full[h], (unsigned)u & 1u);
                const int64_t m0 = t * kFmT;
                if (rows_live) {
                    tmap_store_2d(&tm_out, (int)m0, row0 + 64 * h, stg + 8192u * h);
                    if (m0 + 16 < P.n_out) tmap_store_2d(&tm_out, (int)(m0 + 16), row0 + 64 * h, stg + 16384 + 8192u * h);
                }
                bulk_commit();
                bulk_wait_read_all();
                mbar_arrive(&bar_stg_free[h]);
            }
            bulk_wait_all();
        }
      }
    }
}

}  // namespace sigops
