// K3 (fastest path) — biquad cascades fed by tensor-map TMA.
//
// Same arithmetic and the same WARM decomposition as k_iir_tma.cuh (chunk k >= 1 starts Wc
// frames early from zero state and discards those outputs; DSP.jl `filt!(DF2TFilter{SOS})`
// reached from src/filters.jl:252-255).  What changes is who moves the data.  In k_iir_tma
// every lane issues its own bulk copies — measured, those two instructions and the scalar
// code around them are 40 % of the kernel's stall samples.  Here the 32 lanes of a warp are
// 32 consecutive ROWS (a row = one channel of one instance) working on the SAME time chunk, so
// a stage of the warp is a rectangular box of the [rows][frames] matrix and moves with ONE
// elected-lane instruction:
//     cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes   (load)
//     cp.async.bulk.tensor.3d.global.shared::cta.bulk_group                          (store)
// The matrix is described as [row][frame/16][16] so that the innermost extent is 128 bytes, the
// widest the 128-byte swizzle allows; the box (16, 5, 32) is 640 contiguous bytes of each of
// 32 rows.  With the swizzle a lane reading its own row 16 bytes at a time hits 8 different
// bank groups per quarter warp (conflict free) without any padding.  Out-of-range coordinates
// are handled by the TMA unit: frames past the end of the input read as zeros (the reference's
// zero padding), frames past the end of the output and rows past the last one are clipped on
// store.
//
// Measured on B200 (config 2; k_iir_tma = 0.776 ms), warps x stages x frames per stage:
//   8 x 2 x 48   0.773 ms   k_iir_tma's shape: a third fewer instructions, same time; 4 x 4 and 6 x 3
//                           stagings and L2 prefetch of longer row pieces do not move it either — the
//                           limit is what HBM delivers for ~38 000 concurrent 384-byte streams
//   6 x 2 x 64   0.753 ms   longer pieces help (4-way bank conflicts from the even block count)
//   4 x 2 x 80   0.732 ms   <- used: 640-byte pieces; 0.718 ms inside bench.py = 84 % of the measured copy peak
//   4 x 2 x 112  0.837 ms,  2 x 2 x 192  1.39 ms   (too few lanes for the FP64 dependency chains)
// One copy instruction per stage is what makes long pieces affordable; the per-lane kernel's copy
// cost is per copy and it needs 8 warps to hide it.  SIGOPS_NO_TMAP=1 switches this kernel off.
//
// Eligibility (checked by the host): Float64 in/out, constant-gain epilogue, every row of the
// wave at base + row*stride (true for staged host batches and for one batch tensor), frame
// counts that are multiples of 16, WARM mode.
#pragma once
#include <cuda.h>

#include "k_iir_tma.cuh"

namespace sigops {

constexpr int kTmSub = 16;                       // Float64 frames per 128-byte box row (the widest swizzled row)
#ifndef TMSUBS
#define TMSUBS 5                                 // (tuning builds override the shape with -DTMSUBS/-DTMW/-DTMS)
#endif
// 80-frame stages: 640 contiguous bytes per row and copy.  An odd number of blocks per row also keeps
// the swizzle key (blocks*row + block) mod 8 different for 8 consecutive rows (4 blocks: 4-way conflicts).
constexpr int kTmSubsPerStage = TMSUBS;                  // Float64 shape
constexpr int kTmStageCols = kTmSub * kTmSubsPerStage;   // Float64 frames per stage
constexpr int kTmSubBytes = 32 * 128;                    // one box row block: 32 rows x 128 bytes
// Float32 shape: the bytes per sample halve while the FP64 work per sample stays, so the kernel is
// bound by its dependency chains — twice the warps, 3-block stages (96 frames, 384 bytes per row)
constexpr int kTmSubsPerStageF32 = 3, kTmWarpsF32 = 8;
// fused row-invariant programs (config 5: 5 general biquads + 4 elementwise operations per sample): the FP64
// dependency chains are long, so twice the warps on 48-frame stages, like the Float32 shape
constexpr int kTmSubsPerStageLv = 3, kTmWarpsLv = 8;
constexpr int kTmMaxLeafOps = 4;                        // fused row-invariant operations before / after the cascade
constexpr size_t tm_smem_bytes(int nw, int ns, int subs, bool lv = false, int sub = kTmSub) {   // + 1024-byte alignment slack
    return (size_t)nw * ns * subs * kTmSubBytes + 1024 + (lv ? (size_t)nw * 2 * kTmMaxLeafOps * subs * sub * sizeof(double) : 0);
}

struct IirTmapParams {
    const BufRef* bufrefs;
    double* scalars;
    int nbuf, nscalars;
    int out_buf, sumsq_slot;
    int nch;
    int64_t nrows;
    int64_t N, L, Wc;          // frames, chunk length, warm-up (both multiples of the stage)
    int64_t cpr;               // chunks per row
    int64_t nunits;            // row groups * cpr
    double gain, scale, scale2;     // y = ((cascade * gain) * scale) * scale2: the epilogue's constants, applied in order
    double coef[kIirMaxSections][5];
    // Fused elementwise programs whose leaves do not depend on the row (constants, generators, ramps — e.g.
    // BASELINE config 5: x * (0.5 sin + 0.5) before the cascade, y * ramp_on * ramp_off + tone after it):
    // ops[0 .. n_in_ops) combine the loaded sample with their leaf, ops[4 .. 4 + n_ep_ops) the filter output.  A
    // closure function f(x) (FN1) or g(x, constant) (FN2) takes an op slot and no leaf vector (e.g. abs before an
    // envelope follower's lowpass, tanh after a filter).
    int n_in_ops, n_ep_ops;
    sigops_instr ops[2 * kTmMaxLeafOps];
};

__device__ __forceinline__ void tmap_load_3d(void* smem_dst, const CUtensorMap* tm, int c0, int c1, int c2, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(tm), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tmap_store_3d(const CUtensorMap* tm, int c0, int c1, int c2, const void* smem_src) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%1, %2, %3}], [%4];" ::"l"(tm), "r"(c0), "r"(c1), "r"(c2),
                 "r"(smem_u32(smem_src))
                 : "memory");
}

// 16 frames of the lane's row through the cascade, in place in a swizzled box.  `row` points at the
// lane's 128-byte box row, `key` = address bits 7-9 of that row: 16-byte chunk j lives at chunk
// j ^ key.  Float64: the row is one 16-frame block (8 chunks).  Float32: it holds two (blk = 0, 1; 4
// chunks each); samples are widened on load, the state and all arithmetic stay Float64 like the
// reference's DF2T filter state, and results are rounded on store.
// Returns sum(out^2) over the first `nvalid` outputs as stored.
// acc[k] = acc[k] (op) v[k] for 16 frames, the operator decoded once (v: warp-uniform values in shared memory)
// (FN1 / FN2 with a constant: acc[k] = f(acc[k]) or g(acc[k], d0), no leaf vector)
template <bool FN>
__device__ __forceinline__ void apply_leaf16(const sigops_instr& I, double* acc, const double* v) {
    if (FN && (I.op == SIGOPS_OP_FN1 || I.op == SIGOPS_OP_FN2)) {
        efn_vec<16>(I.fn, acc, [&](int) { return I.d0; }, I.d1);
        return;
    }
    switch (I.op) {
        case SIGOPS_OP_ADD:
#pragma unroll
            for (int k = 0; k < 16; ++k) acc[k] = acc[k] + v[k];
            break;
        case SIGOPS_OP_SUB:
#pragma unroll
            for (int k = 0; k < 16; ++k) acc[k] = acc[k] - v[k];
            break;
        case SIGOPS_OP_MUL:
#pragma unroll
            for (int k = 0; k < 16; ++k) acc[k] = acc[k] * v[k];
            break;
        default:
#pragma unroll
            for (int k = 0; k < 16; ++k) acc[k] = acc[k] / v[k];
            break;
    }
}

// LV: 0 none, 1 row-invariant leaf operations, 2 the same with closure functions among them
template <int M, bool UNITB, class T, int LV = 0>
__device__ __forceinline__ double cascade16_swz(Cascade<M>& f, unsigned char* row, int key, int blk, double gain, double sc, double sc2,
                                                int nvalid, bool want_ss, const IirTmapParams* P = nullptr, const double* lv = nullptr,
                                                int lvpitch = 0, unsigned skip = 0u) {
    double xr[16];
    if (sizeof(T) == 8) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const double2 v = *reinterpret_cast<const double2*>(row + ((j ^ key) << 4));
            xr[2 * j] = v.x; xr[2 * j + 1] = v.y;
        }
    } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float4 v = *reinterpret_cast<const float4*>(row + (((4 * blk + j) ^ key) << 4));
            xr[4 * j] = v.x; xr[4 * j + 1] = v.y; xr[4 * j + 2] = v.z; xr[4 * j + 3] = v.w;
        }
    }
    // (bit j of `skip`: operation j multiplies / divides by a leaf that is exactly 1 over this whole stage — a ramp
    //  outside its short region — which is the identity, bit for bit)
    if (LV) {
        for (int j = 0; j < P->n_in_ops; ++j)
            if (!((skip >> j) & 1u)) apply_leaf16<LV == 2>(P->ops[j], xr, lv + j * lvpitch);
    }
    double pipe[M], out[16];
#pragma unroll
    for (int t = 0; t < 16 + M - 1; ++t) {
#pragma unroll
        for (int j = M - 1; j >= 0; --j) {
            const int k = t - j;
            if (k >= 0 && k < 16) {
                const double in = (j == 0) ? xr[k] : pipe[j - 1];
                pipe[j] = biquad_step<M, UNITB>(f, j, in);
                if (j == M - 1) out[k] = pipe[j] * gain;
            }
        }
    }
    // y = ((cascade * gain) * sc) * sc2, the epilogue's constants in order; a factor of exactly 1 is skipped (identity)
    if (sc != 1.0) {
#pragma unroll
        for (int k = 0; k < 16; ++k) out[k] *= sc;
    }
    if (sc2 != 1.0) {
#pragma unroll
        for (int k = 0; k < 16; ++k) out[k] *= sc2;
    }
    if (LV) {
        for (int j = 0; j < P->n_ep_ops; ++j)
            if (!((skip >> (kTmMaxLeafOps + j)) & 1u))
                apply_leaf16<LV == 2>(P->ops[kTmMaxLeafOps + j], out, lv + (kTmMaxLeafOps + j) * lvpitch);
    }
    if (sizeof(T) == 8) {
#pragma unroll
        for (int j = 0; j < 8; ++j) *reinterpret_cast<double2*>(row + ((j ^ key) << 4)) = make_double2(out[2 * j], out[2 * j + 1]);
    } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float4 v = make_float4((float)out[4 * j], (float)out[4 * j + 1], (float)out[4 * j + 2], (float)out[4 * j + 3]);
            *reinterpret_cast<float4*>(row + (((4 * blk + j) ^ key) << 4)) = v;
            out[4 * j] = v.x; out[4 * j + 1] = v.y; out[4 * j + 2] = v.z; out[4 * j + 3] = v.w;
        }
    }
    double ss = 0.0;
    if (want_ss) {                                   // only when a Normpower follows (warp-uniform)
#pragma unroll
        for (int k = 0; k < 16; ++k)
            if (nvalid >= 16 || k < nvalid) ss = fma(out[k], out[k], ss);
    }
    return ss;
}

// NW warps per block, NS stages per warp (NS - 1 loads in flight while one stage is filtered), SUBS
// 128-byte blocks per row and stage (odd: keeps the swizzle key distinct for 8 consecutive rows).
// value of a row-invariant leaf at frame n (the interpreter's exact per-frame formulas)
__device__ __forceinline__ double rowinv_leaf(const sigops_instr* I, int64_t n) {
    return I->leaf == SIGOPS_LEAF_CONST ? I->d0 : leaf_value_slow(I, nullptr, n, 0);
}

template <int M, bool UNITB, int NW, int NS, int SUBS, class T, int LV = 0>
__global__ void __launch_bounds__(NW * 32, 1)
k_iir_tmap(const __grid_constant__ IirTmapParams P, const __grid_constant__ CUtensorMap tm_in,
           const __grid_constant__ CUtensorMap tm_out) {
    constexpr int SUB = 128 / (int)sizeof(T);        // frames per 128-byte box row: 16 or 32
    constexpr int SC = SUB * SUBS;                   // frames per stage
    constexpr int kStageB = SUBS * kTmSubBytes;      // bytes per stage
    extern __shared__ unsigned char tm_smem_raw[];
    __shared__ uint64_t bars[NW][NS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // 1024-byte aligned stage buffers (the swizzle pattern is a function of address bits 4-9)
    // (an offset into the shared array, not a pointer rebuilt from an integer: the latter turns every access of
    //  the kernel into a generic LD/ST)
    unsigned char* base = tm_smem_raw + ((1024u - (smem_u32(tm_smem_raw) & 1023u)) & 1023u);
    unsigned char* const stage0 = base + (size_t)warp * NS * kStageB;
    auto stage_of = [&](int b) { return stage0 + b * kStageB; };
    // (LV) the block's leaf vectors, double-buffered over stages: [2][2 * kTmMaxLeafOps][SC] doubles.  They depend on
    // the frame only, so the warps of a block are given the SAME chunk of NW consecutive row groups and evaluate
    // each value once per block (one leaf evaluation per thread and stage instead of four, all on the critical
    // path of a kernel that is bound by its FP64 dependency chains: 30 % of the stall samples before).
    double* const lvbuf = reinterpret_cast<double*>(base + (size_t)NW * NS * kStageB);

    int64_t grp, k;
    bool active = true;
    if (LV) {
        const int64_t ngroups = P.nunits / P.cpr;
        k = (int64_t)blockIdx.x % P.cpr;
        grp = ((int64_t)blockIdx.x / P.cpr) * NW + warp;
        active = grp < ngroups;                                        // (idle warps still take part in the leaf vectors)
    } else {
        const int64_t unit = (int64_t)blockIdx.x * NW + warp;         // (row group, chunk)
        if (unit >= P.nunits) return;
        grp = unit / P.cpr;
        k = unit % P.cpr;
    }
    const int64_t row = grp * 32 + lane;
    const bool live = row < P.nrows;
    const int64_t pre = k >= 1 ? P.Wc : 0;
    int64_t len = P.N - k * P.L;
    len = len > P.L ? P.L : len;                                       // >= 1 by construction of cpr
    const int64_t work = len + pre;
    const int64_t start = k * P.L - pre;                               // frame of stage 0, column 0
    const int64_t nstage = (work + SC - 1) / SC;
    const int c1 = (int)(grp * 32);

    if (lane == 0) {
        for (int b = 0; b < NS; ++b) mbar_init(&bars[warp][b], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    fence_async_smem();
    __syncwarp();

    Cascade<M> f;
    {
        // same coefficient set-up as Cascade::init, from this kernel's parameter block
#pragma unroll
        for (int j = 0; j < M; ++j) {
            f.b0[j] = P.coef[j][0]; f.b1[j] = P.coef[j][1]; f.b2[j] = P.coef[j][2];
            f.a1[j] = P.coef[j][3]; f.a2[j] = P.coef[j][4];
            f.s1[j] = 0.0; f.s2[j] = 0.0;
        }
    }

    // One tensor instruction per stage: box = (128 bytes, 5 blocks, 32 rows) of the
    // [row][frame/SUB][SUB] view, i.e. 640 contiguous bytes per row.
    auto issue_load = [&](int64_t h) {
        if (lane == 0 && active) {
            const int b = (int)(h % NS);
            mbar_expect_tx(&bars[warp][b], kStageB);
            tmap_load_3d(stage_of(b), &tm_in, 0, (int)((start + h * SC) / SUB), c1, &bars[warp][b]);
        }
    };

    double ss = 0.0;
    const bool want_ss = P.sumsq_slot >= 0;
    unsigned parity = 0u;
    for (int64_t h = 0; h < NS - 1 && h < nstage; ++h) issue_load(h);
    for (int64_t h = 0; h < nstage; ++h) {
        const int b = (int)(h % NS);
        if (active) mbar_wait(&bars[warp][b], (parity >> b) & 1u);
        parity ^= 1u << b;
        const int64_t off = h * SC;
        // smem box layout: [row][block][128 bytes]; the 128-byte swizzle XORs the 16-byte chunk index
        // with address bits 7-9 = (blocks_per_stage*row + block) mod 8
        unsigned char* rowp = stage_of(b) + lane * (SUBS * 128);
        const bool keep = off >= pre;                                  // pre is a multiple of the stage
        double s3 = 0.0;
        unsigned skip = 0u;
        const double* lvs = lvbuf + (h & 1) * (2 * kTmMaxLeafOps * SC);
        if (LV) {
            // the leaves of the fused programs: every thread of the block evaluates at most a few values of the stage
            // (the interpreter's exact per-frame formulas), all rows then read them back as broadcasts.  One block
            // barrier per stage: the buffer written now was last read two stages ago, before the previous barrier.
            double* lvw = lvbuf + (h & 1) * (2 * kTmMaxLeafOps * SC);
            const int nops = P.n_in_ops + P.n_ep_ops;
            const int64_t n0 = start + off;
            unsigned ones = 0u;                                        // ramps are 1 outside a short region
            for (int jj = 0; jj < nops; ++jj) {
                const int j = jj < P.n_in_ops ? jj : kTmMaxLeafOps + jj - P.n_in_ops;
                const sigops_instr* I = &P.ops[j];
                bool one = false;
                if (I->leaf == SIGOPS_LEAF_RAMP_ON) one = n0 + I->i0 > I->i1;
                else if (I->leaf == SIGOPS_LEAF_RAMP_OFF) one = n0 + (SC - 1) + I->i0 <= I->i1;
                if (one) {
                    ones |= 1u << j;
                    if (I->op == SIGOPS_OP_MUL || I->op == SIGOPS_OP_DIV) skip |= 1u << j;
                }
            }
            for (int v = threadIdx.x; v < nops * SC; v += NW * 32) {
                const int jj = v / SC, fr = v - jj * SC;
                const int j = jj < P.n_in_ops ? jj : kTmMaxLeafOps + jj - P.n_in_ops;
                if (((skip >> j) & 1u) || (LV == 2 && P.ops[j].op >= SIGOPS_OP_FN1)) continue;   // (functions: no vector)
                lvw[j * SC + fr] = ((ones >> j) & 1u) ? 1.0 : rowinv_leaf(&P.ops[j], n0 + fr);
            }
            __syncthreads();
        }
        if (!active) continue;
#pragma unroll
        for (int s = 0; s < SUBS; ++s) {
#pragma unroll
            for (int blk = 0; blk < SUB / 16; ++blk) {
                const int64_t rem = work - off - s * SUB - blk * 16;   // outputs of this block that exist
                s3 += cascade16_swz<M, UNITB, T, LV>(f, rowp + s * 128, (SUBS * lane + s) & 7, blk, P.gain, P.scale, P.scale2,
                                                     rem >= 16 ? 16 : (rem > 0 ? (int)rem : 0), want_ss, &P, lvs + s * SUB + blk * 16, SC, skip);
            }
            if (s == 0 && h + NS - 1 < nstage) {
                // the stage filtered one iteration ago went to a tensor store: once the TMA unit has
                // read it, refill it (issued after the first block so the wait is off the critical path)
                if (lane == 0) bulk_wait_read_all();
                issue_load(h + NS - 1);
            }
        }
        // the stage was rewritten in place through the generic proxy; the next thing to touch it
        // is the TMA unit (store now, or the refill two iterations on)
        fence_async_smem();
        __syncwarp();
        if (keep) {
            ss += s3;
            if (lane == 0) {
                // frames past N and rows past the last one are clipped by the tensor bounds
                tmap_store_3d(&tm_out, 0, (int)((start + off) / SUB), c1, stage_of(b));
                bulk_commit();
            }
        }
        __syncwarp();
    }
    if (lane == 0 && active) bulk_wait_all();
    if (P.sumsq_slot >= 0 && live && active) {
        const int64_t inst = row / P.nch;
        atomicAdd(P.scalars + (size_t)inst * P.nscalars + P.sumsq_slot, ss);
    }
}

}  // namespace sigops
