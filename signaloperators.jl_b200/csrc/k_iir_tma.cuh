// K3 (fast path) — biquad cascades with TMA bulk copies (UBLKCP) as the data mover.
//
// Same MAIN / CARRY / FIX decomposition as k_iir.cuh, specialised for the common
// shape of `Filt(x, ...) |> Amplify(c) |> sink` on Float64 data: plain Float64 buffer
// in, Float64 buffer out, constant-gain epilogue, 16-byte aligned channels.
//
// Every lane is an independent stream: lane = one chunk of one channel.  The chunk
// moves through two private 48-frame shared-memory stages:
//     cp.async.bulk global -> shared (384 B, mbarrier complete_tx)        [TMA load]
//     cascade in place on the stage (register-blocked, software-pipelined)
//     cp.async.bulk shared -> global (384 B, bulk_group)                   [TMA store]
// When the cascade's zero-input response dies out within Wc < L frames the kernel runs
// in WARM mode instead: chunk k >= 1 starts Wc frames early from zero state and simply
// discards those outputs — after Wc frames its state equals the sequential filter's to
// 2^-64 of full scale — so one launch produces final results and no CARRY/FIX pass,
// state array or second trip over the data is needed.
// Each global access is a contiguous 384-byte segment, no thread ever waits on
// another lane's data, and while a stage is being filtered the next one is already in
// flight.  Chunks are numbered over (instance, channel, chunk) jointly, so a warp's 32
// lanes may belong to different channels and the grid can be sized to whole waves.
#pragma once
#include "k_iir.cuh"
#include "ptx.cuh"

namespace sigops {

constexpr int kTmaWarps = 8;
constexpr int kTmaThreads = kTmaWarps * 32;
constexpr int kStageCols = 48;                 // frames per stage (384 B)
static_assert(kStageCols % 16 == 0, "stage = whole 16-frame register blocks");
constexpr int kStagePitch = kStageCols + 2;    // doubles: rows keep 16-B alignment; (cols+2)*2 = 4 mod 32 words makes
                                               // lane=row 128-bit accesses bank-conflict free
constexpr int kStageBytes = kStageCols * 8;
// per warp: [stage 0/1][lane][kStagePitch] doubles, then two mbarriers per lane
constexpr size_t kTmaSmemBytes = (size_t)kTmaThreads * 2 * kStagePitch * sizeof(double) + (size_t)kTmaThreads * 2 * sizeof(uint64_t);

// Fused elementwise programs of the TMA kernel (PROG variants): the input program sees the
// frame just loaded as LEAF_STAGE (e.g. `load * modulator`), the epilogue sees the filter
// output as LEAF_STAGE (e.g. `y * ramp_on * ramp_off + tone`).  Neither may read another
// buffer or an RMS slot (the planner falls back to k_iir for those).
struct TmaProg {
    const sigops_instr* in_prog;  const double* in_lc;  const double2* in_rot;  int in_len;
    const sigops_instr* ep_prog;  const double* ep_lc;  const double2* ep_rot;  int ep_len;
};

// 16 frames (one third of a stage) through the cascade (cascade_frames, out as in cascade_tile of k_iir.cuh).
// Returns sum(out^2) of the 16 outputs.  n0 = signal frame of p[0], c = channel, keep = the
// outputs will be stored (PROG only).
template <int M, bool ZERO_IN, bool UNITB, bool PROG>
__device__ __forceinline__ double cascade16(Cascade<M>& f, double* p, double gain, double sc,
                                            const TmaProg& T, int64_t n0, int c, bool keep = true) {
    double xr[16];
#pragma unroll
    for (int k = 0; k < 16; k += 2) {
        const double2 v = *reinterpret_cast<const double2*>(p + k);
        xr[k] = v.x; xr[k + 1] = v.y;
    }
    if (PROG && T.in_len > 0) {
        double t[16];
        Env env{nullptr, nullptr, 0};
        eval_program<16>(T.in_prog, T.in_lc, T.in_rot, T.in_len, env, n0, 1, c, xr, t, nullptr, 0);
#pragma unroll
        for (int k = 0; k < 16; ++k) xr[k] = t[k];
    }
    double pipe[M], out[16];
    cascade_frames<M, 16, ZERO_IN, UNITB>(f, xr, pipe, [&](int k, double y) {
        out[k] = ZERO_IN ? fma(y, gain, xr[k]) * sc : (y * gain) * sc;
    });
    if (PROG && T.ep_len > 0 && keep) {      // warm-up outputs are discarded: no epilogue
        double t[16];
        Env env{nullptr, nullptr, 0};
        eval_program<16>(T.ep_prog, T.ep_lc, T.ep_rot, T.ep_len, env, n0, 1, c, out, t, nullptr, 0);
#pragma unroll
        for (int k = 0; k < 16; ++k) out[k] = t[k];
    }
    double ss = 0.0;
#pragma unroll
    for (int k = 0; k < 16; k += 2) {
        *reinterpret_cast<double2*>(p + k) = make_double2(out[k], out[k + 1]);
        ss = fma(out[k], out[k], ss);
        ss = fma(out[k + 1], out[k + 1], ss);
    }
    return ss;
}

struct IirTmaParams {
    IirParams base;
    int64_t cpr;            // chunks per channel
    int64_t total_chunks;   // rows * cpr
};

template <int M, int MODE, bool UNITB, bool PROG>
__global__ void __launch_bounds__(kTmaThreads, 1)
k_iir_tma(const __grid_constant__ IirTmaParams Q) {
    const IirParams& P = Q.base;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ sigops_instr sp_in[PROG ? SIGOPS_MAX_PROG : 1], sp_ep[PROG ? SIGOPS_MAX_PROG : 1];
    __shared__ double lc_in[PROG ? SIGOPS_MAX_PROG : 1], lc_ep[PROG ? SIGOPS_MAX_PROG : 1];
    __shared__ double2 lr_in[PROG ? SIGOPS_MAX_PROG : 1], lr_ep[PROG ? SIGOPS_MAX_PROG : 1];
    TmaProg T{sp_in, lc_in, lr_in, PROG ? P.in_prog_len : 0, sp_ep, lc_ep, lr_ep, PROG ? P.epi_prog_len : 0};
    if (PROG) {
        Env env0{nullptr, nullptr, 0};
        prepare_program(P.instrs + P.in_prog_start, P.in_prog_len, sp_in, lc_in, lr_in, env0, 1);
        prepare_program(P.instrs + P.epi_prog_start, P.epi_prog_len, sp_ep, lc_ep, lr_ep, env0, 1);
        __syncthreads();
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // per warp: [stage 0/1][lane][kStagePitch] doubles (lane stride 132 words = 4 mod 32 banks:
    // 128-bit lane=row accesses are conflict free), then two mbarriers per lane
    double* warp_base = reinterpret_cast<double*>(smem_raw) + (size_t)warp * 2 * 32 * kStagePitch;
    double* const stage_a = warp_base + (size_t)lane * kStagePitch;
    double* const stage_b = stage_a + (size_t)32 * kStagePitch;
    uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<double*>(smem_raw) + (size_t)kTmaThreads * 2 * kStagePitch) +
                     (size_t)(warp * 32 + lane) * 2;

    const int64_t g = ((int64_t)blockIdx.x * kTmaWarps + warp) * 32 + lane;     // my chunk
    const bool active = g < Q.total_chunks;
    const int64_t gg = active ? g : 0;
    const int64_t row = gg / Q.cpr, k = gg % Q.cpr;
    const int inst = (int)(row / P.nch), c = (int)(row % P.nch);
    const BufRef ib = P.bufrefs[(size_t)inst * P.nbuf + P.plain_in_buf];
    const BufRef ob = P.bufrefs[(size_t)inst * P.nbuf + P.out_buf];
    const int64_t L = P.L;
    const double* xin = reinterpret_cast<const double*>(ib.ptr) + (int64_t)c * ib.ld + k * L;
    double* yout = reinterpret_cast<double*>(ob.ptr) + (int64_t)c * ob.ld + k * L;
    // frames of this chunk that exist in the output / in the input buffer
    int64_t len = P.N - k * L;
    len = len < 0 ? 0 : (len > L ? L : len);
    int64_t in_len = P.plain_in_len - k * L;
    in_len = in_len < 0 ? 0 : (in_len > len ? len : in_len);
    if (!active) { len = 0; in_len = 0; }
    // WARM: the lane starts `pre` frames before its chunk (those outputs are discarded)
    const int64_t pre = (MODE == IIR_WARM && k >= 1) ? P.Wc : 0;
    // FIX only touches the first Wc frames of chunks >= 1
    const int64_t work = (MODE == IIR_FIX) ? ((k >= 1) ? (len < P.Wc ? len : P.Wc) : 0) : (len > 0 ? len + pre : 0);
    int64_t src_len = work;                                  // frames the source really holds from gsrc on
    if (MODE != IIR_FIX) {
        src_len = P.plain_in_len - (k * L - pre);
        src_len = src_len < 0 ? 0 : (src_len > work ? work : src_len);
        if (!active) src_len = 0;
    }
    const double* gsrc = (MODE == IIR_FIX) ? yout : xin - pre;
    double* const gdst = yout - pre;                          // stage h of the lane lands at gdst + h*kStageCols
    const int64_t nstage = (work + kStageCols - 1) / kStageCols;

    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    fence_mbarrier_init();
    fence_async_smem();
    __syncwarp();

    Cascade<M> f;
    f.init(P.coef);
    if (MODE == IIR_FIX && active && k >= 1) load_carried_state(f, P, Q.total_chunks, g);
    const double sc_final = P.epi_scale[0] * P.epi_scale[1];
    const int64_t raw_frames = (MODE == IIR_MAIN && k >= 1) ? P.Wc : 0;   // MAIN leaves these un-scaled for FIX
    const int64_t skip_frames = pre;                                       // WARM: nothing is stored before this
    double ss = 0.0;
    unsigned parity = 0u, pending = 0u;      // bit b: mbarrier phase / TMA load in flight for stage b

    // Stage h of my chunk -> shared.  Full stages go through the TMA; a ragged
    // last stage (or input shorter than the output: zero padding) is copied by the lane.
    auto issue_load = [&](int64_t h) {
        const unsigned b = (unsigned)(h & 1);
        double* dst = b ? stage_b : stage_a;
        const int64_t off = h * kStageCols;
        const int64_t have = src_len - off;          // frames available from the source
        if (have >= kStageCols) {
            mbar_expect_tx(&bars[b], kStageBytes);
            bulk_load(dst, gsrc + off, kStageBytes, &bars[b]);
            pending |= 1u << b;
        } else {
            for (int i = 0; i < kStageCols; ++i) dst[i] = (i < have) ? gsrc[off + i] : 0.0;
            pending &= ~(1u << b);
        }
    };

    if (nstage > 0) issue_load(0);
    for (int64_t h = 0; h < nstage; ++h) {
        const unsigned b = (unsigned)(h & 1);
        double* buf = b ? stage_b : stage_a;
        if (pending & (1u << b)) {
            mbar_wait(&bars[b], (parity >> b) & 1u);
            parity ^= 1u << b;
        }
        const int64_t off = h * kStageCols;
        const double sc = (off < raw_frames) ? 1.0 : sc_final;      // Wc is a multiple of the stage
        const int64_t nstage0 = k * L - pre + off;                 // signal frame of buf[0]
        double s4;
        if (PROG) s4 = 0.0;
        else s4 = cascade16<M, MODE == IIR_FIX, UNITB, PROG>(f, buf, P.gain, sc, T, nstage0, c);
        // the other stage was handed to a bulk store one iteration ago: once the TMA has
        // read it, start filling it with the next stage
        if (h + 1 < nstage) {
            bulk_wait_read_all();
            issue_load(h + 1);
        }
        if (PROG) {          // the interpreter is big: keep one copy of it (all three blocks in one loop)
#pragma unroll 1
            for (int q = 0; q < kStageCols; q += 16)
                s4 += cascade16<M, MODE == IIR_FIX, UNITB, PROG>(f, buf + q, P.gain, sc, T, nstage0 + q, c, off >= skip_frames);
        } else {
#pragma unroll
            for (int q = 16; q < kStageCols; q += 16)
                s4 += cascade16<M, MODE == IIR_FIX, UNITB, PROG>(f, buf + q, P.gain, sc, T, nstage0 + q, c);
        }
        const int64_t rem = work - off;
        if (off < skip_frames) {
            // warm-up stage: outputs are not part of this chunk (pre is a multiple of the stage)
        } else if (rem >= kStageCols) {
            fence_async_smem();
            bulk_store(gdst + off, buf, kStageBytes);
            bulk_commit();
            if (off >= raw_frames) ss += s4;
        } else {
            for (int i = 0; i < (int)rem; ++i) {
                const double w = buf[i];
                gdst[off + i] = w;
                if (off >= raw_frames) ss = fma(w, w, ss);
            }
        }
    }
    bulk_wait_all();

    if (MODE == IIR_MAIN && active && P.state_zs) store_final_state(f, P.state_zs, Q.total_chunks, g);
    if (P.sumsq_slot >= 0) {
        // lanes of a warp may belong to different instances: one atomic per lane that has data
        if (active && work > 0) atomicAdd(P.scalars + (size_t)inst * P.nscalars + P.sumsq_slot, ss);
    }
}

}  // namespace sigops
