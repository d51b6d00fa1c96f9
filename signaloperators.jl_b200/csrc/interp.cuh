// Elementwise program interpreter shared by every kernel (K1 and the fused
// prologues/epilogues of the IIR and FIR kernels).
//
// Replaces, per output sample, the reference's recursive `frame(x,block,i)` walk:
//   MapSignal.frame      src/mapsignal.jl:249-272
//   SignalFunction frame src/functions.jl:53-60
//   RampSignal frame     src/ramps.jl:56-72
//   NumberBlock/PadBlock/CutBlock/AppendBlock/ArrayBlock frames
//     src/numbers.jl:62-64, src/padding.jl:210-214, src/cutting.jl:217-218,
//     src/appending.jl:89-90, src/arrays.jl:118-119
// All index plumbing (offsets, valid lengths, pads) was resolved by the host
// planner; the device only sees pure leaves evaluated at (n,c).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "../../include/signalops.h"

namespace sigops {

struct BufRef {            // one buffer of one instance
    void*   ptr;
    int64_t ld;
    int32_t dtype;
    int32_t nch;
};

// Everything a block needs to evaluate leaves for one instance.
struct Env {
    const BufRef* bufs;        // [nbuf] for this instance (shared memory copy)
    const double* scalars;     // [nscalars] for this instance (global)
    int64_t inst;              // index of the instance in the whole call (all waves, all devices): noise stream offset
};

__device__ __forceinline__ double load_elem(const void* p, int dtype, int64_t i) {
    if (dtype == SIGOPS_F64) return __ldg(reinterpret_cast<const double*>(p) + i);
    if (dtype == SIGOPS_F32) return (double)__ldg(reinterpret_cast<const float*>(p) + i);
    return (double)__ldg(reinterpret_cast<const long long*>(p) + i);
}

__device__ __forceinline__ double store_elem(void* p, int dtype, int64_t i, double v) {
    if (dtype == SIGOPS_F64) { reinterpret_cast<double*>(p)[i] = v; return v; }
    if (dtype == SIGOPS_F32) { float f = (float)v; reinterpret_cast<float*>(p)[i] = f; return (double)f; }
    long long q = (long long)v; reinterpret_cast<long long*>(p)[i] = q; return (double)q;
}

__device__ __forceinline__ double apply_fn(int fn, double x, double a, double b) {
    switch (fn) {
        case SIGOPS_FN_SIN: return sin(x);
        case SIGOPS_FN_COS: return cos(x);
        case SIGOPS_FN_SAW: return x / 3.141592653589793 - 1.0;
        case SIGOPS_FN_AFFINE_SIN: return a * sin(x) + b;
        case SIGOPS_FN_AFFINE_COS: return a * cos(x) + b;
        case SIGOPS_FN_IDENTITY: return x;
        case SIGOPS_FN_SINRAMP: return sinpi(0.5 * x);
    }
    return 0.0;
}

// src/functions.jl:53-60 — evaluated in exactly this operation order
__device__ __forceinline__ double gen_value(const sigops_instr& I, int64_t k) {
    const double t = (double)k / I.d0;
    if (I.flags & SIGOPS_FLAG_HAS_OMEGA) {
        const double u = t * I.d1 + I.d2;
        if (I.fn == SIGOPS_FN_SIN) return sinpi(2.0 * u);
        // u % 1.0 (truncated remainder, src/functions.jl:56) == u - trunc(u) exactly, without fmod's loop
        return apply_fn(I.fn, 6.283185307179586 * (u - trunc(u)), I.d3, I.d4);
    }
    if (I.fn == SIGOPS_FN_SIN) return sinpi(2.0 * (t + I.d2));
    return apply_fn(I.fn, t + I.d2, I.d3, I.d4);
}

// `Signal(randn; rng)` on the device (src/functions.jl:98-114): frame k (1-based) of noise stream `stream` under `seed`, a
// pure function of its arguments — Philox4x32-10 (Salmon et al., SC'11) on counter ((k-1)>>1, stream), key seed, then
// Box-Muller: r cos(2 pi u2) for odd k, r sin(2 pi u2) for even k.  host/philox.py is the same function in numpy.
static __device__ __noinline__ double randn_value(int64_t seed, int64_t stream, int64_t k) {
    const uint64_t pair = (uint64_t)(k - 1) >> 1, st = (uint64_t)stream, sd = (uint64_t)seed;
    uint32_t c0 = (uint32_t)pair, c1 = (uint32_t)(pair >> 32), c2 = (uint32_t)st, c3 = (uint32_t)(st >> 32);
    uint32_t k0 = (uint32_t)sd, k1 = (uint32_t)(sd >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    const double u1 = ((double)((((uint64_t)c1 << 32) | c0) >> 11) + 0.5) * (1.0 / 9007199254740992.0);
    const double u2 = ((double)((((uint64_t)c3 << 32) | c2) >> 11) + 0.5) * (1.0 / 9007199254740992.0);
    const double r = sqrt(-2.0 * log(u1));
    double sn, cs;
    sincospi(2.0 * u2, &sn, &cs);
    return r * ((k & 1) ? cs : sn);
}

// Per-frame evaluation of the leaves that have no vector fast path (padded / non-Float64
// buffers, channel sums, non-sinusoidal generators, frames inside a ramp).  Deliberately not
// inlined: the 64-bit divisions and libm calls in here would otherwise be replicated V times
// at every call site and push the kernels out of the instruction cache.
static __device__ __noinline__ double leaf_value_slow(const sigops_instr* Ip, const BufRef* bufs, int64_t n, int c, int64_t inst = 0) {
    const sigops_instr& I = *Ip;
    switch (I.leaf) {
        case SIGOPS_LEAF_BUF: {
            const BufRef b = bufs[I.buf];
            int64_t idx = n + I.i0;
            const int pad = (I.flags >> 1) & 3;
            if (idx < 0 || idx >= I.i1) {
                if (pad == SIGOPS_PAD_CONST || idx < 0 || I.i1 <= 0) return I.d0;
                if (pad == SIGOPS_PAD_CYCLE) idx = idx % I.i1;
                else if (pad == SIGOPS_PAD_MIRROR) {
                    const int64_t cnt = idx / I.i1, rem = idx % I.i1;
                    idx = (cnt & 1) ? (I.i1 - 1 - rem) : rem;
                } else idx = I.i1 - 1;
            }
            const int ch = c * I.c_mul + I.c_off;
            return load_elem(b.ptr, b.dtype, (int64_t)ch * b.ld + idx);
        }
        case SIGOPS_LEAF_CHANSUM: {
            const BufRef b = bufs[I.buf];
            const int64_t idx = n + I.i0;
            if (idx < 0 || idx >= I.i1) return I.d0;
            double s = load_elem(b.ptr, b.dtype, idx);
            for (int ch = 1; ch < (int)I.i2; ++ch) s += load_elem(b.ptr, b.dtype, (int64_t)ch * b.ld + idx);
            return s;
        }
        case SIGOPS_LEAF_GEN:
            return gen_value(I, n + I.i0);
        case SIGOPS_LEAF_RANDN:
            return randn_value(I.i1, I.i2 + inst, n + I.i0);
        case SIGOPS_LEAF_RAMP_ON: {
            const int64_t k = n + I.i0;
            if (k > I.i1) return 1.0;
            return apply_fn(I.fn, (double)(k - 1) / (double)I.i1, 0.0, 0.0);
        }
        case SIGOPS_LEAF_RAMP_OFF: {
            const int64_t k = n + I.i0;
            if (k <= I.i1) return 1.0;
            return apply_fn(I.fn, 1.0 - (double)(k - I.i1) / (double)I.i2, 0.0, 0.0);
        }
    }
    return 0.0;
}


// V frames of a sinusoidal generator, `nstride` apart: exact (reference formula,
// src/functions.jl:53-60) for the first, angle addition for the rest.
template <int V>
__device__ __forceinline__ void gen_trig_values(const sigops_instr& I, double2 rot, int64_t k0, double* out) {
    const double t = (double)k0 / I.d0;
    double s, c;
    if (I.flags & SIGOPS_FLAG_HAS_OMEGA) {
        const double u = t * I.d1 + I.d2;
        if (I.fn == SIGOPS_FN_SIN) sincospi(2.0 * u, &s, &c);
        else sincos(6.283185307179586 * (u - trunc(u)), &s, &c);   // u % 1.0 exactly, see gen_value
    } else if (I.fn == SIGOPS_FN_SIN) {
        sincospi(2.0 * (t + I.d2), &s, &c);
    } else {
        sincos(t + I.d2, &s, &c);
    }
    // cos-type generators track (cos, -sin): the same rotation then advances either pair
    double x = s, y = c;
    if (I.fn == SIGOPS_FN_COS || I.fn == SIGOPS_FN_AFFINE_COS) { x = c; y = -s; }
    if (I.fn == SIGOPS_FN_SIN || I.fn == SIGOPS_FN_COS) {
#pragma unroll
        for (int j = 0; j < V; ++j) {
            out[j] = x;
            const double x2 = fma(x, rot.y, y * rot.x), y2 = fma(y, rot.y, -x * rot.x);
            x = x2; y = y2;
        }
    } else {
        const double a = I.d3, b = I.d4;
#pragma unroll
        for (int j = 0; j < V; ++j) {
            out[j] = a * x + b;
            const double x2 = fma(x, rot.y, y * rot.x), y2 = fma(y, rot.y, -x * rot.x);
            x = x2; y = y2;
        }
    }
}

__device__ __forceinline__ bool gen_is_trig(const sigops_instr& I) {
    return I.fn == SIGOPS_FN_SIN || I.fn == SIGOPS_FN_COS || I.fn == SIGOPS_FN_AFFINE_SIN || I.fn == SIGOPS_FN_AFFINE_COS;
}

// Per-block preparation: copy the program to shared memory and fold the leaves
// that do not depend on (n,c) (constants, Normpower divisors) into leafconst[].
// For sinusoidal generators leafrot[] gets (sin, cos) of the phase advance between two
// consecutive frames a thread evaluates (`nstride` frames apart): eval_program evaluates
// the first frame with the reference's formula and reaches the next ones by angle
// addition — 4 FMAs instead of a Float64 sin() per sample, exact to a few ulp.
__device__ __forceinline__ void prepare_program(const sigops_instr* __restrict__ gprog, int len,
                                                sigops_instr* sprog, double* leafconst, double2* leafrot,
                                                const Env& env, int64_t nstride) {
    for (int i = threadIdx.x; i < len; i += blockDim.x) {
        sigops_instr I = gprog[i];
        sprog[i] = I;
        double v = 0.0;
        double2 rot = make_double2(0.0, 1.0);
        if (I.leaf == SIGOPS_LEAF_CONST) v = I.d0;
        // rms = sqrt(mean(x^2)) over the whole N x C matrix, src/filters.jl:304
        else if (I.leaf == SIGOPS_LEAF_RMS) v = sqrt(env.scalars[I.buf] / I.d0);
        if (I.leaf == SIGOPS_LEAF_CONST || I.leaf == SIGOPS_LEAF_RMS) {
            // divisions by a block-uniform value (Normpower: x ./ rms) use its reciprocal, see div_uniform;
            // rot.x = 0 marks divisors outside the range where that is exact
            const double a = fabs(v);
            rot.x = (a > 1e-150 && a < 1e150) ? 1.0 / v : 0.0;
        }
        else if (I.leaf == SIGOPS_LEAF_GEN && gen_is_trig(I)) {
            const double w = (I.flags & SIGOPS_FLAG_HAS_OMEGA) ? I.d1 : 1.0;     // cycles per second
            double cyc = (double)nstride / I.d0 * w;                             // cycles per step
            if (!(I.flags & SIGOPS_FLAG_HAS_OMEGA) && I.fn != SIGOPS_FN_SIN) cyc *= 0.15915494309189535;  // fn(t): radians
            sincospi(2.0 * cyc, &rot.x, &rot.y);
        }
        leafconst[i] = v;
        leafrot[i] = rot;
    }
}

// a / k for a block-uniform k with r = RN(1/k): one Newton step on the residual gives the correctly
// rounded quotient (Markstein), i.e. the same bits as the IEEE division the reference performs, for
// 3 FP64 instructions instead of ~20.  Callers fall back to `/` when r == 0 (k tiny, huge, 0, inf, nan).
__device__ __forceinline__ double div_uniform(double a, double k, double r) {
    const double q = a * r;
    const double e = fma(-k, q, a);
    return fma(e, r, q);
}

__device__ __forceinline__ double binop(int op, double a, double b) {
    switch (op) {
        case SIGOPS_OP_ADD: case SIGOPS_OP_POPADD: return a + b;
        case SIGOPS_OP_SUB: case SIGOPS_OP_POPSUB: return a - b;
        case SIGOPS_OP_MUL: case SIGOPS_OP_POPMUL: return a * b;
        default: return a / b;
    }
}

// ---- OperateOn closure functions (SIGOPS_EFN_*), Julia's Base semantics on Float64 ----
// Julia `min` / `max` (base/math.jl): a NaN operand wins, and -0.0 orders below 0.0.  CUDA's fmin/fmax drop NaNs.
__device__ __forceinline__ double jl_min(double a, double b) {
    if (a != a || b != b) return a + b;
    return a == b ? (signbit(a) ? a : b) : (a < b ? a : b);
}
__device__ __forceinline__ double jl_max(double a, double b) {
    if (a != a || b != b) return a + b;
    return a == b ? (signbit(a) ? b : a) : (a > b ? a : b);
}

// Every function but the four efn_vec keeps in line, out of line for the reason leaf_value_slow is: inlined at
// every V-wide call site libm bodies took the fused IIR kernels from 7k to 54k SASS instructions (DESIGN §3 K1),
// and even the one-instruction roundings nearly double the fused kernels' code when each gets a V-wide case.
static __device__ __noinline__ double efn_slow(int fn, double a, double b) {
    switch (fn) {
        case SIGOPS_EFN_SIGN: return (a > 0.0) ? 1.0 : ((a < 0.0) ? -1.0 : a);       // keeps +-0 and NaN
        case SIGOPS_EFN_FLOOR: return floor(a);
        case SIGOPS_EFN_CEIL: return ceil(a);
        case SIGOPS_EFN_TRUNC: return trunc(a);
        case SIGOPS_EFN_ROUND: return rint(a);
        case SIGOPS_EFN_COPYSIGN: return copysign(a, b);
        case SIGOPS_EFN_SQRT: return sqrt(a);
        case SIGOPS_EFN_EXP: return exp(a);
        case SIGOPS_EFN_EXP2: return exp2(a);
        case SIGOPS_EFN_EXPM1: return expm1(a);
        case SIGOPS_EFN_LOG: return log(a);
        case SIGOPS_EFN_LOG2: return log2(a);
        case SIGOPS_EFN_LOG10: return log10(a);
        case SIGOPS_EFN_LOG1P: return log1p(a);
        case SIGOPS_EFN_SIN: return sin(a);
        case SIGOPS_EFN_COS: return cos(a);
        case SIGOPS_EFN_TAN: return tan(a);
        case SIGOPS_EFN_TANH: return tanh(a);
        case SIGOPS_EFN_SINH: return sinh(a);
        case SIGOPS_EFN_COSH: return cosh(a);
        case SIGOPS_EFN_ATAN: return atan(a);
        case SIGOPS_EFN_CBRT: return cbrt(a);
        case SIGOPS_EFN_REM: return fmod(a, b);
        case SIGOPS_EFN_MOD: {
            const double r = fmod(a, b);
            if (r == 0.0) return copysign(r, b);
            return ((r > 0.0) != (b > 0.0)) ? r + b : r;
        }
        case SIGOPS_EFN_POW: return pow(a, b);
        case SIGOPS_EFN_HYPOT: return hypot(a, b);
    }
    return __longlong_as_double(0x7ff8000000000000LL);
}

// a[j] = f(a[j]) (FN1: b(j), c = the instruction's d0, d1) or g(a[j], b(j)) (FN2, POPFN2) for V values; the function
// is decoded once.  abs, clamp, min and max (envelopes, clipping, rectifiers) run in line, everything else is one
// efn_slow call per value.
template <int V, class B>
__device__ __forceinline__ void efn_vec(int fn, double* a, B b, double c) {
#define SIGOPS_EFN_LOOP(expr) _Pragma("unroll") for (int j = 0; j < V; ++j) { const double x = a[j]; a[j] = (expr); } break
    switch (fn) {
        case SIGOPS_EFN_ABS: SIGOPS_EFN_LOOP(fabs(x));
        case SIGOPS_EFN_CLAMP: SIGOPS_EFN_LOOP(x > c ? c : (x < b(j) ? b(j) : x));
        case SIGOPS_EFN_MIN: SIGOPS_EFN_LOOP(jl_min(x, b(j)));
        case SIGOPS_EFN_MAX: SIGOPS_EFN_LOOP(jl_max(x, b(j)));
        default: SIGOPS_EFN_LOOP(efn_slow(fn, x, b(j)));
    }
#undef SIGOPS_EFN_LOOP
}

// V frames of a buffer leaf, `nstride` apart.  The common case (Float64, every frame
// inside the valid range) is V plain loads off one base pointer; everything else falls
// back to the per-frame path (pads, other sample types).
template <int V>
__device__ __forceinline__ void buf_values(const sigops_instr& I, const sigops_instr* Ip, const Env& env, int64_t n0,
                                           int64_t nstride, int c, double* out) {
    const BufRef b = env.bufs[I.buf];
    const int64_t idx0 = n0 + I.i0;
    const int ch = c * I.c_mul + I.c_off;
    if (b.dtype == SIGOPS_F64 && idx0 >= 0 && idx0 + (V - 1) * nstride < I.i1) {
        const double* p = reinterpret_cast<const double*>(b.ptr) + (int64_t)ch * b.ld + idx0;
#pragma unroll
        for (int j = 0; j < V; ++j) out[j] = __ldg(p + j * nstride);
        return;
    }
    if (b.dtype == SIGOPS_F32 && idx0 >= 0 && idx0 + (V - 1) * nstride < I.i1) {
        const float* p = reinterpret_cast<const float*>(b.ptr) + (int64_t)ch * b.ld + idx0;
#pragma unroll
        for (int j = 0; j < V; ++j) out[j] = (double)__ldg(p + j * nstride);
        return;
    }
#pragma unroll
    for (int j = 0; j < V; ++j) out[j] = leaf_value_slow(Ip, env.bufs, n0 + j * nstride, c);
}

// Evaluate a program for V samples n[j] = n0 + j*nstride of channel c (nstride must be
// the stride prepare_program was given).  `stack` is this thread's spill area, laid out
// [depth][V] with stride `sstride` doubles between consecutive slots (so neighbouring
// threads interleave and stay bank-conflict free).  Each instruction is decoded once
// (copied to registers) and its leaf is evaluated for all V frames by a vector routine.
// FN: the program may hold closure functions (FN1 / FN2 / POPFN2).  The hot kernels have a variant without them, chosen
// by the host from the plan, so that programs without functions keep their registers and spill-free code.
template <int V, bool FN = true>
__device__ __forceinline__ void eval_program(const sigops_instr* sprog, const double* leafconst,
                                             const double2* leafrot, int len, const Env& env,
                                             int64_t n0, int64_t nstride, int c, const double* stageval,
                                             double* acc, double* stack, int sstride) {
    int sp = 0;
#pragma unroll
    for (int j = 0; j < V; ++j) acc[j] = 0.0;
    for (int pc = 0; pc < len; ++pc) {
        const sigops_instr I = sprog[pc];
        const int op = I.op;
        if (op <= SIGOPS_OP_DIV || (FN && op == SIGOPS_OP_FN2)) {
            double v[V];
            switch (I.leaf) {
                case SIGOPS_LEAF_CONST:
                case SIGOPS_LEAF_RMS: {
                    const double k = leafconst[pc];
                    const double r = leafrot[pc].x;
                    if (op == SIGOPS_OP_DIV && r != 0.0) {
#pragma unroll
                        for (int j = 0; j < V; ++j) {
                            const double q = div_uniform(acc[j], k, r);
                            // the Newton step loses its footing only when the quotient leaves the normal range
                            acc[j] = (fabs(q) < 1e290 && (fabs(q) > 1e-290 || acc[j] == 0.0)) ? q : acc[j] / k;
                        }
                        continue;
                    }
#pragma unroll
                    for (int j = 0; j < V; ++j) v[j] = k;
                    break;
                }
                case SIGOPS_LEAF_BUF:
                    buf_values<V>(I, &sprog[pc], env, n0, nstride, c, v);
                    break;
                case SIGOPS_LEAF_STAGE:
#pragma unroll
                    for (int j = 0; j < V; ++j) v[j] = stageval[j];
                    break;
                case SIGOPS_LEAF_GEN:
                    if (V > 1 && gen_is_trig(I)) {
                        gen_trig_values<V>(I, leafrot[pc], n0 + I.i0, v);
                        break;
                    }
                    if (V <= 8 && (I.fn == SIGOPS_FN_SAW || I.fn == SIGOPS_FN_IDENTITY) && (I.flags & SIGOPS_FLAG_HAS_OMEGA)) {
                        // sawtooth / phase ramps: cheap enough to evaluate in line (the map kernel only)
#pragma unroll
                        for (int j = 0; j < V; ++j) {
                            const double u = ((double)(n0 + I.i0 + j * nstride) / I.d0) * I.d1 + I.d2;
                            const double x = 6.283185307179586 * (u - trunc(u));
                            v[j] = I.fn == SIGOPS_FN_SAW ? x / 3.141592653589793 - 1.0 : x;
                        }
                        break;
                    }
                    // fall through
                default: {
                    // ramps are 1 outside a short region: decide once for the V frames
                    bool ones = false;
                    if (I.leaf == SIGOPS_LEAF_RAMP_ON) ones = n0 + I.i0 > I.i1;
                    else if (I.leaf == SIGOPS_LEAF_RAMP_OFF) ones = n0 + (V - 1) * nstride + I.i0 <= I.i1;
                    if (ones) {
#pragma unroll
                        for (int j = 0; j < V; ++j) v[j] = 1.0;
                    } else {
#pragma unroll
                        for (int j = 0; j < V; ++j) v[j] = leaf_value_slow(&sprog[pc], env.bufs, n0 + j * nstride, c, env.inst);
                    }
                }
            }
            switch (op) {
                case SIGOPS_OP_LOAD:
#pragma unroll
                    for (int j = 0; j < V; ++j) acc[j] = v[j];
                    break;
                case SIGOPS_OP_ADD:
#pragma unroll
                    for (int j = 0; j < V; ++j) acc[j] += v[j];
                    break;
                case SIGOPS_OP_SUB:
#pragma unroll
                    for (int j = 0; j < V; ++j) acc[j] -= v[j];
                    break;
                case SIGOPS_OP_MUL:
#pragma unroll
                    for (int j = 0; j < V; ++j) acc[j] *= v[j];
                    break;
                case SIGOPS_OP_FN2:
                    if constexpr (FN) efn_vec<V>(I.fn, acc, [&](int j) { return v[j]; }, 0.0);
                    break;
                default:
#pragma unroll
                    for (int j = 0; j < V; ++j) acc[j] /= v[j];
            }
        } else if (op == SIGOPS_OP_PUSH) {
#pragma unroll
            for (int j = 0; j < V; ++j) stack[(sp * V + j) * sstride] = acc[j];
            ++sp;
        } else if (op <= SIGOPS_OP_POPDIV) {
            --sp;
#pragma unroll
            for (int j = 0; j < V; ++j) acc[j] = binop(op, stack[(sp * V + j) * sstride], acc[j]);
        } else if (op == SIGOPS_OP_NEG) {
#pragma unroll
            for (int j = 0; j < V; ++j) acc[j] = -acc[j];
        } else if (op == SIGOPS_OP_CAST_F32) {
#pragma unroll
            for (int j = 0; j < V; ++j) acc[j] = (double)(float)acc[j];
        } else if (op == SIGOPS_OP_CAST_I64) {
#pragma unroll
            for (int j = 0; j < V; ++j) acc[j] = (double)(long long)acc[j];
        } else if (FN && op == SIGOPS_OP_FN1) {
            efn_vec<V>(I.fn, acc, [&](int) { return I.d0; }, I.d1);
        } else if (FN && op == SIGOPS_OP_POPFN2) {
            --sp;
            double l[V];
#pragma unroll
            for (int j = 0; j < V; ++j) l[j] = stack[(sp * V + j) * sstride];
            efn_vec<V>(I.fn, l, [&](int j) { return acc[j]; }, 0.0);
#pragma unroll
            for (int j = 0; j < V; ++j) acc[j] = l[j];
        }
    }
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

}  // namespace sigops
