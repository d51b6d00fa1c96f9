/*
 * signalops.h — C ABI of libsignalops_cuda.so, the B200 materialisation engine
 * behind `sink(x, ::GPUSink)`.
 *
 * Nothing comparable exists in the reference (pure Julia, no ccall).  Each entry
 * point names the reference interface it stands in for on the GPU path:
 *
 *   sigops_plan_create      what `sink(x,T,::SinkCut)` decides before the loop:
 *                           process_sink_params + initsink shapes
 *                           (src/sink.jl:87-99,115-121) and the per-node block
 *                           set-up (`FilterBlock(x)` src/filters.jl:204-211,
 *                           `initblock(::NormedSignal)` src/filters.jl:296-309)
 *   sigops_plan_run         `sink!(result,x)` — the block-pull loop and
 *                           `sink_helper!` (src/sink.jl:158-168,225-267)
 *   sigops_plan_run_device  same loop with inputs/outputs already resident in HBM
 *   sigops_last_error       Julia `error(msg)` -> ErrorException (SURVEY.md §8b)
 *
 * Conventions: plain pointers and sizes only; 0 = success, negative = failure
 * (message via sigops_last_error); never throws or aborts across the boundary;
 * the caller owns every host buffer, the library owns all device memory it
 * allocates; no pointer is retained after a call returns.  Sample buffers are
 * channel-planar (Julia column-major `nframes x nchannels`): element (n,c) is
 * at ptr[c*ld + n].
 */
#ifndef SIGNALOPS_H
#define SIGNALOPS_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SIGOPS_ABI_VERSION 1

/* ---- status codes -------------------------------------------------------- */
#define SIGOPS_OK 0
#define SIGOPS_ERR_INVALID (-1)     /* malformed plan / bad argument          */
#define SIGOPS_ERR_UNSUPPORTED (-2) /* valid but not lowered to the GPU path  */
#define SIGOPS_ERR_CUDA (-3)        /* CUDA runtime failure                   */
#define SIGOPS_ERR_NOMEM (-4)

/* ---- sample types -------------------------------------------------------- */
#define SIGOPS_F32 1
#define SIGOPS_F64 2
#define SIGOPS_I64 3
#define SIGOPS_I16 4                 /* PCM16: only as the file-side encoding of an interleaved host buffer */
/* Host buffers of sigops_plan_run may be given in WAV data-chunk layout: OR this into `dtype`.  The
 * buffer is then frame-interleaved ([frame][channel], `ld` ignored) in the encoding of the low byte
 * (F32 / F64 / I16) and the library transposes and converts on the device — results leave the GPU
 * already in file layout (`sink(x,"file.wav")`, src/sink.jl:139-142 + src/WAV.jl:3-7), files enter it
 * as they are on disk (`Signal("file.wav")`, src/WAV.jl:8-15).  The plan's buffer must be F32 or F64. */
#define SIGOPS_INTERLEAVED 0x100

typedef struct sigops_ctx sigops_ctx;
typedef struct sigops_plan sigops_plan;

typedef struct sigops_buffer {
    void*   ptr;       /* host pointer (run) or device pointer (run_device) */
    int64_t nframes;
    int32_t nchannels;
    int32_t dtype;     /* SIGOPS_F32 / F64 / I64 */
    int64_t ld;        /* elements between consecutive channels (>= nframes) */
} sigops_buffer;

typedef struct sigops_stats {
    double  gpu_ms;        /* device time of the kernels of the slowest device (CUDA events) */
    double  h2d_ms;        /* host->device copies, slowest device (0 for run_device)          */
    double  d2h_ms;
    double  wall_ms;       /* host wall clock of the whole call                               */
    int64_t launches;      /* kernels launched by this call (all devices)                     */
    int64_t h2d_bytes;
    int64_t d2h_bytes;
    int64_t out_samples;   /* frames*channels*instances written                               */
} sigops_stats;

/* ---- entry points -------------------------------------------------------- */
int sigops_abi_version(void);
int sigops_device_count(int* count);

/* devices: CUDA ordinals to shard batches over (NULL/0 -> device 0 only). */
int sigops_ctx_create(const int* devices, int ndev, sigops_ctx** out);
void sigops_ctx_destroy(sigops_ctx* ctx);

/* Last error of this ctx; ctx == NULL returns the calling thread's last
 * ctx-less error (e.g. from a failed sigops_ctx_create). Never NULL. */
const char* sigops_last_error(sigops_ctx* ctx);

/* Parse + validate the plan bytes (format below), upload coefficient tables,
 * pre-compute the IIR chunking / FIR index tables.  Plans are immutable and
 * reusable for any number of runs with buffers of the declared shapes. */
int sigops_plan_create(sigops_ctx* ctx, const void* plan, size_t nbytes, sigops_plan** out);
void sigops_plan_destroy(sigops_plan* plan);

/* Run `ninst` independent instances of the plan.  `in` holds ninst*n_inputs
 * descriptors (instance-major), `out` ninst*n_outputs.  Host buffers;
 * instances are split into contiguous ranges over the ctx devices (no
 * collective); blocks until every output has been written. */
int sigops_plan_run(sigops_plan* plan, int64_t ninst,
                    const sigops_buffer* in, sigops_buffer* out, sigops_stats* stats);

/* Ragged batch: `ninst` instances of a plan built for the longest of them, each with its own lengths.  Every
 * host buffer may hold fewer frames than the plan declares (`nframes` <= the plan's; same channels and sample
 * type, no SIGOPS_INTERLEAVED); `temp_frames` holds ninst*n_temps valid frame counts of the temps, instance-
 * major.  An instance's results are the first frames of what the plan computes from its inputs extended with
 * zeros, with every buffer read as zero past the instance's valid frames and each sum of squares taken over the
 * instance's valid frames of its stage's output: exactly the instance's own plan, for plans whose lengths are
 * the only difference (the host lowering checks that).  Each RMS leaf divides by d0 * (the instance's frames x
 * channels) / (the plan's), so every RMS leaf of one scalar slot must carry the same d0.  Instances run longest
 * first (in the caller's order when the plan draws device noise) and devices take about equal output samples.
 * Only the instance's valid output frames are written.  Costs over an equal-length batch: one reduction pass
 * per sum of squares, the zero tails and the frames each wave computes past its shorter instances' lengths. */
int sigops_plan_run_ragged(sigops_plan* plan, int64_t ninst, const sigops_buffer* in, sigops_buffer* out,
                           const int64_t* temp_frames, sigops_stats* stats);

/* Page-locked host memory for sample buffers.  `sigops_plan_run` accepts ANY host pointer: page-locked
 * memory (from here, cudaHostAlloc or cudaHostRegister) is read and written by the DMA engines directly;
 * pageable memory (a plain Julia `Array`, malloc) is staged through the library's own pinned ring by a few
 * copy threads, which costs about a third of the end-to-end throughput.  The glue allocates the RESULT of
 * `sink(x, GPUSink())` here (the reference allocates it itself at src/sink.jl:115-121, so there is no
 * caller array to honour) and releases it from the array's finalizer. */
int sigops_host_alloc(size_t bytes, void** out);
int sigops_host_free(void* ptr);

/* Same, with every buffer already resident on ctx device `dev_index`.  Work is
 * enqueued on `cuda_stream` (a cudaStream_t; NULL = the library's own stream)
 * and the call returns without synchronising when a stream is given.  All calls on one ctx device share
 * one workspace; the library orders them itself (an event behind every call, waited for by the next call
 * on a different stream), so asynchronous calls on several streams are safe but do not overlap. */
int sigops_plan_run_device(sigops_plan* plan, int dev_index, int64_t ninst,
                           const sigops_buffer* in, sigops_buffer* out,
                           void* cuda_stream, sigops_stats* stats);

/* Introspection used by tests/bench: kernels one run launches, and the
 * algorithmic HBM bytes of one instance (SURVEY.md §8d accounting). */
int sigops_plan_launch_count(sigops_plan* plan, int64_t* launches);
int sigops_plan_algorithmic_bytes(sigops_plan* plan, int64_t* bytes_per_instance);

/* Per-launch timing for the roofline report: when enabled every kernel launch is
 * bracketed by CUDA events on its own stream.  collect() synchronises the device
 * and sums elapsed ms / launch counts by kernel kind
 * (0 map, 1 iir main, 2 iir carry, 3 iir fix, 4 fir), then clears the record. */
#define SIGOPS_KERNEL_KINDS 5
int sigops_ctx_set_profiling(sigops_ctx* ctx, int enabled);
int sigops_profile_collect(sigops_ctx* ctx, int dev_index, double* ms_by_kind, int64_t* count_by_kind, int nkinds);

/* Measured FP64 FMA and HBM copy peaks of ctx device `dev_index` (micro-benchmarks
 * used for the roofline denominators; SURVEY.md §6 asks for the FP64 one). */
int sigops_measure_peaks(sigops_ctx* ctx, int dev_index, double* dfma_per_s, double* copy_gbs);

/* =========================================================================
 * Plan byte format (little endian, every section 8-byte aligned, in order):
 *
 *   sigops_plan_header
 *   sigops_bufdesc   x (n_inputs + n_temps + n_outputs)   buffer ids in this order
 *   sigops_tabledesc x n_tables
 *   sigops_instr     x n_instrs
 *   sigops_piece     x n_pieces
 *   sigops_stage     x n_stages                           executed in order
 *   double           x n_table_doubles                    coefficient blob
 *
 * Frame indices are 0-based; `n` below is the output frame of the stage, `c`
 * its channel.  All arithmetic is Float64; loads convert, stores round.
 * ========================================================================= */
#define SIGOPS_MAGIC 0x504F4753u /* "SGOP" */
#define SIGOPS_PLAN_VERSION 1u

typedef struct sigops_plan_header {
    uint32_t magic, version;
    uint32_t n_inputs, n_temps, n_outputs;
    uint32_t n_scalars;       /* per-instance Float64 accumulators (sum of squares) */
    uint32_t n_tables, n_instrs, n_pieces, n_stages;
    uint64_t n_table_doubles;
} sigops_plan_header;

typedef struct sigops_bufdesc {
    int64_t nframes;
    int32_t nchannels;
    int32_t dtype;
} sigops_bufdesc;

typedef struct sigops_tabledesc {
    int64_t offset;  /* in doubles into the blob */
    int64_t count;
} sigops_tabledesc;

/* ---- elementwise programs: an accumulator machine ------------------------
 * acc is the running value; a leaf is evaluated at (n,c).
 *   LOAD leaf        acc = leaf
 *   ADD/SUB/MUL/DIV  acc = acc (op) leaf
 *   PUSH             save acc on a small stack (depth <= SIGOPS_MAX_STACK)
 *   POPADD/...       acc = popped (op) acc
 *   NEG, CAST_F32    unary on acc
 *   FN1              acc = f(acc)          f = SIGOPS_EFN_* in `fn`, no leaf; d0, d1 = constant
 *                                          parameters (CLAMP: lo, hi)
 *   FN2              acc = g(acc, leaf)    g in `fn`: the leaf must not read `fn` itself, so only
 *                                          CONST, BUF, CHANSUM, RMS, STAGE and RANDN leaves
 *   POPFN2           acc = g(popped, acc)  (generator and ramp operands: PUSH ... POPFN2)
 * Julia's left-to-right `((a+b)+c)` order is kept by construction
 * (src/mapsignal.jl:249-255). */
enum {
    SIGOPS_OP_LOAD = 1, SIGOPS_OP_ADD, SIGOPS_OP_SUB, SIGOPS_OP_MUL, SIGOPS_OP_DIV,
    SIGOPS_OP_PUSH, SIGOPS_OP_POPADD, SIGOPS_OP_POPSUB, SIGOPS_OP_POPMUL, SIGOPS_OP_POPDIV,
    SIGOPS_OP_NEG, SIGOPS_OP_CAST_F32, SIGOPS_OP_CAST_I64,
    SIGOPS_OP_FN1, SIGOPS_OP_FN2, SIGOPS_OP_POPFN2
};
#define SIGOPS_MAX_STACK 4
#define SIGOPS_MAX_PROG 48

enum {
    SIGOPS_LEAF_NONE = 0,
    SIGOPS_LEAF_CONST,      /* d0                                                            */
    SIGOPS_LEAF_BUF,        /* buf[(c*c_mul+c_off)*ld + idx], idx=n+i0; outside [0,i1): pad   */
    SIGOPS_LEAF_CHANSUM,    /* sum over channels 0..i2-1 of buf at idx (ToChannels(1))        */
    SIGOPS_LEAF_GEN,        /* SignalFunction frame, k = n+i0 (1-based); fn, d0=fs d1=w d2=phi*/
    SIGOPS_LEAF_RAMP_ON,    /* k=n+i0 (1-based); i1=L: k<=L ? fn((k-1)/L) : 1                 */
    SIGOPS_LEAF_RAMP_OFF,   /* k=n+i0; i1=n0, i2=L: k<=n0 ? 1 : fn(1-(k-n0)/L)                */
    SIGOPS_LEAF_RMS,        /* sqrt(scalar[buf]/d0)  (Normpower divisor, d0 = N*C)            */
    SIGOPS_LEAF_STAGE,      /* the value the enclosing IIR/FIR stage just computed at (n,c)   */
    SIGOPS_LEAF_RANDN       /* `Signal(randn; rng)` (src/functions.jl:98-114) on the device: N(0,1) as a pure function
                               of (seed = i1, stream = i2 + index of the instance in the call, frame k = n+i0, 1-based):
                               Philox4x32-10 on counter (k-1)>>1, stream / key seed, Box-Muller, cos for odd k, sin for even */
};

/* pad modes of LEAF_BUF (flags bits 1..2), src/padding.jl:110-192 */
#define SIGOPS_PAD_CONST 0     /* value d0 */
#define SIGOPS_PAD_CYCLE 1
#define SIGOPS_PAD_MIRROR 2
#define SIGOPS_PAD_LAST 3
#define SIGOPS_FLAG_HAS_OMEGA 1u

/* generator / ramp functions (`fn` field) */
enum {
    SIGOPS_FN_SIN = 1,     /* Julia `sin`: sinpi(2u) special case (src/functions.jl:57-60) */
    SIGOPS_FN_COS,         /* cos(x)                                                       */
    SIGOPS_FN_SAW,         /* x/pi - 1                (README sawtooth)                    */
    SIGOPS_FN_AFFINE_SIN,  /* d3*sin(x) + d4          (README AM modulator)                */
    SIGOPS_FN_AFFINE_COS,  /* d3*cos(x) + d4                                               */
    SIGOPS_FN_IDENTITY,    /* x                                                            */
    SIGOPS_FN_SINRAMP      /* sinpi(0.5x)             (src/ramps.jl:4)                     */
};

/* elementwise functions of OperateOn closures (`fn` of FN1 / FN2 / POPFN2), Julia's Base semantics on
 * Float64 (src/mapsignal.jl:131-145 calls the closure per sample).  Where Julia throws a DomainError
 * (sqrt(-1.0), log(-1.0), a non-integer power of a negative number) the device returns NaN.
 * Exact: ABS .. CLAMP and MIN .. MOD.  Within a few ulp of Julia's libm: EXP .. CBRT, POW, HYPOT. */
enum {
    /* unary (FN1) */
    SIGOPS_EFN_ABS = 1, SIGOPS_EFN_SIGN, SIGOPS_EFN_FLOOR, SIGOPS_EFN_CEIL, SIGOPS_EFN_TRUNC,
    SIGOPS_EFN_ROUND,      /* ties to even (Julia `round`, numpy `rint`)                  */
    SIGOPS_EFN_SQRT,       /* correctly rounded                                           */
    SIGOPS_EFN_CLAMP,      /* clamp(x, d0, d1): x > d1 ? d1 : x < d0 ? d0 : x (NaN stays) */
    SIGOPS_EFN_EXP, SIGOPS_EFN_EXP2, SIGOPS_EFN_EXPM1, SIGOPS_EFN_LOG, SIGOPS_EFN_LOG2, SIGOPS_EFN_LOG10,
    SIGOPS_EFN_LOG1P, SIGOPS_EFN_SIN, SIGOPS_EFN_COS, SIGOPS_EFN_TAN, SIGOPS_EFN_TANH, SIGOPS_EFN_SINH,
    SIGOPS_EFN_COSH, SIGOPS_EFN_ATAN, SIGOPS_EFN_CBRT,
    /* binary (FN2, POPFN2): g(a, b) */
    SIGOPS_EFN_MIN = 32,   /* Julia `min`: NaN propagates, -0.0 < 0.0 (not fmin)          */
    SIGOPS_EFN_MAX,        /* Julia `max`, likewise                                       */
    SIGOPS_EFN_COPYSIGN,
    SIGOPS_EFN_REM,        /* fmod                                                        */
    SIGOPS_EFN_MOD,        /* Julia `mod`: rem, + b when the signs differ, 0 takes b's sign */
    SIGOPS_EFN_POW, SIGOPS_EFN_HYPOT
};
#define SIGOPS_EFN_UNARY_LAST SIGOPS_EFN_CBRT
#define SIGOPS_EFN_BINARY_LAST SIGOPS_EFN_HYPOT

typedef struct sigops_instr {
    uint8_t op, leaf, fn, flags;
    int32_t buf;           /* buffer id / scalar slot */
    int32_t c_mul, c_off;
    int64_t i0, i1, i2;
    double  d0, d1, d2, d3, d4;
} sigops_instr;            /* 80 bytes */

typedef struct sigops_piece {
    int64_t out_start, out_len;   /* frames [out_start, out_start+out_len) */
    int32_t ch_start, ch_count;   /* channels of the output this piece writes */
    int32_t prog_start, prog_len; /* into the instr array */
} sigops_piece;            /* 32 bytes */

enum { SIGOPS_STAGE_MAP = 1, SIGOPS_STAGE_IIR = 2, SIGOPS_STAGE_FIR = 3 };
enum { SIGOPS_FIR_ARBITRARY = 1, SIGOPS_FIR_RATIONAL = 2, SIGOPS_FIR_DECIMATOR = 3 };

typedef struct sigops_stage {
    int32_t kind;
    int32_t out_buf;
    int32_t sumsq_slot;              /* accumulate sum(out^2) here, -1 = none           */
    int32_t piece_start, n_pieces;   /* MAP: pieces tiling the output                   */
    int32_t in_prog_start, in_prog_len;    /* IIR/FIR: program producing the input x[n] */
    int32_t epi_prog_start, epi_prog_len;  /* IIR/FIR: program over LEAF_STAGE (0 = store as is) */
    int32_t nchannels;               /* IIR/FIR rows per instance                       */
    int64_t n_in, n_out;             /* frames in / out per channel                     */
    /* IIR: DF2T cascade y = g * sos_M(...sos_1(x))  (DSP.jl _filt!, SURVEY.md App. B.2) */
    int32_t n_sections;
    int32_t coef_table;              /* M rows of [b0 b1 b2 a1 a2]                      */
    double  gain;
    /* FIR: polyphase kernels (DSP.jl stream_filt.jl, SURVEY.md App. B.4) */
    int32_t fir_kind;
    int32_t n_phases, taps_per_phase;
    int32_t pfb_table;               /* [n_phases][taps_per_phase], window order         */
    int32_t dpfb_table;              /* same for the derivative bank, -1 if none         */
    int32_t interpolation, decimation;
    int32_t reserved0;
    int64_t input_deficit;           /* kernel.inputDeficit after setphase! (1-based)    */
    double  rate;                    /* FIRArbitrary.rate                                */
    double  phase0;                  /* phiAccumulator (arbitrary) or phiIdx (rational)  */
} sigops_stage;            /* 128 bytes */

#ifdef __cplusplus
}
#endif
#endif /* SIGNALOPS_H */
