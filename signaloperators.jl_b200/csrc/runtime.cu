// libsignalops_cuda.so — host runtime behind the C ABI of include/signalops.h.
//
// Plan parsing/validation, per-device workspaces, stage launch order, batch
// sharding over devices (no collectives: instances are independent, SURVEY.md
// §8e) and the host<->device pipeline of `sigops_plan_run`.
#include <algorithm>
#include <array>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <future>
#include <unordered_map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/signalops.h"
#include "common.h"
#include "launchers.h"
#include "k_iir_carry.cuh"
#include "k_fir.cuh"
#include "k_fir_mma.cuh"
#include "k_fir_tmap.cuh"
#include "k_iir_tmap.cuh"
#include "k_map.cuh"
#include "k_wav.cuh"

static_assert(sizeof(sigops_instr) == 80, "ABI: sigops_instr");
static_assert(sizeof(sigops_piece) == 32, "ABI: sigops_piece");
static_assert(sizeof(sigops_stage) == 128, "ABI: sigops_stage");
static_assert(sizeof(sigops_plan_header) == 48, "ABI: sigops_plan_header");
static_assert(sizeof(sigops_bufdesc) == 16, "ABI: sigops_bufdesc");

using namespace sigops;

namespace {

thread_local std::string g_tls_error = "";

size_t elem_size(int dtype) { return (dtype & 0xff) == SIGOPS_F32 ? 4 : ((dtype & 0xff) == SIGOPS_I16 ? 2 : 8); }
int64_t round_up(int64_t v, int64_t m) { return (v + m - 1) / m * m; }

// Grow-only device arena (one per pipeline slot); reset at the start of a wave.
struct Arena {
    char* base = nullptr;
    size_t cap = 0, used = 0;
    void reset() { used = 0; }
    void reserve(size_t bytes) {
        if (bytes <= cap) return;
        if (base) CUDA_OK(cudaFree(base));
        base = nullptr;
        cap = 0;
        CUDA_OK(cudaMalloc(&base, bytes));
        cap = bytes;
    }
    void* take(size_t bytes) {
        size_t off = (used + 255) & ~size_t(255);
        if (off + bytes > cap) fail(SIGOPS_ERR_NOMEM, "internal: arena overflow (%zu > %zu)", off + bytes, cap);
        used = off + bytes;
        return base + off;
    }
    void* take_packed(size_t bytes) {      // 16-byte granularity: consecutive takes stay adjacent
        size_t off = (used + 15) & ~size_t(15);
        if (off + bytes > cap) fail(SIGOPS_ERR_NOMEM, "internal: arena overflow (%zu > %zu)", off + bytes, cap);
        used = off + bytes;
        return base + off;
    }
    void release() {
        if (base) cudaFree(base);
        base = nullptr;
        cap = used = 0;
    }
};

constexpr int kTableRing = 4;

struct Slot {
    cudaStream_t stream = nullptr;
    Arena arena;
    // pinned staging for the BufRef table: a small ring, each entry guarded by the event recorded behind
    // its upload, so that a new table never waits for the stream to drain
    void* pinned[kTableRing] = {};
    size_t pinned_cap[kTableRing] = {};
    cudaEvent_t pinned_ev[kTableRing] = {};
    int pinned_next = 0;
    std::vector<char> last_table; // contents last uploaded (skip identical re-uploads)
    void* last_table_dev = nullptr;
    cudaEvent_t ev[6] = {};
    // everything a call enqueues on this slot ends with this event; the next user of the slot (possibly on
    // another stream) waits for it before touching the arena, the table or the IIR state
    cudaEvent_t busy = nullptr;
    cudaStream_t busy_stream = nullptr;
    bool busy_valid = false;
    // the prepared launches of a wave captured as a CUDA graph (replayed when the same plan runs on the same
    // buffers again and profiling is off)
    cudaGraphExec_t graph = nullptr;
    cudaStream_t graph_stream = nullptr;
    int replays = 0;
    // per-launch timing (sigops_ctx_set_profiling): (start, stop, kernel kind)
    // prepared launches of the last wave (replayed when the same plan runs on the same buffers)
    struct Prepared {
        int kind;
        std::function<void(cudaStream_t)> fn;
    };
    std::vector<Prepared> cache_launches;
    uint64_t cache_plan = 0;      // plan uid
    int64_t cache_ninst = -1;
    int64_t cache_inst0 = 0;      // (plans with noise leaves: the launches carry the wave's first instance index)
    std::vector<cudaEvent_t> prof_pool;
    std::vector<int> prof_kind;
    size_t prof_used = 0;
};

enum { KIND_MAP = 0, KIND_IIR_MAIN, KIND_IIR_CARRY, KIND_IIR_FIX, KIND_FIR, KIND_COUNT };

struct ProfScope {          // brackets one kernel launch with events when profiling is on
    Slot* slot = nullptr;
    cudaStream_t st = nullptr;
    ProfScope(Slot& s, bool on, cudaStream_t stream, int kind) {
        if (!on) return;
        slot = &s;
        st = stream;
        if (s.prof_used + 2 > s.prof_pool.size()) {
            for (int i = 0; i < 2; ++i) {
                cudaEvent_t e;
                CUDA_OK(cudaEventCreate(&e));
                s.prof_pool.push_back(e);
            }
        }
        s.prof_kind.push_back(kind);
        CUDA_OK(cudaEventRecord(s.prof_pool[s.prof_used], st));
    }
    ~ProfScope() {
        if (!slot) return;
        cudaEventRecord(slot->prof_pool[slot->prof_used + 1], st);
        slot->prof_used += 2;
    }
};

constexpr int kHostSlots = 3;       // staging buffers of the host-buffer pipeline (H2D | kernels | D2H in flight at once)

// Pinned staging ring for caller arrays that are NOT page-locked (a Julia `Array`, a numpy array):
// worker threads copy user memory <-> pinned chunks, the DMA engines move pinned <-> device.
struct PinnedStage {
    char* base = nullptr;
    size_t cap = 0;
    void reserve(size_t bytes) {
        if (bytes <= cap) return;
        if (base) cudaFreeHost(base);
        base = nullptr;
        cap = 0;
        CUDA_OK(cudaHostAlloc((void**)&base, bytes, cudaHostAllocDefault));
        cap = bytes;
    }
    void release() {
        if (base) cudaFreeHost(base);
        base = nullptr;
        cap = 0;
    }
};

struct Device {
    int ordinal = 0;
    int sm_count = 148;
    Slot slots[kHostSlots];
    cudaStream_t s_in = nullptr, s_out = nullptr;          // copy streams of the host-buffer pipeline
    cudaEvent_t ev_in[kHostSlots] = {}, ev_k[kHostSlots] = {}, ev_out[kHostSlots] = {};
    cudaEvent_t ev_t[kHostSlots][4] = {};                    // timing: H2D start/stop, D2H start/stop
    PinnedStage stage_in[kHostSlots], stage_out[kHostSlots];
};

// ---- per-stage derived data ---------------------------------------------------

struct IirDerived {
    int M = 0;
    int64_t W = 0;                 // decay length of the zero-input response (frames)
    bool plain_in = false;
    int plain_buf = -1;
    int64_t plain_len = 0;
    bool fast = false;             // k_iir_fast applies (f64 in/out, constant-gain epilogue)
    bool fast32 = false;           // same shape on Float32 buffers: k_iir_tmap<float> applies
    bool tma_prog = false;         // k_iir_tma<PROG>: one plain f64 buffer + buffer-free programs
    int prog_in_start = 0, prog_in_len = 0;   // input program with the buffer leaf turned into LEAF_STAGE
    bool rowinv = false;           // tma_prog whose other leaves depend on the frame only: k_iir_tmap with leaf vectors
    std::vector<sigops_instr> rv_in, rv_ep;   // those operations, in order (<= kTmMaxLeafOps each)
    bool unitb = false;            // every section has b0 == 1 and b2 == 1 exactly
    int n_scale = 0;
    double scale[2] = {1.0, 1.0};
};

struct FirDerived {
    std::vector<int64_t> xi0;
    std::vector<double> phi;
    std::vector<int32_t> poff;   // k_fir_mma: (phase index - 1) * taps_per_phase
    std::vector<double> alpha;   //            fractional phase
    int dpad = 0, pmax = 0;      // window shift inside 8 outputs; positions of a 64-output tile
    int pmax32 = 0;              // positions of a 32-output tile
    int ring32 = 0;              // k_fir_mma: positions resident while a tile is multiplied and the next two are loaded
    int in_buf = -1;
    int64_t in_len = 0;
    bool epi_const = true;       // epilogue = none or LOAD STAGE (MUL CONST){1,2}: folded into the taps
    double epi_scale = 1.0;
    int64_t period = 0;          // outputs after which index pattern and taps repeat (multiple of 32), 0 = they do not
    int64_t epoch_tiles = 0;     // the Float64 phase accumulator drifts (linearly, ~1e-15 per output): the period table is
    int64_t n_epochs = 0;        // rebuilt every epoch_tiles tiles so that the phase stays within 2e-10 of the table's
};

struct StageRT {
    sigops_stage st;
    IirDerived iir;
    FirDerived fir;
};

struct PlanDev {               // device-resident constants of a plan
    bool ready = false;
    sigops_instr* instrs = nullptr;
    double* blob = nullptr;
    std::vector<int64_t*> xi0;  // per stage
    std::vector<double*> phi;
    std::vector<int32_t*> poff;
    std::vector<double*> alpha;
    std::unordered_map<uint64_t, double*> carry;   // (stage, chunk length) -> device copy of the L-step transition matrix
    std::unordered_map<uint64_t, double*> bands;   // (stage, ks) -> merged tap bands of one period (k_fir_tmap)
};

}  // namespace

struct sigops_ctx {
    std::vector<Device> devs;
    std::string err;
    std::mutex mu;
    size_t ws_budget = size_t(16) << 30;
    bool profiling = false;
};

struct sigops_plan {
    sigops_ctx* ctx = nullptr;
    sigops_plan_header h{};
    std::vector<sigops_bufdesc> bufs;
    std::vector<sigops_tabledesc> tables;
    std::vector<sigops_instr> instrs;
    std::vector<sigops_piece> pieces;
    std::vector<StageRT> stages;
    std::vector<double> blob;
    std::vector<PlanDev> dev;
    int nbuf() const { return (int)bufs.size(); }
    int max_stack = 0;
    bool has_randn = false;        // some program draws device noise (LEAF_RANDN): launches depend on the wave's first instance index
    bool has_fn = false;           // some program applies closure functions (FN1 / FN2 / POPFN2): k_map's variant with them
    uint64_t uid = 0;
};

namespace {

// ---- plan validation ----------------------------------------------------------

// LOAD, ADD .. DIV and FN2 evaluate a leaf
bool op_has_leaf(int op) { return (op >= SIGOPS_OP_LOAD && op <= SIGOPS_OP_DIV) || op == SIGOPS_OP_FN2; }

int program_stack_depth(const sigops_plan& p, int start, int len, bool allow_stage, const char* what) {
    if (len < 0 || start < 0 || (size_t)start + len > p.instrs.size())
        fail(SIGOPS_ERR_INVALID, "%s: program range [%d,+%d) outside the instruction array", what, start, len);
    if (len > SIGOPS_MAX_PROG)
        fail(SIGOPS_ERR_UNSUPPORTED, "%s: program of %d instructions exceeds SIGOPS_MAX_PROG=%d", what, len, SIGOPS_MAX_PROG);
    int sp = 0, maxsp = 0;
    for (int i = 0; i < len; ++i) {
        const sigops_instr& I = p.instrs[start + i];
        if (I.op < SIGOPS_OP_LOAD || I.op > SIGOPS_OP_POPFN2) fail(SIGOPS_ERR_INVALID, "%s: bad opcode %d", what, I.op);
        if (i == 0 && I.op != SIGOPS_OP_LOAD) fail(SIGOPS_ERR_INVALID, "%s: program must start with LOAD", what);
        if (I.op == SIGOPS_OP_FN1 && (I.fn < SIGOPS_EFN_ABS || I.fn > SIGOPS_EFN_UNARY_LAST))
            fail(SIGOPS_ERR_UNSUPPORTED, "%s: unary function %d", what, I.fn);
        if ((I.op == SIGOPS_OP_FN2 || I.op == SIGOPS_OP_POPFN2) && (I.fn < SIGOPS_EFN_MIN || I.fn > SIGOPS_EFN_BINARY_LAST))
            fail(SIGOPS_ERR_UNSUPPORTED, "%s: binary function %d", what, I.fn);
        // FN2 keeps its function in `fn`, so its leaf must be one that does not read `fn` (generators and ramps do)
        if (I.op == SIGOPS_OP_FN2 && (I.leaf == SIGOPS_LEAF_GEN || I.leaf == SIGOPS_LEAF_RAMP_ON || I.leaf == SIGOPS_LEAF_RAMP_OFF))
            fail(SIGOPS_ERR_INVALID, "%s: FN2 on a generator or ramp leaf (use PUSH ... POPFN2)", what);
        if (op_has_leaf(I.op)) {
            switch (I.leaf) {
                case SIGOPS_LEAF_CONST: break;
                case SIGOPS_LEAF_BUF:
                case SIGOPS_LEAF_CHANSUM: {
                    if (I.buf < 0 || I.buf >= p.nbuf()) fail(SIGOPS_ERR_INVALID, "%s: leaf reads buffer %d of %d", what, I.buf, p.nbuf());
                    const sigops_bufdesc& b = p.bufs[I.buf];
                    if (I.i1 > b.nframes) fail(SIGOPS_ERR_INVALID, "%s: leaf valid length %lld exceeds buffer frames %lld", what, (long long)I.i1, (long long)b.nframes);
                    if (I.leaf == SIGOPS_LEAF_CHANSUM && (I.i2 < 1 || I.i2 > b.nchannels)) fail(SIGOPS_ERR_INVALID, "%s: CHANSUM over %lld channels of %d", what, (long long)I.i2, b.nchannels);
                    if (I.leaf == SIGOPS_LEAF_BUF && (I.c_mul < 0 || I.c_mul > 1 || I.c_off < -65536)) fail(SIGOPS_ERR_INVALID, "%s: bad channel map", what);
                    break;
                }
                case SIGOPS_LEAF_GEN:
                    if (!(I.d0 > 0)) fail(SIGOPS_ERR_INVALID, "%s: generator needs a positive frame rate", what);
                    if (I.fn < SIGOPS_FN_SIN || I.fn > SIGOPS_FN_IDENTITY) fail(SIGOPS_ERR_UNSUPPORTED, "%s: generator fn %d", what, I.fn);
                    break;
                case SIGOPS_LEAF_RAMP_ON:
                case SIGOPS_LEAF_RAMP_OFF:
                    if (I.fn != SIGOPS_FN_SINRAMP && I.fn != SIGOPS_FN_IDENTITY) fail(SIGOPS_ERR_UNSUPPORTED, "%s: ramp fn %d", what, I.fn);
                    if ((I.leaf == SIGOPS_LEAF_RAMP_ON ? I.i1 : I.i2) < 1) fail(SIGOPS_ERR_INVALID, "%s: ramp length must be >= 1", what);
                    break;
                case SIGOPS_LEAF_RMS:
                    if (I.buf < 0 || I.buf >= (int)p.h.n_scalars) fail(SIGOPS_ERR_INVALID, "%s: scalar slot %d of %u", what, I.buf, p.h.n_scalars);
                    break;
                case SIGOPS_LEAF_STAGE:
                    if (!allow_stage) fail(SIGOPS_ERR_INVALID, "%s: LEAF_STAGE outside an epilogue", what);
                    break;
                case SIGOPS_LEAF_RANDN: break;
                default: fail(SIGOPS_ERR_INVALID, "%s: bad leaf kind %d", what, I.leaf);
            }
        } else if (I.op == SIGOPS_OP_PUSH) {
            if (++sp > SIGOPS_MAX_STACK) fail(SIGOPS_ERR_UNSUPPORTED, "%s: expression nests deeper than SIGOPS_MAX_STACK", what);
            maxsp = std::max(maxsp, sp);
        } else if (I.op <= SIGOPS_OP_POPDIV || I.op == SIGOPS_OP_POPFN2) {
            if (--sp < 0) fail(SIGOPS_ERR_INVALID, "%s: POP on empty stack", what);
        }
    }
    if (sp != 0) fail(SIGOPS_ERR_INVALID, "%s: unbalanced PUSH/POP", what);
    return maxsp;
}

// zero-input decay length of the cascade: the frame after which neither the
// output nor any state exceeds 2^-64 of its peak, for every unit initial state.
int64_t decay_length(const double (*c)[5], int M, double g, int64_t limit) {
    const int S = 2 * M;
    std::vector<double> st((size_t)S * S, 0.0);
    for (int b = 0; b < S; ++b) st[(size_t)b * S + b] = 1.0;
    double peak = 1.0;
    int64_t last = 0;
    const double thresh = std::ldexp(1.0, -64);
    for (int64_t k = 0; k < limit; ++k) {
        double norm = 0.0;
        for (int b = 0; b < S; ++b) {
            double* s = &st[(size_t)b * S];
            double y = 0.0;
            for (int j = 0; j < M; ++j) {
                const double xi = y;
                y = s[2 * j] + c[j][0] * xi;
                s[2 * j] = s[2 * j + 1] + c[j][1] * xi - c[j][3] * y;
                s[2 * j + 1] = c[j][2] * xi - c[j][4] * y;
                norm = std::max(norm, std::max(std::fabs(s[2 * j]), std::fabs(s[2 * j + 1])));
            }
            norm = std::max(norm, std::fabs(y));
        }
        if (!(norm == norm) || std::isinf(norm)) return limit;   // unstable filter: never decays
        peak = std::max(peak, norm);
        if (norm > thresh * peak) last = k + 1;
        else if (k - last > 256) break;
    }
    return std::min(limit, last + 1);
}

// L-step state transition matrix of the cascade (row-major S x S).
std::vector<double> transition_matrix(const double (*c)[5], int M, int64_t L) {
    const int S = 2 * M;
    std::vector<double> AL((size_t)S * S);
    for (int b = 0; b < S; ++b) {
        std::vector<double> s(S, 0.0);
        s[b] = 1.0;
        for (int64_t k = 0; k < L; ++k) {
            double y = 0.0;
            for (int j = 0; j < M; ++j) {
                const double xi = y;
                y = s[2 * j] + c[j][0] * xi;
                s[2 * j] = s[2 * j + 1] + c[j][1] * xi - c[j][3] * y;
                s[2 * j + 1] = c[j][2] * xi - c[j][4] * y;
            }
        }
        for (int i = 0; i < S; ++i) AL[(size_t)i * S + b] = s[i];
    }
    return AL;
}

void derive_iir(sigops_plan& p, StageRT& s, int idx) {
    const sigops_stage& st = s.st;
    char what[64];
    snprintf(what, sizeof what, "stage %d (IIR)", idx);
    if (st.n_sections < 1 || st.n_sections > kIirMaxSections)
        fail(SIGOPS_ERR_UNSUPPORTED, "%s: %d biquad sections (1..%d supported per stage)", what, st.n_sections, kIirMaxSections);
    if (st.coef_table < 0 || st.coef_table >= (int)p.tables.size() || p.tables[st.coef_table].count != 5 * st.n_sections)
        fail(SIGOPS_ERR_INVALID, "%s: coefficient table must hold 5*M doubles", what);
    if (st.n_in != st.n_out) fail(SIGOPS_ERR_INVALID, "%s: n_in != n_out", what);
    s.iir.M = st.n_sections;
    const double* t = p.blob.data() + p.tables[st.coef_table].offset;
    double c[kIirMaxSections][5];
    for (int j = 0; j < st.n_sections; ++j)
        for (int k = 0; k < 5; ++k) c[j][k] = t[j * 5 + k];
    s.iir.unitb = true;
    for (int j = 0; j < st.n_sections; ++j) s.iir.unitb = s.iir.unitb && c[j][0] == 1.0 && c[j][2] == 1.0;
    s.iir.W = decay_length(c, st.n_sections, st.gain, std::max<int64_t>(32, std::min<int64_t>(st.n_out, 1 << 18)));
    if (st.in_prog_len == 1) {
        const sigops_instr& I = p.instrs[st.in_prog_start];
        if (I.op == SIGOPS_OP_LOAD && I.leaf == SIGOPS_LEAF_BUF && I.i0 == 0 && I.c_mul == 1 && I.c_off == 0 &&
            ((I.flags >> 1) & 3) == SIGOPS_PAD_CONST && I.d0 == 0.0) {
            s.iir.plain_in = true;
            s.iir.plain_buf = I.buf;
            s.iir.plain_len = I.i1;
        }
    }
    // FAST path: Float64 buffer in, Float64 out, epilogue = LOAD STAGE (MUL CONST){0,2}
    bool epi_ok = st.epi_prog_len == 0;
    if (st.epi_prog_len >= 1 && st.epi_prog_len <= 3) {
        const sigops_instr* E = &p.instrs[st.epi_prog_start];
        epi_ok = E[0].op == SIGOPS_OP_LOAD && E[0].leaf == SIGOPS_LEAF_STAGE;
        for (int i = 1; i < st.epi_prog_len && epi_ok; ++i) {
            epi_ok = E[i].op == SIGOPS_OP_MUL && E[i].leaf == SIGOPS_LEAF_CONST;
            if (epi_ok) s.iir.scale[s.iir.n_scale++] = E[i].d0;
        }
        if (!epi_ok) s.iir.n_scale = 0;
    }
    s.iir.fast = epi_ok && s.iir.plain_in && p.bufs[s.iir.plain_buf].dtype == SIGOPS_F64 &&
                 p.bufs[st.out_buf].dtype == SIGOPS_F64;
    // Float32 in and out (state and arithmetic stay Float64): the same epilogue shape, with the
    // final rounding to Float32 that the store performs anyway
    if (!epi_ok && st.epi_prog_len >= 2 && st.epi_prog_len <= 4 && s.iir.plain_in &&
        p.bufs[s.iir.plain_buf].dtype == SIGOPS_F32 && p.bufs[st.out_buf].dtype == SIGOPS_F32) {
        const sigops_instr* E = &p.instrs[st.epi_prog_start];
        const int n = st.epi_prog_len - 1;
        bool ok = E[0].op == SIGOPS_OP_LOAD && E[0].leaf == SIGOPS_LEAF_STAGE && E[n].op == SIGOPS_OP_CAST_F32;
        int ns = 0;
        double sc[2] = {1.0, 1.0};
        for (int i = 1; i < n && ok; ++i) {
            ok = E[i].op == SIGOPS_OP_MUL && E[i].leaf == SIGOPS_LEAF_CONST;
            if (ok) sc[ns++] = E[i].d0;
        }
        if (ok) {
            s.iir.fast32 = true;
            s.iir.n_scale = ns;
            s.iir.scale[0] = sc[0]; s.iir.scale[1] = sc[1];
        }
    } else if (epi_ok && s.iir.plain_in && p.bufs[s.iir.plain_buf].dtype == SIGOPS_F32 && p.bufs[st.out_buf].dtype == SIGOPS_F32)
        s.iir.fast32 = true;
    // TMA + fused programs: the input program reads exactly one plain Float64 buffer, nothing else
    // in either program touches a buffer or an RMS slot
    if (!s.iir.fast && p.bufs[st.out_buf].dtype == SIGOPS_F64) {
        int nbuf_leaves = 0, bufpc = -1;
        bool ok = true;
        auto scan = [&](int start, int len, bool is_input) {
            for (int i = 0; i < len; ++i) {
                const sigops_instr& I = p.instrs[start + i];
                if (!op_has_leaf(I.op)) { if (I.op == SIGOPS_OP_PUSH) ok = false; continue; }   // no stack in this path
                if (I.leaf == SIGOPS_LEAF_RMS || I.leaf == SIGOPS_LEAF_CHANSUM || I.leaf == SIGOPS_LEAF_RANDN) ok = false;
                if (I.leaf == SIGOPS_LEAF_BUF) {
                    if (!is_input) { ok = false; continue; }
                    ++nbuf_leaves;
                    bufpc = start + i;
                    if (!(I.i0 == 0 && I.c_mul == 1 && I.c_off == 0 && ((I.flags >> 1) & 3) == SIGOPS_PAD_CONST && I.d0 == 0.0 &&
                          p.bufs[I.buf].dtype == SIGOPS_F64))
                        ok = false;
                }
            }
        };
        scan(st.in_prog_start, st.in_prog_len, true);
        scan(st.epi_prog_start, st.epi_prog_len, false);
        if (ok && nbuf_leaves == 1) {
            s.iir.tma_prog = true;
            s.iir.plain_buf = p.instrs[bufpc].buf;
            s.iir.plain_len = p.instrs[bufpc].i1;
            s.iir.prog_in_start = (int)p.instrs.size();
            s.iir.prog_in_len = st.in_prog_len;
            for (int i = 0; i < st.in_prog_len; ++i) {
                sigops_instr I = p.instrs[st.in_prog_start + i];
                if (st.in_prog_start + i == bufpc) { I.leaf = SIGOPS_LEAF_STAGE; I.buf = 0; }
                p.instrs.push_back(I);
            }
            if (s.iir.prog_in_len == 1) s.iir.prog_in_len = 0;      // bare load: nothing to evaluate
            // Row-invariant form: `LOAD buffer, (op leaf)*` before and `LOAD stage, (op leaf)*` after the cascade,
            // every leaf a constant, generator or ramp (the same value for all rows at a frame); closure functions
            // f(acc) and g(acc, constant) take an operation slot and no leaf vector
            auto rowinv_ops = [&](int start, int len, std::vector<sigops_instr>& ops) {
                for (int i = 1; i < len; ++i) {
                    const sigops_instr& I = p.instrs[start + i];
                    if (I.op == SIGOPS_OP_FN1 || (I.op == SIGOPS_OP_FN2 && I.leaf == SIGOPS_LEAF_CONST)) {
                        ops.push_back(I);
                        continue;
                    }
                    if (I.op < SIGOPS_OP_ADD || I.op > SIGOPS_OP_DIV) return false;
                    if (I.leaf != SIGOPS_LEAF_CONST && I.leaf != SIGOPS_LEAF_GEN && I.leaf != SIGOPS_LEAF_RAMP_ON &&
                        I.leaf != SIGOPS_LEAF_RAMP_OFF)
                        return false;
                    ops.push_back(I);
                }
                return (int)ops.size() <= kTmMaxLeafOps;
            };
            const bool in_first = bufpc == st.in_prog_start && p.instrs[bufpc].op == SIGOPS_OP_LOAD;
            const bool ep_first = st.epi_prog_len == 0 || (p.instrs[st.epi_prog_start].op == SIGOPS_OP_LOAD &&
                                                           p.instrs[st.epi_prog_start].leaf == SIGOPS_LEAF_STAGE);
            s.iir.rowinv = in_first && ep_first && rowinv_ops(st.in_prog_start, st.in_prog_len, s.iir.rv_in) &&
                           rowinv_ops(st.epi_prog_start, st.epi_prog_len, s.iir.rv_ep);
        }
    }
}

constexpr size_t kFirSmemLimit = 200 * 1024;
constexpr size_t kFirMmaSmemLimit = 220 * 1024;
constexpr size_t kFirTmSmemLimit = 232448 - 512;   // 227 KB per block minus the kernel's static barriers
constexpr int kFirT = 64;     // k_fir's tile (outputs), the table padding granularity (largest tile)

// k_fir<G, 8> geometry: merged-tap rows, window pitch and dynamic shared memory.  Eight warps make a 64-output
// tile (measured on B200, config 3: 3.8 ms against 4.7 ms with four warps and 32-output tiles — the smaller tile's
// extra halo and per-tile set-up cost more than overlapping two blocks per SM buys)
struct FirGeom {
    int hbase, tpad, xpitch;
    size_t smem;
};
FirGeom fir_geometry(const FirDerived& f, int tapsper, int G, int max_stack) {
    FirGeom g;
    constexpr int W = 8, T = 8 * W, ypitch = T + 2;
    g.hbase = (f.dpad + 2) & ~1;                                   // even, >= dmax + 1
    g.tpad = (g.hbase + tapsper + f.dpad + 5 + 8) & ~1;            // + 8: slack read by the 4-pair unrolled tail
    const int need = f.pmax + 4 + 8;                             // positions of a tile (+ even start, pair tail rounded to a pair, unroll slack)
    g.xpitch = need + ((2 - need % 4) + 4) % 4;                    // = 2 mod 4: lane=row 128-bit reads conflict free
    const size_t xrows = (size_t)std::max(g.xpitch, ypitch);
    g.smem = ((size_t)T * g.tpad + (size_t)32 * G * xrows + (size_t)max_stack * 2 * W * 32) * sizeof(double);
    return g;
}
size_t fir_smem_bytes(const FirDerived& f, int tapsper, int G, int max_stack) { return fir_geometry(f, tapsper, G, max_stack).smem; }

void derive_fir(sigops_plan& p, StageRT& s, int idx) {
    const sigops_stage& st = s.st;
    char what[64];
    snprintf(what, sizeof what, "stage %d (FIR)", idx);
    if (st.taps_per_phase < 1 || st.n_phases < 1) fail(SIGOPS_ERR_INVALID, "%s: empty filter bank", what);
    if (st.taps_per_phase > 1024) fail(SIGOPS_ERR_UNSUPPORTED, "%s: %d taps per phase (<= 1024 supported)", what, st.taps_per_phase);
    auto check_table = [&](int id, const char* nm) {
        if (id < 0 || id >= (int)p.tables.size() || p.tables[id].count != (int64_t)st.n_phases * st.taps_per_phase)
            fail(SIGOPS_ERR_INVALID, "%s: %s table must hold n_phases*taps_per_phase doubles", what, nm);
    };
    check_table(st.pfb_table, "pfb");
    if (st.dpfb_table >= 0) check_table(st.dpfb_table, "dpfb");
    if (st.input_deficit < 1) fail(SIGOPS_ERR_INVALID, "%s: input_deficit must be >= 1", what);
    if (st.in_prog_len != 1) fail(SIGOPS_ERR_UNSUPPORTED, "%s: input must be a materialised buffer", what);
    const sigops_instr& I = p.instrs[st.in_prog_start];
    if (!(I.op == SIGOPS_OP_LOAD && I.leaf == SIGOPS_LEAF_BUF && I.i0 == 0 && I.c_mul == 1 && I.c_off == 0 &&
          ((I.flags >> 1) & 3) == SIGOPS_PAD_CONST && I.d0 == 0.0))
        fail(SIGOPS_ERR_UNSUPPORTED, "%s: input must be a bare zero-padded buffer load", what);
    s.fir.in_buf = I.buf;
    s.fir.in_len = I.i1;
    s.fir.epi_const = st.epi_prog_len == 0;
    if (st.epi_prog_len >= 2 && st.epi_prog_len <= 3) {
        const sigops_instr* E = &p.instrs[st.epi_prog_start];
        bool ok = E[0].op == SIGOPS_OP_LOAD && E[0].leaf == SIGOPS_LEAF_STAGE;
        double sc = 1.0;
        for (int i = 1; i < st.epi_prog_len && ok; ++i) {
            ok = E[i].op == SIGOPS_OP_MUL && E[i].leaf == SIGOPS_LEAF_CONST;
            sc *= E[i].d0;
        }
        s.fir.epi_const = ok;
        if (ok) s.fir.epi_scale = sc;
    }

    // Replay the kernel's index recurrence (DSP.jl stream_filt.jl `filt!`/`update`).
    const int64_t nout = st.n_out;
    const int64_t padded = round_up(std::max<int64_t>(nout, 1), kFirT);
    s.fir.xi0.resize(padded);
    s.fir.phi.resize(padded);
    int64_t x = st.input_deficit;              // 1-based index of the newest sample
    if (st.fir_kind == SIGOPS_FIR_ARBITRARY) {
        if (st.dpfb_table < 0) fail(SIGOPS_ERR_INVALID, "%s: arbitrary-rate kernel needs the derivative bank", what);
        if (!(st.rate > 0)) fail(SIGOPS_ERR_INVALID, "%s: rate must be positive", what);
        const double nphi = (double)st.n_phases;
        const double delta = nphi / st.rate;
        double acc = st.phase0;
        if (!(acc >= 1.0 && acc < nphi + 1.0)) fail(SIGOPS_ERR_INVALID, "%s: phase accumulator outside [1,Nphi+1)", what);
        for (int64_t m = 0; m < nout; ++m) {
            s.fir.xi0[m] = x - 1;
            s.fir.phi[m] = acc;
            acc += delta;
            if (acc > nphi) {
                x += (int64_t)std::floor((acc - 1.0) / nphi);
                acc = std::fmod(acc - 1.0, nphi) + 1.0;
            }
        }
    } else if (st.fir_kind == SIGOPS_FIR_RATIONAL) {
        const int p_ = st.interpolation, q = st.decimation;
        if (p_ != st.n_phases || q < 1) fail(SIGOPS_ERR_INVALID, "%s: rational kernel needs n_phases == interpolation", what);
        int64_t ph = (int64_t)st.phase0;
        if (ph < 1 || ph > p_) fail(SIGOPS_ERR_INVALID, "%s: phase index outside 1..p", what);
        const int step = q % p_;
        for (int64_t m = 0; m < nout; ++m) {
            s.fir.xi0[m] = x - 1;
            s.fir.phi[m] = (double)ph;
            x += (ph + q - 1) / p_;
            const int64_t v = ph + step;
            ph = v > p_ ? v - p_ : v;
        }
    } else if (st.fir_kind == SIGOPS_FIR_DECIMATOR) {
        if (st.n_phases != 1 || st.decimation < 1) fail(SIGOPS_ERR_INVALID, "%s: decimator needs one phase", what);
        for (int64_t m = 0; m < nout; ++m) {
            s.fir.xi0[m] = x - 1;
            s.fir.phi[m] = 1.0;
            x += st.decimation;
        }
    } else
        fail(SIGOPS_ERR_INVALID, "%s: unknown FIR kind %d", what, st.fir_kind);
    for (int64_t m = nout; m < padded; ++m) {
        s.fir.xi0[m] = nout ? s.fir.xi0[nout - 1] : 0;
        s.fir.phi[m] = 1.0;
    }
    // the tensor-core kernel takes the phase split into bank row and fraction (same arithmetic as
    // k_fir.cuh: fl = floor(phi), alpha = phi - fl), so its helper warps need no FP64 instruction
    s.fir.poff.resize(padded);
    s.fir.alpha.resize(padded);
    for (int64_t m = 0; m < padded; ++m) {
        const double fl = std::floor(s.fir.phi[m]);
        s.fir.poff[m] = (int32_t)(((int64_t)fl - 1) * st.taps_per_phase);
        s.fir.alpha[m] = s.fir.phi[m] - fl;
    }
    // Period of the resampler (rational ratios, e.g. 44.1 <-> 48 kHz: 160 outputs per 147 inputs): the index pattern must
    // repeat EXACTLY over the whole output and the phase to 1e-9 (the Float64 accumulator drifts by ~1e-13 and may sit on
    // either side of an integer phase: the merged taps are continuous across it).  k_fir_tmap then reads the merged tap
    // bands of one period from a table instead of rebuilding them for every tile.
    s.fir.period = 0;
    if (nout >= 128) {
        const double nphi_ = (double)st.n_phases;
        auto same = [&](int64_t m, int64_t P, int64_t dx) {
            if (s.fir.xi0[m + P] - s.fir.xi0[m] != dx) return false;
            const double d = std::fabs(s.fir.phi[m + P] - s.fir.phi[m]);
            return d <= 1e-9 && std::floor(s.fir.phi[m]) >= 1.0 && s.fir.phi[m] < nphi_ + 1.0;
        };
        for (int64_t P = 32; P <= 8192 && 2 * P <= nout && !s.fir.period; P += 32) {
            const int64_t dx = s.fir.xi0[P] - s.fir.xi0[0];
            bool ok = true;
            for (int64_t m = 0; m < std::min<int64_t>(nout - P, 2 * P) && ok; ++m) ok = same(m, P, dx);
            if (!ok) continue;
            for (int64_t m = 2 * P; m + P < nout && ok; ++m) ok = same(m, P, dx);
            if (ok) s.fir.period = P;
            else break;                        // repeats for two periods, then drifts apart: no exact period
        }
    }
    if (s.fir.period) {
        // Epochs: DSP.jl's accumulator `acc += delta` is reproduced step by step (parity with the reference includes
        // its rounding drift: 4e-9 in phase over a one-minute signal, 1e-9 of the output).  One table per epoch, taken
        // from the epoch's own first period, keeps the phase within 2e-10 of the table's (5e-11 of the output).
        const int64_t P = s.fir.period, ptiles = P / 32, ntile = (nout + 31) / 32;
        bool ok = false;
        for (int64_t nep = 1; nep <= 4096 && !ok; nep *= 2) {
            int64_t E = round_up((ntile + nep - 1) / nep, ptiles);
            E = std::max(E, ptiles);
            int64_t last = 0;                               // last epoch whose reference period lies inside the output
            while ((last + 1) * E * 32 + P <= nout) ++last;
            double worst = 0.0;
            for (int64_t m = 0; m < nout; ++m) {
                const int64_t e = std::min<int64_t>((m / 32) / E, last), start = e * E * 32;
                worst = std::max(worst, std::fabs(s.fir.phi[m] - s.fir.phi[start + (m - start) % P]));
            }
            if (worst <= 2e-10) {
                ok = true;
                s.fir.epoch_tiles = E;
                s.fir.n_epochs = last + 1;
            }
        }
        if (!ok) s.fir.period = 0;
    }
    int64_t dpad = 0, span = 0;
    for (int64_t m = 0; m + kFirR - 1 < padded; ++m) dpad = std::max(dpad, s.fir.xi0[m + kFirR - 1] - s.fir.xi0[m]);
    for (int64_t m = 0; m < padded; m += kFirT) span = std::max(span, s.fir.xi0[m + kFirT - 1] - s.fir.xi0[m]);
    int64_t span32 = 0;
    for (int64_t m = 0; m < padded; m += 32) span32 = std::max(span32, s.fir.xi0[m + 31] - s.fir.xi0[m]);
    s.fir.dpad = (int)dpad;
    s.fir.pmax = (int)(span + st.taps_per_phase);
    s.fir.pmax32 = (int)(span32 + st.taps_per_phase);
    // k_fir_mma keeps the windows of tile t-1 (being multiplied) and tile t (being loaded) in its ring
    int64_t ring = 0;
    for (int64_t t = 0; t * kFmT < padded; ++t) {
        const int64_t tn = (t + 2) * kFmT <= padded ? t + 1 : t;      // loads run up to one tile ahead
        const int64_t over = round_up(dpad + st.taps_per_phase, 4) - st.taps_per_phase;     // positions read past a window (zero taps)
        const int64_t need = (s.fir.xi0[tn * kFmT + kFmT - 1] + 2 + over) & ~int64_t(1);
        const int64_t p0 = (s.fir.xi0[(t > 0 ? t - 1 : 0) * kFmT] - st.taps_per_phase + 1) & ~int64_t(1);
        ring = std::max(ring, need - p0);
    }
    s.fir.ring32 = (int)std::min<int64_t>(ring, 1 << 30);
    if (fir_smem_bytes(s.fir, st.taps_per_phase, 1, SIGOPS_MAX_STACK) > kFirSmemLimit)
        fail(SIGOPS_ERR_UNSUPPORTED, "%s: resampling ratio %g with %d taps/phase needs %zu bytes of shared memory per block",
             what, st.rate, st.taps_per_phase, fir_smem_bytes(s.fir, st.taps_per_phase, 1, SIGOPS_MAX_STACK));
}

void parse_plan(sigops_plan& p, const void* bytes, size_t nbytes) {
    const char* cur = (const char*)bytes;
    const char* end = cur + nbytes;
    auto take = [&](void* dst, size_t n, const char* what) {
        if ((size_t)(end - cur) < n) fail(SIGOPS_ERR_INVALID, "plan truncated while reading %s", what);
        memcpy(dst, cur, n);
        cur += n;
    };
    take(&p.h, sizeof p.h, "header");
    if (p.h.magic != SIGOPS_MAGIC) fail(SIGOPS_ERR_INVALID, "bad plan magic 0x%08x", p.h.magic);
    if (p.h.version != SIGOPS_PLAN_VERSION) fail(SIGOPS_ERR_INVALID, "plan version %u, library speaks %u", p.h.version, SIGOPS_PLAN_VERSION);
    const uint64_t nb = (uint64_t)p.h.n_inputs + p.h.n_temps + p.h.n_outputs;
    if (nb == 0 || nb > kMaxBufs) fail(SIGOPS_ERR_UNSUPPORTED, "plan uses %llu buffers (1..%d supported)", (unsigned long long)nb, kMaxBufs);
    if (p.h.n_outputs < 1) fail(SIGOPS_ERR_INVALID, "plan has no output");
    if (p.h.n_stages < 1 || p.h.n_stages > 4096) fail(SIGOPS_ERR_INVALID, "plan has %u stages", p.h.n_stages);
    if (p.h.n_instrs > (1u << 20) || p.h.n_pieces > (1u << 20) || p.h.n_tables > (1u << 16) ||
        p.h.n_table_doubles > (uint64_t(1) << 31) || p.h.n_scalars > 4096)
        fail(SIGOPS_ERR_INVALID, "plan section counts out of range");
    p.bufs.resize(nb);
    take(p.bufs.data(), nb * sizeof(sigops_bufdesc), "buffer descriptors");
    p.tables.resize(p.h.n_tables);
    take(p.tables.data(), p.h.n_tables * sizeof(sigops_tabledesc), "table descriptors");
    p.instrs.resize(p.h.n_instrs);
    take(p.instrs.data(), p.h.n_instrs * sizeof(sigops_instr), "instructions");
    p.pieces.resize(p.h.n_pieces);
    take(p.pieces.data(), p.h.n_pieces * sizeof(sigops_piece), "pieces");
    std::vector<sigops_stage> st(p.h.n_stages);
    take(st.data(), p.h.n_stages * sizeof(sigops_stage), "stages");
    p.blob.resize(p.h.n_table_doubles);
    take(p.blob.data(), p.h.n_table_doubles * sizeof(double), "coefficient blob");
    if (cur != end) fail(SIGOPS_ERR_INVALID, "%zu trailing bytes after the plan", (size_t)(end - cur));

    for (auto& b : p.bufs) {
        if (b.nframes < 0 || b.nchannels < 1 || b.nchannels > 65535) fail(SIGOPS_ERR_INVALID, "buffer with %lld frames x %d channels", (long long)b.nframes, b.nchannels);
        if (b.dtype != SIGOPS_F32 && b.dtype != SIGOPS_F64 && b.dtype != SIGOPS_I64) fail(SIGOPS_ERR_INVALID, "unknown sample type %d", b.dtype);
    }
    for (auto& t : p.tables)
        if (t.offset < 0 || t.count < 0 || (uint64_t)(t.offset + t.count) > p.h.n_table_doubles) fail(SIGOPS_ERR_INVALID, "table outside the blob");

    p.stages.resize(st.size());
    for (size_t i = 0; i < st.size(); ++i) {
        StageRT& s = p.stages[i];
        s.st = st[i];
        const sigops_stage& g = s.st;
        char what[64];
        snprintf(what, sizeof what, "stage %zu", i);
        if (g.out_buf < (int)p.h.n_inputs || g.out_buf >= p.nbuf()) fail(SIGOPS_ERR_INVALID, "%s: output buffer %d is not a temp/output", what, g.out_buf);
        if (g.sumsq_slot >= (int)p.h.n_scalars) fail(SIGOPS_ERR_INVALID, "%s: scalar slot %d of %u", what, g.sumsq_slot, p.h.n_scalars);
        const sigops_bufdesc& ob = p.bufs[g.out_buf];
        if (g.kind == SIGOPS_STAGE_MAP) {
            if (g.n_pieces < 1 || g.n_pieces > kMaxPieces) fail(SIGOPS_ERR_UNSUPPORTED, "%s: %d pieces (1..%d supported)", what, g.n_pieces, kMaxPieces);
            if (g.piece_start < 0 || (size_t)g.piece_start + g.n_pieces > p.pieces.size()) fail(SIGOPS_ERR_INVALID, "%s: piece range", what);
            for (int k = 0; k < g.n_pieces; ++k) {
                const sigops_piece& pc = p.pieces[g.piece_start + k];
                if (pc.out_start < 0 || pc.out_len < 0 || pc.out_start + pc.out_len > ob.nframes) fail(SIGOPS_ERR_INVALID, "%s: piece %d outside the output (%lld+%lld > %lld)", what, k, (long long)pc.out_start, (long long)pc.out_len, (long long)ob.nframes);
                if (pc.ch_start < 0 || pc.ch_count < 1 || pc.ch_start + pc.ch_count > ob.nchannels) fail(SIGOPS_ERR_INVALID, "%s: piece %d channel range", what, k);
                p.max_stack = std::max(p.max_stack, program_stack_depth(p, pc.prog_start, pc.prog_len, false, what));
                if (pc.prog_len < 1) fail(SIGOPS_ERR_INVALID, "%s: empty program", what);
            }
        } else if (g.kind == SIGOPS_STAGE_IIR || g.kind == SIGOPS_STAGE_FIR) {
            if (g.nchannels != ob.nchannels || g.n_out != ob.nframes) fail(SIGOPS_ERR_INVALID, "%s: stage shape %lldx%d != output buffer %lldx%d", what, (long long)g.n_out, g.nchannels, (long long)ob.nframes, ob.nchannels);
            if (g.in_prog_len < 1) fail(SIGOPS_ERR_INVALID, "%s: missing input program", what);
            p.max_stack = std::max(p.max_stack, program_stack_depth(p, g.in_prog_start, g.in_prog_len, false, what));
            p.max_stack = std::max(p.max_stack, program_stack_depth(p, g.epi_prog_start, g.epi_prog_len, true, what));
            // an epilogue that is just "LOAD the stage value" (a fused plain copy) is no epilogue
            if (g.epi_prog_len == 1 && p.instrs[g.epi_prog_start].op == SIGOPS_OP_LOAD &&
                p.instrs[g.epi_prog_start].leaf == SIGOPS_LEAF_STAGE)
                s.st.epi_prog_len = 0;
            if (g.kind == SIGOPS_STAGE_IIR) derive_iir(p, s, (int)i);
            else derive_fir(p, s, (int)i);
        } else
            fail(SIGOPS_ERR_INVALID, "%s: unknown kind %d", what, g.kind);
    }
    for (const sigops_instr& I : p.instrs) {
        if (op_has_leaf(I.op) && I.leaf == SIGOPS_LEAF_RANDN) p.has_randn = true;
        if (I.op >= SIGOPS_OP_FN1) p.has_fn = true;
    }
}

// ---- device-side plan constants -------------------------------------------------

void ensure_plan_dev(sigops_plan& p, int di) {
    PlanDev& d = p.dev[di];
    if (d.ready) return;
    CUDA_OK(cudaSetDevice(p.ctx->devs[di].ordinal));
    if (!p.instrs.empty()) {
        CUDA_OK(cudaMalloc(&d.instrs, p.instrs.size() * sizeof(sigops_instr)));
        CUDA_OK(cudaMemcpy(d.instrs, p.instrs.data(), p.instrs.size() * sizeof(sigops_instr), cudaMemcpyHostToDevice));
    }
    if (!p.blob.empty()) {
        CUDA_OK(cudaMalloc(&d.blob, p.blob.size() * sizeof(double)));
        CUDA_OK(cudaMemcpy(d.blob, p.blob.data(), p.blob.size() * sizeof(double), cudaMemcpyHostToDevice));
    }
    d.xi0.assign(p.stages.size(), nullptr);
    d.phi.assign(p.stages.size(), nullptr);
    d.poff.assign(p.stages.size(), nullptr);
    d.alpha.assign(p.stages.size(), nullptr);
    for (size_t i = 0; i < p.stages.size(); ++i) {
        const FirDerived& f = p.stages[i].fir;
        if (p.stages[i].st.kind != SIGOPS_STAGE_FIR) continue;
        CUDA_OK(cudaMalloc(&d.xi0[i], f.xi0.size() * sizeof(int64_t)));
        CUDA_OK(cudaMalloc(&d.phi[i], f.phi.size() * sizeof(double)));
        CUDA_OK(cudaMemcpy(d.xi0[i], f.xi0.data(), f.xi0.size() * sizeof(int64_t), cudaMemcpyHostToDevice));
        CUDA_OK(cudaMemcpy(d.phi[i], f.phi.data(), f.phi.size() * sizeof(double), cudaMemcpyHostToDevice));
        CUDA_OK(cudaMalloc(&d.poff[i], f.poff.size() * sizeof(int32_t)));
        CUDA_OK(cudaMalloc(&d.alpha[i], f.alpha.size() * sizeof(double)));
        CUDA_OK(cudaMemcpy(d.poff[i], f.poff.data(), f.poff.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
        CUDA_OK(cudaMemcpy(d.alpha[i], f.alpha.data(), f.alpha.size() * sizeof(double), cudaMemcpyHostToDevice));
    }
    d.ready = true;
}

void free_plan_dev(sigops_plan& p) {
    for (size_t di = 0; di < p.dev.size(); ++di) {
        PlanDev& d = p.dev[di];
        if (!d.ready) continue;
        cudaSetDevice(p.ctx->devs[di].ordinal);
        cudaFree(d.instrs);
        cudaFree(d.blob);
        for (auto q : d.xi0) cudaFree(q);
        for (auto q : d.phi) cudaFree(q);
        for (auto q : d.poff) cudaFree(q);
        for (auto q : d.alpha) cudaFree(q);
        for (auto& kv : d.carry) cudaFree(kv.second);
        d.carry.clear();
        for (auto& kv : d.bands) cudaFree(kv.second);
        d.bands.clear();
        d.ready = false;
    }
}

// ---- IIR chunking ---------------------------------------------------------------

struct IirLaunch {
    int blocks_per_row;
    int64_t L, Wc, nchunks;
    bool need_matrix;
    double cost = 0.0;       // the flat and tensor-map choosers' estimate, in lane-frames
};

// Chunking for k_iir_tma: chunks are numbered over all rows jointly, so L can be chosen
// freely (multiple of the stage).  Cost model in units of one lane-frame, blocks running in whole
// waves of one block per SM:
//   WARM (W < L)          one launch, every lane walks L + Wc frames
//   MAIN + CARRY + FIX    (W >= L) two passes over L frames each, plus the carry's walk along the
//                         chunks of a row (one 2Mx2M mat-vec each, ~3 frame-times) and two more launches
// Measured on B200 (README scene, W = 3307: WARM L = 3360 -> 0.375 ms, MAIN/CARRY/FIX L = 240 ->
// 0.035 + 0.042 + 0.034 ms; 512 such rows: 0.735 ms vs 0.29 ms).
IirLaunch choose_iir_chunking_flat(const StageRT& s, int64_t rows, int sm_count, bool allow_matrix = true) {
    const int64_t N = s.st.n_out;
    const int64_t W64 = round_up(std::max<int64_t>(s.iir.W, 1), kStageCols);
    const int64_t jmax = std::max<int64_t>(1, (N + kStageCols - 1) / kStageCols);
    double best = 1e300;
    int64_t bestL = kStageCols * jmax;
    const int64_t step = std::max<int64_t>(1, jmax / 4096);
    for (int64_t j = 1; j <= jmax; j += step) {
        const int64_t L = j * kStageCols;
        const int64_t cpr = (N + L - 1) / L;
        const bool matrix = cpr > 1 && W64 >= L;
        if (matrix && !allow_matrix && j + step <= jmax) continue;
        const int64_t blocks = (((rows * cpr) + 31) / 32 + kTmaWarps - 1) / kTmaWarps;
        const int64_t waves = (blocks + sm_count - 1) / sm_count;
        double cost;
        if (matrix) cost = (double)waves * (2.0 * (double)L + 1200.0) + 3.0 * (double)cpr + 400.0;
        else cost = (double)waves * ((double)L + (cpr > 1 ? (double)W64 : 0.0) + 600.0);
        if (N % L) cost *= 1.02;                                     // ragged last chunk takes the scalar path
        if (cost < best) { best = cost; bestL = L; }
    }
    IirLaunch r;
    r.blocks_per_row = 0;
    r.L = bestL;
    r.nchunks = (N + bestL - 1) / bestL;
    r.Wc = std::min(W64, r.L);
    r.need_matrix = r.nchunks > 1 && s.iir.W >= r.L;
    r.cost = best;
    return r;
}

// Chunking for k_iir_tmap: lanes = rows, one group of 32 rows per warp, blocks of `nw` warps in whole waves of one
// block per SM; a lane walks L + Wc frames with Wc = Wst (the kernel only runs WARM, so L > Wst).  With fused
// row-invariant programs the warps of a block share a chunk (see k_iir_tmap).
IirLaunch choose_tmap_chunking(int64_t N, int64_t rows, int64_t stage_cols, int64_t Wst, int nw, bool rowinv, int sm_count) {
    const int64_t groups = (rows + 31) / 32;
    const int64_t jmax = std::max<int64_t>(1, (N + stage_cols - 1) / stage_cols);
    double best = 1e300;
    int64_t bestL = 0;
    for (int64_t j = Wst / stage_cols + 1; j <= jmax; j += std::max<int64_t>(1, jmax / 4096)) {
        const int64_t L = j * stage_cols, cpr = (N + L - 1) / L;
        const int64_t blocks = rowinv ? cpr * ((groups + nw - 1) / nw) : (groups * cpr + nw - 1) / nw;
        const int64_t waves = (blocks + sm_count - 1) / sm_count;
        const double cost = (double)waves * ((double)L + (cpr > 1 ? (double)Wst : 0.0) + 600.0);
        if (cost < best) { best = cost; bestL = L; }
    }
    return IirLaunch{0, bestL, Wst, bestL ? (N + bestL - 1) / bestL : 0, false, best};
}

IirLaunch choose_iir_chunking(const StageRT& s, int64_t rows, int sm_count) {
    const int64_t N = s.st.n_out;
    const int64_t W32 = round_up(std::max<int64_t>(s.iir.W, 1), 32);
    const int64_t target_blocks = (int64_t)sm_count * 4;
    int bpr = 1;
    auto Lof = [&](int b) { return std::max<int64_t>(32, round_up((N + (int64_t)b * kIirThreads - 1) / ((int64_t)b * kIirThreads), 32)); };
    const int64_t Lmin = std::max<int64_t>(256, std::min<int64_t>(4 * W32, 8192));
    while (rows * bpr < target_blocks && Lof(bpr * 2) >= Lmin && bpr < 4096) bpr *= 2;
    IirLaunch r;
    r.blocks_per_row = bpr;
    r.L = Lof(bpr);
    // a chunk shorter than the decay length would force the MAIN+CARRY+FIX path over every frame:
    // prefer fewer, longer chunks (idle lanes) as long as a row still splits into >= 8 of them
    if (r.L <= W32 && 2 * W32 <= N / 8) r.L = round_up(2 * W32, 32);
    r.nchunks = (N + r.L - 1) / r.L;
    r.Wc = std::min(W32, r.L);
    r.need_matrix = s.iir.W >= r.L;
    return r;
}

// ---- one wave of instances on one device ------------------------------------------

struct WaveIO {
    int64_t ninst;
    const sigops_buffer* in;   // device pointers, [ninst][n_inputs]
    const sigops_buffer* out;  // [ninst][n_outputs]
    int64_t inst0 = 0;         // index of the wave's first instance in the whole call (LEAF_RANDN streams)
};

size_t temp_bytes_per_instance(const sigops_plan& p) {
    size_t total = 0;
    for (uint32_t t = 0; t < p.h.n_temps; ++t) {
        const sigops_bufdesc& b = p.bufs[p.h.n_inputs + t];
        total += (size_t)round_up(round_up(std::max<int64_t>(b.nframes, 1), 16) * b.nchannels * (int64_t)elem_size(b.dtype), 256);
    }
    return total;
}

size_t iir_state_bytes(const sigops_plan& p, int64_t ninst, int sm_count) {
    size_t total = 0;   // every IIR stage of a wave takes its own state arrays from the arena
    for (auto& s : p.stages) {
        if (s.st.kind != SIGOPS_STAGE_IIR) continue;
        const int64_t rows = ninst * s.st.nchannels;
        const IirLaunch a = choose_iir_chunking(s, rows, sm_count);
        size_t slots = (size_t)rows * a.blocks_per_row * kIirThreads;
        if (s.iir.fast || s.iir.tma_prog) slots = std::max(slots, (size_t)rows * choose_iir_chunking_flat(s, rows, sm_count).nchunks);
        total += (size_t)2 * (2 * s.iir.M) * slots * sizeof(double) + 4096 + 1024;
    }
    return total;
}

size_t wave_workspace_bytes(const sigops_plan& p, int64_t ninst, int sm_count) {
    return temp_bytes_per_instance(p) * ninst + iir_state_bytes(p, ninst, sm_count) +
           (size_t)ninst * p.nbuf() * sizeof(BufRef) + (size_t)ninst * std::max<uint32_t>(p.h.n_scalars, 1) * sizeof(double) +
           (1 << 16);
}

// ---- stage launch planning ------------------------------------------------------
// One planner per stage kind turns a stage of the wave into prepared launches.  Every choice depends on the plan,
// the wave's BufRef table, the device and the SIGOPS_NO_* switches (read per wave) alone.

struct Wave {                 // what the wave knows when its stages are planned
    sigops_plan& p;
    PlanDev& pd;
    int sm_count;
    const BufRef* refs;       // host copy of the wave's BufRef table, [ninst][nbuf]
    BufRef* d_refs;           // its device copy
    double* scalars;          // [ninst][nscal], zeroed at the start of the wave
    int nbuf, nscal;
    int64_t ninst, inst0;
    size_t si;                // stage being planned
    Arena& arena;             // IIR state
    cudaStream_t stream;      // (the synchronous SIGOPS_FIR_DBG launches)
    std::vector<Slot::Prepared>& launches;
    void add(int kind, std::function<void(cudaStream_t)> fn) const { launches.push_back({kind, std::move(fn)}); }
};

// Every instance's rows of buffer `buf` start on a 16-byte boundary (several channels: an even number of
// elements apart), and with `f64` hold Float64: what the bulk copies of the TMA and tensor-core kernels need.
bool rows_aligned(const BufRef* refs, int64_t ninst, int nbuf, int buf, bool f64) {
    for (int64_t i = 0; i < ninst; ++i) {
        const BufRef& r = refs[i * nbuf + buf];
        if (((uintptr_t)r.ptr & 15) || (r.nch > 1 && (r.ld & 1)) || (f64 && r.dtype != SIGOPS_F64)) return false;
    }
    return true;
}

// Every row of buffer `buf` in the wave at base + row*stride with 16-byte aligned base and stride, all of type
// `dtype` (one batch tensor, or the library's own staging): one 2-D tensor map covers the buffer of the whole wave.
bool strided_matrix(const BufRef* refs, int64_t ninst, int nbuf, int buf, int elem_bytes, int dtype, char** base, int64_t* stride) {
    const BufRef& r0 = refs[buf];
    *base = (char*)r0.ptr;
    *stride = r0.ld * elem_bytes;
    if ((*stride & 15) || ((uintptr_t)*base & 15) || r0.dtype != dtype) return false;
    for (int64_t i = 0; i < ninst; ++i) {
        const BufRef& rb = refs[i * nbuf + buf];
        if (rb.ld != r0.ld || rb.nch != r0.nch || rb.dtype != dtype || (char*)rb.ptr != *base + (int64_t)i * r0.nch * *stride)
            return false;
    }
    return true;
}

// Segments along the time axis of the tensor-core FIR kernels (grid = segments x row groups): whole waves of one
// block per SM; a segment pays about three tiles of start-up (first window, pipeline fill).
int64_t choose_tiles_per_segment(int64_t ntiles, int64_t groups, int sm_count) {
    int64_t best_tps = ntiles;
    double best_cost = 1e300;
    for (int w = 1; w <= 8; ++w) {
        int64_t nseg = std::max<int64_t>(1, std::min<int64_t>(ntiles, ((int64_t)w * sm_count + groups - 1) / groups));
        const int64_t tps = (ntiles + nseg - 1) / nseg;
        nseg = (ntiles + tps - 1) / tps;
        const int64_t waves = (groups * nseg + sm_count - 1) / sm_count;
        const double cost = (double)waves * (double)(tps + 3);
        if (cost < best_cost) { best_cost = cost; best_tps = tps; }
    }
    return best_tps;
}

// Merged tap bands of one period of a periodic resampler for k_fir_tmap, one table per epoch ([tile][4 groups][ks][8],
// columns XOR-swizzled like the helper warps write them, the constant-gain epilogue folded in): built and uploaded
// once per plan, stage, band height and device.
const double* period_bands(const Wave& w, int ks) {
    const uint64_t key = ((uint64_t)w.si << 16) | (uint64_t)ks;
    auto it = w.pd.bands.find(key);
    if (it != w.pd.bands.end()) return it->second;
    const sigops_plan& p = w.p;
    const StageRT& s = p.stages[w.si];
    const sigops_stage& g = s.st;
    const int64_t Pp = s.fir.period;
    const double* hp = p.blob.data() + p.tables[g.pfb_table].offset;
    const double* hd = g.dpfb_table >= 0 ? p.blob.data() + p.tables[g.dpfb_table].offset : nullptr;
    const size_t per_epoch = (size_t)(Pp / 8) * ks * 8;
    std::vector<double> tab(per_epoch * (size_t)s.fir.n_epochs, 0.0);
    for (int64_t e = 0; e < s.fir.n_epochs; ++e) {
        const int64_t start = e * s.fir.epoch_tiles * kFmT;          // the epoch's own first period
        for (int64_t q = 0; q < Pp; ++q) {
            const int64_t m = start + q, m0 = m & ~int64_t(7);
            const int n = (int)(m - m0), stn = (int)(s.fir.xi0[m] - s.fir.xi0[m0]);
            double* band = tab.data() + per_epoch * (size_t)e + (size_t)((q & ~int64_t(7)) / 8) * ks * 8;
            for (int t = 0; t < g.taps_per_phase && stn + t < ks; ++t) {
                const double pf = hp[s.fir.poff[m] + t] * s.fir.epi_scale;
                const double h = hd ? std::fma(hd[s.fir.poff[m] + t] * s.fir.epi_scale, s.fir.alpha[m], pf) : pf;
                const int k = stn + t;
                band[k * 8 + (n ^ (((k >> 1) & 1) << 2))] = h;
            }
        }
    }
    double* dptr = nullptr;
    CUDA_OK(cudaMalloc(&dptr, tab.size() * sizeof(double)));
    CUDA_OK(cudaMemcpy(dptr, tab.data(), tab.size() * sizeof(double), cudaMemcpyHostToDevice));
    w.pd.bands.emplace(key, dptr);
    return dptr;
}

// Tuning aid (SIGOPS_FIR_DBG=1): `launch` runs a FIR kernel once with per-block cycle counters ([nblocks][8]); the
// counters summed over the blocks, per tile.
std::array<double, 8> fir_cycles_per_tile(cudaStream_t stream, size_t nblocks, int64_t tiles_per_seg,
                                          const std::function<void(long long*)>& launch) {
    long long* dbg = nullptr;
    CUDA_OK(cudaMalloc(&dbg, nblocks * 8 * sizeof(long long)));
    CUDA_OK(cudaMemset(dbg, 0, nblocks * 8 * sizeof(long long)));
    launch(dbg);
    CUDA_OK(cudaStreamSynchronize(stream));
    std::vector<long long> h(nblocks * 8);
    CUDA_OK(cudaMemcpy(h.data(), dbg, h.size() * sizeof(long long), cudaMemcpyDeviceToHost));
    cudaFree(dbg);
    std::array<double, 8> sum{};
    for (size_t b = 0; b < nblocks; ++b)
        for (int k = 0; k < 8; ++k) sum[k] += (double)h[b * 8 + k];
    const double per = 1.0 / ((double)nblocks * (double)tiles_per_seg);
    for (double& v : sum) v *= per;
    return sum;
}

// One launch with `smem` bytes of dynamic shared memory (opted in once per kernel, size and device).
template <class... P, class... A>
void launch_dyn_smem(void (*kernel)(P...), dim3 grid, int threads, size_t smem, cudaStream_t st, const A&... args) {
    ensure_dyn_smem(kernel, smem);
    kernel<<<grid, threads, smem, st>>>(args...);
}

void plan_map_stage(const Wave& w) {
    const sigops_plan& p = w.p;
    const sigops_stage& g = p.stages[w.si].st;
    MapParams P{};
    P.instrs = w.pd.instrs; P.bufrefs = w.d_refs; P.scalars = w.scalars; P.inst0 = w.inst0;
    P.nbuf = w.nbuf; P.nscalars = w.nscal;
    P.out_buf = g.out_buf; P.sumsq_slot = g.sumsq_slot; P.out_nch = p.bufs[g.out_buf].nchannels;
    P.n_pieces = g.n_pieces;
    // frames per block: four 2048-frame passes amortise the per-block set-up, unless that would
    // leave the GPU with fewer than a few blocks per SM
    int64_t subs = 0;
    for (int k = 0; k < g.n_pieces; ++k)
        subs += (p.pieces[g.piece_start + k].out_len + kMapSub - 1) / kMapSub * p.pieces[g.piece_start + k].ch_count;
    P.passes = subs * w.ninst >= (int64_t)kMapPasses * w.sm_count * 8 ? kMapPasses : 1;
    const int64_t per_block = (int64_t)kMapSub * P.passes;
    int tiles = 0;
    for (int k = 0; k < g.n_pieces; ++k) {
        P.pieces[k] = p.pieces[g.piece_start + k];
        P.tile_prefix[k] = tiles;
        tiles += (int)((P.pieces[k].out_len + per_block - 1) / per_block);
    }
    P.tile_prefix[g.n_pieces] = tiles;
    if (tiles == 0) return;
    const size_t stack_map = p.max_stack ? (size_t)p.max_stack * kMapV * kMapThreads * sizeof(double) : 0;
    const bool fn = p.has_fn;
    if (stack_map > 16 * 1024) ensure_dyn_smem(fn ? k_map<true> : k_map<false>, stack_map);
    for (int64_t i0 = 0; i0 < w.ninst; i0 += 65535) {
        const int64_t ni = std::min<int64_t>(65535, w.ninst - i0);
        MapParams Q = P;
        Q.bufrefs = w.d_refs + i0 * w.nbuf;
        Q.scalars = w.scalars + i0 * w.nscal;
        dim3 grid(tiles, P.out_nch, (unsigned)ni);
        w.add(KIND_MAP, [=](cudaStream_t st) {
            if (fn) k_map<true><<<grid, kMapThreads, stack_map, st>>>(Q);
            else k_map<false><<<grid, kMapThreads, stack_map, st>>>(Q);
        });
    }
}

// Tensor-map IIR kernel (k_iir_tmap.cuh; SIGOPS_NO_TMAP=1 switches it off): lanes = rows.  Needs every row of the
// wave at base + row*stride for both buffers, enough rows to fill warps, and a filter that decays within a chunk
// (WARM).  `tma`: the stage could take the per-lane TMA kernel.  Returns whether this one applies.
bool plan_iir_tmap(const Wave& w, bool tma) {
    const StageRT& s = w.p.stages[w.si];
    const sigops_stage& g = s.st;
    const int64_t rows = w.ninst * g.nchannels;
    const bool f32 = s.iir.fast32;
    const bool rowinv = tma && s.iir.tma_prog && s.iir.rowinv && !getenv("SIGOPS_NO_TMAP_LEAVES");
    const int esz = f32 ? 4 : 8;
    const int stage_cols = f32 ? 32 * kTmSubsPerStageF32 : (rowinv ? kTmSub * kTmSubsPerStageLv : kTmStageCols);
    if (!((tma && s.iir.fast) || f32 || rowinv) || getenv("SIGOPS_NO_TMAP") || !iir_tmap_available() ||
        !(rows % 32 == 0 || rows >= 256) || rows * 32 >= (int64_t(1) << 31) || g.n_out >= (int64_t(1) << 30))
        return false;
    char *bin = nullptr, *bout = nullptr;
    int64_t sin_ = 0, sout = 0;
    const int dtype = f32 ? SIGOPS_F32 : SIGOPS_F64;
    const int64_t Wst = round_up(std::max<int64_t>(s.iir.W, 1), stage_cols);
    if (!strided_matrix(w.refs, w.ninst, w.nbuf, s.iir.plain_buf, esz, dtype, &bin, &sin_) ||
        !strided_matrix(w.refs, w.ninst, w.nbuf, g.out_buf, esz, dtype, &bout, &sout) || 2 * Wst > g.n_out)
        return false;
    const int64_t N = g.n_out, groups = (rows + 31) / 32;
    const int nw = f32 ? kTmWarpsF32 : (rowinv ? kTmWarpsLv : kTmWarps);
    const IirLaunch c = choose_tmap_chunking(N, rows, stage_cols, Wst, nw, rowinv, w.sm_count);
    // A slowly decaying filter is better served by k_iir_tma's short chunks and carry pass.
    // Both estimates are in lane-frames; a lane-frame takes about max(100, 0.82 * lanes per SM)
    // cycles (measured: 210 with 256 lanes, 102 with 128), which makes them comparable.
    auto frame_cycles = [](int lanes) { return std::max(100.0, 0.82 * lanes); };
    const bool tmap_wins = c.cost * frame_cycles(32 * nw) <=
                           choose_iir_chunking_flat(s, rows, w.sm_count).cost * frame_cycles(32 * kTmaWarps);
    TensorMapBlob mi, mo;
    // (a Float32 stage has no other fast kernel to fall back on: take this one whenever it applies)
    if (!(c.L > Wst && (tmap_wins || f32 || rowinv) &&
          iir_tmap_encode(&mi, bin, std::min<int64_t>(s.iir.plain_len, N), rows, sin_, esz, rowinv ? kTmSubsPerStageLv : 0) &&
          iir_tmap_encode(&mo, bout, N, rows, sout, esz, rowinv ? kTmSubsPerStageLv : 0)))
        return false;
    IirTmapParams T{};
    T.bufrefs = w.d_refs; T.scalars = w.scalars; T.nbuf = w.nbuf; T.nscalars = w.nscal;
    T.out_buf = g.out_buf; T.sumsq_slot = g.sumsq_slot; T.nch = g.nchannels; T.nrows = rows;
    T.N = N; T.L = c.L; T.Wc = Wst;
    T.cpr = c.nchunks;
    T.nunits = groups * T.cpr;
    T.gain = g.gain;
    T.scale = s.iir.scale[0];          // (applied one after the other, like the reference's nested maps)
    T.scale2 = s.iir.scale[1];
    if (rowinv) {
        T.scale = T.scale2 = 1.0;
        T.n_in_ops = (int)s.iir.rv_in.size();
        T.n_ep_ops = (int)s.iir.rv_ep.size();
        for (int j = 0; j < T.n_in_ops; ++j) T.ops[j] = s.iir.rv_in[j];
        for (int j = 0; j < T.n_ep_ops; ++j) T.ops[kTmMaxLeafOps + j] = s.iir.rv_ep[j];
    }
    const double* tc = w.p.blob.data() + w.p.tables[g.coef_table].offset;
    for (int j = 0; j < s.iir.M; ++j)
        for (int k = 0; k < 5; ++k) T.coef[j][k] = tc[j * 5 + k];
    const int M_ = s.iir.M;
    const bool unitb = s.iir.unitb;
    dim3 tgrid((unsigned)(rowinv ? T.cpr * ((groups + nw - 1) / nw) : (T.nunits + nw - 1) / nw));
    if (getenv("SIGOPS_DEBUG"))
        fprintf(stderr, "[sigops] IIR stage %zu: tensor-map%s rows=%lld N=%lld M=%d W=%lld L=%lld chunks/row=%lld blocks=%u\n", w.si,
                f32 ? " (Float32)" : (rowinv ? " (fused row-invariant programs)" : ""),
                (long long)rows, (long long)N, M_, (long long)s.iir.W, (long long)T.L, (long long)T.cpr, tgrid.x);
    w.add(KIND_IIR_MAIN, [=](cudaStream_t st) { launch_iir_tmap(f32, M_, unitb, tgrid, st, T, &mi, &mo); });
    return true;
}

// IIR: the tensor-map kernel, else per-lane TMA (with fused programs or plain; WARM or MAIN + CARRY + FIX), else
// cp.async (Float64 rows that are not 16-byte aligned), else the generic program-carrying kernel.
void plan_iir_stage(const Wave& w) {
    const sigops_plan& p = w.p;
    const StageRT& s = p.stages[w.si];
    const sigops_stage& g = s.st;
    if (g.n_out == 0) return;
    const int64_t rows = w.ninst * g.nchannels;
    // TMA path: fast-path stage whose every channel starts on a 16-byte boundary
    bool tma = (s.iir.fast || s.iir.tma_prog) && rows_aligned(w.refs, w.ninst, w.nbuf, s.iir.plain_buf, false) &&
               rows_aligned(w.refs, w.ninst, w.nbuf, g.out_buf, false);
    if (plan_iir_tmap(w, tma)) return;
    // (the program-carrying TMA kernel has no MAIN/FIX form: keep it to chunkings it can run)
    IirLaunch c = tma ? choose_iir_chunking_flat(s, rows, w.sm_count, !s.iir.tma_prog) : choose_iir_chunking(s, rows, w.sm_count);
    // the program-carrying TMA kernel only exists in the single-launch WARM form
    bool tprog = tma && s.iir.tma_prog;
    if (tprog && c.need_matrix) {
        tma = tprog = false;
        c = choose_iir_chunking(s, rows, w.sm_count);
    }
    IirParams P{};
    P.instrs = w.pd.instrs; P.bufrefs = w.d_refs; P.scalars = w.scalars; P.inst0 = w.inst0;
    P.nbuf = w.nbuf; P.nscalars = w.nscal;
    P.out_buf = g.out_buf; P.sumsq_slot = g.sumsq_slot;
    P.in_prog_start = g.in_prog_start; P.in_prog_len = g.in_prog_len;
    P.epi_prog_start = g.epi_prog_start; P.epi_prog_len = g.epi_prog_len;
    P.plain_in_buf = (s.iir.plain_in || tprog) ? s.iir.plain_buf : -1;
    P.plain_in_len = s.iir.plain_len;
    P.nch = g.nchannels; P.blocks_per_row = c.blocks_per_row;
    P.N = g.n_out; P.L = c.L; P.Wc = c.Wc;
    P.slots_per_row = tma ? c.nchunks : (int64_t)c.blocks_per_row * kIirThreads;
    P.M = s.iir.M; P.gain = g.gain;
    const double* t = p.blob.data() + p.tables[g.coef_table].offset;
    for (int j = 0; j < s.iir.M; ++j)
        for (int k = 0; k < 5; ++k) P.coef[j][k] = t[j * 5 + k];
    const size_t nslots = (size_t)rows * P.slots_per_row;
    const int S = 2 * s.iir.M;
    P.state_zs = (double*)w.arena.take(nslots * S * sizeof(double));
    P.state_in = (double*)w.arena.take(nslots * S * sizeof(double));
    P.n_epi_scale = s.iir.n_scale;
    P.epi_scale[0] = s.iir.scale[0]; P.epi_scale[1] = s.iir.scale[1];
    P.carry_is_shift = c.need_matrix ? 0 : 1;
    IirTmaParams Q{};
    Q.base = P; Q.cpr = c.nchunks; Q.total_chunks = rows * c.nchunks;
    if (tprog) {
        Q.base.in_prog_start = s.iir.prog_in_start; Q.base.in_prog_len = s.iir.prog_in_len;
        Q.base.n_epi_scale = 0; Q.base.epi_scale[0] = Q.base.epi_scale[1] = 1.0;
    }
    if (getenv("SIGOPS_DEBUG"))
        fprintf(stderr, "[sigops] IIR stage %zu: %s rows=%lld N=%lld M=%d W=%lld L=%lld chunks/row=%lld Wc=%lld matrix=%d\n", w.si,
                tma ? "tma" : (s.iir.fast ? "cp.async" : "generic"), (long long)rows, (long long)g.n_out, s.iir.M,
                (long long)s.iir.W, (long long)c.L, (long long)c.nchunks, (long long)c.Wc, (int)c.need_matrix);
    const int64_t tma_blocks = ((Q.total_chunks + 31) / 32 + kTmaWarps - 1) / kTmaWarps;
    dim3 grid((unsigned)(tma ? tma_blocks : rows * c.blocks_per_row));
    const bool warm = tma && !c.need_matrix;     // single self-contained launch
    const size_t stack_iir = p.max_stack ? (size_t)p.max_stack * kIirV * kIirThreads * sizeof(double) : 0;
    const int M_ = s.iir.M;
    const bool unitb = s.iir.unitb, fast = s.iir.fast;
    w.add(KIND_IIR_MAIN, [=](cudaStream_t st) {
        if (warm) launch_iir_tma_any(LAUNCH_WARM, tprog, M_, unitb, grid, st, Q);
        else if (tma) launch_iir_tma_any(LAUNCH_MAIN, false, M_, unitb, grid, st, Q);
        else if (fast) launch_iir_cpasync(LAUNCH_MAIN, M_, unitb, grid, st, P);
        else launch_iir_generic(LAUNCH_MAIN, M_, grid, stack_iir, st, P);
    });
    if (c.nchunks <= 1 || warm) return;
    if (c.need_matrix) {
        CarryParams C{};
        C.state_zs = P.state_zs; C.state_in = P.state_in;
        C.nrows = rows; C.slots_per_row = P.slots_per_row; C.nchunks = c.nchunks; C.M2 = S;
        // L-step transition matrix: computed and uploaded once per (stage, chunk length) and device
        const uint64_t akey = ((uint64_t)w.si << 40) ^ (uint64_t)c.L;
        double*& dAL = w.pd.carry[akey];
        if (!dAL) {
            std::vector<double> AL = transition_matrix(P.coef, s.iir.M, c.L);
            CUDA_OK(cudaMalloc(&dAL, AL.size() * sizeof(double)));
            CUDA_OK(cudaMemcpy(dAL, AL.data(), AL.size() * sizeof(double), cudaMemcpyHostToDevice));
        }
        C.AL = dAL;
        const unsigned cblocks = (unsigned)((rows + 3) / 4);        // one warp per row
        w.add(KIND_IIR_CARRY, [=](cudaStream_t st) { k_iir_carry<<<cblocks, 128, 0, st>>>(C); });
    }
    w.add(KIND_IIR_FIX, [=](cudaStream_t st) {
        if (tma) launch_iir_tma_any(LAUNCH_FIX, false, M_, unitb, grid, st, Q);
        else if (fast) launch_iir_cpasync(LAUNCH_FIX, M_, unitb, grid, st, P);
        else launch_iir_generic(LAUNCH_FIX, M_, grid, stack_iir, st, P);
    });
}

// Tensor-map FIR kernel (k_fir_tmap.cuh; SIGOPS_NO_FIR_TMAP=1 switches it off): every row of the wave at base +
// row*stride, more than 64 rows, band <= 64 positions, a tile's window inside the ring.  Returns whether it applies.
bool plan_fir_tmap(const Wave& w, const FirParams& P) {
    const StageRT& s = w.p.stages[w.si];
    const sigops_stage& g = s.st;
    const int64_t rows = P.nrows;
    if (rows <= 64 || getenv("SIGOPS_NO_FIR_TMAP") || !iir_tmap_available() || rows >= (int64_t(1) << 31) ||
        g.n_out >= (int64_t(1) << 31) || s.fir.in_len >= (int64_t(1) << 31))
        return false;
    // a group's band starts at its first window position; the helpers build it in blocks of 8 rows
    const int ks = (int)round_up(s.fir.dpad + g.taps_per_phase, 8);
    const int win_slots = (s.fir.pmax32 + 3 + 14) / 16 + 1;      // worst alignment of a tile's window (+ 3 positions read past it)
    const bool has_d = P.dpfb != nullptr;
    // periodic resamplers read the merged tap bands of a tile from the period tables: no banks in shared
    // memory then, which buys one more ring slot
    const double* bands_g = nullptr;
    int period_tiles = 0;
    if (s.fir.period > 0 && g.sumsq_slot < 0 && !getenv("SIGOPS_NO_FIR_BANDS") &&
        (size_t)(s.fir.period / 8) * ks * 64 * (size_t)s.fir.n_epochs <= (size_t(96) << 20)) {
        bands_g = period_bands(w, ks);
        period_tiles = (int)(s.fir.period / kFmT);
    }
    const int64_t tabd = bands_g ? 0 : (int64_t)g.n_phases * g.taps_per_phase;
    int nslot = kFtMaxSlots;
    while (nslot > win_slots + 1 && fir_tm_smem_bytes(nslot, ks, (int)tabd, has_d) > kFirTmSmemLimit) --nslot;
    char *bin = nullptr, *bout = nullptr;
    int64_t sin_ = 0, sout = 0;
    TensorMapBlob mi, mo;
    if (!(ks <= kFtMaxKs && nslot >= win_slots + 1 && fir_tm_smem_bytes(nslot, ks, (int)tabd, has_d) <= kFirTmSmemLimit &&
          strided_matrix(w.refs, w.ninst, w.nbuf, s.fir.in_buf, 8, SIGOPS_F64, &bin, &sin_) &&
          strided_matrix(w.refs, w.ninst, w.nbuf, g.out_buf, 8, SIGOPS_F64, &bout, &sout) && s.fir.in_len >= 1 &&
          tmap_encode_2d_f64(&mi, bin, s.fir.in_len, rows, sin_, kFtSlotPos, kFtRows) &&
          tmap_encode_2d_f64(&mo, bout, g.n_out, rows, sout, 16, kFtRows / 2)))
        return false;
    FirTmParams T{};
    T.scalars = w.scalars; T.nscalars = w.nscal; T.sumsq_slot = g.sumsq_slot; T.nch = g.nchannels;
    T.nrows = rows; T.n_out = g.n_out; T.tapsper = g.taps_per_phase; T.ks = ks; T.nslot = nslot;
    T.ntiles = (g.n_out + kFmT - 1) / kFmT;
    T.pfb = P.pfb; T.dpfb = P.dpfb; T.xi0 = P.xi0; T.poff = w.pd.poff[w.si]; T.alpha = w.pd.alpha[w.si];
    T.tab_doubles = (int)tabd;
    T.bands_g = bands_g; T.period_tiles = period_tiles;
    T.epoch_tiles = s.fir.epoch_tiles; T.n_epochs = (int)s.fir.n_epochs;
    T.gain = s.fir.epi_scale;
    if (const char* e = getenv("SIGOPS_FIR_EXP")) T.exp = atoi(e);
    const int64_t groups = (rows + kFtRows - 1) / kFtRows;
    if (groups > 65535) return false;
    T.tiles_per_seg = choose_tiles_per_segment(T.ntiles, groups, w.sm_count);
    const int64_t nseg = (T.ntiles + T.tiles_per_seg - 1) / T.tiles_per_seg;
    const size_t smem = fir_tm_smem_bytes(nslot, ks, (int)tabd, has_d);
    dim3 tgrid((unsigned)nseg, (unsigned)groups);
    if (getenv("SIGOPS_DEBUG")) {
        fprintf(stderr, "[sigops] FIR stage %zu: tensor-map rows=%lld n_out=%lld taps=%d ks=%d slots=%d (window %d) grid=%lldx%lld tiles/seg=%lld smem=%zu gain=%g period=%lld outputs%s\n",
                w.si, (long long)rows, (long long)g.n_out, T.tapsper, ks, nslot, win_slots, (long long)nseg, (long long)groups,
                (long long)T.tiles_per_seg, smem, T.gain, (long long)s.fir.period, bands_g ? " (tap bands from the period tables)" : "");
        if (bands_g) fprintf(stderr, "[sigops]   %lld epochs of %lld tiles\n", (long long)s.fir.n_epochs, (long long)s.fir.epoch_tiles);
    }
    if (getenv("SIGOPS_FIR_DBG")) {
        const auto c = fir_cycles_per_tile(w.stream, (size_t)nseg * groups, T.tiles_per_seg, [&](long long* dbg) {
            FirTmParams D = T;
            D.dbg = dbg;
            launch_dyn_smem(k_fir_tmap<false, true>, tgrid, kFtThreads, smem, w.stream, D, *(const CUtensorMap*)&mi,
                            *(const CUtensorMap*)&mo);
        });
        fprintf(stderr, "[sigops] FIR tmap cycles/tile  compute: set-up %.0f (of it wait_taps %.0f) staging %.0f (of it wait_stg %.0f) total %.0f | helper: wait_done %.0f build %.0f\n",
                c[1], c[0], c[6], c[2], c[3], c[4], c[5]);
    }
    const auto kernel = g.sumsq_slot >= 0 ? k_fir_tmap<true> : k_fir_tmap<false>;
    w.add(KIND_FIR, [=](cudaStream_t st) {
        launch_dyn_smem(kernel, tgrid, kFtThreads, smem, st, T, *(const CUtensorMap*)&mi, *(const CUtensorMap*)&mo);
    });
    return true;
}

// Per-row tensor-core FIR kernel (k_fir_mma.cuh: 8 compute warps, RB/16 row fragments each).  Returns whether it applies.
bool plan_fir_mma(const Wave& w, const FirParams& P) {
    const StageRT& s = w.p.stages[w.si];
    const sigops_stage& g = s.st;
    const int64_t rows = P.nrows;
    FirMmaParams Q{};
    Q.bufrefs = w.d_refs; Q.scalars = w.scalars; Q.nbuf = w.nbuf; Q.nscalars = w.nscal;
    Q.in_buf = s.fir.in_buf; Q.out_buf = g.out_buf; Q.sumsq_slot = g.sumsq_slot;
    Q.in_len = s.fir.in_len; Q.nch = g.nchannels; Q.nrows = rows; Q.n_out = g.n_out;
    Q.tapsper = g.taps_per_phase;
    Q.ks = (int)round_up(s.fir.dpad + g.taps_per_phase, 4);
    Q.ring = s.fir.ring32;
    Q.pitch = Q.ring + ((4 - Q.ring % 16) + 16) % 16;
    Q.pfb = P.pfb; Q.dpfb = P.dpfb; Q.xi0 = P.xi0; Q.poff = w.pd.poff[w.si]; Q.alpha = w.pd.alpha[w.si];
    Q.ntiles = (g.n_out + kFmT - 1) / kFmT;
    Q.gain = s.fir.epi_scale;
    // both polyphase banks ride along in shared memory when that leaves the ring its room
    const int64_t tabd = (int64_t)g.n_phases * g.taps_per_phase;
    const size_t tab_bytes = (size_t)tabd * 8 * (P.dpfb ? 2 : 1);
    Q.tab_doubles = (int)tabd;
    if (tab_bytes > 48 * 1024) return false;      // banks too large to ride along in shared memory
    auto smem_for = [&](int RBx) {
        return (size_t)RBx * Q.pitch * 8 + (size_t)2 * 4 * Q.ks * kFmHbPitch * 8 + tab_bytes;
    };
    // rows per block RB: as many as the batch fills and shared memory holds
    int RB = rows > 64 ? 128 : (rows > 32 ? 64 : 32);
    while (RB > 32 && smem_for(RB) > kFirMmaSmemLimit) RB >>= 1;
    const int64_t groups = (rows + RB - 1) / RB;
    if (smem_for(RB) > kFirMmaSmemLimit || groups > 65535) return false;
    Q.tiles_per_seg = choose_tiles_per_segment(Q.ntiles, groups, w.sm_count);
    const int64_t nseg = (Q.ntiles + Q.tiles_per_seg - 1) / Q.tiles_per_seg;
    const size_t smem = smem_for(RB);
    dim3 grid((unsigned)nseg, (unsigned)groups);
    if (getenv("SIGOPS_DEBUG"))
        fprintf(stderr, "[sigops] FIR stage %zu: mma rows=%lld n_out=%lld taps=%d ks=%d ring=%d pitch=%d rows/block=%d grid=%lldx%lld tiles/seg=%lld smem=%zu\n",
                w.si, (long long)rows, (long long)g.n_out, Q.tapsper, Q.ks, Q.ring, Q.pitch, RB, (long long)nseg,
                (long long)groups, (long long)Q.tiles_per_seg, smem);
    if (getenv("SIGOPS_FIR_DBG")) {
        const auto c = fir_cycles_per_tile(w.stream, (size_t)nseg * groups, Q.tiles_per_seg, [&](long long* dbg) {
            FirMmaParams D = Q;
            D.dbg = dbg;
            if (RB == 128) launch_dyn_smem(k_fir_mma<8, 2, false>, grid, 16 * 32, smem, w.stream, D);
        });
        fprintf(stderr, "[sigops] FIR cycles/tile  aux: wait_done %.0f extend %.0f taps %.0f | compute: wait_taps %.0f wait_data %.0f dmma %.0f store %.0f\n",
                c[0], c[1], c[2], c[3], c[4], c[5], c[6]);
    }
    const bool ssq = Q.sumsq_slot >= 0;
    const auto kernel = RB == 128 ? (ssq ? k_fir_mma<8, 2, true> : k_fir_mma<8, 2, false>)
                      : RB == 64  ? (ssq ? k_fir_mma<4, 2, true> : k_fir_mma<4, 2, false>)
                                  : (ssq ? k_fir_mma<2, 2, true> : k_fir_mma<2, 2, false>);
    w.add(KIND_FIR, [=](cudaStream_t st) { launch_dyn_smem(kernel, grid, 16 * 32, smem, st, Q); });
    return true;
}

// FIR: the tensor-core kernels for plain Float64 rows on 16-byte boundaries with no epilogue or a constant gain
// (k_fir_tmap, else k_fir_mma), else the scalar-FMA kernel k_fir.
void plan_fir_stage(const Wave& w) {
    const sigops_plan& p = w.p;
    const StageRT& s = p.stages[w.si];
    const sigops_stage& g = s.st;
    if (g.n_out == 0) return;
    const int64_t rows = w.ninst * g.nchannels;
    FirParams P{};
    P.instrs = w.pd.instrs; P.bufrefs = w.d_refs; P.scalars = w.scalars; P.inst0 = w.inst0;
    P.nbuf = w.nbuf; P.nscalars = w.nscal;
    P.out_buf = g.out_buf; P.sumsq_slot = g.sumsq_slot;
    P.in_buf = s.fir.in_buf; P.in_len = s.fir.in_len;
    P.epi_prog_start = g.epi_prog_start; P.epi_prog_len = g.epi_prog_len;
    P.nch = g.nchannels; P.nrows = rows; P.n_out = g.n_out;
    P.tapsper = g.taps_per_phase;
    P.pfb = w.pd.blob + p.tables[g.pfb_table].offset;
    P.dpfb = g.dpfb_table >= 0 ? w.pd.blob + p.tables[g.dpfb_table].offset : nullptr;
    P.xi0 = w.pd.xi0[w.si]; P.phi = w.pd.phi[w.si];
    const bool mma = s.fir.epi_const && !getenv("SIGOPS_NO_FIR_MMA") &&
                     p.bufs[s.fir.in_buf].dtype == SIGOPS_F64 && p.bufs[g.out_buf].dtype == SIGOPS_F64 &&
                     rows_aligned(w.refs, w.ninst, w.nbuf, s.fir.in_buf, true) && rows_aligned(w.refs, w.ninst, w.nbuf, g.out_buf, true);
    if (mma && (plan_fir_tmap(w, P) || plan_fir_mma(w, P))) return;
    // rows per thread: as many as fit in shared memory, but no more than the batch can fill
    int G = 4;
    while (G > 1 && (fir_smem_bytes(s.fir, g.taps_per_phase, G, p.max_stack) > kFirSmemLimit || rows <= 16 * G)) G >>= 1;
    const FirGeom geo = fir_geometry(s.fir, g.taps_per_phase, G, p.max_stack);
    P.hbase = geo.hbase; P.tpad = geo.tpad; P.xpitch = geo.xpitch;
    const size_t smem = geo.smem;
    const int64_t tiles = (g.n_out + kFirT - 1) / kFirT;
    const int64_t groups = (rows + 32 * G - 1) / (32 * G);
    if (groups > 65535) fail(SIGOPS_ERR_UNSUPPORTED, "FIR stage over more than %d rows per wave", 65535 * 32 * G);
    dim3 grid((unsigned)tiles, (unsigned)groups);
    if (getenv("SIGOPS_DEBUG"))
        fprintf(stderr, "[sigops] FIR stage %zu: scalar rows=%lld n_out=%lld taps=%d G=%d tiles=%lld smem=%zu\n", w.si,
                (long long)rows, (long long)g.n_out, g.taps_per_phase, G, (long long)tiles, smem);
    const auto kernel = G == 4 ? k_fir<4, 8> : (G == 2 ? k_fir<2, 8> : k_fir<1, 8>);
    w.add(KIND_FIR, [=](cudaStream_t st) { launch_dyn_smem(kernel, grid, 256, smem, st, P); });
}

// Enqueue every stage of the plan for one wave. Returns kernels launched.
int64_t enqueue_wave(sigops_plan& p, int di, Slot& slot, cudaStream_t stream, const WaveIO& io) {
    Device& dev = p.ctx->devs[di];
    PlanDev& pd = p.dev[di];
    const int nbuf = p.nbuf();
    const int64_t ninst = io.ninst;
    const int nscal = std::max<uint32_t>(p.h.n_scalars, 1);
    // -- workspace carve-up
    const size_t temp_stride = temp_bytes_per_instance(p);
    char* temps = temp_stride ? (char*)slot.arena.take(temp_stride * ninst) : nullptr;
    double* scalars = (double*)slot.arena.take((size_t)ninst * nscal * sizeof(double));
    BufRef* d_refs = (BufRef*)slot.arena.take((size_t)ninst * nbuf * sizeof(BufRef));
    CUDA_OK(cudaMemsetAsync(scalars, 0, (size_t)ninst * nscal * sizeof(double), stream));

    // -- BufRef table (instance-major)
    const size_t table_bytes = (size_t)ninst * nbuf * sizeof(BufRef);
    std::vector<char> table(table_bytes);
    BufRef* refs = (BufRef*)table.data();
    for (int64_t i = 0; i < ninst; ++i) {
        size_t toff = 0;
        for (int b = 0; b < nbuf; ++b) {
            BufRef& r = refs[i * nbuf + b];
            const sigops_bufdesc& bd = p.bufs[b];
            memset(&r, 0, sizeof r);
            if (b < (int)p.h.n_inputs) {
                const sigops_buffer& ib = io.in[i * p.h.n_inputs + b];
                r.ptr = ib.ptr; r.ld = ib.ld; r.dtype = ib.dtype; r.nch = ib.nchannels;
            } else if (b < (int)(p.h.n_inputs + p.h.n_temps)) {
                const int64_t ld = round_up(std::max<int64_t>(bd.nframes, 1), 16);
                r.ptr = temps + (size_t)i * temp_stride + toff;
                r.ld = ld; r.dtype = bd.dtype; r.nch = bd.nchannels;
                toff += (size_t)round_up(ld * bd.nchannels * (int64_t)elem_size(bd.dtype), 256);
            } else {
                const sigops_buffer& ob = io.out[i * p.h.n_outputs + (b - p.h.n_inputs - p.h.n_temps)];
                r.ptr = ob.ptr; r.ld = ob.ld; r.dtype = ob.dtype; r.nch = ob.nchannels;
            }
        }
    }
    bool table_changed = false;
    if (slot.last_table_dev != (void*)d_refs || slot.last_table != table) {
        // next entry of the pinned ring; its previous upload (kTableRing waves ago) has long completed
        const int r = slot.pinned_next;
        slot.pinned_next = (r + 1) % kTableRing;
        if (!slot.pinned_ev[r]) CUDA_OK(cudaEventCreateWithFlags(&slot.pinned_ev[r], cudaEventDisableTiming));
        else CUDA_OK(cudaEventSynchronize(slot.pinned_ev[r]));
        if (slot.pinned_cap[r] < table_bytes) {
            if (slot.pinned[r]) cudaFreeHost(slot.pinned[r]);
            slot.pinned[r] = nullptr;
            slot.pinned_cap[r] = 0;
            CUDA_OK(cudaMallocHost(&slot.pinned[r], table_bytes));
            slot.pinned_cap[r] = table_bytes;
        }
        memcpy(slot.pinned[r], table.data(), table_bytes);
        CUDA_OK(cudaMemcpyAsync(d_refs, slot.pinned[r], table_bytes, cudaMemcpyHostToDevice, stream));
        CUDA_OK(cudaEventRecord(slot.pinned_ev[r], stream));
        slot.last_table.swap(table);
        slot.last_table_dev = d_refs;
        table_changed = true;
    }
    // Same plan on the same buffers as last time: replay the prepared launches (all the
    // chunking / alignment / table decisions below are pure functions of those).
    auto replay = [&]() -> int64_t {
        for (auto& L : slot.cache_launches) {
            ProfScope ps(slot, p.ctx->profiling, stream, L.kind);
            L.fn(stream);
            CUDA_OK(cudaGetLastError());
        }
        return (int64_t)slot.cache_launches.size();
    };
    auto drop_graph = [&]() {
        if (slot.graph) cudaGraphExecDestroy(slot.graph);
        slot.graph = nullptr;
        slot.replays = 0;
    };
    if (!table_changed && slot.cache_plan == p.uid && slot.cache_ninst == ninst && (!p.has_randn || slot.cache_inst0 == io.inst0)) {
        // Same plan on the same buffers again: from the second replay on, the scalar reset and every launch of
        // the wave go out as ONE cudaGraphLaunch (plans of several small stages are launch-latency bound).
        static const bool no_graph = getenv("SIGOPS_NO_GRAPH") != nullptr;
        const bool want_graph = !no_graph && !p.ctx->profiling && slot.cache_launches.size() >= 2;
        if (want_graph && slot.graph && slot.graph_stream == stream) {
            CUDA_OK(cudaGraphLaunch(slot.graph, stream));
            return (int64_t)slot.cache_launches.size();
        }
        if (want_graph && ++slot.replays >= 2) {
            drop_graph();
            cudaGraph_t gr = nullptr;
            if (cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
                cudaMemsetAsync(scalars, 0, (size_t)ninst * nscal * sizeof(double), stream);
                for (auto& L : slot.cache_launches) L.fn(stream);
                const cudaError_t ce = cudaStreamEndCapture(stream, &gr);
                if (ce == cudaSuccess && gr && cudaGraphInstantiate(&slot.graph, gr, 0) == cudaSuccess) slot.graph_stream = stream;
                else slot.graph = nullptr;
                if (gr) cudaGraphDestroy(gr);
            }
            cudaGetLastError();
            if (slot.graph) {
                // (the eager memset issued above for this run is harmless: the graph repeats it)
                CUDA_OK(cudaGraphLaunch(slot.graph, stream));
                return (int64_t)slot.cache_launches.size();
            }
        }
        return replay();
    }
    drop_graph();
    slot.cache_launches.clear();
    slot.cache_plan = 0;
    // (slot.last_table now holds this wave's table)
    Wave w{p, pd, dev.sm_count, (const BufRef*)slot.last_table.data(), d_refs, scalars, nbuf, nscal, ninst, io.inst0, 0,
           slot.arena, stream, slot.cache_launches};
    for (w.si = 0; w.si < p.stages.size(); ++w.si) {
        switch (p.stages[w.si].st.kind) {
            case SIGOPS_STAGE_MAP: plan_map_stage(w); break;
            case SIGOPS_STAGE_IIR: plan_iir_stage(w); break;
            default: plan_fir_stage(w);
        }
    }
    slot.cache_plan = p.uid;
    slot.cache_ninst = ninst;
    slot.cache_inst0 = io.inst0;
    return replay();
}

void validate_io(const sigops_plan& p, int64_t ninst, const sigops_buffer* in, const sigops_buffer* out, bool allow_wav = false) {
    if (ninst < 0) fail(SIGOPS_ERR_INVALID, "negative instance count");
    if (ninst > 0 && ((p.h.n_inputs && !in) || !out)) fail(SIGOPS_ERR_INVALID, "null buffer array");
    for (int64_t i = 0; i < ninst; ++i) {
        for (uint32_t b = 0; b < p.h.n_inputs + p.h.n_outputs; ++b) {
            const bool isin = b < p.h.n_inputs;
            const sigops_buffer& ub = isin ? in[i * p.h.n_inputs + b] : out[i * p.h.n_outputs + (b - p.h.n_inputs)];
            const sigops_bufdesc& bd = isin ? p.bufs[b] : p.bufs[p.h.n_temps + b];
            const bool wav = (ub.dtype & SIGOPS_INTERLEAVED) != 0;
            const int enc = ub.dtype & 0xff;
            const bool type_ok = wav ? (allow_wav && (enc == SIGOPS_F32 || enc == SIGOPS_F64 || enc == SIGOPS_I16) &&
                                        (bd.dtype == SIGOPS_F32 || bd.dtype == SIGOPS_F64))
                                     : ub.dtype == bd.dtype;
            if (ub.nframes != bd.nframes || ub.nchannels != bd.nchannels || !type_ok)
                fail(SIGOPS_ERR_INVALID, "instance %lld %s %u: buffer is %lldx%d type %d, plan expects %lldx%d type %d",
                     (long long)i, isin ? "input" : "output", isin ? b : b - p.h.n_inputs, (long long)ub.nframes, ub.nchannels,
                     ub.dtype, (long long)bd.nframes, bd.nchannels, bd.dtype);
            if (!wav && ub.ld < ub.nframes) fail(SIGOPS_ERR_INVALID, "instance %lld: ld %lld < nframes %lld", (long long)i, (long long)ub.ld, (long long)ub.nframes);
            if (!ub.ptr && ub.nframes > 0) fail(SIGOPS_ERR_INVALID, "instance %lld: null buffer pointer", (long long)i);
        }
    }
}

int64_t count_out_samples(const sigops_plan& p, int64_t ninst) {
    int64_t n = 0;
    for (uint32_t b = 0; b < p.h.n_outputs; ++b) {
        const sigops_bufdesc& bd = p.bufs[p.h.n_inputs + p.h.n_temps + b];
        n += bd.nframes * bd.nchannels;
    }
    return n * ninst;
}

// Device-resident run: waves bounded by the workspace budget, all on `stream`.
int64_t run_device_resident(sigops_plan& p, int di, int64_t ninst, const sigops_buffer* in,
                            const sigops_buffer* out, cudaStream_t stream, Slot& slot) {
    Device& dev = p.ctx->devs[di];
    CUDA_OK(cudaSetDevice(dev.ordinal));
    ensure_plan_dev(p, di);
    if (ninst == 0) return 0;
    int64_t wave = ninst;
    while (wave > 1 && wave_workspace_bytes(p, wave, dev.sm_count) > p.ctx->ws_budget) wave = (wave + 1) / 2;
    const size_t need = wave_workspace_bytes(p, wave, dev.sm_count);
    if (need > slot.arena.cap) {
        CUDA_OK(cudaStreamSynchronize(stream));
        slot.arena.reserve(need);
        slot.last_table_dev = nullptr;
    }
    int64_t launches = 0;
    for (int64_t i0 = 0; i0 < ninst; i0 += wave) {
        slot.arena.reset();
        WaveIO io{std::min(wave, ninst - i0), in ? in + i0 * p.h.n_inputs : nullptr, out + i0 * p.h.n_outputs, i0};
        launches += enqueue_wave(p, di, slot, stream, io);
    }
    return launches;
}

// Copy buffer `b` of `w` consecutive instances between host and device staging.  A buffer whose
// rows are dense (ld == nframes on both sides) is one contiguous block.  `merge`: blocks of consecutive
// instances that are adjacent on both sides go as ONE cudaMemcpyAsync — only valid when the host side
// is a single allocation (the library's pinned ring); adjacent caller arrays may be separate page-locked
// allocations, which one copy must not span.
int64_t copy_runs(const sigops_buffer* host, const sigops_buffer* dev, int64_t w, uint32_t nb, bool to_device, cudaStream_t st,
                  bool merge) {
    int64_t total = 0;
    for (uint32_t b = 0; b < nb; ++b) {
        int64_t i = 0;
        while (i < w) {
            const sigops_buffer& hb = host[i * nb + b];
            const sigops_buffer& db = dev[i * nb + b];
            const size_t es = elem_size(hb.dtype);
            if (hb.nframes == 0) { ++i; continue; }
            const bool dense = hb.ld == hb.nframes && db.ld == hb.nframes;
            if (!dense) {
                if (to_device) CUDA_OK(cudaMemcpy2DAsync(db.ptr, db.ld * es, hb.ptr, hb.ld * es, hb.nframes * es, hb.nchannels, cudaMemcpyHostToDevice, st));
                else CUDA_OK(cudaMemcpy2DAsync(hb.ptr, hb.ld * es, db.ptr, db.ld * es, hb.nframes * es, hb.nchannels, cudaMemcpyDeviceToHost, st));
                total += hb.nframes * hb.nchannels * (int64_t)es;
                ++i;
                continue;
            }
            const size_t bytes = (size_t)hb.nframes * hb.nchannels * es;
            int64_t j = i + 1;
            while (merge && j < w && (char*)host[j * nb + b].ptr == (char*)hb.ptr + (j - i) * bytes &&
                   (char*)dev[j * nb + b].ptr == (char*)db.ptr + (j - i) * bytes)
                ++j;
            if (to_device) CUDA_OK(cudaMemcpyAsync(db.ptr, hb.ptr, bytes * (j - i), cudaMemcpyHostToDevice, st));
            else CUDA_OK(cudaMemcpyAsync(hb.ptr, db.ptr, bytes * (j - i), cudaMemcpyDeviceToHost, st));
            total += (int64_t)bytes * (j - i);
            i = j;
        }
    }
    return total;
}

// ---- host-buffer run: H2D | stages | D2H on three streams, three staging buffers per device ----------

struct HostRunResult {
    int64_t launches = 0, h2d = 0, d2h = 0;
    double gpu_ms = 0, h2d_ms = 0, d2h_ms = 0;
    int staged_waves = 0;
    int code = 0;
    std::string msg;
};

// Is this caller pointer page-locked (cudaHostAlloc / cudaHostRegister / sigops_host_alloc)?  Anything else is
// pageable memory, which the DMA engines cannot read directly: cudaMemcpyAsync would fall back to a staged,
// synchronous copy (measured on the B200 box: 11 GB/s H2D, 22 GB/s D2H instead of 55/57).
bool is_pinned(const void* ptr) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, ptr) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
}

// memcpy of `n` (dst, src, bytes) pieces spread over a few threads (host DRAM: ~15 GB/s per thread, ~50 with 8)
struct CopyPiece { char* dst; const char* src; size_t bytes; };
void parallel_copy(const std::vector<CopyPiece>& pieces, int nthreads) {
    size_t total = 0;
    for (auto& c : pieces) total += c.bytes;
    if (total == 0) return;
    nthreads = (int)std::max<size_t>(1, std::min<size_t>(nthreads, total >> 22));      // >= 4 MB per thread
    if (nthreads == 1) {
        for (auto& c : pieces) memcpy(c.dst, c.src, c.bytes);
        return;
    }
    const size_t share = (total + nthreads - 1) / nthreads;
    std::vector<std::thread> th;
    for (int t = 0; t < nthreads; ++t) {
        th.emplace_back([&, t] {
            size_t lo = share * t, hi = std::min(total, lo + share), pos = 0;       // my byte range of the concatenation
            for (auto& c : pieces) {
                const size_t a = std::max(lo, pos), b = std::min(hi, pos + c.bytes);
                if (a < b) memcpy(c.dst + (a - pos), c.src + (a - pos), b - a);
                pos += c.bytes;
                if (pos >= hi) break;
            }
        });
    }
    for (auto& t : th) t.join();
}

int copy_threads(int ndev) {
    if (const char* e = getenv("SIGOPS_COPY_THREADS")) return std::max(1, atoi(e));
    const int hw = (int)std::thread::hardware_concurrency();
    return std::max(1, std::min(8, (hw > 0 ? hw : 8) / std::max(1, ndev)));
}

void run_host_on_device(sigops_plan& p, int di, int64_t i_begin, int64_t i_end, const sigops_buffer* in,
                        sigops_buffer* out, HostRunResult& res) {
    Device& dev = p.ctx->devs[di];
    try {
        CUDA_OK(cudaSetDevice(dev.ordinal));
        ensure_plan_dev(p, di);
        const int64_t ninst = i_end - i_begin;
        if (ninst <= 0) return;
        const uint32_t nin = p.h.n_inputs, nout = p.h.n_outputs;
        // bytes of device staging one instance needs, and of host data it moves
        size_t io_bytes = 0, in_host = 0, out_host = 0;
        for (uint32_t b = 0; b < nin + nout; ++b) {
            const sigops_bufdesc& bd = b < nin ? p.bufs[b] : p.bufs[p.h.n_temps + b];
            io_bytes += (size_t)round_up(round_up(std::max<int64_t>(bd.nframes, 1), 16) * bd.nchannels * (int64_t)elem_size(bd.dtype), 256);
            (b < nin ? in_host : out_host) += (size_t)bd.nframes * bd.nchannels * elem_size(bd.dtype);
        }
        // WAV-layout host buffers need a device scratch area next to the planar buffer
        bool any_wav = false;
        for (uint32_t b = 0; b < nin; ++b) any_wav = any_wav || (in[i_begin * nin + b].dtype & SIGOPS_INTERLEAVED);
        for (uint32_t b = 0; b < nout; ++b) any_wav = any_wav || (out[i_begin * nout + b].dtype & SIGOPS_INTERLEAVED);
        if (any_wav) { io_bytes *= 2; in_host *= 2; out_host *= 2; }   // (a Float64 file for a Float32 plan buffer is twice its size)
        // page-locked caller memory is copied from / to directly; anything else goes through the pinned ring
        bool pinned_in = true, pinned_out = true;
        for (int64_t i : {i_begin, i_end - 1}) {
            for (uint32_t b = 0; b < nin; ++b)
                if (in[i * nin + b].nframes > 0 && !is_pinned(in[i * nin + b].ptr)) pinned_in = false;
            for (uint32_t b = 0; b < nout; ++b)
                if (out[i * nout + b].nframes > 0 && !is_pinned(out[i * nout + b].ptr)) pinned_out = false;
        }
        if (getenv("SIGOPS_FORCE_STAGING")) pinned_in = pinned_out = false;
        const size_t budget = p.ctx->ws_budget / kHostSlots;
        int64_t wave = ninst;
        auto need_for = [&](int64_t w) { return wave_workspace_bytes(p, w, dev.sm_count) + io_bytes * w + (size_t)w * (nin + nout) * sizeof(sigops_buffer); };
        // several waves when the batch allows it, so that H2D of wave k+1, the kernels of wave k and D2H of wave
        // k-1 overlap (the first H2D and the last D2H are exposed: 1/nwaves of the copy time)
        int nwaves = 16;
        if (const char* e = getenv("SIGOPS_HOST_WAVES")) nwaves = std::max(1, atoi(e));
        if (ninst >= 2 * nwaves) wave = (ninst + nwaves - 1) / nwaves;
        while (wave > 1 && need_for(wave) > budget) wave = (wave + 1) / 2;
        // pageable callers: bound the pinned ring (page-locking costs ~0.6 s per GB, once per context)
        const size_t stage_cap = size_t(512) << 20;
        if (!pinned_in) while (wave > 1 && in_host * wave > stage_cap) wave = (wave + 1) / 2;
        if (!pinned_out) while (wave > 1 && out_host * wave > stage_cap) wave = (wave + 1) / 2;
        const int nthreads = copy_threads((int)p.ctx->devs.size());
        for (int s = 0; s < kHostSlots; ++s) {
            Slot& slot = dev.slots[s];
            if (slot.busy_valid) CUDA_OK(cudaEventSynchronize(slot.busy));        // an earlier asynchronous run_device on this slot
            slot.busy_valid = false;
            if (need_for(wave) > slot.arena.cap) {
                CUDA_OK(cudaStreamSynchronize(slot.stream));
                slot.arena.reserve(need_for(wave));
                slot.last_table_dev = nullptr;
            }
            if (!pinned_in) dev.stage_in[s].reserve(in_host * wave);
            if (!pinned_out) dev.stage_out[s].reserve(out_host * wave);
        }
        struct InFlight { int64_t i0 = 0, w = 0; bool live = false; std::vector<CopyPiece> drain; std::future<void> drained; };
        InFlight fl[kHostSlots];
        // din/dout: the planar device buffers the stages see; c*_u / c*_d: what is copied (the same buffer, or for
        // a WAV-layout host buffer its raw interleaved bytes and a device scratch area next to the planar one)
        std::vector<sigops_buffer> din, dout, cin_u, cin_d, cout_u, cout_d, hin, hout;
        struct WavJob { WavParams P; };
        std::vector<WavJob> wav_in, wav_out;
        auto finish = [&](int s) {      // wave in staging buffer s: wait for its D2H, account, drain the pinned ring
            InFlight& f = fl[s];
            if (!f.live) return;
            if (f.drained.valid()) f.drained.get();          // pageable results: the background drain of this buffer (rethrows)
            CUDA_OK(cudaEventSynchronize(dev.ev_out[s]));
            float ms = 0;
            cudaEventElapsedTime(&ms, dev.ev_t[s][0], dev.ev_t[s][1]); res.h2d_ms += ms;
            cudaEventElapsedTime(&ms, dev.ev_in[s], dev.ev_k[s]); res.gpu_ms += ms;
            cudaEventElapsedTime(&ms, dev.ev_t[s][2], dev.ev_t[s][3]); res.d2h_ms += ms;
            if (!f.drain.empty()) parallel_copy(f.drain, nthreads);
            f.drain.clear();
            f.live = false;
        };
        // device staging of one side of a wave: planar buffers first (buffer-major: the same buffer of consecutive
        // instances is contiguous, which the tensor-map kernels and merged copies rely on), WAV scratch after them
        auto stage_side = [&](Slot& slot, const sigops_buffer* user, int64_t w, uint32_t nb, uint32_t desc0, bool input,
                              std::vector<sigops_buffer>& dbufs, std::vector<sigops_buffer>& cu, std::vector<sigops_buffer>& cd,
                              std::vector<WavJob>& jobs) {
            dbufs.assign((size_t)w * nb, sigops_buffer{});
            cu.assign((size_t)w * nb, sigops_buffer{});
            cd.assign((size_t)w * nb, sigops_buffer{});
            jobs.clear();
            for (uint32_t b = 0; b < nb; ++b)
                for (int64_t i = 0; i < w; ++i) {
                    const sigops_buffer& ub = user[i * nb + b];
                    const sigops_bufdesc& bd = p.bufs[desc0 + b];
                    sigops_buffer& db = dbufs[i * nb + b];
                    db = ub;
                    db.dtype = bd.dtype;
                    db.ld = round_up(std::max<int64_t>(ub.nframes, 1), 16);
                    db.ptr = slot.arena.take_packed((size_t)db.ld * ub.nchannels * elem_size(bd.dtype));
                    cu[i * nb + b] = ub;
                    cd[i * nb + b] = db;
                }
            for (uint32_t b = 0; b < nb; ++b)
                for (int64_t i = 0; i < w; ++i) {
                    const sigops_buffer& ub = user[i * nb + b];
                    if (!(ub.dtype & SIGOPS_INTERLEAVED)) continue;
                    const int enc = ub.dtype & 0xff;
                    const int64_t total = ub.nframes * ub.nchannels;
                    void* scratch = slot.arena.take_packed((size_t)std::max<int64_t>(total, 1) * elem_size(enc));
                    cu[i * nb + b] = sigops_buffer{ub.ptr, total, 1, enc, total};
                    cd[i * nb + b] = sigops_buffer{scratch, total, 1, enc, total};
                    const sigops_buffer& db = dbufs[i * nb + b];
                    WavParams W{};
                    W.src = input ? scratch : db.ptr;
                    W.dst = input ? db.ptr : scratch;
                    W.nframes = ub.nframes; W.nch = ub.nchannels; W.ld = db.ld;
                    W.planar_dtype = db.dtype; W.file_dtype = enc;
                    jobs.push_back({W});
                }
        };
        // dense copy of the copy views into / out of the pinned ring (one piece per channel row)
        auto ring_views = [&](char* ring, const std::vector<sigops_buffer>& cu, int64_t w, uint32_t nb, std::vector<sigops_buffer>& hv,
                              std::vector<CopyPiece>& pieces, bool to_ring) {
            hv.assign((size_t)w * nb, sigops_buffer{});
            pieces.clear();
            char* cur = ring;
            for (uint32_t b = 0; b < nb; ++b)
                for (int64_t i = 0; i < w; ++i) {
                    const sigops_buffer& ub = cu[i * nb + b];
                    sigops_buffer& hb = hv[i * nb + b];
                    hb = ub;
                    hb.ld = ub.nframes;
                    hb.ptr = cur;
                    const size_t es = elem_size(ub.dtype), row = (size_t)ub.nframes * es;
                    for (int c = 0; c < ub.nchannels; ++c) {
                        char* r = cur + c * row;
                        char* u = (char*)ub.ptr + (size_t)c * ub.ld * es;
                        if (to_ring) pieces.push_back({r, u, row});
                        else pieces.push_back({u, r, row});
                    }
                    cur += row * ub.nchannels;
                }
        };
        int k = 0;
        for (int64_t i0 = 0; i0 < ninst; i0 += wave, ++k) {
            const int s = k % kHostSlots;
            Slot& slot = dev.slots[s];
            const int64_t w = std::min(wave, ninst - i0);
            finish(s);                  // the buffer's previous wave has left the device (and the pinned ring)
            slot.arena.reset();
            stage_side(slot, in + (i_begin + i0) * nin, w, nin, 0, true, din, cin_u, cin_d, wav_in);
            stage_side(slot, out + (i_begin + i0) * nout, w, nout, nin + p.h.n_temps, false, dout, cout_u, cout_d, wav_out);
            // ---- H2D on the copy-in stream
            const sigops_buffer* src = cin_u.data();
            if (!pinned_in && nin) {
                std::vector<CopyPiece> pieces;                     // user arrays -> pinned ring, by worker threads
                ring_views(dev.stage_in[s].base, cin_u, w, nin, hin, pieces, true);
                parallel_copy(pieces, nthreads);
                src = hin.data();
                ++res.staged_waves;
            }
            CUDA_OK(cudaEventRecord(dev.ev_t[s][0], dev.s_in));
            res.h2d += copy_runs(src, cin_d.data(), w, nin, true, dev.s_in, !pinned_in);
            CUDA_OK(cudaEventRecord(dev.ev_t[s][1], dev.s_in));
            CUDA_OK(cudaEventRecord(dev.ev_in[s], dev.s_in));
            // ---- stages on the slot's stream (WAV-layout inputs are transposed / decoded first, outputs encoded last)
            CUDA_OK(cudaStreamWaitEvent(slot.stream, dev.ev_in[s], 0));
            for (auto& j : wav_in) launch_wav(false, j.P, slot.stream);
            WaveIO io{w, din.data(), dout.data(), i_begin + i0};
            res.launches += enqueue_wave(p, di, slot, slot.stream, io) + (int64_t)wav_in.size() + (int64_t)wav_out.size();
            for (auto& j : wav_out) launch_wav(true, j.P, slot.stream);
            CUDA_OK(cudaGetLastError());
            CUDA_OK(cudaEventRecord(dev.ev_k[s], slot.stream));
            // ---- D2H on the copy-out stream
            CUDA_OK(cudaStreamWaitEvent(dev.s_out, dev.ev_k[s], 0));
            const sigops_buffer* dst = cout_u.data();
            fl[s].drain.clear();
            if (!pinned_out) {
                ring_views(dev.stage_out[s].base, cout_u, w, nout, hout, fl[s].drain, false);
                dst = hout.data();
            }
            CUDA_OK(cudaEventRecord(dev.ev_t[s][2], dev.s_out));
            res.d2h += copy_runs(dst, cout_d.data(), w, nout, false, dev.s_out, !pinned_out);
            CUDA_OK(cudaEventRecord(dev.ev_t[s][3], dev.s_out));
            CUDA_OK(cudaEventRecord(dev.ev_out[s], dev.s_out));
            fl[s].i0 = i0; fl[s].w = w; fl[s].live = true;
            if (!fl[s].drain.empty()) {
                // pageable results leave the pinned ring on a background thread as soon as the wave's D2H has
                // landed, while this thread stages the next waves' inputs: copy-in and copy-out of the caller's
                // memory overlap instead of taking turns (the ring buffer is not touched again before finish(s))
                fl[s].drained = std::async(std::launch::async, [&dev, s, nthreads, pieces = std::move(fl[s].drain)] {
                    CUDA_OK(cudaSetDevice(dev.ordinal));
                    CUDA_OK(cudaEventSynchronize(dev.ev_out[s]));
                    parallel_copy(pieces, nthreads);
                });
                fl[s].drain.clear();
            }
        }
        for (int j = 0; j < kHostSlots; ++j) finish((k + j) % kHostSlots);      // oldest first
    } catch (const Failure& f) {
        res.code = f.code;
        res.msg = f.msg;
        for (int s = 0; s < kHostSlots; ++s) cudaStreamSynchronize(dev.slots[s].stream);
        cudaStreamSynchronize(dev.s_in);
        cudaStreamSynchronize(dev.s_out);
    }
}

// ---- micro-benchmarks for the roofline denominators ---------------------------------

__global__ void k_dfma_peak(double* out, int iters, double a, double b) {
    double x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
    for (int i = 0; i < iters; ++i) {
        x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
        x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
    }
    out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
}

__global__ void k_copy_peak(const double2* __restrict__ src, double2* __restrict__ dst, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) dst[i] = src[i];
}

template <class F>
int guarded(sigops_ctx* ctx, F&& f) {
    try {
        f();
        return SIGOPS_OK;
    } catch (const Failure& e) {
        if (ctx) {
            std::lock_guard<std::mutex> lk(ctx->mu);
            ctx->err = e.msg;
        } else
            g_tls_error = e.msg;
        return e.code;
    } catch (const std::bad_alloc&) {
        if (ctx) ctx->err = "host allocation failed";
        else g_tls_error = "host allocation failed";
        return SIGOPS_ERR_NOMEM;
    } catch (const std::exception& e) {
        if (ctx) ctx->err = e.what();
        else g_tls_error = e.what();
        return SIGOPS_ERR_INVALID;
    }
}

}  // namespace

// =====================================================================================
// C ABI
// =====================================================================================

extern "C" {

int sigops_abi_version(void) { return SIGOPS_ABI_VERSION; }

int sigops_device_count(int* count) {
    return guarded(nullptr, [&] {
        if (!count) fail(SIGOPS_ERR_INVALID, "null argument");
        int n = 0;
        cudaError_t e = cudaGetDeviceCount(&n);
        if (e != cudaSuccess) {
            cudaGetLastError();
            n = 0;
        }
        *count = n;
    });
}

int sigops_ctx_create(const int* devices, int ndev, sigops_ctx** out) {
    return guarded(nullptr, [&] {
        if (!out) fail(SIGOPS_ERR_INVALID, "null argument");
        *out = nullptr;
        int have = 0;
        cudaError_t e = cudaGetDeviceCount(&have);
        if (e != cudaSuccess || have == 0) {
            cudaGetLastError();
            fail(SIGOPS_ERR_CUDA, "no CUDA device available (%s); the GPU sink has no CPU fallback",
                 e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
        }
        std::vector<int> ords;
        if (!devices || ndev <= 0) ords.push_back(0);
        else ords.assign(devices, devices + ndev);
        auto ctx = std::make_unique<sigops_ctx>();
        for (int o : ords) {
            if (o < 0 || o >= have) fail(SIGOPS_ERR_INVALID, "device ordinal %d of %d", o, have);
            cudaDeviceProp prop;
            CUDA_OK(cudaGetDeviceProperties(&prop, o));
            if (prop.major < 10) fail(SIGOPS_ERR_UNSUPPORTED, "device %d is sm_%d%d; this library is built for sm_100a only", o, prop.major, prop.minor);
            Device d;
            d.ordinal = o;
            d.sm_count = prop.multiProcessorCount;
            CUDA_OK(cudaSetDevice(o));
            for (int s = 0; s < kHostSlots; ++s) {
                CUDA_OK(cudaStreamCreateWithFlags(&d.slots[s].stream, cudaStreamNonBlocking));
                for (auto& ev : d.slots[s].ev) CUDA_OK(cudaEventCreate(&ev));
                CUDA_OK(cudaEventCreateWithFlags(&d.slots[s].busy, cudaEventDisableTiming));
                CUDA_OK(cudaEventCreate(&d.ev_in[s]));
                CUDA_OK(cudaEventCreate(&d.ev_k[s]));
                CUDA_OK(cudaEventCreate(&d.ev_out[s]));
                for (auto& ev : d.ev_t[s]) CUDA_OK(cudaEventCreate(&ev));
            }
            CUDA_OK(cudaStreamCreateWithFlags(&d.s_in, cudaStreamNonBlocking));
            CUDA_OK(cudaStreamCreateWithFlags(&d.s_out, cudaStreamNonBlocking));
            ctx->devs.push_back(std::move(d));
        }
        if (const char* b = getenv("SIGOPS_WS_BYTES")) ctx->ws_budget = std::max<size_t>(size_t(64) << 20, strtoull(b, nullptr, 10));
        *out = ctx.release();
    });
}

void sigops_ctx_destroy(sigops_ctx* ctx) {
    if (!ctx) return;
    for (auto& d : ctx->devs) {
        cudaSetDevice(d.ordinal);
        if (d.s_in) cudaStreamSynchronize(d.s_in);
        if (d.s_out) cudaStreamSynchronize(d.s_out);
        for (auto& s : d.slots) {
            if (s.stream) cudaStreamSynchronize(s.stream);
            if (s.busy_valid) cudaEventSynchronize(s.busy);
            if (s.graph) cudaGraphExecDestroy(s.graph);
            s.arena.release();
            for (int r = 0; r < kTableRing; ++r) {
                if (s.pinned[r]) cudaFreeHost(s.pinned[r]);
                if (s.pinned_ev[r]) cudaEventDestroy(s.pinned_ev[r]);
            }
            for (auto& ev : s.ev)
                if (ev) cudaEventDestroy(ev);
            if (s.busy) cudaEventDestroy(s.busy);
            for (auto& ev : s.prof_pool) cudaEventDestroy(ev);
            if (s.stream) cudaStreamDestroy(s.stream);
        }
        for (int s = 0; s < kHostSlots; ++s) {
            d.stage_in[s].release();
            d.stage_out[s].release();
            if (d.ev_in[s]) cudaEventDestroy(d.ev_in[s]);
            if (d.ev_k[s]) cudaEventDestroy(d.ev_k[s]);
            if (d.ev_out[s]) cudaEventDestroy(d.ev_out[s]);
            for (auto& ev : d.ev_t[s])
                if (ev) cudaEventDestroy(ev);
        }
        if (d.s_in) cudaStreamDestroy(d.s_in);
        if (d.s_out) cudaStreamDestroy(d.s_out);
    }
    delete ctx;
}

const char* sigops_last_error(sigops_ctx* ctx) {
    if (!ctx) return g_tls_error.c_str();
    std::lock_guard<std::mutex> lk(ctx->mu);
    g_tls_error = ctx->err;
    return g_tls_error.c_str();
}

int sigops_plan_create(sigops_ctx* ctx, const void* plan, size_t nbytes, sigops_plan** out) {
    return guarded(ctx, [&] {
        if (!ctx || !plan || !out) fail(SIGOPS_ERR_INVALID, "null argument");
        *out = nullptr;
        auto p = std::make_unique<sigops_plan>();
        static std::atomic<uint64_t> next_uid{1};
        p->uid = next_uid++;
        p->ctx = ctx;
        parse_plan(*p, plan, nbytes);
        p->dev.resize(ctx->devs.size());
        *out = p.release();
    });
}

void sigops_plan_destroy(sigops_plan* plan) {
    if (!plan) return;
    free_plan_dev(*plan);
    delete plan;
}

int sigops_plan_run_device(sigops_plan* plan, int dev_index, int64_t ninst, const sigops_buffer* in,
                           sigops_buffer* out, void* cuda_stream, sigops_stats* stats) {
    if (!plan) return SIGOPS_ERR_INVALID;
    return guarded(plan->ctx, [&] {
        sigops_ctx* ctx = plan->ctx;
        if (dev_index < 0 || dev_index >= (int)ctx->devs.size()) fail(SIGOPS_ERR_INVALID, "device index %d of %zu", dev_index, ctx->devs.size());
        validate_io(*plan, ninst, in, out);
        std::lock_guard<std::mutex> lk(ctx->mu);
        Device& dev = ctx->devs[dev_index];
        Slot& slot = dev.slots[0];
        cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : slot.stream;
        auto t0 = std::chrono::steady_clock::now();
        CUDA_OK(cudaSetDevice(dev.ordinal));
        // every call shares this slot's workspace (temps, scalars, IIR state, BufRef table): work enqueued by an
        // earlier call on ANOTHER stream must have finished with it first
        if (slot.busy_valid && slot.busy_stream != st) CUDA_OK(cudaStreamWaitEvent(st, slot.busy, 0));
        if (stats) CUDA_OK(cudaEventRecord(slot.ev[4], st));
        const int64_t launches = run_device_resident(*plan, dev_index, ninst, in, out, st, slot);
        if (stats) CUDA_OK(cudaEventRecord(slot.ev[5], st));
        CUDA_OK(cudaEventRecord(slot.busy, st));
        slot.busy_stream = st;
        slot.busy_valid = true;
        if (!cuda_stream || stats) CUDA_OK(cudaStreamSynchronize(st));
        if (stats) {
            memset(stats, 0, sizeof *stats);
            float ms = 0;
            CUDA_OK(cudaEventElapsedTime(&ms, slot.ev[4], slot.ev[5]));
            stats->gpu_ms = ms;
            stats->launches = launches;
            stats->out_samples = count_out_samples(*plan, ninst);
            stats->wall_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        }
    });
}

int sigops_plan_run(sigops_plan* plan, int64_t ninst, const sigops_buffer* in, sigops_buffer* out,
                    sigops_stats* stats) {
    if (!plan) return SIGOPS_ERR_INVALID;
    return guarded(plan->ctx, [&] {
        sigops_ctx* ctx = plan->ctx;
        validate_io(*plan, ninst, in, out, true);
        std::unique_lock<std::mutex> lk(ctx->mu);
        auto t0 = std::chrono::steady_clock::now();
        const int nd = (int)ctx->devs.size();
        std::vector<HostRunResult> res(nd);
        std::vector<std::thread> th;
        for (int d = 0; d < nd; ++d) {
            const int64_t b = ninst * d / nd, e = ninst * (d + 1) / nd;
            if (nd == 1) run_host_on_device(*plan, d, b, e, in, out, res[d]);
            else th.emplace_back([&, d, b, e] { run_host_on_device(*plan, d, b, e, in, out, res[d]); });
        }
        for (auto& t : th) t.join();
        lk.unlock();
        for (auto& r : res)
            if (r.code) throw Failure{r.code, r.msg};
        if (stats) {
            memset(stats, 0, sizeof *stats);
            for (auto& r : res) {
                stats->gpu_ms = std::max(stats->gpu_ms, r.gpu_ms);
                stats->h2d_ms = std::max(stats->h2d_ms, r.h2d_ms);
                stats->d2h_ms = std::max(stats->d2h_ms, r.d2h_ms);
                stats->launches += r.launches;
                stats->h2d_bytes += r.h2d;
                stats->d2h_bytes += r.d2h;
            }
            stats->out_samples = count_out_samples(*plan, ninst);
            stats->wall_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        }
    });
}

int sigops_host_alloc(size_t bytes, void** out) {
    return guarded(nullptr, [&] {
        if (!out) fail(SIGOPS_ERR_INVALID, "null argument");
        *out = nullptr;
        if (bytes == 0) return;
        CUDA_OK(cudaHostAlloc(out, bytes, cudaHostAllocPortable));
    });
}

int sigops_host_free(void* ptr) {
    return guarded(nullptr, [&] {
        if (ptr) CUDA_OK(cudaFreeHost(ptr));
    });
}

int sigops_plan_launch_count(sigops_plan* plan, int64_t* launches) {
    if (!plan) return SIGOPS_ERR_INVALID;
    return guarded(plan->ctx, [&] {
        if (!launches) fail(SIGOPS_ERR_INVALID, "null argument");
        int64_t n = 0;
        for (auto& s : plan->stages) {
            if (s.st.kind == SIGOPS_STAGE_IIR) n += s.st.n_out > 0 ? 3 : 0;   // upper bound: main + carry + fix
            else n += 1;
        }
        *launches = n;
    });
}

int sigops_plan_algorithmic_bytes(sigops_plan* plan, int64_t* bytes) {
    if (!plan) return SIGOPS_ERR_INVALID;
    return guarded(plan->ctx, [&] {
        if (!bytes) fail(SIGOPS_ERR_INVALID, "null argument");
        // SURVEY.md §8d: every stage writes its output once and reads each distinct
        // buffer it references once per output sample (generators/constants/ramps cost 0).
        int64_t total = 0;
        auto prog_reads = [&](int start, int len, int64_t frames, int nch) {
            int64_t b = 0;
            for (int i = 0; i < len; ++i) {
                const sigops_instr& I = plan->instrs[start + i];
                if (!op_has_leaf(I.op)) continue;
                if (I.leaf == SIGOPS_LEAF_BUF) b += frames * nch * (int64_t)elem_size(plan->bufs[I.buf].dtype);
                if (I.leaf == SIGOPS_LEAF_CHANSUM) b += frames * I.i2 * (int64_t)elem_size(plan->bufs[I.buf].dtype);
            }
            return b;
        };
        for (auto& s : plan->stages) {
            const sigops_stage& g = s.st;
            const sigops_bufdesc& ob = plan->bufs[g.out_buf];
            if (g.kind == SIGOPS_STAGE_MAP) {
                for (int k = 0; k < g.n_pieces; ++k) {
                    const sigops_piece& pc = plan->pieces[g.piece_start + k];
                    total += pc.out_len * pc.ch_count * (int64_t)elem_size(ob.dtype);
                    total += prog_reads(pc.prog_start, pc.prog_len, pc.out_len, pc.ch_count);
                }
            } else {
                total += g.n_out * g.nchannels * (int64_t)elem_size(ob.dtype);
                total += prog_reads(g.in_prog_start, g.in_prog_len, g.n_in, g.nchannels);
                total += prog_reads(g.epi_prog_start, g.epi_prog_len, g.n_out, g.nchannels);
            }
        }
        *bytes = total;
    });
}

int sigops_ctx_set_profiling(sigops_ctx* ctx, int enabled) {
    return guarded(ctx, [&] {
        if (!ctx) fail(SIGOPS_ERR_INVALID, "null argument");
        std::lock_guard<std::mutex> lk(ctx->mu);
        ctx->profiling = enabled != 0;
        for (auto& d : ctx->devs)
            for (auto& s : d.slots) {
                s.prof_used = 0;
                s.prof_kind.clear();
            }
    });
}

int sigops_profile_collect(sigops_ctx* ctx, int dev_index, double* ms_by_kind, int64_t* count_by_kind, int nkinds) {
    return guarded(ctx, [&] {
        if (!ctx || dev_index < 0 || dev_index >= (int)ctx->devs.size() || !ms_by_kind || !count_by_kind)
            fail(SIGOPS_ERR_INVALID, "bad argument");
        std::lock_guard<std::mutex> lk(ctx->mu);
        for (int k = 0; k < nkinds; ++k) { ms_by_kind[k] = 0; count_by_kind[k] = 0; }
        Device& dev = ctx->devs[dev_index];
        CUDA_OK(cudaSetDevice(dev.ordinal));
        CUDA_OK(cudaDeviceSynchronize());
        for (auto& s : dev.slots) {
            for (size_t i = 0; i < s.prof_kind.size(); ++i) {
                float ms = 0;
                CUDA_OK(cudaEventElapsedTime(&ms, s.prof_pool[2 * i], s.prof_pool[2 * i + 1]));
                const int k = s.prof_kind[i];
                if (k < nkinds) { ms_by_kind[k] += ms; count_by_kind[k] += 1; }
            }
            s.prof_used = 0;
            s.prof_kind.clear();
        }
    });
}

int sigops_measure_peaks(sigops_ctx* ctx, int dev_index, double* dfma_per_s, double* copy_gbs) {
    return guarded(ctx, [&] {
        if (!ctx || dev_index < 0 || dev_index >= (int)ctx->devs.size()) fail(SIGOPS_ERR_INVALID, "bad device index");
        std::lock_guard<std::mutex> lk(ctx->mu);
        Device& dev = ctx->devs[dev_index];
        CUDA_OK(cudaSetDevice(dev.ordinal));
        cudaStream_t st = dev.slots[0].stream;
        cudaEvent_t e0 = dev.slots[0].ev[4], e1 = dev.slots[0].ev[5];
        if (dfma_per_s) {
            const int blocks = dev.sm_count * 8, threads = 256, iters = 1 << 14;
            double* d = nullptr;
            CUDA_OK(cudaMalloc(&d, (size_t)blocks * threads * sizeof(double)));
            double best = 0;
            for (int rep = 0; rep < 5; ++rep) {
                CUDA_OK(cudaEventRecord(e0, st));
                k_dfma_peak<<<blocks, threads, 0, st>>>(d, iters, 0.999999, 1e-9);
                CUDA_OK(cudaEventRecord(e1, st));
                CUDA_OK(cudaStreamSynchronize(st));
                float ms = 0;
                CUDA_OK(cudaEventElapsedTime(&ms, e0, e1));
                best = std::max(best, (double)blocks * threads * iters * 8.0 / (ms * 1e-3));
            }
            cudaFree(d);
            *dfma_per_s = best;
        }
        if (copy_gbs) {
            const size_t n = size_t(1) << 26;   // 2 x 1 GiB
            double2 *a = nullptr, *b = nullptr;
            CUDA_OK(cudaMalloc(&a, n * sizeof(double2)));
            CUDA_OK(cudaMalloc(&b, n * sizeof(double2)));
            CUDA_OK(cudaMemsetAsync(a, 0, n * sizeof(double2), st));
            double best = 0;
            for (int rep = 0; rep < 6; ++rep) {
                CUDA_OK(cudaEventRecord(e0, st));
                k_copy_peak<<<dev.sm_count * 16, 512, 0, st>>>(a, b, n);
                CUDA_OK(cudaEventRecord(e1, st));
                CUDA_OK(cudaStreamSynchronize(st));
                float ms = 0;
                CUDA_OK(cudaEventElapsedTime(&ms, e0, e1));
                if (rep) best = std::max(best, 2.0 * n * sizeof(double2) / (ms * 1e-3) / 1e9);
            }
            cudaFree(a);
            cudaFree(b);
            *copy_gbs = best;
        }
    });
}

}  // extern "C"
