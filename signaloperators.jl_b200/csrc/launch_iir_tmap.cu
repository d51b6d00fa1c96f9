// Instantiations of k_iir_tmap (tensor-map TMA) and the host side of its tensor maps.
#include "common.h"
#include "launchers.h"
#include "k_iir_tmap.cuh"

namespace sigops {
namespace {

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess)
            p = nullptr;
        cudaGetLastError();
        return (EncodeTiledFn)p;
    }();
    return fn;
}

template <int M, int NW, int NS, int SUBS, class T, int LV>
void launch_cfg(bool unitb, dim3 grid, cudaStream_t st, const IirTmapParams& P, const CUtensorMap& a, const CUtensorMap& b) {
    constexpr size_t smem = tm_smem_bytes(NW, NS, SUBS, LV != 0, 128 / (int)sizeof(T));
    if (unitb) {
        ensure_dyn_smem(k_iir_tmap<M, true, NW, NS, SUBS, T, LV>, smem);
        k_iir_tmap<M, true, NW, NS, SUBS, T, LV><<<grid, NW * 32, smem, st>>>(P, a, b);
    } else {
        ensure_dyn_smem(k_iir_tmap<M, false, NW, NS, SUBS, T, LV>, smem);
        k_iir_tmap<M, false, NW, NS, SUBS, T, LV><<<grid, NW * 32, smem, st>>>(P, a, b);
    }
}

template <int M>
void launch_m(bool f32, bool unitb, dim3 grid, cudaStream_t st, const IirTmapParams& P, const CUtensorMap& a, const CUtensorMap& b) {
    const bool lv = P.n_in_ops + P.n_ep_ops > 0;
    bool fn = false;                   // a closure function among the fused operations: the variant that applies them
    for (int j = 0; j < 2 * kTmMaxLeafOps; ++j) fn = fn || P.ops[j].op == SIGOPS_OP_FN1 || P.ops[j].op == SIGOPS_OP_FN2;
    if (f32) launch_cfg<M, kTmWarpsF32, kTmStages, kTmSubsPerStageF32, float, 0>(unitb, grid, st, P, a, b);
    else if (lv && fn) launch_cfg<M, kTmWarpsLv, kTmStages, kTmSubsPerStageLv, double, 2>(unitb, grid, st, P, a, b);
    else if (lv) launch_cfg<M, kTmWarpsLv, kTmStages, kTmSubsPerStageLv, double, 1>(unitb, grid, st, P, a, b);
    else launch_cfg<M, kTmWarps, kTmStages, kTmSubsPerStage, double, 0>(unitb, grid, st, P, a, b);
}

}  // namespace

bool iir_tmap_available() { return encode_fn() != nullptr; }

// [rows][frames] matrix of Float64 (elem_bytes 8) or Float32 (4) samples, row r at
// base + r*row_stride_bytes, described as [row][frame/S][S] with S = 128 bytes of samples;
// box = (S, blocks per stage, 32), 128-byte swizzle.  `frames` must be a multiple of S.
bool iir_tmap_encode(void* out_map, void* base, int64_t frames, int64_t rows, int64_t row_stride_bytes, int elem_bytes, int subs_override) {
    EncodeTiledFn fn = encode_fn();
    const int S = 128 / elem_bytes;
    if (!fn || (elem_bytes != 4 && elem_bytes != 8) || frames % S) return false;
    const cuuint64_t gdim[3] = {(cuuint64_t)S, (cuuint64_t)(frames / S), (cuuint64_t)rows};
    const cuuint64_t gstr[2] = {128, (cuuint64_t)row_stride_bytes};
    const cuuint32_t box[3] = {(cuuint32_t)S, (cuuint32_t)(subs_override > 0 ? subs_override : (elem_bytes == 8 ? kTmSubsPerStage : kTmSubsPerStageF32)), 32u};
    const cuuint32_t estr[3] = {1u, 1u, 1u};
    const CUresult r = fn((CUtensorMap*)out_map, elem_bytes == 8 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT64 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, base,
                          gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                          CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS;
}

// [rows][dim0] matrix of Float64 samples, row r at base + r*row_stride_bytes; box = (box0 samples, box1 rows),
// 128-byte swizzle (box0*8 <= 128), zero fill outside the tensor.  Used by k_fir_tmap.
bool tmap_encode_2d_f64(void* out_map, void* base, int64_t dim0, int64_t rows, int64_t row_stride_bytes, int box0, int box1) {
    EncodeTiledFn fn = encode_fn();
    if (!fn || dim0 < 1 || rows < 1 || box0 * 8 > 128 || box1 > 256 || (row_stride_bytes & 15) || ((uintptr_t)base & 15)) return false;
    const cuuint64_t gdim[2] = {(cuuint64_t)dim0, (cuuint64_t)rows};
    const cuuint64_t gstr[1] = {(cuuint64_t)row_stride_bytes};
    const cuuint32_t box[2] = {(cuuint32_t)box0, (cuuint32_t)box1};
    const cuuint32_t estr[2] = {1u, 1u};
    const CUresult r = fn((CUtensorMap*)out_map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, base, gdim, gstr, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS;
}

void launch_iir_tmap(bool f32, int M, bool unitb, dim3 grid, cudaStream_t st, const IirTmapParams& P, const void* map_in,
                     const void* map_out) {
    const CUtensorMap& a = *(const CUtensorMap*)map_in;
    const CUtensorMap& b = *(const CUtensorMap*)map_out;
    switch (M) {
        case 1: launch_m<1>(f32, unitb, grid, st, P, a, b); break;
        case 2: launch_m<2>(f32, unitb, grid, st, P, a, b); break;
        case 3: launch_m<3>(f32, unitb, grid, st, P, a, b); break;
        case 4: launch_m<4>(f32, unitb, grid, st, P, a, b); break;
        case 5: launch_m<5>(f32, unitb, grid, st, P, a, b); break;
        case 6: launch_m<6>(f32, unitb, grid, st, P, a, b); break;
        case 7: launch_m<7>(f32, unitb, grid, st, P, a, b); break;
        case 8: launch_m<8>(f32, unitb, grid, st, P, a, b); break;
        default: fail(SIGOPS_ERR_UNSUPPORTED, "IIR cascade of %d sections", M);
    }
    CUDA_OK(cudaGetLastError());
}

}  // namespace sigops
