// Kernel launchers compiled in their own translation units (the IIR kernels are
// instantiated for 1..8 sections x several modes; separate objects build in parallel).
#pragma once
#include <cuda_runtime.h>

#include <type_traits>

#include "common.h"
#include "k_iir.cuh"
#include "k_iir_tma.cuh"

namespace sigops {

enum { LAUNCH_MAIN = 0, LAUNCH_FIX = 1, LAUNCH_WARM = 2 };

// f(std::integral_constant<int, M>{}) for the cascade lengths the IIR kernels are instantiated for
template <class F>
void with_sections(int M, F&& f) {
    switch (M) {
        case 1: f(std::integral_constant<int, 1>{}); break;
        case 2: f(std::integral_constant<int, 2>{}); break;
        case 3: f(std::integral_constant<int, 3>{}); break;
        case 4: f(std::integral_constant<int, 4>{}); break;
        case 5: f(std::integral_constant<int, 5>{}); break;
        case 6: f(std::integral_constant<int, 6>{}); break;
        case 7: f(std::integral_constant<int, 7>{}); break;
        case 8: f(std::integral_constant<int, 8>{}); break;
        default: fail(SIGOPS_ERR_UNSUPPORTED, "IIR cascade of %d sections", M);
    }
}

// generic program-carrying kernel (k_iir)
void launch_iir_generic(int mode, int M, dim3 grid, size_t smem, cudaStream_t st, const IirParams& P);
// cp.async fast path for unaligned Float64 buffers (k_iir_fast)
void launch_iir_cpasync(int mode, int M, bool unitb, dim3 grid, cudaStream_t st, const IirParams& P);
// TMA bulk-copy kernel (k_iir_tma); `prog` selects the variant with fused programs (WARM only)
void launch_iir_tma_any(int mode, bool prog, int M, bool unitb, dim3 grid, cudaStream_t st, const IirTmaParams& Q);
// the variant with fused programs for M sections, instantiated in launch_iir_tma_prog.cu
template <int M>
void launch_iir_tma_prog(dim3 grid, cudaStream_t st, const IirTmaParams& Q);


// tensor-map TMA kernel (k_iir_tmap, WARM mode, constant-gain epilogue).  The maps are opaque
// 128-byte CUtensorMap objects (64-byte aligned), encoded in launch_iir_tmap.cu.
struct IirTmapParams;
struct alignas(64) TensorMapBlob { unsigned char bytes[128]; };
bool iir_tmap_available();
bool tmap_encode_2d_f64(void* out_map, void* base, int64_t dim0, int64_t rows, int64_t row_stride_bytes, int box0, int box1);
bool iir_tmap_encode(void* out_map, void* base, int64_t frames, int64_t rows, int64_t row_stride_bytes, int elem_bytes, int subs_override = 0);
constexpr int kTmWarps = 4, kTmStages = 2;     // warps per block, stages per warp (160 KB of stages)
void launch_iir_tmap(bool f32, int M, bool unitb, dim3 grid, cudaStream_t st, const IirTmapParams& P, const void* map_in,
                     const void* map_out);

}  // namespace sigops
