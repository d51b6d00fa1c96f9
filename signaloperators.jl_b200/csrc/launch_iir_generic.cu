// Instantiations of the general IIR kernels: k_iir (program-carrying) and k_iir_fast (cp.async).
#include "common.h"
#include "launchers.h"

namespace sigops {
namespace {
template <int MODE>
void launch_iir(int M, dim3 grid, size_t smem, cudaStream_t st, const IirParams& P) {
    with_sections(M, [&](auto m) {
        if (smem > 0) ensure_dyn_smem(k_iir<m, MODE>, smem);
        k_iir<m, MODE><<<grid, kIirThreads, smem, st>>>(P);
    });
    CUDA_OK(cudaGetLastError());
}

template <int MODE>
void launch_iir_fast(int M, bool unitb, dim3 grid, cudaStream_t st, const IirParams& P) {
    with_sections(M, [&](auto m) {
        if (unitb) k_iir_fast<m, MODE, true><<<grid, kIirThreads, 0, st>>>(P);
        else k_iir_fast<m, MODE, false><<<grid, kIirThreads, 0, st>>>(P);
    });
    CUDA_OK(cudaGetLastError());
}

}  // namespace

void launch_iir_generic(int mode, int M, dim3 grid, size_t smem, cudaStream_t st, const IirParams& P) {
    if (mode == LAUNCH_MAIN) launch_iir<IIR_MAIN>(M, grid, smem, st, P);
    else launch_iir<IIR_FIX>(M, grid, smem, st, P);
}

void launch_iir_cpasync(int mode, int M, bool unitb, dim3 grid, cudaStream_t st, const IirParams& P) {
    if (mode == LAUNCH_MAIN) launch_iir_fast<IIR_MAIN>(M, unitb, grid, st, P);
    else launch_iir_fast<IIR_FIX>(M, unitb, grid, st, P);
}

}  // namespace sigops
