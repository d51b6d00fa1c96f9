// Instantiations of k_iir_tma without fused programs (MAIN / FIX / WARM).
#include "common.h"
#include "launchers.h"

namespace sigops {
namespace {
template <int MODE>
void launch_iir_tma(int M, bool unitb, dim3 grid, cudaStream_t st, const IirTmaParams& Q) {
    with_sections(M, [&](auto m) {
        if (unitb) {
            ensure_dyn_smem(k_iir_tma<m, MODE, true, false>, kTmaSmemBytes);
            k_iir_tma<m, MODE, true, false><<<grid, kTmaThreads, kTmaSmemBytes, st>>>(Q);
        } else {
            ensure_dyn_smem(k_iir_tma<m, MODE, false, false>, kTmaSmemBytes);
            k_iir_tma<m, MODE, false, false><<<grid, kTmaThreads, kTmaSmemBytes, st>>>(Q);
        }
    });
    CUDA_OK(cudaGetLastError());
}
}  // namespace

void launch_iir_tma_any(int mode, bool prog, int M, bool unitb, dim3 grid, cudaStream_t st, const IirTmaParams& Q) {
    if (prog) {
        if (mode != LAUNCH_WARM) fail(SIGOPS_ERR_UNSUPPORTED, "internal: program-carrying TMA kernel is WARM only");
        with_sections(M, [&](auto m) { launch_iir_tma_prog<m>(grid, st, Q); });
    } else if (mode == LAUNCH_WARM) launch_iir_tma<IIR_WARM>(M, unitb, grid, st, Q);
    else if (mode == LAUNCH_MAIN) launch_iir_tma<IIR_MAIN>(M, unitb, grid, st, Q);
    else launch_iir_tma<IIR_FIX>(M, unitb, grid, st, Q);
}

}  // namespace sigops
