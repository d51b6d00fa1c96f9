// Instantiations of k_iir_tma<..., PROG = true> (fused input / epilogue programs, WARM mode).
// Compiled once per pair of section counts (-DSIGOPS_PROG_GROUP=g covers M = 2g+1, 2g+2): the
// embedded interpreter makes each instantiation slow to build.  No b0 = b2 = 1 specialisation:
// the programs dominate these kernels.
#include "common.h"
#include "launchers.h"

#ifndef SIGOPS_PROG_GROUP
#error "compile with -DSIGOPS_PROG_GROUP=0..3"
#endif

namespace sigops {

template <int M>
void launch_iir_tma_prog(dim3 grid, cudaStream_t st, const IirTmaParams& Q) {
    ensure_dyn_smem(k_iir_tma<M, IIR_WARM, false, true>, kTmaSmemBytes);
    k_iir_tma<M, IIR_WARM, false, true><<<grid, kTmaThreads, kTmaSmemBytes, st>>>(Q);
    CUDA_OK(cudaGetLastError());
}

template void launch_iir_tma_prog<2 * SIGOPS_PROG_GROUP + 1>(dim3, cudaStream_t, const IirTmaParams&);
template void launch_iir_tma_prog<2 * SIGOPS_PROG_GROUP + 2>(dim3, cudaStream_t, const IirTmaParams&);

}  // namespace sigops
