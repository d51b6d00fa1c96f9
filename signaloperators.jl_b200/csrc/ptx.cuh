// PTX wrappers shared by the IIR and FIR kernels: mbarriers, bulk and tensor-map copies, cp.async,
// the FP64 tensor-core MMA and explicit shared-memory accesses.  Each instruction form is written once;
// where a kernel keeps shared-memory addresses as 32-bit shared-window addresses (k_fir_tmap), that is
// the form defined here and the pointer form calls it.
#pragma once
#include <cuda.h>

#include <cstdint>

namespace sigops {

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }

// ---- mbarriers
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbarrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) { mbar_arrive(smem_u32(bar)); }
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra LAB_DONE;\n"
        "bra LAB_WAIT;\n"
        "LAB_DONE:\n"
        "}\n" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) { mbar_wait(smem_u32(bar), parity); }
// the barrier counts the calling thread's cp.async copies in and completes them as they land
__device__ __forceinline__ void cp_async_mbar_arrive(uint64_t* bar) {
    asm volatile("cp.async.mbarrier.arrive.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// ---- bulk copies (completion of loads: complete_tx on an mbarrier; of stores: bulk groups)
__device__ __forceinline__ void bulk_load(unsigned smem_dst, const void* gsrc, unsigned bytes, unsigned bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_dst),
                 "l"(gsrc), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gsrc, unsigned bytes, uint64_t* bar) {
    bulk_load(smem_u32(smem_dst), gsrc, bytes, smem_u32(bar));
}
__device__ __forceinline__ void bulk_store(void* gdst, const void* smem_src, unsigned bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_u32(smem_src)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// generic-proxy writes to shared memory become visible to the TMA unit (and the other way round)
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- tensor-map copies
__device__ __forceinline__ void tmap_load_2d(unsigned smem_dst, const CUtensorMap* tm, int c0, int c1, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(smem_dst),
                 "l"(tm), "r"(c0), "r"(c1), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tmap_store_2d(const CUtensorMap* tm, int c0, int c1, unsigned smem_src) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];" ::"l"(tm), "r"(c0), "r"(c1), "r"(smem_src)
                 : "memory");
}
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

// ---- cp.async
__device__ __forceinline__ void cp_async8(double* smem_dst, const double* gmem_src, bool valid) {
    const unsigned dst = (unsigned)__cvta_generic_to_shared(smem_dst);
    const int src_size = valid ? 8 : 0;       // src_size 0 => the 8 bytes are zero-filled, nothing is read
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(dst), "l"(gmem_src), "r"(src_size) : "memory");
}
__device__ __forceinline__ void cp_async16(double* smem_dst, const double* gmem_src, int src_bytes) {
    const unsigned dst = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(gmem_src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait_group() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// ---- FP64 tensor cores: C (8x8, two elements per lane) += A (8x4) * B (4x8), one element of each per lane
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
// sum over the four lanes of a quad (lane ^ 1, lane ^ 2): the lanes that share a row of a DMMA fragment
__device__ __forceinline__ double quad_sum(double v) {
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    return v;
}

// ---- shared memory through 32-bit shared-window addresses
__device__ __forceinline__ double lds_f64(unsigned a) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts_f64(unsigned a, double v) { asm volatile("st.shared.f64 [%0], %1;" ::"r"(a), "d"(v) : "memory"); }
__device__ __forceinline__ void sts_v2f64(unsigned a, double x, double y) {
    asm volatile("st.shared.v2.f64 [%0], {%1, %2};" ::"r"(a), "d"(x), "d"(y) : "memory");
}

}  // namespace sigops
