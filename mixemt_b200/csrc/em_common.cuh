// What the two translation units of the EM fit share: the control block of a restart, the
// PTX helpers of the fp64-row (em_kernels.cuh) and class-tile (em_tiles.cuh) kernels, and the
// launch helper of em.cu and em_tiles.cu.
#pragma once

#include <stdint.h>
#include <stdlib.h>

#include "common.cuh"

namespace mxb {

// Device-resident control block: lets every kernel of an iteration early-exit
// once the run has converged, so iterations can be enqueued ahead of the host.
constexpr int kDoneNeedsLogStep = 4;

struct EmState {
    int done;            // 0 running, 1 converged, 2 max_iter reached, 3 peer time-out,
                         // 4 the current iteration must be redone in log space
    int cur;             // index of the current (input) proportions buffer
    int bad;             // rows that cannot be carried in linear space (row_needs_logspace)
    int pad;
    long long iters;
    long long max_iter;
    double tol;
    double delta;
};

// ---- small PTX helpers ------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;"
                 ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra WAIT_DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "WAIT_DONE:\n\t"
        "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// 1-D bulk async copy global -> shared, completion counted on an mbarrier.
__device__ __forceinline__ void bulk_load(void *dst_smem, const void *src, uint32_t bytes,
                                          uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
        ::"r"(smem_u32(dst_smem)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void mbar_expect_tx_u32(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait_u32(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra WAIT_DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "WAIT_DONE:\n\t"
        "}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_load_u32(uint32_t dst_smem, const void *src, uint32_t bytes,
                                              uint32_t bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
        ::"r"(dst_smem), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

// Programmatic dependent launch: a kernel launched with the stream-serialization attribute
// may start while its predecessor in the stream is still running; it must not touch what the
// predecessor writes before pdl_wait().  Both are no-ops in a plain launch.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

__device__ __forceinline__ void mbar_init_fence() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_u32(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// loads through 32-bit shared-window addresses (record base, warp-uniform, + per-thread offset:
// ptxas folds the sum into the [R + UR] form of LDS)
__device__ __forceinline__ uint2 lds_v2_u32(uint32_t addr) {
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ double2 lds_v2_f64(uint32_t addr) {
    double2 v;
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(addr) : "memory");
    return v;
}

inline bool pdl_enabled() {   // MXB_EM_NO_PDL=1 turns the attribute off (plain stream order)
    static const bool on = getenv("MXB_EM_NO_PDL") == nullptr;
    return on;
}
// Launch in plain stream order, or (pdl) with the programmatic-stream-serialization attribute
// (see pdl_wait): the kernel may then be scheduled before its predecessor in the stream has
// finished.
template <typename... KArgs, typename... Args>
cudaError_t launch_kernel(bool pdl, void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem,
                          cudaStream_t s, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl && pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

}  // namespace mxb
