// ptx.cuh — the asynchronous-copy and synchronisation primitives of the SpMV kernels (spmv.cu, gather.cu, peer.cu):
// TMA bulk copies (cp.async.bulk) with mbarrier completion, bulk groups for the shared -> global direction, the L2
// bulk prefetch and cache policy, programmatic dependent launch, and the device flag barrier between ranks.
#pragma once

#include <cstdint>

namespace spl {

__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}

// ---- mbarrier.  A kernel initialises its barriers, then calls mbar_init_fence() once before any other thread or a
// bulk copy uses them.
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_init_fence() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

// ---- bulk copies.  global -> shared completes on an mbarrier (complete_tx bytes); shared -> global goes into the
// thread's bulk group: commit, then wait until the stores are written (bulk_wait_all) or until all but the newest
// group have read their shared-memory source (bulk_wait_read_but_one).
__device__ __forceinline__ void tma_bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s_hint(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar,
                                                  uint64_t policy) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
            smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
        : "memory");
}
__device__ __forceinline__ void tma_bulk_s2g(void *dst_gmem, const void *src_smem, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem),
                 "r"(smem_u32(src_smem)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read_but_one() {
    asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
}

// ---- L2: bulk prefetch, and the eviction policy of data read once (a matrix stream should not push the re-read x
// out of L2)
__device__ __forceinline__ void l2_prefetch_bulk(const void *gmem, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(gmem), "r"(bytes) : "memory");
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}

// ---- programmatic dependent launch
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void griddep_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

__device__ __forceinline__ uint32_t ld_acquire_gpu(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ uint64_t global_timer_ns() {
    uint64_t t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// ---- the flag barrier between ranks.  Every rank owns a block of flag words in peer-visible memory; word g of
// rank r's block holds the last epoch at which rank g arrived.  Arrival: make this rank's earlier writes visible
// system-wide, then release-store the epoch into word `rank` of the peer's block.  Wait: acquire-load the own
// block's word of one peer until it reaches the epoch (wrap-around safe), bounded by `timeout_ns` so that a missing
// peer never hangs the GPU: on a timeout *failed is set and the call returns false.
__device__ __forceinline__ void flag_arrive(uint32_t *peer_block, int rank, uint32_t epoch) {
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(peer_block + rank), "r"(epoch) : "memory");
}
__device__ __forceinline__ bool flag_wait(const uint32_t *slot, uint32_t epoch, uint64_t timeout_ns, unsigned sleep_ns,
                                          uint32_t *failed) {
    const uint64_t t0 = global_timer_ns();
    for (;;) {
        uint32_t v;
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(slot) : "memory");
        if ((int32_t)(v - epoch) >= 0) return true;
        if (global_timer_ns() - t0 > timeout_ns) {
            atomicExch(failed, 1u);
            return false;
        }
        __nanosleep(sleep_ns);
    }
}

}  // namespace spl
