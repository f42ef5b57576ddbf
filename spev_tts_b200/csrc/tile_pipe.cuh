// tile_pipe.cuh -- persistent-tile plumbing shared by the FFT kernels: cp.async (LDGSTS) helpers
// with zero fill, the 4-slot tile-descriptor ring, L2 prefetch and programmatic-dependent-launch
// hooks.
#pragma once
#include "spev_internal.cuh"

namespace spev {

struct BatchView {
    int n_ftiles, n_ctiles;
    const spev_tile* ftiles;
    const spev_tile* ctiles;
};

static BatchView view_of(const spev_batch* b) {
    BatchView v;
    v.n_ftiles = b->n_ftiles; v.n_ctiles = b->n_ctiles;
    v.ftiles = b->ftiles; v.ctiles = b->ctiles;
    return v;
}

constexpr float kTiny = 1.17549435e-38f;   // np.finfo(np.float32).tiny
constexpr int kRing = 4;

// ---------------------------------------------------------------------------------------
// cp.async helpers (LDGSTS): zero-fill through the src-size operand
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem, int src_bytes) {
    const unsigned s = static_cast<unsigned>(__cvta_generic_to_shared(smem));
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async4(void* smem, const void* gmem, int src_bytes) {
    const unsigned s = static_cast<unsigned>(__cvta_generic_to_shared(smem));
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;\n" ::"r"(s), "l"(gmem), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;\n" ::: "memory"); }

// Warp-cooperative L2 prefetch of [p, p+bytes): moves DRAM->L2 traffic off the critical path
// (issued at tile start, consumed after the FFT phase), no registers or shared memory needed.
__device__ __forceinline__ void warp_prefetch_l2(const void* p, int bytes, int lane) {
    const uintptr_t base = reinterpret_cast<uintptr_t>(p) & ~static_cast<uintptr_t>(127);
    const int n = static_cast<int>((reinterpret_cast<uintptr_t>(p) + bytes - base + 127) >> 7);
    for (int i = lane; i < n; i += 32)
        asm volatile("prefetch.global.L2 [%0];\n" ::"l"(base + (static_cast<uintptr_t>(i) << 7)));
}

__device__ __forceinline__ void fetch_desc(spev_tile* slot, const spev_tile* g) {
    static_assert(sizeof(spev_tile) == 48, "spev_tile must be 48 bytes");
    if (threadIdx.x == 0) {
        cp_async16(reinterpret_cast<char*>(slot), reinterpret_cast<const char*>(g), 16);
        cp_async16(reinterpret_cast<char*>(slot) + 16, reinterpret_cast<const char*>(g) + 16, 16);
        cp_async16(reinterpret_cast<char*>(slot) + 32, reinterpret_cast<const char*>(g) + 32, 16);
    }
}

// Programmatic dependent launch: a kernel launched with the stream-serialization attribute may
// start while its predecessor is still draining; everything before pdl_wait() must only touch
// data the predecessor does not write (constant tables, tile descriptors).
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;\n" ::: "memory"); }

// ---------------------------------------------------------------------------------------
// shared-memory mbarriers, completed by the bulk asynchronous copies below
// (waits are bounded: a protocol bug traps instead of hanging)
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_addr(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void bar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_addr(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void bar_wait(uint64_t* bar, uint32_t parity) {
    const uint32_t addr = smem_addr(bar);
    uint32_t done = 0;
    for (uint32_t spin = 0; !done; ++spin) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.acquire.cta.shared::cta.b64 p, [%1], %2, %3;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}\n"
            : "=r"(done) : "r"(addr), "r"(parity), "r"(200000u) : "memory");   // sleep in hardware (<= 200 us) instead of polling
        if (spin > (1u << 22)) asm volatile("trap;\n");
    }
}

// Bulk asynchronous copy global -> shared (the TMA unit's 1-D path): one instruction moves up to a whole row,
// needs no registers and no LSU issue slots, and signals an mbarrier with the byte count.  Addresses and size must
// be multiples of 16 bytes.
__device__ __forceinline__ void bar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
                 ::"r"(smem_addr(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_addr(bar)) : "memory");
}
// L2 eviction policies (createpolicy): the Griffin-Lim loop streams 106 MB of momentum spectra per iteration through
// an L2 that could otherwise keep its 73 MB producer -> consumer working set (S, pair segments, y) resident.
__device__ __forceinline__ uint64_t l2_policy_evict_first() {   // streaming data
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;\n" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {    // data read again soon
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;\n" : "=l"(p));
    return p;
}
__device__ __forceinline__ void bulk_g2s_hint(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar, uint64_t pol) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;\n"
                 ::"r"(smem_addr(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_addr(bar)), "l"(pol) : "memory");
}
__device__ __forceinline__ void st_hint(float2* p, float2 v, uint64_t pol) {
    asm volatile("st.global.L2::cache_hint.v2.f32 [%0], {%1, %2}, %3;\n" ::"l"(p), "f"(v.x), "f"(v.y), "l"(pol) : "memory");
}
__device__ __forceinline__ void st_hint(float* p, float v, uint64_t pol) {
    asm volatile("st.global.L2::cache_hint.f32 [%0], %1, %2;\n" ::"l"(p), "f"(v), "l"(pol) : "memory");
}
// generic-proxy accesses (LDS/STS) before this point are ordered before later async-proxy (bulk copy) accesses
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory"); }

// Dynamic work distribution without a reset between launches: the counter only ever grows; launch number j of a
// kernel draws tickets base_j, base_j + 1, ... where base_j is computed on the host.  Every worker (warp or CTA)
// stops at its first ticket >= n_work, so a launch consumes exactly n_work + n_workers tickets.
__device__ __forceinline__ unsigned draw_ticket(unsigned* counter, unsigned base) { return atomicAdd(counter, 1u) - base; }

// Persistent-loop bookkeeping shared by the kernels: prologue of the descriptor ring.
__device__ __forceinline__ int ring_prologue(spev_tile* s_ring, const spev_tile* tiles, int n_tiles) {
    const int first = blockIdx.x, stride = gridDim.x;
    const int my_n = first < n_tiles ? (n_tiles - first + stride - 1) / stride : 0;
    for (int j = 0; j < 3 && j < my_n; ++j) fetch_desc(s_ring + j, tiles + first + j * stride);
    cp_async_commit();
    cp_async_wait_all();
    __syncthreads();
    return my_n;
}

}  // namespace spev
