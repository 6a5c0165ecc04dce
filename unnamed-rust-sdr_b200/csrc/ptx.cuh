// ptx.cuh -- the Blackwell (sm_100a) PTX wrappers of the tensor-core and TMA kernels: mbarriers, cp.async, TMA bulk and
// tensor copies, tcgen05 MMA / TMEM, elect.sync, shared-memory matrix and instruction descriptors, and the host-side
// resolution of cuTensorMapEncodeTiled.  Every kernel spells these instructions through this header only.
#pragma once
#include <cuda.h>  // CUtensorMap and the cuTensorMapEncodeTiled prototype only: the entry point is resolved at run time
#include <cuda_runtime.h>
#include <stdint.h>

namespace sdr {

#ifdef __CUDACC__

// ---- addresses -------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier --------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
// makes the initialised barriers visible to the other threads and to the async proxy
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done = 0;
    while (!done)
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
                     : "=r"(done) : "r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}

// ---- async proxy -----------------------------------------------------------------------------------------------------
// this thread's generic-proxy accesses of shared memory before later async-proxy ones (tensor copies, tcgen05.mma)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// the same for every state space: global stores (acquired from other SMs) before this thread's tensor-copy reads of them
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }

// ---- cp.async --------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void cp_async16_s(uint32_t dst, const void *src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gmem_src) {
    cp_async16_s(smem_u32(smem_dst), gmem_src);
}
__device__ __forceinline__ void cp_async8(void *smem_dst, const void *gmem_src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async4(void *smem_dst, const void *gmem_src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(smem_dst)), "l"(gmem_src) : "memory");
}
// reads src_bytes (0 or 8) bytes and zero-fills the rest of the 8
__device__ __forceinline__ void cp_async8_zfill(uint32_t dst, const void *src, uint32_t src_bytes) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
// one arrival on the mbarrier once all of this thread's earlier cp.asyncs have landed (no pending-count increment)
__device__ __forceinline__ void cp_async_arrive_noinc(uint32_t bar) {
    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// ---- TMA: global -> shared, completion in bytes on an mbarrier --------------------------------------------------------
// non-tensor form: one linear bulk copy.  SASS: UBLKCP.
__device__ __forceinline__ void tma_bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
// tensor copies of one box of a tensor map.  SASS: UTMALDG.
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap *tm, int c0, int c1, int c2, uint32_t bar) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                 ::"r"(dst), "l"(tm), "r"(c0), "r"(c1), "r"(c2), "r"(bar) : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap *tm, int c0, int c1, int c2, int c3, uint32_t bar) {
    asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
                 ::"r"(dst), "l"(tm), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(bar) : "memory");
}

// ---- tcgen05 ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// one arrival on the mbarrier once this thread's earlier tcgen05.mma have completed
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc], u8 x s8 -> s32; the accumulate flag is fixed at compile time (no setp on
// the issuing thread's critical path)
template <bool ACC>
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc) {
    if (ACC)
        asm volatile("{\n .reg .pred p;\n setp.eq.u32 p, 1, 1;\n tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n}\n"
                     ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc) : "memory");
    else
        asm volatile("{\n .reg .pred p;\n setp.eq.u32 p, 1, 0;\n tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n}\n"
                     ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc) : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc], bf16 x bf16 -> f32
template <bool ACC>
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc) {
    if (ACC)
        asm volatile("{\n .reg .pred p;\n setp.eq.u32 p, 1, 1;\n tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}\n"
                     ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc) : "memory");
    else
        asm volatile("{\n .reg .pred p;\n setp.eq.u32 p, 1, 0;\n tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}\n"
                     ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc) : "memory");
}
// 8 consecutive columns of one TMEM lane per thread
__device__ __forceinline__ void tmem_ld_32x32b_x8(uint32_t taddr, uint32_t *v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_16x256b_x2(uint32_t taddr, uint32_t (&v)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.16x256b.x2.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// whole warp: allocate COLS TMEM columns (base address written to shared memory at dst) and give up the permit, so
// that the other CTA on the SM can allocate too
template <int COLS>
__device__ __forceinline__ void tmem_alloc(uint32_t dst) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst), "n"(COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(COLS) : "memory");
}
// one lane of a converged warp (elect.sync): unlike `lane == 0`, ptxas KNOWS a single thread follows the branch, so the
// tcgen05.mma operands stay in uniform registers and no per-instruction election loop is emitted around them
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n .reg .pred p;\n elect.sync _|p, 0xffffffff;\n selp.u32 %0, 1, 0, p;\n}\n" : "=r"(pred));
    return pred != 0;
}

// ---- descriptors -----------------------------------------------------------------------------------------------------
// shared-memory matrix descriptor (K-major): start address, leading / stride byte offsets (16-byte units), version 1
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo, uint32_t layout) {
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)((lbo >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((sbo >> 4) & 0x3FFFu) << 32) | ((uint64_t)1 << 46) | ((uint64_t)layout << 61);
}
// K-major rows of PITCH_BYTES: the descriptor's layout type and the XOR that places byte offset o of the flat copy
// (16: no swizzle, 32: SWIZZLE_32B, 64: SWIZZLE_64B; the XOR depends on the absolute address, so overlapping rows agree)
template <int PITCH_BYTES> struct SmemLayout;
template <> struct SmemLayout<16> { static constexpr uint32_t type = 0; __device__ static uint32_t swz(uint32_t o) { return o; } };
template <> struct SmemLayout<32> { static constexpr uint32_t type = 6; __device__ static uint32_t swz(uint32_t o) { return o ^ (((o >> 7) & 1u) << 4); } };
template <> struct SmemLayout<64> { static constexpr uint32_t type = 4; __device__ static uint32_t swz(uint32_t o) { return o ^ (((o >> 7) & 3u) << 4); } };

#endif  // __CUDACC__

// tcgen05 instruction descriptors (dense, K-major A and B): D type at bits 4-5, A type 7-9, B type 10-12, N >> 3 at 17,
// M >> 4 at 24
__host__ __device__ constexpr uint32_t idesc_u8s8_s32(int M, int N) {  // s32 += u8 x s8
    return (2u << 4) | (0u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__host__ __device__ constexpr uint32_t idesc_bf16_f32(int M, int N) {  // f32 += bf16 x bf16
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// ---- host ------------------------------------------------------------------------------------------------------------
// cuTensorMapEncodeTiled, resolved through the runtime (no link-time dependency on libcuda); null = not available
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
inline EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = []() -> EncodeTiledFn {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) {
            cudaGetLastError();
            return nullptr;
        }
        return (EncodeTiledFn)p;
    }();
    return fn;
}

}  // namespace sdr
