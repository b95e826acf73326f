/*
 * ba_port.h — the few spellings that differ between the product build (nvcc, sm_100a) and the development-time
 * thread emulation used by tests/emu (g++ -DBA_EMU, see tests/emu/cuda_emu.h; never part of libba_cuda.so).
 */
#ifndef BA_PORT_H
#define BA_PORT_H

#ifdef BA_EMU
#include "cuda_emu.h"
#define BA_SHARED(name) unsigned char* name = emu::tls().cta->smem
#define BA_LAUNCH(kern, grid, block, smem, stream, ...)                                  \
    do {                                                                                  \
        if (emu::launch_allowed((const void*)(kern), (size_t)(smem)))                     \
            emu::launch(dim3(grid), dim3(block), (size_t)(smem), [=]() { kern(__VA_ARGS__); }); \
    } while (0)
#define BA_BAR_SYNC(id, count) emu::bar_named((id), (count))
#define BA_CTA_SYNC_ONCE(id, threads) __syncthreads()
/* cp.async: global -> shared without passing through registers; synchronous in the emulation */
#define BA_CP_ASYNC_8(smem_ptr, gmem_ptr) memcpy((smem_ptr), (gmem_ptr), 8)
#define BA_CP_ASYNC_4(smem_ptr, gmem_ptr) memcpy((smem_ptr), (gmem_ptr), 4)
#define BA_CP_ASYNC_16(smem_ptr, gmem_ptr) memcpy((smem_ptr), (gmem_ptr), 16)
#define BA_CP_ASYNC_COMMIT() ((void)0)
#define BA_CP_ASYNC_WAIT(n) ((void)0)
/* mbarrier + bulk copy: the emulated copy is done by the issuing thread on the spot; every use in the kernels has a
 * __syncthreads() between the issue and the first read, so the wait has nothing left to do */
#define BA_MBAR_INIT(bar, count) ((void)(bar))
#define BA_FENCE_MBAR_INIT() ((void)0)
#define BA_MBAR_EXPECT_TX(bar, bytes) ((void)(bar))
#define BA_BULK_G2S(dst, src, bytes, bar) memcpy((dst), (src), (bytes))
#define BA_MBAR_WAIT(bar, parity) ((void)(bar))
/* flags in shared memory that one warp of a CTA publishes and another polls (the chunk FIFO between the demodulator's stages) */
#define BA_FLAG_LOAD(p) __atomic_load_n((p), __ATOMIC_ACQUIRE)
#define BA_FLAG_STORE(p, v) __atomic_store_n((p), (v), __ATOMIC_RELEASE)
#define BA_SPIN_PAUSE() std::this_thread::yield()
static inline unsigned atomicAdd(unsigned* p, unsigned v) {
    return __atomic_fetch_add(p, v, __ATOMIC_RELAXED);
}
/* peer access between emulated devices (one address space: every pair can reach each other).  BA_EMU_NO_PEER set to a
 * non-zero value makes cudaDeviceCanAccessPeer answer 0, so that a test can see the engine refuse a GPU pair without it. */
enum { cudaErrorPeerAccessAlreadyEnabled = 704 };
static inline cudaError_t cudaDeviceCanAccessPeer(int* can, int d, int peer) {
    const char* v = getenv("BA_EMU_NO_PEER");
    if (d < 0 || d >= emu::device_count() || peer < 0 || peer >= emu::device_count())
        return cudaErrorInvalidValue;
    *can = (d != peer && !(v && atoi(v) != 0)) ? 1 : 0;
    return cudaSuccess;
}
static inline cudaError_t cudaDeviceEnablePeerAccess(int peer, unsigned) {
    if (peer < 0 || peer >= emu::device_count() || peer == emu::current_device())
        return cudaErrorInvalidValue;
    return cudaSuccess;
}
static inline unsigned __byte_perm(unsigned x, unsigned y, unsigned s) {
    const unsigned long long src = ((unsigned long long)y << 32) | x;
    unsigned r = 0;
    for (int i = 0; i < 4; i++)
        r |= (unsigned)((src >> (8 * ((s >> (4 * i)) & 7))) & 0xffu) << (8 * i);
    return r;
}
#else
#include <cuda_runtime.h>
#define BA_SHARED(name) extern __shared__ __align__(16) unsigned char name[]
#define BA_LAUNCH(kern, grid, block, smem, stream, ...) kern<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__)
#define BA_BAR_SYNC(id, count) asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory")
/* every thread of the CTA, before any subset starts using barrier `id` with its own count (a completed barrier can be reused with another count) */
#define BA_CTA_SYNC_ONCE(id, threads) BA_BAR_SYNC((id), (threads))
/* flags in shared memory that one warp of a CTA publishes and another polls (the chunk FIFO between the demodulator's stages):
 * release/acquire at CTA scope orders the slot's contents with the counter */
static __device__ __forceinline__ int ba_flag_load(const int* p) {
    int v;
    asm volatile("ld.acquire.cta.shared.b32 %0, [%1];" : "=r"(v) : "r"((unsigned)__cvta_generic_to_shared(p)) : "memory");
    return v;
}
static __device__ __forceinline__ void ba_flag_store(int* p, int v) {
    asm volatile("st.release.cta.shared.b32 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(p)), "r"(v) : "memory");
}
#define BA_FLAG_LOAD(p) ba_flag_load(p)
#define BA_FLAG_STORE(p, v) ba_flag_store((p), (v))
/* a chunk of the demodulator's pipelines takes well under a microsecond: no sleep between polls */
#define BA_SPIN_PAUSE() ((void)0)
#define BA_CP_ASYNC_8(smem_ptr, gmem_ptr) \
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(smem_ptr)), "l"(gmem_ptr) : "memory")
#define BA_CP_ASYNC_4(smem_ptr, gmem_ptr) \
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((unsigned)__cvta_generic_to_shared(smem_ptr)), "l"(gmem_ptr) : "memory")
#define BA_CP_ASYNC_16(smem_ptr, gmem_ptr) \
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(smem_ptr)), "l"(gmem_ptr) : "memory")
#define BA_CP_ASYNC_COMMIT() asm volatile("cp.async.commit_group;" ::: "memory")
#define BA_CP_ASYNC_WAIT(n) asm volatile("cp.async.wait_group %0;" ::"n"(n) : "memory")
/* mbarrier + TMA bulk copy (global -> shared, 16-byte granules, completion counted in bytes on the mbarrier) */
#define BA_MBAR_INIT(bar, count) \
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"((unsigned)(count)) : "memory")
#define BA_FENCE_MBAR_INIT() asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory")
#define BA_MBAR_EXPECT_TX(bar, bytes) \
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"((unsigned)(bytes)) : "memory")
#define BA_BULK_G2S(dst, src, bytes, bar)                                                                                    \
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(         \
                     (unsigned)__cvta_generic_to_shared(dst)),                                                               \
                 "l"(src), "r"((unsigned)(bytes)), "r"((unsigned)__cvta_generic_to_shared(bar))                           \
                 : "memory")
#define BA_MBAR_WAIT(bar, parity)                                                                       \
    asm volatile(                                                                                       \
        "{\n"                                                                                           \
        ".reg .pred P1;\n"                                                                              \
        "LAB_WAIT:\n"                                                                                   \
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"                                      \
        "@P1 bra DONE;\n"                                                                               \
        "bra LAB_WAIT;\n"                                                                               \
        "DONE:\n"                                                                                       \
        "}" ::"r"((unsigned)__cvta_generic_to_shared(bar)),                                             \
        "r"((unsigned)(parity))                                                                         \
        : "memory")
#endif

#endif
