// Shared device helpers for libvn_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdarg>
#include <cstdio>

#include "vn_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libvn_b200 is written for sm_100a (B200) only"
#endif

namespace vn {

void set_error(const char *fmt, ...);
// Counts a kernel launch whose enqueue returned `e`; VN_ECUDA with `what` in vn_last_error when it failed.
int32_t launch_result(const char *what, cudaError_t e);
// Whether every pointer is 16-byte aligned (a null pointer is).
template <typename... P>
inline bool aligned16(const P *...p) {
    return ((reinterpret_cast<uintptr_t>(p) | ... | uintptr_t(0)) & 15) == 0;
}
int sm_count();  // multiprocessors of the current device (cached per device)
// Raises the kernel's dynamic shared-memory limit on the current device to `bytes` unless an earlier call did; a size
// is remembered only once the attribute was set.  VN_ECUDA with a message when it cannot be set.
int32_t ensure_smem(const void *kernel, int bytes);
template <typename... KArgs>
int32_t ensure_smem(void (*kernel)(KArgs...), int bytes) {
    return ensure_smem(reinterpret_cast<const void *>(kernel), bytes);
}
// CTAs of `smem` bytes of dynamic shared memory that fit on one SM (220 KB usable, ~1 KB reserved per CTA), 1 .. cap.
inline int ctas_per_sm(int smem, int cap = 32) {
    const int fit = (220 * 1024) / (smem + 1024);
    return fit < 1 ? 1 : (fit < cap ? fit : cap);
}

// Launches kernel(args...) on `stream` and counts it.  programmatic: the kernel may be scheduled while its predecessor
// in the stream is still running (programmatic dependent launch); it synchronises itself with griddepcontrol.wait.
template <typename... KArgs, typename... Args>
int32_t launch(void (*kernel)(KArgs...), const char *name, dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
               bool programmatic, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = programmatic ? 1 : 0;
    cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
    const cudaError_t last = cudaGetLastError();  // also clears what a failed launch left behind
    return launch_result(name, e != cudaSuccess ? e : last);
}
// All float leaves of one step in one launch (vn_rollout.cu); in_step = enqueued by vn_env_reset / vn_env_step* right
// after the kernels that wrote `desc` (programmatic launch, releases its stream successor early).
int32_t launch_float_leaves(const vn_store_t *store, const vn_float_leaf_t *leaves, int32_t n_leaves, const int32_t *desc,
                            int32_t n, int32_t h, int32_t w, void *stream, bool in_step);

#define VN_REQUIRE(cond, ...)            \
    do {                                 \
        if (!(cond)) {                   \
            ::vn::set_error(__VA_ARGS__); \
            return VN_EINVAL;            \
        }                                \
    } while (0)

// ---------------------------------------------------------------- 16-byte streaming loads / stores
// Frames are read once per gather from the HBM-resident store (read-only for the kernel's lifetime):
// ld.global.nc + L1::no_allocate keeps them out of L1; the batch rows are written once and consumed by
// a later kernel (the policy), so they go straight to L2.
__device__ __forceinline__ int4 ld_stream16(const void *p) {
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ void st_stream16(void *p, const int4 &v) {
    asm volatile("st.global.L1::no_allocate.v4.s32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z),
                 "r"(v.w)
                 : "memory");
}

// ---------------------------------------------------------------- splitmix64 frame hash (scenes.py)
__host__ __device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ull;
    uint64_t z = x;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
__host__ __device__ __forceinline__ uint64_t frame_key(uint64_t seed, uint32_t scene, uint64_t state, uint32_t plane) {
    uint64_t k = splitmix64(seed ^ ((uint64_t)scene * 0xD1B54A32D192ED03ull));
    k = splitmix64(k ^ (state * 0x8CB92BA72F3D8DD7ull));
    return splitmix64(k ^ (uint64_t)(plane + 1));
}

// ---------------------------------------------------------------- Philox4x32-10 (counter-based RNG)
struct Philox4 {
    uint32_t v[4];
};
__device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                                 uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0;
        c1 = lo1;
        c2 = n2;
        c3 = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    Philox4 o;
    o.v[0] = c0;
    o.v[1] = c1;
    o.v[2] = c2;
    o.v[3] = c3;
    return o;
}

// ---------------------------------------------------------------- mbarrier + bulk async copy (TMA engine)
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
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
// global -> shared, completion counted in bytes on the mbarrier
__device__ __forceinline__ void bulk_g2s(void *smem_dst, const void *gmem_src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// shared -> global, tracked by the per-thread bulk async-group
__device__ __forceinline__ void bulk_s2g(void *gmem_dst, const void *smem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst),
                 "r"(smem_u32(smem_src)), "r"(bytes)
                 : "memory");
}
// L2 cache-policy variants.  The store is re-read across envs and steps while a batch row is written once and
// consumed later by another kernel: loads are tagged evict_last and stores evict_first so that, when store +
// batch exceed the 126 MB L2, it is the written rows that leave first and the frames that stay.
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ void bulk_g2s_hint(void *smem_dst, const void *gmem_src, uint32_t bytes, uint64_t *bar,
                                              uint64_t policy) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
            smem_u32(smem_dst)),
        "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
        : "memory");
}
__device__ __forceinline__ void bulk_s2g_hint(void *gmem_dst, const void *smem_src, uint32_t bytes, uint64_t policy) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;" ::"l"(gmem_dst),
                 "r"(smem_u32(smem_src)), "r"(bytes), "l"(policy)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

}  // namespace vn
