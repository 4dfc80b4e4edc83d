// b200sd -- shared device/host helpers for the sm_100a kernels.
// Inline-PTX wrappers for mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld)
// and small bf16 utilities.  Everything here is written for sm_100a only.
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/b200sd.h"

typedef __nv_bfloat16 bf16;

// ----------------------------------------------------------------------------------------------
// host-side error plumbing (no exceptions cross the C ABI)
// ----------------------------------------------------------------------------------------------
void b200sd_set_error(const char* fmt, ...);

#define B200SD_REQUIRE(cond, ...)                       \
    do {                                                \
        if (!(cond)) {                                  \
            b200sd_set_error(__VA_ARGS__);              \
            return B200SD_ERR_INVALID;                  \
        }                                               \
    } while (0)

#define B200SD_CUDA(call)                                                                   \
    do {                                                                                    \
        cudaError_t e__ = (call);                                                           \
        if (e__ != cudaSuccess) {                                                           \
            b200sd_set_error("%s:%d CUDA error %s", __FILE__, __LINE__, cudaGetErrorString(e__)); \
            return B200SD_ERR_CUDA;                                                         \
        }                                                                                   \
    } while (0)

#define B200SD_LAUNCH_CHECK() B200SD_CUDA(cudaGetLastError())

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

// number of SMs of the current device (cached)
int b200sd_num_sms();

// Encode a tiled TMA descriptor (driver entry point fetched through the runtime; no -lcuda needed).
// dims/strides are innermost-first; strides are in bytes for dims 1..rank-1.
int b200sd_make_tmap(CUtensorMap* out, const void* base, int rank, const uint64_t* dims,
                     const uint64_t* strides_bytes, const uint32_t* box, CUtensorMapSwizzle swizzle,
                     CUtensorMapDataType dtype = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16);

#ifdef __CUDACC__
// The opt-in to > 48 KB of dynamic shared memory is a per-DEVICE attribute of a kernel function: set it once per (kernel
// instantiation, device), under a mutex (the C ABI may be called from several threads, and a process may drive several GPUs).
// (Keyed on the kernel's ADDRESS, not on its type: instantiations of one kernel template share a function-pointer type.)
cudaError_t b200sd_opt_in_smem_impl(const void* kernel, int bytes, bool max_carveout);
template <typename K>
static inline cudaError_t b200sd_opt_in_smem(K kernel, int bytes, bool max_carveout = false) {
    return b200sd_opt_in_smem_impl(reinterpret_cast<const void*>(kernel), bytes, max_carveout);
}

// ----------------------------------------------------------------------------------------------
// device helpers
// ----------------------------------------------------------------------------------------------
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}\n"
        : "=r"(pred));
    return pred != 0;
}

// ---- mbarrier ----
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
// orders this thread's async-proxy accesses to GLOBAL memory (completed TMA stores) before its later generic-proxy accesses
__device__ __forceinline__ void fence_proxy_async_global() {
    asm volatile("fence.proxy.async.global;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug must never hang the GPU box -- trap after ~2 s instead.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 4000000000LL) {
            printf("b200sd: mbarrier wait timed out (block %d,%d thread %d)\n", blockIdx.x, blockIdx.y,
                   threadIdx.x);
            __trap();
        }
    }
}

// ---- TMA ----
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2,
                                            int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], "
        "[%2];" ::"r"(smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}

// ---- TMA store: smem tile -> global through a tensor map (bulk async-group completion) ----
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(m)),
                 "r"(smem_u32(src)), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// wait until at most N of this thread's committed bulk groups are still READING their smem source
template <int N>
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
// wait until at most N committed bulk groups are still in flight at all (writes performed)
template <int N>
__device__ __forceinline__ void tma_store_wait() { asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory"); }

// ---- CTA-pair (cta_group::2) variants: both CTAs of a pair issue their own loads into their own smem, the
// transaction bytes are signalled on the LEADER's mbarrier (a shared::cluster address obtained with mapa) ----
__device__ __forceinline__ uint32_t mapa_u32(uint32_t local_smem_addr, uint32_t cta_rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_smem_addr), "r"(cta_rank));
    return r;
}
__device__ __forceinline__ void tma_load_2d_cg2(void* dst, const CUtensorMap* m, uint32_t bar_cluster_addr, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_3d_cg2(void* dst, const CUtensorMap* m, uint32_t bar_cluster_addr, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d_cg2(void* dst, const CUtensorMap* m, uint32_t bar_cluster_addr, int c0, int c1, int c2,
                                                int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], "
        "[%2];" ::"r"(smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tmem_alloc_cg2(uint32_t* dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish_cg2() {
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_cg2(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem of both CTAs] (+)= A * B^T with M = 256 (128 rows per CTA), B rows split across the pair; leader CTA only
__device__ __forceinline__ void umma_bf16_ss_cg2(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                                 uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrive (once all previously issued MMAs of this thread completed) on the same mbarrier of every CTA in `cta_mask`
__device__ __forceinline__ void umma_commit_cg2(uint64_t* bar, uint16_t cta_mask) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
                 "h"(cta_mask)
                 : "memory");
}

// ---- tcgen05 ----
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
                 "r"(ncols)
                 : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, bf16 inputs, fp32 accumulate, issued by ONE thread.
__device__ __forceinline__ void umma_bf16_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                             uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]^T
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                             uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n" ::"r"(tmem_d),
        "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrive on an mbarrier once all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// 32 lanes x 16 consecutive 32-bit columns -> 16 registers / thread (thread i <-> lane base+i)
__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, "
        "%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x8(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr)
                 : "memory");
}

// UMMA shared-memory descriptor, K-major operand, 128-byte swizzle, 64 bf16 (=128 B) per row,
// 8-row groups 1024 B apart (the layout a SWIZZLE_128B TMA box of inner extent 64 produces).
__device__ __forceinline__ uint64_t umma_desc_k_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);  // start address  [0,14)
    d |= (uint64_t)1 << 16;                       // LBO (unused for swizzled K-major) = 1
    d |= (uint64_t)(1024 >> 4) << 32;             // SBO = 1024 B   [32,46)
    d |= (uint64_t)1 << 46;                       // descriptor version (Blackwell)
    d |= (uint64_t)2 << 61;                       // SWIZZLE_128B
    return d;
}
// UMMA shared-memory descriptor, MN-major operand, 128-byte swizzle: rows are 64 contiguous M/N elements
// (128 B), 8 consecutive k-rows form a 1024-byte swizzle atom (SBO = 1024 between k-groups), the next 64
// M/N elements start `lbo_bytes` further (one SWIZZLE_128B TMA box of inner extent 64 per 64 columns).
__device__ __forceinline__ uint64_t umma_desc_mn_sw128(uint32_t smem_addr, uint32_t lbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
// instruction descriptor: bf16 x bf16 -> f32, both K-major, M=128, N=n (bit 15 / 16: A / B is MN-major)
__device__ __forceinline__ uint32_t umma_idesc_bf16(uint32_t m, uint32_t n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((n >> 3) << 17) | ((m >> 4) << 24);
}

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

}  // namespace ptx

__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
    __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float2 unpack_bf16x2(uint32_t u) {
    __nv_bfloat162 v = *reinterpret_cast<__nv_bfloat162*>(&u);
    return __bfloat1622float2(v);
}
// 8 consecutive elements <-> float[8]; DT = B200SD_F32 (2 x 16 B) or B200SD_BF16 (16 B)
template <int DT>
__device__ __forceinline__ void ld8(const void* p, size_t i, float (&v)[8]) {
    if constexpr (DT == B200SD_F32) {
        const float4* q = reinterpret_cast<const float4*>(static_cast<const float*>(p) + i);
        const float4 a = __ldg(q), b = __ldg(q + 1);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
        v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    } else {
        const uint4 u = __ldg(reinterpret_cast<const uint4*>(static_cast<const bf16*>(p) + i));
        float2 f;
        f = unpack_bf16x2(u.x); v[0] = f.x; v[1] = f.y;
        f = unpack_bf16x2(u.y); v[2] = f.x; v[3] = f.y;
        f = unpack_bf16x2(u.z); v[4] = f.x; v[5] = f.y;
        f = unpack_bf16x2(u.w); v[6] = f.x; v[7] = f.y;
    }
}
template <int DT>
__device__ __forceinline__ void st8(void* p, size_t i, const float (&v)[8]) {
    if constexpr (DT == B200SD_F32) {
        float4* q = reinterpret_cast<float4*>(static_cast<float*>(p) + i);
        q[0] = make_float4(v[0], v[1], v[2], v[3]);
        q[1] = make_float4(v[4], v[5], v[6], v[7]);
    } else {
        uint4 u;
        u.x = pack_bf16x2(v[0], v[1]);
        u.y = pack_bf16x2(v[2], v[3]);
        u.z = pack_bf16x2(v[4], v[5]);
        u.w = pack_bf16x2(v[6], v[7]);
        *reinterpret_cast<uint4*>(static_cast<bf16*>(p) + i) = u;
    }
}
__device__ __forceinline__ float silu_f(float x) { return x / (1.0f + __expf(-x)); }
__device__ __forceinline__ float gelu_erf_f(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752f)); }

// erf GELU on 2 MUFU + ~12 FMA-pipe instructions: Phi(x) = 1/2 erfc(-x / sqrt 2) with erfc(z) = poly(t) exp(-z^2), t = 1 / (1 + p z)
// (Abramowitz-Stegun 7.1.26, |error| <= 1.5e-7 on erfc).  Computing through erfc keeps the left tail free of cancellation;
// the absolute error on gelu(x) stays below 3e-7 |x|, far under the bf16 rounding of the result it feeds.
__device__ __forceinline__ float gelu_erf_fast(float x) {
    const float z = fabsf(x) * 0.70710678118654752f;
    float t;   // rcp.approx (1 ulp): __frcp_rn would pull in an IEEE slow path with a call per element
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f, z, 1.0f)));
    float poly = fmaf(1.061405429f, t, -1.453152027f);
    poly = fmaf(poly, t, 1.421413741f);
    poly = fmaf(poly, t, -0.284496736f);
    poly = fmaf(poly, t, 0.254829592f);
    float ex;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(ex) : "f"(-1.4426950408889634f * z * z));
    const float e = poly * t * ex;   // erfc(z)
    const float phi = x < 0.f ? 0.5f * e : fmaf(-0.5f, e, 1.0f);
    return x * phi;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
#endif  // __CUDACC__
