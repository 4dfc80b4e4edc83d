// b200sd -- GroupNorm(+SiLU, + fused channel concat) and LayerNorm over NHWC bf16 activations.
// Both are bandwidth-bound passes over L2-resident activations (<= 21 MB at CFG batch 2).
#include <atomic>

#include <algorithm>


#include "common.cuh"

extern std::atomic<long long> g_b200sd_launches;
#define COUNT_LAUNCH() g_b200sd_launches.fetch_add(1, std::memory_order_relaxed)

namespace {

// hi / lo split of an fp32 vector for the fp32-accuracy path: hi = bf16(y), lo = bf16(y - hi); y = hi + lo to ~2^-17
__device__ __forceinline__ void st8_lo(bf16* lo, size_t i, const float (&y)[8]) {
    float r[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = y[j] - __bfloat162float(__float2bfloat16(y[j]));
    st8<B200SD_BF16>(lo, i, r);
}

constexpr int kGnThreads = 256;
constexpr int kMaxSlabs = 128;
constexpr int kCounterFloats = 1024;  // per-image arrival counters (batch <= 1024), must start zeroed
constexpr int kMaxGroups = 32;

// ---- pass 1: per-(image, group) mean / rstd ---------------------------------------------------------
// grid (slabs, batch).  Each thread owns ONE 16-byte channel vector (8 channels) and walks down the
// pixels of its slab with several independent loads in flight; per-thread sums are folded into
// shared per-group accumulators once at the end, each block publishes its partials, and the
// last block of an image (arrival counter, self-cleaning) reduces the slabs in a fixed order
// (deterministic) and writes mean / rstd.
template <int DT>
__global__ void __launch_bounds__(1024) gn_stats_kernel(const void* __restrict__ x0, const void* __restrict__ x1,
                                                        int C0, int C1, float* __restrict__ partial,
                                                        float* __restrict__ mean_rstd, unsigned int* __restrict__ counters,
                                                        int hw, int groups, int pix_per_slab, int rows_per_pass,
                                                        float eps) {
    __shared__ float s_sum[kMaxGroups], s_sq[kMaxGroups];
    __shared__ bool s_last;
    extern __shared__ float s_part[];  // [2][rows_per_pass][C] per-thread channel sums (deterministic fold)
    const int C = C0 + C1;
    const int C8 = C / 8;
    const int cpg = C / groups;
    const int b = blockIdx.y, slab = blockIdx.x, slabs = gridDim.x;
    const int vec = threadIdx.x % C8;
    const int prow = threadIdx.x / C8;
    const int c = vec * 8;
    const void* src;
    size_t off;
    int pitch;
    if (c < C0) { src = x0; off = (size_t)b * hw * C0 + c; pitch = C0; }
    else { src = x1; off = (size_t)b * hw * C1 + (c - C0); pitch = C1; }
    const int p_begin = slab * pix_per_slab;
    const int p_end = min(p_begin + pix_per_slab, hw);
    float s[8], ss[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { s[j] = 0.f; ss[j] = 0.f; }
    if (prow < rows_per_pass) {
#pragma unroll 4
        for (int pp = p_begin + prow; pp < p_end; pp += rows_per_pass) {
            float f[8];
            ld8<DT>(src, off + (size_t)pp * pitch, f);
#pragma unroll
            for (int j = 0; j < 8; ++j) { s[j] += f[j]; ss[j] += f[j] * f[j]; }
        }
        float* ps = s_part + (size_t)prow * C + c;
        float* pq = s_part + (size_t)(rows_per_pass + prow) * C + c;
#pragma unroll
        for (int j = 0; j < 8; ++j) { ps[j] = s[j]; pq[j] = ss[j]; }
    }
    __syncthreads();
    if (threadIdx.x < groups) {
        // fixed-order fold of the group's channels over the pixel rows of this block
        float a = 0.f, q = 0.f;
        for (int r = 0; r < rows_per_pass; ++r) {
            const float* ps = s_part + (size_t)r * C + threadIdx.x * cpg;
            const float* pq = s_part + (size_t)(rows_per_pass + r) * C + threadIdx.x * cpg;
            for (int j = 0; j < cpg; ++j) { a += ps[j]; q += pq[j]; }
        }
        s_sum[threadIdx.x] = a;
        s_sq[threadIdx.x] = q;
    }
    __syncthreads();
    if (threadIdx.x < groups) {
        float* dst = partial + (((size_t)b * slabs + slab) * groups + threadIdx.x) * 2;
        __stcg(dst, s_sum[threadIdx.x]);
        __stcg(dst + 1, s_sq[threadIdx.x]);
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned int prev = atomicAdd(counters + b, 1u);
        s_last = (prev == (unsigned int)slabs - 1);
        if (s_last) counters[b] = 0;
    }
    __syncthreads();
    if (s_last) {
        // 8 threads per group walk the slabs (fixed assignment -> deterministic), then a shuffle tree
        __threadfence();
        const int g = threadIdx.x >> 3, part = threadIdx.x & 7;
        double sum = 0.0, sq = 0.0;
        if (g < groups) {
            for (int i = part; i < slabs; i += 8) {
                const float* srcp = partial + (((size_t)b * slabs + i) * groups + g) * 2;
                sum += (double)__ldcg(srcp);
                sq += (double)__ldcg(srcp + 1);
            }
        }
#pragma unroll
        for (int o = 4; o > 0; o >>= 1) {
            sum += __shfl_xor_sync(0xffffffffu, sum, o);
            sq += __shfl_xor_sync(0xffffffffu, sq, o);
        }
        if (g < groups && part == 0) {
            const double cnt = (double)hw * cpg;
            const double mean = sum / cnt;
            double var = sq / cnt - mean * mean;
            if (var < 0.0) var = 0.0;
            mean_rstd[((size_t)b * groups + g) * 2] = (float)mean;
            mean_rstd[((size_t)b * groups + g) * 2 + 1] = (float)(1.0 / sqrt(var + (double)eps));
        }
    }
}

// ---- pass 2: normalise + affine (+ SiLU), write the concatenated bf16 tensor --------------------
template <int DT>
__global__ void __launch_bounds__(kGnThreads) gn_apply_kernel(const void* __restrict__ x0, const void* __restrict__ x1,
                                                              int C0, int C1, const float* __restrict__ gamma,
                                                              const float* __restrict__ beta, bf16* __restrict__ out,
                                                              bf16* __restrict__ raw_out, bf16* __restrict__ out_lo,
                                                              bf16* __restrict__ raw_lo,
                                                              const float* __restrict__ mean_rstd, int hw,
                                                              int groups, int silu, int pix_per_block) {
    extern __shared__ float2 s_ab[];  // per-channel (scale, shift)
    const int C = C0 + C1;
    const int cpg = C / groups;
    const int b = blockIdx.y;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        const int g = c / cpg;
        const float mean = __ldg(mean_rstd + ((size_t)b * groups + g) * 2);
        const float rstd = __ldg(mean_rstd + ((size_t)b * groups + g) * 2 + 1);
        const float a = rstd * __ldg(gamma + c);
        s_ab[c] = make_float2(a, __ldg(beta + c) - mean * a);
    }
    __syncthreads();
    const int vec_per_pix = C / 8;
    const int p_begin = blockIdx.x * pix_per_block;
    const int p_end = min(p_begin + pix_per_block, hw);
    const int total = (p_end - p_begin) * vec_per_pix;
#pragma unroll 4
    for (int i = threadIdx.x; i < total; i += blockDim.x) {
        const int p = p_begin + i / vec_per_pix;
        const int c = (i % vec_per_pix) * 8;
        float f[8], y[8];
        if (c < C0) ld8<DT>(x0, ((size_t)b * hw + p) * C0 + c, f);
        else ld8<DT>(x1, ((size_t)b * hw + p) * C1 + (c - C0), f);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float2 ab = s_ab[c + j];
            y[j] = f[j] * ab.x + ab.y;
            if (silu) y[j] = silu_f(y[j]);
        }
        st8<B200SD_BF16>(out, ((size_t)b * hw + p) * C + c, y);
        if (raw_out) st8<B200SD_BF16>(raw_out, ((size_t)b * hw + p) * C + c, f);  // bf16 copy of [x0|x1] (1x1 shortcut operand)
        if (out_lo) st8_lo(out_lo, ((size_t)b * hw + p) * C + c, y);
        if (raw_lo) st8_lo(raw_lo, ((size_t)b * hw + p) * C + c, f);
    }
}


// ---- fused GroupNorm: ONE kernel, one thread-block cluster per (image, set of G adjacent groups) ------------
// The CL CTAs of a cluster split the pixels.  Pass 1: every thread owns one 8-channel vector column and
// walks its pixels accumulating per-channel sums; a fixed-order fold gives this CTA's per-group partials,
// which the cluster exchanges through distributed shared memory (fixed rank order: deterministic).
// Pass 2 re-reads the same slab (L1/L2-hot), normalises, applies affine (+SiLU) and writes bf16 (+ the raw copy).
__device__ __forceinline__ void gn_cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ float gn_ld_dsmem(const float* local, uint32_t rank) {
    uint32_t raddr;
    float v;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(raddr) : "r"(ptx::smem_u32(local)), "r"(rank));
    asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(raddr) : "memory");
    return v;
}

template <int DT>
__global__ void __launch_bounds__(512) gn_fused_kernel(const void* __restrict__ x0, const void* __restrict__ x1, int C0,
                                                       int C1, const float* __restrict__ gamma,
                                                       const float* __restrict__ beta, bf16* __restrict__ out,
                                                       bf16* __restrict__ raw_out, bf16* __restrict__ out_lo,
                                                       bf16* __restrict__ raw_lo, int hw, int groups, int G, int CL,
                                                       int pix_per_cta, int R, float eps, int silu,
                                                       float* __restrict__ stats_out) {
    extern __shared__ float gsm[];  // [2][R][Cg] per-thread channel sums | [Cg] scale | [Cg] shift
    __shared__ float s_cta[2 * kMaxGroups];   // this CTA's (sum, sumsq) per group of the set
    __shared__ float s_mr[2 * kMaxGroups];    // (mean, rstd) per group of the set
    const int C = C0 + C1;
    const int cpg = C / groups;
    const int Cg = G * cpg;          // channels of this group set (multiple of 8)
    const int VC = Cg / 8;
    const int rank = blockIdx.x;     // cluster spans gridDim.x == CL
    const int set = blockIdx.y, b = blockIdx.z;
    const int c_base = set * Cg;
    float* s_part = gsm;
    float2* s_ab = reinterpret_cast<float2*>(gsm + 2 * R * Cg);
    const int vec = threadIdx.x % VC, prow = threadIdx.x / VC;
    const bool active = prow < R;
    const int c = c_base + vec * 8;  // global channel of this thread's vector
    const void* src;
    size_t off;
    int pitch;
    if (c < C0) { src = x0; off = (size_t)b * hw * C0 + c; pitch = C0; }
    else { src = x1; off = (size_t)b * hw * C1 + (c - C0); pitch = C1; }
    const int p_begin = rank * pix_per_cta;
    const int p_end = min(p_begin + pix_per_cta, hw);

    // ---- pass 1 ----
    if (active) {
        float s[8], ss[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) { s[j] = 0.f; ss[j] = 0.f; }
#pragma unroll 4
        for (int pp = p_begin + prow; pp < p_end; pp += R) {
            float f[8];
            ld8<DT>(src, off + (size_t)pp * pitch, f);
#pragma unroll
            for (int j = 0; j < 8; ++j) { s[j] += f[j]; ss[j] += f[j] * f[j]; }
        }
        float* ps = s_part + (size_t)prow * Cg + vec * 8;
        float* pq = s_part + (size_t)(R + prow) * Cg + vec * 8;
#pragma unroll
        for (int j = 0; j < 8; ++j) { ps[j] = s[j]; pq[j] = ss[j]; }
    }
    __syncthreads();
    // fixed-order parallel fold: rows -> K row-chunks -> channels -> groups
    {
        const int K = max(1, min(R, (int)blockDim.x / (2 * Cg)));      // row chunks reduced in parallel
        float* s_red = reinterpret_cast<float*>(s_ab);                  // [2][K][Cg] scratch (s_ab is built later)
        for (int t = threadIdx.x; t < 2 * K * Cg; t += blockDim.x) {
            const int which = t / (K * Cg), k = (t / Cg) % K, i = t % Cg;
            float a = 0.f;
            for (int r = k; r < R; r += K) a += s_part[(size_t)(which * R + r) * Cg + i];
            s_red[t] = a;
        }
        __syncthreads();
        for (int t = threadIdx.x; t < 2 * Cg; t += blockDim.x) {
            const int which = t / Cg, i = t % Cg;
            float a = 0.f;
            for (int k = 0; k < K; ++k) a += s_red[(which * K + k) * Cg + i];
            s_part[which * Cg + i] = a;   // reuse row 0 of s_part: per-channel totals [2][Cg]
        }
        __syncthreads();
        for (int t = threadIdx.x; t < 2 * G; t += blockDim.x) {
            const int which = t / G, g = t % G;
            float a = 0.f;
            for (int j = 0; j < cpg; ++j) a += s_part[which * Cg + g * cpg + j];
            s_cta[2 * g + which] = a;
        }
    }
    if (CL > 1) gn_cluster_sync(); else __syncthreads();
    if (threadIdx.x < G) {
        double sum = 0.0, sq = 0.0;
        if (CL > 1) {
            for (int r = 0; r < CL; ++r) {
                sum += (double)gn_ld_dsmem(&s_cta[2 * threadIdx.x], r);
                sq += (double)gn_ld_dsmem(&s_cta[2 * threadIdx.x + 1], r);
            }
        } else {
            sum = s_cta[2 * threadIdx.x];
            sq = s_cta[2 * threadIdx.x + 1];
        }
        const double cnt = (double)hw * cpg;
        const double mean = sum / cnt;
        double var = sq / cnt - mean * mean;
        if (var < 0.0) var = 0.0;
        s_mr[2 * threadIdx.x] = (float)mean;
        s_mr[2 * threadIdx.x + 1] = (float)(1.0 / sqrt(var + (double)eps));
        if (stats_out != nullptr && rank == 0) {   // kept for the backward pass
            stats_out[((size_t)b * groups + set * G + threadIdx.x) * 2] = s_mr[2 * threadIdx.x];
            stats_out[((size_t)b * groups + set * G + threadIdx.x) * 2 + 1] = s_mr[2 * threadIdx.x + 1];
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < Cg; i += blockDim.x) {
        const int g = i / cpg;
        const float a = s_mr[2 * g + 1] * __ldg(gamma + c_base + i);
        s_ab[i] = make_float2(a, __ldg(beta + c_base + i) - s_mr[2 * g] * a);
    }
    __syncthreads();

    // ---- pass 2 ----
    if (active) {
#pragma unroll 4
        for (int pp = p_begin + prow; pp < p_end; pp += R) {
            float f[8], y[8];
            ld8<DT>(src, off + (size_t)pp * pitch, f);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float2 ab = s_ab[vec * 8 + j];
                y[j] = f[j] * ab.x + ab.y;
                if (silu) y[j] = silu_f(y[j]);
            }
            const size_t o = ((size_t)b * hw + pp) * C + c;
            st8<B200SD_BF16>(out, o, y);
            if (raw_out) st8<B200SD_BF16>(raw_out, o, f);
            if (out_lo) st8_lo(out_lo, o, y);
            if (raw_lo) st8_lo(raw_lo, o, f);
        }
    }
    if (CL > 1) gn_cluster_sync();  // peers may still be reading s_cta
}

// ---- GroupNorm from producer-side statistics: the GEMM that wrote x0 (/ x1) also wrote, per CTA, the column sums and sums
// of squares of the rows it stored (gemm_tcgen05.cu, KParams::gn_part).  No statistics pass over the tensor and no cluster:
// every CTA folds the partial rows of its image for its own channels (fixed order: deterministic), then does the apply
// pass of gn_fused_kernel over its pixel slab.  part*: [image][ppi][2][ld] floats.
template <int DT>
__global__ void __launch_bounds__(512) gn_parts_kernel(const void* __restrict__ x0, const void* __restrict__ x1, int C0, int C1,
                                                       const float* __restrict__ part0, int ppi0, int ld0,
                                                       const float* __restrict__ part1, int ppi1, int ld1,
                                                       const float* __restrict__ gamma, const float* __restrict__ beta,
                                                       bf16* __restrict__ out, bf16* __restrict__ raw_out, int hw, int groups, int G,
                                                       int pix_per_cta, int R, float eps, int silu, float* __restrict__ stats_out) {
    extern __shared__ float gsm[];  // [2][Cg] per-channel totals | [Cg] (scale, shift)
    __shared__ float s_grp[2 * kMaxGroups];
    __shared__ float s_mr[2 * kMaxGroups];
    const int C = C0 + C1;
    const int cpg = C / groups;
    const int Cg = G * cpg;
    const int VC = Cg / 8;
    const int slab = blockIdx.x, set = blockIdx.y, b = blockIdx.z;
    const int c_base = set * Cg;
    float* s_tot = gsm;
    float2* s_ab = reinterpret_cast<float2*>(gsm + 2 * Cg);
    // fold the partial rows: nq thread groups take every nq-th row (8 loads in flight each), then a fixed-order fold
    float* s_red = gsm + 4 * Cg;    // [nq][2 * Cg]
    const int nq = max(1, (int)blockDim.x / (2 * Cg));
    for (int t = threadIdx.x; t < nq * 2 * Cg; t += blockDim.x) {
        const int q = t / (2 * Cg), v = t % (2 * Cg);
        const int which = v / Cg, c = c_base + v % Cg;
        const float* pp;
        int n, stride;
        if (c < C0) { pp = part0 + ((size_t)b * ppi0 * 2 + which) * ld0 + c; n = ppi0; stride = 2 * ld0; }
        else { pp = part1 + ((size_t)b * ppi1 * 2 + which) * ld1 + (c - C0); n = ppi1; stride = 2 * ld1; }
        float a = 0.f;
#pragma unroll 8
        for (int k = q; k < n; k += nq) a += __ldg(pp + (size_t)k * stride);
        s_red[t] = a;
    }
    __syncthreads();
    for (int t = threadIdx.x; t < 2 * Cg; t += blockDim.x) {
        float a = 0.f;
        for (int q = 0; q < nq; ++q) a += s_red[q * 2 * Cg + t];
        s_tot[t] = a;
    }
    __syncthreads();
    for (int t = threadIdx.x; t < 2 * G; t += blockDim.x) {
        const int which = t / G, g = t % G;
        float a = 0.f;
        for (int j = 0; j < cpg; ++j) a += s_tot[which * Cg + g * cpg + j];
        s_grp[2 * g + which] = a;
    }
    __syncthreads();
    if (threadIdx.x < G) {
        const double cnt = (double)hw * cpg;
        const double mean = (double)s_grp[2 * threadIdx.x] / cnt;
        double var = (double)s_grp[2 * threadIdx.x + 1] / cnt - mean * mean;
        if (var < 0.0) var = 0.0;
        s_mr[2 * threadIdx.x] = (float)mean;
        s_mr[2 * threadIdx.x + 1] = (float)(1.0 / sqrt(var + (double)eps));
        if (stats_out != nullptr && slab == 0) {
            stats_out[((size_t)b * groups + set * G + threadIdx.x) * 2] = s_mr[2 * threadIdx.x];
            stats_out[((size_t)b * groups + set * G + threadIdx.x) * 2 + 1] = s_mr[2 * threadIdx.x + 1];
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < Cg; i += blockDim.x) {
        const int g = i / cpg;
        const float a = s_mr[2 * g + 1] * __ldg(gamma + c_base + i);
        s_ab[i] = make_float2(a, __ldg(beta + c_base + i) - s_mr[2 * g] * a);
    }
    __syncthreads();
    const int vec = threadIdx.x % VC, prow = threadIdx.x / VC;
    if (prow >= R) return;
    const int c = c_base + vec * 8;
    const void* src;
    size_t off;
    int pitch;
    if (c < C0) { src = x0; off = (size_t)b * hw * C0 + c; pitch = C0; }
    else { src = x1; off = (size_t)b * hw * C1 + (c - C0); pitch = C1; }
    const int p_begin = slab * pix_per_cta;
    const int p_end = min(p_begin + pix_per_cta, hw);
    float2 ab[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) ab[j] = s_ab[vec * 8 + j];
#pragma unroll 4
    for (int pp = p_begin + prow; pp < p_end; pp += R) {
        float f[8], y[8];
        ld8<DT>(src, off + (size_t)pp * pitch, f);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            y[j] = f[j] * ab[j].x + ab[j].y;
            if (silu) y[j] = silu_f(y[j]);
        }
        const size_t o = ((size_t)b * hw + pp) * C + c;
        st8<B200SD_BF16>(out, o, y);
        if (raw_out) st8<B200SD_BF16>(raw_out, o, f);
    }
}

// ---- LayerNorm: one warp per row, row held in registers (C <= 1280) ------------------------------
template <int PAIRS_PER_LANE, int DT>
__global__ void __launch_bounds__(256) layernorm_kernel(const void* __restrict__ x, const float* __restrict__ gamma,
                                                        const float* __restrict__ beta, bf16* __restrict__ out,
                                                        bf16* __restrict__ out_lo, int rows, int C, float eps) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= rows) return;
    float2 v[PAIRS_PER_LANE];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < PAIRS_PER_LANE; ++i) {
        if constexpr (DT == B200SD_F32)
            v[i] = __ldg(reinterpret_cast<const float2*>(static_cast<const float*>(x) + (size_t)warp * C) + lane + 32 * i);
        else
            v[i] = unpack_bf16x2(__ldg(reinterpret_cast<const uint32_t*>(static_cast<const bf16*>(x) + (size_t)warp * C) + lane + 32 * i));
        s += v[i].x + v[i].y;
    }
    const float mean = warp_sum(s) / (float)C;
    float ss = 0.f;
#pragma unroll
    for (int i = 0; i < PAIRS_PER_LANE; ++i) {
        const float a = v[i].x - mean, b = v[i].y - mean;
        ss += a * a + b * b;
    }
    const float rstd = rsqrtf(warp_sum(ss) / (float)C + eps);
    uint32_t* dst = reinterpret_cast<uint32_t*>(out + (size_t)warp * C);
    const float2* g2 = reinterpret_cast<const float2*>(gamma);
    const float2* b2 = reinterpret_cast<const float2*>(beta);
#pragma unroll
    for (int i = 0; i < PAIRS_PER_LANE; ++i) {
        const float2 g = __ldg(g2 + lane + 32 * i), bb = __ldg(b2 + lane + 32 * i);
        const float y0 = (v[i].x - mean) * rstd * g.x + bb.x, y1 = (v[i].y - mean) * rstd * g.y + bb.y;
        dst[lane + 32 * i] = pack_bf16x2(y0, y1);
        if (out_lo != nullptr)
            reinterpret_cast<uint32_t*>(out_lo + (size_t)warp * C)[lane + 32 * i] =
                pack_bf16x2(y0 - __bfloat162float(__float2bfloat16(y0)), y1 - __bfloat162float(__float2bfloat16(y1)));
    }
}

}  // namespace

extern "C" int b200sd_groupnorm_silu_split(const void* x0, const void* x1, int C0, int C1, const float* gamma,
                                           const float* beta, void* out, void* out_lo, void* raw_out, void* raw_lo,
                                           float* stats_ws, float* stats_out, int batch, int hw, int groups, float eps,
                                           int silu, int in_dtype, b200sd_stream_t stream) {
    B200SD_REQUIRE(raw_lo == nullptr || raw_out != nullptr, "groupnorm: raw_lo needs raw_out");
    B200SD_REQUIRE(x0 && gamma && beta && out && stats_ws, "groupnorm: null pointer");
    if (!x1) C1 = 0;
    const int C = C0 + C1;
    B200SD_REQUIRE(batch > 0 && hw > 0 && batch <= kCounterFloats, "groupnorm: bad batch/hw");
    B200SD_REQUIRE(groups > 0 && groups <= kMaxGroups && C % groups == 0 && (C / groups) % 2 == 0,
                   "groupnorm: C=%d groups=%d unsupported (channels per group must be even)", C, groups);
    B200SD_REQUIRE(C0 % 8 == 0 && C1 % 8 == 0, "groupnorm: channel counts must be multiples of 8");
    B200SD_REQUIRE(C * sizeof(float2) <= 48 * 1024, "groupnorm: C=%d too large", C);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    B200SD_REQUIRE(in_dtype == B200SD_BF16 || in_dtype == B200SD_F32, "groupnorm: bad input dtype");
    {
        // fused single-kernel path
        const int cpg = C / groups;
        int G = 1;
        while ((G * cpg) % 8 != 0 && G < groups) G *= 2;
        while (G * 2 <= groups && groups % (G * 2) == 0 && G * cpg < 32) G *= 2;   // >= 32 channels per pixel segment
        const int Cg = G * cpg;
        // The single-kernel path keeps an image's pixels on at most 8 CTAs per channel set: right for the UNet (<= 2.6 M elements
        // per image, launch latency dominates), hopeless for the VAE's 256^2 / 512^2 levels (33 M elements on 32 CTAs measured
        // 832 us = 0.4 TB/s).  Large images take the two-kernel path below: 128 statistics slabs + 4 apply CTAs per SM.
        if ((Cg % 8) == 0 && groups % G == 0 && Cg / 8 <= 512 && (long)hw * C <= 3000000L) {
            const int VC = Cg / 8;
            const int sets = groups / G;
            int CL = 1;
            while (CL < 8 && (long)batch * sets * CL < b200sd_num_sms() && hw / (CL * 2) >= 32) CL *= 2;
            const int ppc = ceil_div(hw, CL);
            int R = 256 / VC;
            if (R < 1) R = 1;
            if (R > ppc) R = ppc;
            int threads = ((VC * R + 31) / 32) * 32;
            if (threads < 32) threads = 32;
            const size_t smem = ((size_t)2 * R * Cg + 2 * Cg + threads) * sizeof(float);
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3(CL, sets, batch);
            cfg.blockDim = dim3(threads);
            cfg.dynamicSmemBytes = smem;
            cfg.stream = s;
            cudaLaunchAttribute attr[1];
            if (CL > 1) {
                attr[0].id = cudaLaunchAttributeClusterDimension;
                attr[0].val.clusterDim.x = CL;
                attr[0].val.clusterDim.y = 1;
                attr[0].val.clusterDim.z = 1;
                cfg.attrs = attr;
                cfg.numAttrs = 1;
            }
            if (in_dtype == B200SD_F32)
                B200SD_CUDA(cudaLaunchKernelEx(&cfg, gn_fused_kernel<B200SD_F32>, x0, x1, C0, C1, gamma, beta, static_cast<bf16*>(out),
                                               static_cast<bf16*>(raw_out), static_cast<bf16*>(out_lo), static_cast<bf16*>(raw_lo), hw, groups, G, CL, ppc, R, eps,
                                               silu, stats_out));
            else
                B200SD_CUDA(cudaLaunchKernelEx(&cfg, gn_fused_kernel<B200SD_BF16>, x0, x1, C0, C1, gamma, beta, static_cast<bf16*>(out),
                                               static_cast<bf16*>(raw_out), static_cast<bf16*>(out_lo), static_cast<bf16*>(raw_lo), hw, groups, G, CL, ppc, R, eps,
                                               silu, stats_out));
            COUNT_LAUNCH();
            B200SD_LAUNCH_CHECK();
            return B200SD_OK;
        }
    }
    // two-kernel fallback (stats + apply) for channel layouts the fused kernel does not cover
    const int C8 = C / 8;
    B200SD_REQUIRE(C8 <= 1024, "groupnorm: C=%d too large", C);
    const int rows_per_pass = (C8 >= 256) ? 1 : 256 / C8;
    int threads = ((C8 * rows_per_pass + 31) / 32) * 32;
    if (threads < 256) threads = 256;  // the final reduce uses 8 threads per group
    // workspace layout: [batch counters (as uint)] [mean/rstd 2*batch*groups] [partials 2*batch*slabs*groups]
    unsigned int* counters = reinterpret_cast<unsigned int*>(stats_ws);
    float* mean_rstd = stats_ws + kCounterFloats;
    float* partial = mean_rstd + 2 * (size_t)batch * kMaxGroups;
    int slabs = ceil_div(b200sd_num_sms() * 2, batch);
    if (slabs > kMaxSlabs) slabs = kMaxSlabs;
    int pps = ceil_div(hw, slabs);
    pps = ceil_div(pps, rows_per_pass) * rows_per_pass;
    slabs = ceil_div(hw, pps);
    const size_t st_smem = (size_t)2 * rows_per_pass * C * sizeof(float);
    if (in_dtype == B200SD_F32)
        gn_stats_kernel<B200SD_F32><<<dim3(slabs, batch), dim3(threads), st_smem, s>>>(x0, x1, C0, C1, partial,
                                  mean_rstd, counters, hw, groups, pps, rows_per_pass, eps);
    else
        gn_stats_kernel<B200SD_BF16><<<dim3(slabs, batch), dim3(threads), st_smem, s>>>(x0, x1, C0, C1, partial,
                                  mean_rstd, counters, hw, groups, pps, rows_per_pass, eps);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    if (stats_out != nullptr)
        B200SD_CUDA(cudaMemcpyAsync(stats_out, mean_rstd, (size_t)2 * batch * groups * sizeof(float), cudaMemcpyDeviceToDevice, s));
    int blocks = ceil_div(b200sd_num_sms() * 4, batch);
    int ppb = ceil_div(hw, blocks);
    const int min_ppb = ceil_div(kGnThreads * 4, C / 8);  // >= 4 vectors per thread
    if (ppb < min_ppb) ppb = min_ppb;
    blocks = ceil_div(hw, ppb);
    if (in_dtype == B200SD_F32)
        gn_apply_kernel<B200SD_F32><<<dim3(blocks, batch), dim3(kGnThreads), C * sizeof(float2), s>>>(x0, x1, C0, C1,
                                  gamma, beta, static_cast<bf16*>(out), static_cast<bf16*>(raw_out), static_cast<bf16*>(out_lo), static_cast<bf16*>(raw_lo),
                                  mean_rstd, hw, groups, silu, ppb);
    else
        gn_apply_kernel<B200SD_BF16><<<dim3(blocks, batch), dim3(kGnThreads), C * sizeof(float2), s>>>(x0, x1, C0, C1,
                                  gamma, beta, static_cast<bf16*>(out), static_cast<bf16*>(raw_out), static_cast<bf16*>(out_lo), static_cast<bf16*>(raw_lo),
                                  mean_rstd, hw, groups, silu, ppb);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

extern "C" int b200sd_groupnorm_silu(const void* x0, const void* x1, int C0, int C1, const float* gamma,
                                     const float* beta, void* out, void* raw_out, float* stats_ws, int batch, int hw,
                                     int groups, float eps, int silu, int in_dtype, b200sd_stream_t stream) {
    return b200sd_groupnorm_silu_split(x0, x1, C0, C1, gamma, beta, out, nullptr, raw_out, nullptr, stats_ws, nullptr, batch, hw,
                                       groups, eps, silu, in_dtype, stream);
}

extern "C" int b200sd_groupnorm_silu_stats(const void* x0, const void* x1, int C0, int C1, const float* gamma,
                                           const float* beta, void* out, void* raw_out, float* stats_ws, float* stats_out,
                                           int batch, int hw, int groups, float eps, int silu, int in_dtype,
                                           b200sd_stream_t stream) {
    return b200sd_groupnorm_silu_split(x0, x1, C0, C1, gamma, beta, out, nullptr, raw_out, nullptr, stats_ws, stats_out, batch, hw,
                                       groups, eps, silu, in_dtype, stream);
}

// workspace floats needed by b200sd_groupnorm_silu for a given batch: 2 * batch * kMaxSlabs * kMaxGroups
extern "C" int b200sd_groupnorm_workspace_floats(int batch) {
    return kCounterFloats + 2 * batch * kMaxGroups + 2 * batch * kMaxSlabs * kMaxGroups;
}

extern "C" int b200sd_layernorm_split(const void* x, const float* gamma, const float* beta, void* out, void* out_lo, int rows,
                                      int C, float eps, int in_dtype, b200sd_stream_t stream) {
    B200SD_REQUIRE(x && gamma && beta && out, "layernorm: null pointer");
    B200SD_REQUIRE(rows > 0, "layernorm: rows must be positive");
    B200SD_REQUIRE(C % 64 == 0 && C >= 64 && C <= 1280, "layernorm: C=%d unsupported (multiple of 64, <= 1280)", C);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int blocks = ceil_div(rows, 8);
    const void* xi = x;
    B200SD_REQUIRE(in_dtype == B200SD_BF16 || in_dtype == B200SD_F32, "layernorm: bad input dtype");
    bf16* xo = static_cast<bf16*>(out);
    bf16* xl = static_cast<bf16*>(out_lo);
#define LN_CASE(P)                                                                                     \
    case P:                                                                                            \
        if (in_dtype == B200SD_F32)                                                                         \
            layernorm_kernel<P, B200SD_F32><<<dim3(blocks), dim3(256), 0, s>>>(xi, gamma, beta, xo, xl, rows, C, eps); \
        else                                                                                                \
            layernorm_kernel<P, B200SD_BF16><<<dim3(blocks), dim3(256), 0, s>>>(xi, gamma, beta, xo, xl, rows, C, eps); \
        break;
    switch (C / 64) {
        LN_CASE(1) LN_CASE(2) LN_CASE(3) LN_CASE(4) LN_CASE(5) LN_CASE(6) LN_CASE(7) LN_CASE(8) LN_CASE(9) LN_CASE(10)
        LN_CASE(11) LN_CASE(12) LN_CASE(13) LN_CASE(14) LN_CASE(15) LN_CASE(16) LN_CASE(17) LN_CASE(18) LN_CASE(19) LN_CASE(20)
        default:
            B200SD_REQUIRE(false, "layernorm: C=%d unsupported", C);
    }
#undef LN_CASE
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

extern "C" int b200sd_layernorm(const void* x, const float* gamma, const float* beta, void* out, int rows, int C,
                                float eps, int in_dtype, b200sd_stream_t stream) {
    return b200sd_layernorm_split(x, gamma, beta, out, nullptr, rows, C, eps, in_dtype, stream);
}

// GroupNorm (+SiLU, + concat) whose statistics come from the producing GEMMs' gn_part buffers (b200sd_gemm_gn_layout).
// part1 / ppi1 / ld1 describe the producer of x1 (ignored when x1 == NULL).  Returns B200SD_ERR_UNSUPPORTED for channel
// layouts it does not cover (the caller then uses b200sd_groupnorm_silu).
extern "C" int b200sd_groupnorm_silu_parts(const void* x0, const void* x1, int C0, int C1, const float* part0, int ppi0, int ld0,
                                           const float* part1, int ppi1, int ld1, const float* gamma, const float* beta, void* out,
                                           void* raw_out, float* stats_out, int batch, int hw, int groups, float eps, int silu,
                                           int in_dtype, b200sd_stream_t stream) {
    B200SD_REQUIRE(x0 && part0 && gamma && beta && out && ppi0 > 0, "groupnorm_parts: null pointer");
    if (!x1) C1 = 0;
    B200SD_REQUIRE(C1 == 0 || (part1 && ppi1 > 0), "groupnorm_parts: x1 without its statistics");
    const int C = C0 + C1;
    B200SD_REQUIRE(batch > 0 && hw > 0 && groups > 0 && groups <= kMaxGroups && C % groups == 0, "groupnorm_parts: bad shape");
    B200SD_REQUIRE(C0 % 8 == 0 && C1 % 8 == 0, "groupnorm_parts: channel counts must be multiples of 8");
    B200SD_REQUIRE(in_dtype == B200SD_BF16 || in_dtype == B200SD_F32, "groupnorm_parts: bad input dtype");
    const int cpg = C / groups;
    int G = 1;
    while ((G * cpg) % 8 != 0 && G < groups) G *= 2;
    while (G * 2 <= groups && groups % (G * 2) == 0 && G * cpg < 32) G *= 2;
    const int Cg = G * cpg;
    if ((Cg % 8) != 0 || groups % G != 0 || Cg / 8 > 512) return B200SD_ERR_UNSUPPORTED;
    const int VC = Cg / 8, sets = groups / G;
    int slabs = ceil_div(b200sd_num_sms() * 2, batch * sets);   // two CTAs per SM
    if (slabs > hw / 32) slabs = hw / 32;
    if (slabs < 1) slabs = 1;
    const int ppc = ceil_div(hw, slabs);
    slabs = ceil_div(hw, ppc);
    int R = 256 / VC;
    if (R < 1) R = 1;
    if (R > ppc) R = ppc;
    int threads = ((VC * R + 31) / 32) * 32;
    if (threads < 64) threads = 64;
    const size_t smem = ((size_t)4 * Cg + (size_t)std::max(threads, 2 * Cg)) * sizeof(float);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (in_dtype == B200SD_F32)
        gn_parts_kernel<B200SD_F32><<<dim3(slabs, sets, batch), dim3(threads), smem, s>>>(x0, x1, C0, C1, part0, ppi0,
                                  ld0, part1, ppi1, ld1, gamma, beta, static_cast<bf16*>(out), static_cast<bf16*>(raw_out), hw, groups, G,
                                  ppc, R, eps, silu, stats_out);
    else
        gn_parts_kernel<B200SD_BF16><<<dim3(slabs, sets, batch), dim3(threads), smem, s>>>(x0, x1, C0, C1, part0, ppi0,
                                  ld0, part1, ppi1, ld1, gamma, beta, static_cast<bf16*>(out), static_cast<bf16*>(raw_out), hw, groups, G,
                                  ppc, R, eps, silu, stats_out);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}
