// b200sd -- block-wise 8-bit AdamW over the flat kernel-layout buffers: the optimizer the reference uses by default
// (finetune_sd.py:300 use_8bit_adam=True, :407-420 bnb.optim.AdamW8bit(..., min_8bit_size=16384)).
//
// HBM-bound byte work: per parameter 10 B read (p, g fp32 + two 1-byte moment codes) and 8 B written (p fp32, bf16 tensor-core
// copy, two codes; +4 B when the gradient is zeroed in the same pass) against 16 B + 14 (18) B of the fp32-state kernel
// (adamw_flat_kernel in backward.cu).  One persistent CTA per SM slot walks 2048-value blocks (bitsandbytes' block size):
// de-quantise both moments with the block's absmax, Adam update, block max-reduce of the new moments, parameter update, re-quantise
// to the nearest entry of the 256-value dynamic code book.  The code books live in shared memory once per CTA.  Nearest code =
// number of code-book midpoints below x: a per-CTA lookup table indexed by the top 16 bits of x's order-preserving integer key
// (sign, exponent, 7 mantissa bits: 128 bins per octave over 25 octaves) gives the count at the low edge of x's bin, two
// compare against the sorted midpoints finishes it (the dynamic code books put at most one midpoint into a bin; the CTA checks
// that and otherwise takes the generic eight-level search over the midpoints in breadth-first order, which also builds the
// table).  Shared-memory reads per value: 2 to de-quantise, 4 to re-quantise.  Every product / sum is a separately rounded fp32 operation (__f*_rn) in the order of
// oracle/adam8bit_ref.py, which makes the codes, the absmax tables and the parameters bit-identical to the CPU restatement.
// v1 of this kernel (eight-level search per value, one IEEE division per value for the scaling, 6 CTAs per SM requested where
// 4 fit) ran at 2.66 TB/s = 41 % of the measured copy bandwidth (profiles/r02c_elementwise_with_optimizers_v1.json).
#include <atomic>
#include <cmath>

#include "common.cuh"

extern std::atomic<long long> g_b200sd_launches;
#define COUNT_LAUNCH() g_b200sd_launches.fetch_add(1, std::memory_order_relaxed)

namespace {

constexpr int kBlock = 2048;      // values per quantisation block
constexpr int kV = 4;             // values per thread
constexpr int kThreads = kBlock / kV;     // 512: one CTA iteration = one quantisation block
// resident CTAs per SM the kernel is compiled for: 3 -> 40 registers, 48 warps per SM.  4 (32 registers, 24 B of spills,
// 64 warps) measured slower on B200: 420.9 vs 411.5 us per launch (profiles/r02c_adam8bit_variants_v3.txt).
constexpr int kCtasPerSm = 3;
constexpr int kModeSkip = -2;     // chunk_mode: frozen parameter / padding -- untouched
constexpr int kMode8bit = -1;     // chunk_mode: moments stored as codes; >= 0: offset into the compact fp32 moments
// lookup-table bins: q = (order-preserving key of x) >> 16.  Positive x in [2^-24, 1.0078): q in [0xB380, 0xBF80], everything
// smaller shares the bin below them; negative x mirrored: q in [0x407F, 0x4C7F], tiny negatives share the bin 0x4C80.
constexpr int kPosBase = 0xB37F, kNegBase = 0x407F, kNegClamp = 0x4C80;
constexpr int kNPos = 0xBF80 - kPosBase + 1;      // 3074 bins per sign

struct Adam8Consts {
    float beta1, beta2, omb1, omb2, eps_c2, step_size, decay, grad_scale;
    int apply_decay, zero_grad;
};

// number of midpoints strictly below x == index of the nearest code (ties to the lower code); e[] is the BFS layout of the
// 255 sorted midpoints: node k (1-based) has children 2k, 2k + 1
__device__ __forceinline__ int nearest_code(const float* __restrict__ e, float x) {
    int k = 1;
#pragma unroll
    for (int l = 0; l < 8; ++l) k = 2 * k + (x > e[k] ? 1 : 0);
    return k - 256;
}

__device__ __forceinline__ int lut_bin_signed(float x) {
    const uint32_t u = __float_as_uint(x);
    const int q = (int)((u ^ (uint32_t)(((int32_t)u >> 31) | (int32_t)0x80000000)) >> 16);     // negative: ~u, positive: u | 2^31
    // (the outer clamps only matter for inf / NaN moments, i.e. a diverged run: they keep the table index in range)
    return q >= 0x8000 ? min(max(q, kPosBase), 0xBF80) - kPosBase + kNPos : max(min(q, kNegClamp), kNegBase) - kNegBase;
}
__device__ __forceinline__ int lut_bin_unsigned(float x) {       // x >= 0
    return min(max((int)(__float_as_uint(x) >> 16), kPosBase - 0x8000), 0xBF80 - 0x8000) - (kPosBase - 0x8000);
}
// the smallest value of a bin
__device__ __forceinline__ float bin_low_pos(int bp) { return bp == 0 ? 0.f : __uint_as_float((uint32_t)(kPosBase + bp - 0x8000) << 16); }
__device__ __forceinline__ float bin_low_neg(int b) { return __uint_as_float(((0xFFFFu - (uint32_t)(kNegBase + b)) << 16) | 0xFFFFu); }

__global__ void __launch_bounds__(kThreads, kCtasPerSm) adamw8bit_kernel(float* __restrict__ p, float* __restrict__ g,
                                                                         uint8_t* __restrict__ st1, uint8_t* __restrict__ st2,
                                                                         float* __restrict__ absmax1, float* __restrict__ absmax2,
                                                                         const float* __restrict__ qmap1,
                                                                         const float* __restrict__ qmap2,
                                                                         const int32_t* __restrict__ chunk_mode,
                                                                         float* __restrict__ small_m, float* __restrict__ small_v,
                                                                         bf16* __restrict__ wb, int64_t n, int64_t nblocks,
                                                                         Adam8Consts c) {
    __shared__ float q1[256], q2[256], e1[256], e2[256], m1[256], m2[256];
    __shared__ uint8_t lut1[2 * kNPos + 4], lut2[kNPos + 6];
    __shared__ float red1[kThreads / 32], red2[kThreads / 32];
    const int tid = threadIdx.x;
    if (tid < 256) {
        q1[tid] = __ldg(qmap1 + tid);
        q2[tid] = __ldg(qmap2 + tid);
    }
    __syncthreads();
    if (tid < 256) {
        // sorted midpoints (m[255] = +inf: a compare past the end is false) and their breadth-first copy
        m1[tid] = tid < 255 ? __fmul_rn(__fadd_rn(q1[tid], q1[tid + 1]), 0.5f) : __int_as_float(0x7f800000);
        m2[tid] = tid < 255 ? __fmul_rn(__fadd_rn(q2[tid], q2[tid + 1]), 0.5f) : __int_as_float(0x7f800000);
        if (tid >= 1) {
            // BFS node tid at level L (2^L <= tid < 2^(L+1)), j-th of its level, holds the sorted midpoint of rank (2j + 1) 2^(7-L) - 1
            const int L = 31 - __clz(tid), j = tid - (1 << L);
            const int r = (2 * j + 1) * (1 << (7 - L)) - 1;
            e1[tid] = __fmul_rn(__fadd_rn(q1[r], q1[r + 1]), 0.5f);
            e2[tid] = __fmul_rn(__fadd_rn(q2[r], q2[r + 1]), 0.5f);
        } else {
            e1[0] = e2[0] = 0.f;
        }
    }
    __syncthreads();
    // lookup tables: number of midpoints below the low edge of every bin
    for (int b = tid; b < 2 * kNPos; b += kThreads)
        lut1[b] = (uint8_t)nearest_code(e1, b < kNPos ? bin_low_neg(b) : bin_low_pos(b - kNPos));
    for (int b = tid; b < kNPos; b += kThreads) lut2[b] = (uint8_t)nearest_code(e2, bin_low_pos(b));
    __syncthreads();
    // the fast path needs at most one midpoint per bin (true of the dynamic code books) and, to know the sign of a first-moment
    // code without reading it, an ascending code book whose sign-bit entries all come first; anything else -> generic search
    int generic = tid < 255 && (__float_as_uint(q1[tid & 255]) >> 31) == 0 && (__float_as_uint(q1[(tid + 1) & 255]) >> 31) != 0;
    for (int b = tid; b < 2 * kNPos; b += kThreads) generic |= (b + 1 < 2 * kNPos ? (int)lut1[b + 1] : 255) - (int)lut1[b] > 1;
    for (int b = tid; b < kNPos; b += kThreads) generic |= (b + 1 < kNPos ? (int)lut2[b + 1] : 255) - (int)lut2[b] > 1;
    const bool slow = __syncthreads_or(generic) != 0;
    const int nneg = __syncthreads_count(tid < 256 && (__float_as_uint(q1[tid & 255]) >> 31) != 0);
    const int warp = tid >> 5, lane = tid & 31;
    for (int64_t blk = blockIdx.x; blk < nblocks; blk += gridDim.x) {
        const int64_t i0 = blk * kBlock + (int64_t)tid * kV;
        int mode = kModeSkip;
        if (i0 < n) mode = chunk_mode ? __ldg(chunk_mode + (i0 >> 6)) : kMode8bit;
        float S1[kV], S2[kV];
        float lmax1 = 0.f, lmax2 = 0.f;
        if (mode != kModeSkip) {
            float P[kV], G[kV];
            {
                const float4 a = *reinterpret_cast<const float4*>(p + i0), ga = *reinterpret_cast<const float4*>(g + i0);
                P[0] = a.x; P[1] = a.y; P[2] = a.z; P[3] = a.w;
                G[0] = ga.x; G[1] = ga.y; G[2] = ga.z; G[3] = ga.w;
            }
            int64_t so = 0;
            if (mode == kMode8bit) {
                const float a1 = absmax1[blk], a2 = absmax2[blk];
                const uint32_t u1 = *reinterpret_cast<const uint32_t*>(st1 + i0), u2 = *reinterpret_cast<const uint32_t*>(st2 + i0);
#pragma unroll
                for (int j = 0; j < kV; ++j) {
                    S1[j] = __fmul_rn(q1[(u1 >> (8 * j)) & 255u], a1);
                    S2[j] = __fmul_rn(q2[(u2 >> (8 * j)) & 255u], a2);
                }
            } else {
                so = (int64_t)mode + (i0 & 63);
                const float4 a = *reinterpret_cast<const float4*>(small_m + so), va = *reinterpret_cast<const float4*>(small_v + so);
                S1[0] = a.x; S1[1] = a.y; S1[2] = a.z; S1[3] = a.w;
                S2[0] = va.x; S2[1] = va.y; S2[2] = va.z; S2[3] = va.w;
            }
#pragma unroll
            for (int j = 0; j < kV; ++j) {
                const float gv = __fmul_rn(G[j], c.grad_scale);
                S2[j] = __fadd_rn(__fmul_rn(S2[j], c.beta2), __fmul_rn(__fmul_rn(c.omb2, gv), gv));
                S1[j] = __fadd_rn(__fmul_rn(S1[j], c.beta1), __fmul_rn(c.omb1, gv));
                const float upd = __fdiv_rn(S1[j], __fadd_rn(__fsqrt_rn(S2[j]), c.eps_c2));
                P[j] = __fadd_rn(P[j], __fmul_rn(c.step_size, upd));
                if (c.apply_decay) P[j] = __fmul_rn(P[j], c.decay);
            }
            *reinterpret_cast<float4*>(p + i0) = make_float4(P[0], P[1], P[2], P[3]);
            *reinterpret_cast<uint2*>(wb + i0) = make_uint2(pack_bf16x2(P[0], P[1]), pack_bf16x2(P[2], P[3]));
            if (c.zero_grad) *reinterpret_cast<float4*>(g + i0) = make_float4(0.f, 0.f, 0.f, 0.f);
            if (mode == kMode8bit) {
#pragma unroll
                for (int j = 0; j < kV; ++j) {
                    lmax1 = fmaxf(lmax1, fabsf(S1[j]));
                    lmax2 = fmaxf(lmax2, fabsf(S2[j]));
                }
            } else {
                *reinterpret_cast<float4*>(small_m + so) = make_float4(S1[0], S1[1], S1[2], S1[3]);
                *reinterpret_cast<float4*>(small_v + so) = make_float4(S2[0], S2[1], S2[2], S2[3]);
            }
        }
        // new absmax of the block: max over the threads that hold 8-bit moments (every thread takes part in the reduction)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lmax1 = fmaxf(lmax1, __shfl_xor_sync(0xffffffffu, lmax1, o));
            lmax2 = fmaxf(lmax2, __shfl_xor_sync(0xffffffffu, lmax2, o));
        }
        if (lane == 0) { red1[warp] = lmax1; red2[warp] = lmax2; }
        __syncthreads();
        float n1 = red1[0], n2 = red2[0];
#pragma unroll
        for (int w = 1; w < kThreads / 32; ++w) { n1 = fmaxf(n1, red1[w]); n2 = fmaxf(n2, red2[w]); }
        if (mode == kMode8bit) {
            uint32_t o1 = 0u, o2 = 0u;
            const float inv1 = n1 > 0.f ? __fdiv_rn(1.f, n1) : 0.f, inv2 = n2 > 0.f ? __fdiv_rn(1.f, n2) : 0.f;
#pragma unroll
            for (int j = 0; j < kV; ++j) {
                const float x1 = __fmul_rn(S1[j], inv1), x2 = __fmul_rn(S2[j], inv2);
                int c1, c2;
                bool code_neg;
                if (!slow) {
                    c1 = lut1[lut_bin_signed(x1)];
                    c1 += x1 > m1[c1] ? 1 : 0;
                    c2 = lut2[lut_bin_unsigned(x2)];
                    c2 += x2 > m2[c2] ? 1 : 0;
                    code_neg = c1 < nneg;
                } else {
                    c1 = nearest_code(e1, x1);
                    c2 = nearest_code(e2, x2);
                    code_neg = (__float_as_uint(q1[c1]) >> 31) != 0;
                }
                // bitsandbytes: "make sure state1 term has still the same sign after quantization"
                if (code_neg != ((__float_as_uint(S1[j]) >> 31) != 0)) c1 += S1[j] > 0.f ? 1 : -1;
                o1 |= (uint32_t)(c1 & 255) << (8 * j);
                o2 |= (uint32_t)(c2 & 255) << (8 * j);
            }
            *reinterpret_cast<uint32_t*>(st1 + i0) = o1;
            *reinterpret_cast<uint32_t*>(st2 + i0) = o2;
        }
        if (tid == 0) { absmax1[blk] = n1; absmax2[blk] = n2; }
        __syncthreads();      // red1 / red2 are rewritten by the next block
    }
}

}  // namespace

// bnb.optim.AdamW8bit semantics (block-wise dynamic 8-bit moments, fp32 moments for the tensors below min_8bit_size) over the
// n (multiple of 64) parameters of a flat buffer; see include/b200sd.h.
extern "C" int b200sd_adamw8bit_step(float* param, float* grad, uint8_t* state1, uint8_t* state2, float* absmax1, float* absmax2,
                                     const float* qmap1, const float* qmap2, const int32_t* chunk_mode, float* small_exp_avg,
                                     float* small_exp_avg_sq, void* weights_bf16, int64_t n, float lr, float beta1, float beta2,
                                     float eps, float weight_decay, int step, float grad_scale, int zero_grad,
                                     b200sd_stream_t stream) {
    B200SD_REQUIRE(param && grad && state1 && state2 && absmax1 && absmax2 && qmap1 && qmap2 && weights_bf16,
                   "adamw8bit_step: null pointer");
    B200SD_REQUIRE(n > 0 && n % 64 == 0 && step >= 1, "adamw8bit_step: n must be a positive multiple of 64 and step >= 1");
    B200SD_REQUIRE(((reinterpret_cast<uintptr_t>(param) | reinterpret_cast<uintptr_t>(grad) | reinterpret_cast<uintptr_t>(weights_bf16) |
                     reinterpret_cast<uintptr_t>(small_exp_avg) | reinterpret_cast<uintptr_t>(small_exp_avg_sq)) & 15) == 0 &&
                       ((reinterpret_cast<uintptr_t>(state1) | reinterpret_cast<uintptr_t>(state2)) & 7) == 0,
                   "adamw8bit_step: pointers must be 16-byte (codes: 8-byte) aligned");
    static_assert(kV == 4 && kThreads * kV == kBlock, "one thread owns 4 consecutive values of a 2048-value block");
    B200SD_REQUIRE(chunk_mode == nullptr || (small_exp_avg && small_exp_avg_sq),
                   "adamw8bit_step: a chunk table needs the compact fp32 moment buffers of the small tensors");
    const double c1 = 1.0 - pow((double)beta1, (double)step);
    const double c2 = sqrt(1.0 - pow((double)beta2, (double)step));
    Adam8Consts c;
    c.beta1 = beta1;
    c.beta2 = beta2;
    c.omb1 = (float)(1.0 - (double)beta1);
    c.omb2 = (float)(1.0 - (double)beta2);
    c.eps_c2 = (float)((double)eps * c2);
    c.step_size = (float)(-(double)lr * c2 / c1);
    c.decay = (float)(1.0 - (double)lr * (double)weight_decay);
    c.apply_decay = weight_decay > 0.f ? 1 : 0;
    c.grad_scale = grad_scale;
    c.zero_grad = zero_grad;
    const int64_t nblocks = (n + kBlock - 1) / kBlock;
    // persistent grid: exactly the CTAs that are resident at once (a larger grid would run its tail at partial occupancy)
    static int ctas_per_sm = 0;
    if (ctas_per_sm == 0) {
        int v = 0;
        B200SD_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, adamw8bit_kernel, kThreads, 0));
        ctas_per_sm = v > 0 ? v : 1;
    }
    int64_t grid = (int64_t)b200sd_num_sms() * ctas_per_sm;
    if (grid > nblocks) grid = nblocks;
    adamw8bit_kernel<<<dim3((unsigned)grid), dim3(kThreads), 0, static_cast<cudaStream_t>(stream)>>>(param, grad, state1, state2,
        absmax1, absmax2, qmap1, qmap2, chunk_mode, small_exp_avg, small_exp_avg_sq, static_cast<bf16*>(weights_bf16), n, nblocks, c);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}
