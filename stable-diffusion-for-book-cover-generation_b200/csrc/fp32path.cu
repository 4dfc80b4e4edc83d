// b200sd -- kernels of the fp32-accuracy path (BASELINE north_star: "the fp32 path within 1e-4").
//
// The tensor cores stay bf16: every fp32 operand x is carried as the pair (hi, lo) = (bf16(x), bf16(x - hi)), which
// represents x to ~2^-17, and a product A*B is evaluated as A_hi*B_hi + A_lo*B_hi + A_hi*B_lo by running the SAME
// tcgen05 GEMM twice with fp32 accumulation: [A_hi | A_lo] x [B_hi | B_hi]^T (the kernel's two-source K concat) and then
// A_hi x B_lo^T accumulated through the fp32 residual input.  What lives here is everything around those GEMMs that must
// not round to bf16: the (hi, lo) split, GEGLU on fp32 pre-activations, an fp32 CUDA-core flash attention (online softmax,
// never materialising the score matrix), and the time-embedding linears with fp32 weights.
#include <atomic>

#include "common.cuh"

extern std::atomic<long long> g_b200sd_launches;
#define COUNT_LAUNCH() g_b200sd_launches.fetch_add(1, std::memory_order_relaxed)

namespace {

int ew_grid(int64_t total, int threads) {
    int64_t blocks = (total + threads - 1) / threads;
    const int64_t cap = (int64_t)b200sd_num_sms() * 8;
    if (blocks > cap) blocks = cap;
    return (int)(blocks < 1 ? 1 : blocks);
}

__device__ __forceinline__ void split8(const float (&y)[8], float (&hi)[8], float (&lo)[8]) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        hi[j] = __bfloat162float(__float2bfloat16(y[j]));
        lo[j] = y[j] - hi[j];
    }
}

// x fp32 [n] -> hi, lo bf16 [n]
__global__ void split_hi_lo_kernel(const float* __restrict__ x, bf16* __restrict__ hi, bf16* __restrict__ lo, int64_t n8) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (int64_t)gridDim.x * blockDim.x) {
        float v[8], h[8], l[8];
        ld8<B200SD_F32>(x, (size_t)i * 8, v);
        split8(v, h, l);
        st8<B200SD_BF16>(hi, (size_t)i * 8, h);
        st8<B200SD_BF16>(lo, (size_t)i * 8, l);
    }
}

// u fp32 [rows, 2*Ch] = [values | gates] -> (hi, lo) of values * gelu_erf(gates), [rows, Ch]
__global__ void geglu_f32_kernel(const float* __restrict__ u, bf16* __restrict__ hi, bf16* __restrict__ lo, int64_t rows, int Ch8) {
    const int64_t total = rows * Ch8;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t row = i / Ch8;
        const int c = (int)(i % Ch8) * 8;
        float v[8], g[8], o[8], h[8], l[8];
        ld8<B200SD_F32>(u, (size_t)row * Ch8 * 16 + c, v);
        ld8<B200SD_F32>(u, (size_t)row * Ch8 * 16 + (size_t)Ch8 * 8 + c, g);
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = v[j] * (0.5f * g[j] * (1.0f + erff(g[j] * 0.70710678118654752f)));
        split8(o, h, l);
        st8<B200SD_BF16>(hi, (size_t)row * Ch8 * 8 + c, h);
        st8<B200SD_BF16>(lo, (size_t)row * Ch8 * 8 + c, l);
    }
}

// ---- fp32 flash attention on the CUDA cores (accuracy path) -----------------------------------------------------------
// CTA = 64 queries of one (batch, head); 256 threads = 64 queries x 4 lanes.  Per 64-key tile: lane p of a query computes
// the 16 scores of keys p*16.., the 4 lanes combine max / sum with shuffles (online softmax, exp via expf), the
// probabilities go through smem and lane p accumulates the output columns [p*DQ, (p+1)*DQ), DQ = D/4 (D % 4 == 0, <= 160).
constexpr int kFQ = 64, kFK = 64, kFThreads = 256;
template <int DQ>
__global__ void __launch_bounds__(kFThreads) attention_f32_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                                                  const float* __restrict__ v, float* __restrict__ out, int Sq,
                                                                  int Skv, int ldq, int ldk, int ldv, int ldo, float scale) {
    constexpr int D = DQ * 4;
    extern __shared__ float sm[];
    float* sQ = sm;                       // [64][D + 1]
    float* sK = sQ + kFQ * (D + 1);       // [64][D + 1]
    float* sV = sK + kFK * (D + 1);       // [64][D + 1]
    float* sP = sV + kFK * (D + 1);       // [64][65]
    const int b = blockIdx.z, h = blockIdx.y, q0 = blockIdx.x * kFQ;
    const int qi = threadIdx.x >> 2, part = threadIdx.x & 3;
    const float* qg = q + ((size_t)b * Sq + q0) * ldq + h * D;
    const float* kg = k + (size_t)b * Skv * ldk + h * D;
    const float* vg = v + (size_t)b * Skv * ldv + h * D;
    for (int i = threadIdx.x; i < kFQ * D; i += kFThreads) {
        const int r = i / D, c = i % D;
        sQ[r * (D + 1) + c] = (q0 + r < Sq) ? qg[(size_t)r * ldq + c] * scale : 0.f;
    }
    float o[DQ];
#pragma unroll
    for (int i = 0; i < DQ; ++i) o[i] = 0.f;
    float m = -INFINITY, l = 0.f;
    for (int k0 = 0; k0 < Skv; k0 += kFK) {
        __syncthreads();
        for (int i = threadIdx.x; i < kFK * D; i += kFThreads) {
            const int r = i / D, c = i % D;
            const bool ok = k0 + r < Skv;
            sK[r * (D + 1) + c] = ok ? kg[(size_t)(k0 + r) * ldk + c] : 0.f;
            sV[r * (D + 1) + c] = ok ? vg[(size_t)(k0 + r) * ldv + c] : 0.f;
        }
        __syncthreads();
        float s[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) s[j] = 0.f;
        const float* qr = sQ + qi * (D + 1);
        for (int c = 0; c < D; ++c) {
            const float qv = qr[c];
#pragma unroll
            for (int j = 0; j < 16; ++j) s[j] += qv * sK[(part * 16 + j) * (D + 1) + c];
        }
        float mx = -INFINITY;
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            if (k0 + part * 16 + j >= Skv) s[j] = -INFINITY;
            mx = fmaxf(mx, s[j]);
        }
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
        const float mn = fmaxf(m, mx);
        const float corr = expf(m - mn);
        float rs = 0.f;
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const float pv = expf(s[j] - mn);
            rs += pv;
            sP[qi * 65 + part * 16 + j] = pv;
        }
        rs += __shfl_xor_sync(0xffffffffu, rs, 1);
        rs += __shfl_xor_sync(0xffffffffu, rs, 2);
        l = l * corr + rs;
        m = mn;
#pragma unroll
        for (int i = 0; i < DQ; ++i) o[i] *= corr;
        __syncwarp();   // the 4 lanes of a query sit in one warp: their sP row is complete
        const float* pr = sP + qi * 65;
        for (int j = 0; j < kFK; ++j) {
            const float pv = pr[j];
            const float* vr = sV + j * (D + 1) + part * DQ;
#pragma unroll
            for (int i = 0; i < DQ; ++i) o[i] += pv * vr[i];
        }
    }
    if (q0 + qi < Sq) {
        const float inv = 1.0f / l;
        float* dst = out + ((size_t)b * Sq + q0 + qi) * ldo + h * D + part * DQ;
#pragma unroll
        for (int i = 0; i < DQ; ++i) dst[i] = o[i] * inv;
    }
}

template <int DQ>
int launch_attn_f32(const float* q, const float* k, const float* v, float* out, int batch, int heads, int Sq, int Skv, int ldq, int ldk,
                    int ldv, int ldo, float scale, cudaStream_t s) {
    constexpr int D = DQ * 4;
    const size_t smem = ((size_t)3 * 64 * (D + 1) + 64 * 65) * sizeof(float);
    B200SD_CUDA(b200sd_opt_in_smem(attention_f32_kernel<DQ>, (int)smem));
    attention_f32_kernel<DQ><<<dim3(ceil_div(Sq, kFQ), heads, batch), dim3(kFThreads), smem, s>>>(q, k, v, out, Sq, Skv,
                              ldq, ldk, ldv, ldo, scale);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

// small-M linear with fp32 weights (time-embedding MLP of the fp32 path): one warp per output feature
__global__ void __launch_bounds__(256) small_linear_f32_kernel(const float* __restrict__ in, const float* __restrict__ w,
                                                               const float* __restrict__ bias, float* __restrict__ out, int batch,
                                                               int N, int K, int silu_in, int silu_out) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= N) return;
    for (int b = 0; b < batch; ++b) {
        float a = 0.f;
        for (int c = lane; c < K; c += 32) {
            float x = in[(size_t)b * K + c];
            if (silu_in) x = x / (1.0f + expf(-x));
            a += x * __ldg(w + (size_t)warp * K + c);
        }
        a = warp_sum(a);
        if (lane == 0) {
            a += bias ? bias[warp] : 0.f;
            if (silu_out) a = a / (1.0f + expf(-a));
            out[(size_t)b * N + warp] = a;
        }
    }
}

}  // namespace

extern "C" int b200sd_split_hi_lo(const float* x, void* hi, void* lo, int64_t n, b200sd_stream_t stream) {
    B200SD_REQUIRE(x && hi && lo && n > 0 && n % 8 == 0, "split_hi_lo: n must be a positive multiple of 8");
    split_hi_lo_kernel<<<dim3(ew_grid(n / 8, 256)), dim3(256), 0, static_cast<cudaStream_t>(stream)>>>(x,
                              static_cast<bf16*>(hi), static_cast<bf16*>(lo), n / 8);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

extern "C" int b200sd_geglu_f32(const float* u, void* hi, void* lo, int64_t rows, int C_half, b200sd_stream_t stream) {
    B200SD_REQUIRE(u && hi && lo && rows > 0 && C_half > 0 && C_half % 8 == 0, "geglu_f32: bad arguments");
    geglu_f32_kernel<<<dim3(ew_grid(rows * (C_half / 8), 256)), dim3(256), 0, static_cast<cudaStream_t>(stream)>>>(u,
                              static_cast<bf16*>(hi), static_cast<bf16*>(lo), rows, C_half / 8);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}

extern "C" int b200sd_attention_f32(const float* q, const float* k, const float* v, float* out, int batch, int heads, int Sq,
                                    int Skv, int d, int ldq, int ldk, int ldv, int ldo, float scale, b200sd_stream_t stream) {
    B200SD_REQUIRE(q && k && v && out, "attention_f32: null pointer");
    B200SD_REQUIRE(batch > 0 && heads > 0 && Sq > 0 && Skv > 0 && batch <= 65535 && heads <= 65535, "attention_f32: bad sizes");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
#define AF_CASE(DQ) case DQ * 4: return launch_attn_f32<DQ>(q, k, v, out, batch, heads, Sq, Skv, ldq, ldk, ldv, ldo, scale, s);
    switch (d) {
        AF_CASE(2) AF_CASE(4) AF_CASE(8) AF_CASE(10) AF_CASE(16) AF_CASE(20) AF_CASE(32) AF_CASE(40)
    }
#undef AF_CASE
    B200SD_REQUIRE(false, "attention_f32: head dim %d unsupported (8, 16, 32, 40, 64, 80, 128, 160)", d);
}

extern "C" int b200sd_small_linear_f32(const float* in, const float* w, const float* bias, float* out, int batch, int N, int K,
                                       int silu_in, int silu_out, b200sd_stream_t stream) {
    B200SD_REQUIRE(in && w && out && batch > 0 && N > 0 && K > 0, "small_linear_f32: bad arguments");
    small_linear_f32_kernel<<<dim3(ceil_div(N * 32, 256)), dim3(256), 0, static_cast<cudaStream_t>(stream)>>>(in, w, bias,
                              out, batch, N, K, silu_in, silu_out);
    COUNT_LAUNCH();
    B200SD_LAUNCH_CHECK();
    return B200SD_OK;
}
